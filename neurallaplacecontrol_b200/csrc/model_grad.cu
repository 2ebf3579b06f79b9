// Backward pass of NeuralLaplaceModel.forward with per-sample prediction times (w_nl.py:117-145; the loss.backward() of
// train_utils.py:388-407): gradients of a scalar loss with respect to the 16 parameters and to the obs / action inputs,
// fp32 FFMA on the CUDA cores.
//
// Three launches after the per-sample s-point prep that nlc_model_forward_ts runs too (rollout.cu forward_ts_prep_kernel,
// which here also writes the sphere coordinates [theta_s | phi_s] of every sample):
//   1. model_grad_wt_kernel     - row-major ([out][in], state_dict) copies of the five matrices the backward multiplies by
//                                 transposed (W_hh0, W_ih1, W_hh1, W2, the paired W3), so that every product is a coalesced
//                                 "A[rows][k] . W[k][n]" like the forward's;
//   2. model_grad_tile_kernel   - persistent CTAs, tile t of kGradRows samples on CTA t mod grid: recompute the tile's
//                                 forward in fp32 keeping r, z, n, W_hn h + b_hn and h of every GRU cell, the MLP's
//                                 activations and the first-layer input; then the ILT + sphere-map derivatives, the MLP
//                                 backward, linear_out and BPTT through both GRU layers over the reversed window.  Input
//                                 gradients are written per sample; weight gradients are tile-level products accumulated
//                                 into the CTA's own partial (no atomics);
//   3. model_grad_reduce_kernel - sums the per-CTA partials in CTA order and writes every tensor in its state_dict layout.
// The grid, the tile-to-CTA assignment and every summation order depend on K, B and the model's shape only: two calls on
// the same inputs give bit-identical gradients.
//
// The tile's saved activations live in a per-CTA slice of the workspace (B = 8 windows keep 20 KB per sample of GRU
// cell state, so a shared-memory tile would hold 8 samples and re-read every weight matrix from L2 per 8 samples); the
// slice is written and re-read by the same CTA and stays in L1/L2.  Shared memory is left to L1, which caches the weights.
//
// nlc_model_backward_multi (several prediction times per sample, the rows of nlc_model_forward_multi) runs the same tile
// steps as two stages instead - an MLP/ILT stage over the K n_t rows, then an encoder stage over the K samples - see the
// kernels after model_grad_tile_kernel.
//
// Reads only the unfolded weights of ModelDev: b1_fold, ilt_phase, ilt_weight and the mlp2_* images belong to the last
// prediction time a planner folded and are never touched here.
#include <stddef.h>

#include "common.cuh"

namespace nlc {

int launch_forward_ts_prep(nlc_model_s* m, const float* ts, int K, float* row_b1, float* row_tn, float* row_sph, cudaStream_t s);
int encode_history_impl(nlc_model_t m, const float* hist_dev, int hist_ch, int K, int T, int B, float* p_dev, int math_mode,
                        cudaStream_t s);

constexpr int kGradRows = 32;     // samples per tile
constexpr int kGradThreads = 256;
constexpr int kGradGridCap = 148;  // persistent CTAs (one per B200 SM); fixed, so the reduction order does not depend on the device

static inline size_t up4(size_t n) { return (n + 3) / 4 * 4; }
static inline size_t up64(size_t n) { return (n + 63) / 64 * 64; }

// Shapes and offsets shared by host and device.
struct GradShape {
  int nx, nu, gin, H, Hg, G3, S, Lp, in0, in0p, N3, N3p, B;
  // per-CTA partial, "internal" layouts (the ones the products produce): offsets in floats
  int p_wih0, p_whh0, p_bih0, p_bhh0, p_wih1, p_whh1, p_bih1, p_bhh1, p_wout, p_bout, p_w0, p_b0, p_w2, p_b2, p_w4, p_b4, p_total;
  // state_dict layout of the output (named_parameters() order)
  int o_wih0, o_whh0, o_bih0, o_bhh0, o_wih1, o_whh1, o_bih1, o_bhh1, o_wout, o_bout, o_w0, o_b0, o_w2, o_b2, o_w4, o_b4, o_total;
  // per-CTA tile scratch: offsets in floats
  int s_xs, s_gate, s_h, s_gi, s_gh, s_x1, s_a1, s_a2, s_do, s_dz2, s_dz1, s_dh, s_dxt, s_rc, s_total;
  // transposed weight copies
  int w_hh0, w_ih1, w_hh1, w_2, w_3, w_total;
};

static GradShape make_shape(int nx, int nu, int gin, int H, int S, int B) {
  GradShape g;
  g.nx = nx; g.nu = nu; g.gin = gin; g.H = H; g.Hg = H / 2; g.G3 = 3 * g.Hg; g.S = S; g.Lp = nx + 2; g.in0 = 2 * S + g.Lp;
  g.in0p = (int)up4(g.in0); g.N3 = 2 * nx * S; g.N3p = (int)up4(g.N3); g.B = B;
  const int Hg = g.Hg, G3 = g.G3, R = kGradRows;
  int o = 0;
  auto take = [&](int n) { const int at = o; o += (int)up4(n); return at; };
  g.p_wih0 = take(G3 * gin); g.p_whh0 = take(Hg * G3); g.p_bih0 = take(G3); g.p_bhh0 = take(G3);
  g.p_wih1 = take(Hg * G3); g.p_whh1 = take(Hg * G3); g.p_bih1 = take(G3); g.p_bhh1 = take(G3);
  g.p_wout = take(2 * Hg); g.p_bout = take(2); g.p_w0 = take(g.in0p * H); g.p_b0 = take(H);
  g.p_w2 = take(H * H); g.p_b2 = take(H); g.p_w4 = take(H * g.N3p); g.p_b4 = take(g.N3p);
  g.p_total = (int)up64(o);
  o = 0;
  auto put = [&](int n) { const int at = o; o += n; return at; };
  g.o_wih0 = put(G3 * gin); g.o_whh0 = put(G3 * Hg); g.o_bih0 = put(G3); g.o_bhh0 = put(G3);
  g.o_wih1 = put(G3 * Hg); g.o_whh1 = put(G3 * Hg); g.o_bih1 = put(G3); g.o_bhh1 = put(G3);
  g.o_wout = put(2 * Hg); g.o_bout = put(2); g.o_w0 = put(H * g.in0); g.o_b0 = put(H);
  g.o_w2 = put(H * H); g.o_b2 = put(H); g.o_w4 = put(g.N3 * H); g.o_b4 = put(g.N3);
  g.o_total = o;
  o = 0;
  g.s_xs = take(B * R * 4);              // [B steps][R][4]    normalised window entry of step st (entry B-1-st), gin <= 4
  g.s_gate = take(2 * B * R * 4 * Hg);   // [layer][B][R][4Hg] r | z | n | W_hn h + b_hn; overwritten by dr | dz | dn | dghn
  g.s_h = take(2 * B * R * Hg);          // [layer][B][R][Hg]  h after step st
  g.s_gi = take(R * G3);                 // [R][3Hg] input products of the current cell
  g.s_gh = take(R * G3);                 // [R][3Hg] hidden products of the current cell
  g.s_x1 = take(R * g.in0p);             // [R][in0p] first-layer input [theta_s | phi_s | obs_n | p_action | 0]
  g.s_a1 = take(R * H); g.s_a2 = take(R * H);
  g.s_do = take(R * g.N3p);              // [R][N3p] last-layer pre-activations, then their gradients (paired columns)
  g.s_dz2 = take(R * H); g.s_dz1 = take(R * H);
  g.s_dh = take(4 * R * Hg);             // dh0, dh1 and their next-step buffers
  g.s_dxt = take(R * 16);                // [R][Lp] gradient of [obs_n | p_action]
  g.s_rc = take(2 * R);                  // per-row pi t / T and exp(gamma t)/T
  g.s_total = (int)up64(o);
  o = 0;
  g.w_hh0 = take(G3 * Hg); g.w_ih1 = take(G3 * Hg); g.w_hh1 = take(G3 * Hg); g.w_2 = take(H * H); g.w_3 = take(g.N3p * H);
  g.w_total = (int)up64(o);
  return g;
}

struct GradArgs {
  ModelDev m;
  GradShape g;
  const float* obs;       // [K][nx]
  const float* act;       // [K][B][gin]
  const float* gout;      // [K][nx]
  const float* row_b1;    // [K][H]
  const float* row_tn;    // [K]
  const float* row_sph;   // [K][2S]
  const float* wt;        // transposed weight copies
  float* part;            // [grid][p_total]
  float* scratch;         // [grid][s_total]
  float* grad_obs;        // [K][nx] or null
  float* grad_act;        // [K][B][gin] or null
  int K, n_tiles;
};

// ------------------------------------------------------------------------------------------------------------------
// Tile products.  Rows are the kGradRows samples of the tile; every thread owns fixed 4 x 4 output blocks, so an output
// element is always written by the same thread (repeated accumulating calls on one output need no barrier between them).
// ------------------------------------------------------------------------------------------------------------------
enum { kEpiNone = 0, kEpiTanh = 1, kEpiDtanh = 2 };

// C[m][n] (+)= sum_k A[m][k] W[k][n]  (+ bias[n]; kEpiTanh: tanh of it; kEpiDtanh: times 1 - aux[m][n]^2).
// N, Kd, lda, ldw, ldc multiples of 4; W is read-only for the kernel's lifetime.
template <int EPI>
__device__ __forceinline__ void gemm_nn(const float* A, int lda, const float* __restrict__ W, int ldw, int Kd, int N, float* C, int ldc,
                                        bool accumulate, const float* __restrict__ bias = nullptr, const float* aux = nullptr) {
  const int CG = N / 4, items = (kGradRows / 4) * CG;
  for (int it = threadIdx.x; it < items; it += kGradThreads) {
    const int rg = it / CG, cg = it - rg * CG;
    float c[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (accumulate) v = *reinterpret_cast<const float4*>(C + (4 * rg + i) * ldc + 4 * cg);
      else if (bias) v = *reinterpret_cast<const float4*>(bias + 4 * cg);
      c[i][0] = v.x; c[i][1] = v.y; c[i][2] = v.z; c[i][3] = v.w;
    }
#pragma unroll 2
    for (int k = 0; k < Kd; k += 4) {
      float4 a[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = *reinterpret_cast<const float4*>(A + (4 * rg + i) * lda + k);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        const float4 w = __ldg(reinterpret_cast<const float4*>(W + (size_t)(k + kk) * ldw + 4 * cg));
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float av = kk == 0 ? a[i].x : (kk == 1 ? a[i].y : (kk == 2 ? a[i].z : a[i].w));
          c[i][0] = fmaf(av, w.x, c[i][0]);
          c[i][1] = fmaf(av, w.y, c[i][1]);
          c[i][2] = fmaf(av, w.z, c[i][2]);
          c[i][3] = fmaf(av, w.w, c[i][3]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float* dst = C + (4 * rg + i) * ldc + 4 * cg;
      if (EPI == kEpiTanh) {
        for (int j = 0; j < 4; ++j) c[i][j] = tanh_acc(c[i][j]);
      } else if (EPI == kEpiDtanh) {
        const float4 y = *reinterpret_cast<const float4*>(aux + (4 * rg + i) * ldc + 4 * cg);
        c[i][0] *= 1.0f - y.x * y.x; c[i][1] *= 1.0f - y.y * y.y; c[i][2] *= 1.0f - y.z * y.z; c[i][3] *= 1.0f - y.w * y.w;
      }
      *reinterpret_cast<float4*>(dst) = make_float4(c[i][0], c[i][1], c[i][2], c[i][3]);
    }
  }
}

// Weight gradient: P[k][n] += sum_{s in [s0, s1)} sum_m A_s[m][k] D_s[m][col(n)], A_s = A + (s - alag) sA, D_s = D + s sD,
// col(n) = n + (n >= nsplit ? dshift : 0) (skips a gate slot of the saved GRU gradients).  Kd, N, nsplit multiples of 4.
__device__ __forceinline__ void wgrad(float* P, int ldp, const float* A, int lda, int sA, int alag, const float* D, int ldd, int sD,
                                      int s0, int s1, int Kd, int N, int nsplit, int dshift) {
  const int CG = N / 4, items = (Kd / 4) * CG;
  for (int it = threadIdx.x; it < items; it += kGradThreads) {
    const int kg = it / CG, cg = it - kg * CG;
    const int dc = 4 * cg + (4 * cg >= nsplit ? dshift : 0);
    float c[4][4] = {};
    for (int s = s0; s < s1; ++s) {
      const float* As = A + (s - alag) * sA + 4 * kg;
      const float* Ds = D + s * sD + dc;
#pragma unroll 4
      for (int m = 0; m < kGradRows; ++m) {
        const float4 a = *reinterpret_cast<const float4*>(As + m * lda);
        const float4 d = *reinterpret_cast<const float4*>(Ds + m * ldd);
        const float av[4] = {a.x, a.y, a.z, a.w}, dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) c[i][j] = fmaf(av[i], dv[j], c[i][j]);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float4* p = reinterpret_cast<float4*>(P + (4 * kg + i) * ldp + 4 * cg);
      float4 v = *p;
      v.x += c[i][0]; v.y += c[i][1]; v.z += c[i][2]; v.w += c[i][3];
      *p = v;
    }
  }
}

// Bias gradient: P[n] += sum_{s in [s0, s1)} sum_m D_s[m][col(n)]
__device__ __forceinline__ void colsum(float* P, const float* D, int ldd, int sD, int s0, int s1, int N, int nsplit, int dshift) {
  for (int n = threadIdx.x; n < N; n += kGradThreads) {
    const int dc = n + (n >= nsplit ? dshift : 0);
    float acc = 0.0f;
    for (int s = s0; s < s1; ++s)
      for (int m = 0; m < kGradRows; ++m) acc += D[s * sD + m * ldd + dc];
    P[n] += acc;
  }
}

// GRU cell forward (torch.nn.GRU, gate order r, z, n; the same expressions as encode_gru.cu gru_finish).  gi / gh are the
// bias-free products (gh null: zero state); layer 0 (gin inputs) forms gi here from the step's window entry.
__device__ __forceinline__ void gru_cell_fwd(const GradShape& g, const float* __restrict__ b_i, const float* __restrict__ b_h,
                                             const float* __restrict__ w_ih0, const float* xs, const float* gi, const float* gh,
                                             const float* hprev, float* gate, float* hout) {
  const int Hg = g.Hg, G3 = g.G3;
  for (int i = threadIdx.x; i < kGradRows * Hg; i += kGradThreads) {
    const int m = i / Hg, u = i - m * Hg;
    float gir, giz, gin_;
    if (gi) {
      gir = gi[m * G3 + u]; giz = gi[m * G3 + Hg + u]; gin_ = gi[m * G3 + 2 * Hg + u];
    } else {
      float acc[3];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const float* w = w_ih0 + (q * Hg + u) * g.gin;
        float a = 0.0f;
        for (int v = 0; v < g.gin; ++v) a = fmaf(w[v], xs[m * 4 + v], a);
        acc[q] = a;
      }
      gir = acc[0]; giz = acc[1]; gin_ = acc[2];
    }
    const float ghr = gh ? gh[m * G3 + u] : 0.0f, ghz = gh ? gh[m * G3 + Hg + u] : 0.0f, ghn0 = gh ? gh[m * G3 + 2 * Hg + u] : 0.0f;
    const float r = sigmoid_acc((gir + b_i[u]) + (ghr + b_h[u]));
    const float z = sigmoid_acc((giz + b_i[Hg + u]) + (ghz + b_h[Hg + u]));
    const float ghn = ghn0 + b_h[2 * Hg + u];
    const float n = tanh_acc((gin_ + b_i[2 * Hg + u]) + r * ghn);
    const float ho = hprev ? hprev[m * Hg + u] : 0.0f;
    float* gt = gate + m * 4 * Hg;
    gt[u] = r; gt[Hg + u] = z; gt[2 * Hg + u] = n; gt[3 * Hg + u] = ghn;
    hout[m * Hg + u] = fmaf(z, ho - n, n);
  }
}

// GRU cell backward: dh -> (dr_pre, dz_pre, dn_pre, d(W_hn h + b_hn)) in place of the saved gates, dh_prev's direct part.
__device__ __forceinline__ void gru_cell_bwd(const GradShape& g, const float* dh, const float* hprev, float* gate, float* dh_prev) {
  const int Hg = g.Hg;
  for (int i = threadIdx.x; i < kGradRows * Hg; i += kGradThreads) {
    const int m = i / Hg, u = i - m * Hg;
    float* gt = gate + m * 4 * Hg;
    const float r = gt[u], z = gt[Hg + u], n = gt[2 * Hg + u], ghn = gt[3 * Hg + u];
    const float d = dh[m * Hg + u], ho = hprev ? hprev[m * Hg + u] : 0.0f;
    const float dn = d * (1.0f - z) * (1.0f - n * n);
    const float dr = dn * ghn * r * (1.0f - r);
    const float dz = d * (ho - n) * z * (1.0f - z);
    gt[u] = dr; gt[Hg + u] = dz; gt[2 * Hg + u] = dn; gt[3 * Hg + u] = dn * r;
    dh_prev[m * Hg + u] = d * z;
  }
}

// The per-CTA scratch of a tile (GradShape s_* offsets).
struct TileBufs {
  float *xs, *gate, *hs, *gi, *gh, *x1, *a1, *a2, *dob, *dz2, *dz1, *dhb, *dxt, *rc;
};
__device__ __forceinline__ TileBufs tile_bufs(const GradShape& g, float* sc) {
  TileBufs t;
  t.xs = sc + g.s_xs; t.gate = sc + g.s_gate; t.hs = sc + g.s_h; t.gi = sc + g.s_gi; t.gh = sc + g.s_gh; t.x1 = sc + g.s_x1;
  t.a1 = sc + g.s_a1; t.a2 = sc + g.s_a2; t.dob = sc + g.s_do; t.dz2 = sc + g.s_dz2; t.dz1 = sc + g.s_dz1; t.dhb = sc + g.s_dh;
  t.dxt = sc + g.s_dxt; t.rc = sc + g.s_rc;
  return t;
}
// gate [l][st] at (l * B + st) * R * 4Hg, h [l][st] at (l * B + st) * R * Hg
__device__ __forceinline__ float* tile_gate(const GradShape& g, const TileBufs& t, int l, int st) {
  return t.gate + (size_t)(l * g.B + st) * kGradRows * 4 * g.Hg;
}
__device__ __forceinline__ float* tile_h(const GradShape& g, const TileBufs& t, int l, int st) {
  return t.hs + (size_t)(l * g.B + st) * kGradRows * g.Hg;
}

// Normalised window of samples k0 .. k0 + R - 1 (w_nl.py:121); rows past K repeat sample K - 1.
__device__ __forceinline__ void tile_load_window(const GradShape& g, const ModelDev& md, const float* act, int k0, int K, float* xs) {
  const int B = g.B, gin = g.gin, R = kGradRows;
  for (int i = threadIdx.x; i < B * R * 4; i += kGradThreads) {
    const int st = i / (R * 4), m = (i / 4) % R, u = i & 3;
    const int k = min(k0 + m, K - 1), j = B - 1 - st;  // step st reads entry B-1-st (reversed in time, w_nl.py:27)
    xs[i] = u < gin ? (act[((size_t)k * B + j) * gin + u] - md.act_mean[u]) * md.act_inv_std[u] : 0.0f;
  }
}

// Per-row Fourier constants pi t / T and exp(gamma t) / T of rows k0 .. k0 + R - 1 (rollout.cu rollout_nl_kernel: the same).
__device__ __forceinline__ void tile_fourier_consts(const float* row_tn, int k0, int K, float* rc) {
  const int R = kGradRows;
  for (int m = threadIdx.x; m < R; m += kGradThreads) {
    const float tn = row_tn[min(k0 + m, K - 1)];
    const float T = 2.0f * (tn + 1.0e-6f);
    rc[m] = 3.14159265358979f * 1.0e-6f / T;
    rc[R + m] = expf((1.0e-3f + 4.605170185988091f / T) * tn) / T;
  }
}

// Encoder forward (w_nl.py:25-29) of the tile's windows, saving every cell.  Ends on a barrier.
template <int H>
__device__ __forceinline__ void tile_encoder_fwd(const GradShape& g, const ModelDev& md, const TileBufs& t) {
  constexpr int Hg = H / 2, G3 = 3 * Hg;
  const int B = g.B;
  for (int st = 0; st < B; ++st) {
    if (st > 0) {
      gemm_nn<kEpiNone>(tile_h(g, t, 0, st - 1), Hg, md.w_hh0_t, G3, Hg, G3, t.gh, G3, false);
      __syncthreads();
    }
    gru_cell_fwd(g, md.b_ih0, md.b_hh0, md.w_ih0, t.xs + st * kGradRows * 4, nullptr, st > 0 ? t.gh : nullptr,
                 st > 0 ? tile_h(g, t, 0, st - 1) : nullptr, tile_gate(g, t, 0, st), tile_h(g, t, 0, st));
    __syncthreads();
    gemm_nn<kEpiNone>(tile_h(g, t, 0, st), Hg, md.w_ih1_t, G3, Hg, G3, t.gi, G3, false);
    if (st > 0) gemm_nn<kEpiNone>(tile_h(g, t, 1, st - 1), Hg, md.w_hh1_t, G3, Hg, G3, t.gh, G3, false);
    __syncthreads();
    gru_cell_fwd(g, md.b_ih1, md.b_hh1, nullptr, nullptr, t.gi, st > 0 ? t.gh : nullptr, st > 0 ? tile_h(g, t, 1, st - 1) : nullptr,
                 tile_gate(g, t, 1, st), tile_h(g, t, 1, st));
    __syncthreads();
  }
}

// Representation MLP forward (w_nl.py:55-63) from the first-layer input x1 and the Fourier constants rc, the ILT + sphere map
// derivatives against gout, the MLP backward into the partial P, and the gradient of [obs_n | p_action] into dxt.  Rows
// k0 .. k0 + R - 1 of row_b1 [K][H] and gout [K][nx]; rows past K get zero output gradients.  Ends on a barrier.
template <int H>
__device__ __forceinline__ void tile_mlp_fwd_bwd(const GradShape& g, const ModelDev& md, const float* wt, float* P, const TileBufs& t,
                                                 const float* row_b1, const float* gout, int k0, int K) {
  constexpr int R = kGradRows;
  const int S = g.S, nx = g.nx, Lp = g.Lp, in0p = g.in0p, N3p = g.N3p, nP = nx * S;
  const int tid = threadIdx.x;
  const float* W2 = wt + g.w_2;  // [H][H]   (out, in)
  const float* W3 = wt + g.w_3;  // [N3p][H] (paired output column, in)
  float *x1 = t.x1, *a1 = t.a1, *a2 = t.a2, *dob = t.dob, *dz2 = t.dz2, *dz1 = t.dz1, *dxt = t.dxt, *rc = t.rc;
  for (int i = tid; i < R * H; i += kGradThreads) {  // the s-columns are in row_b1 (forward_ts_prep_kernel)
    const int m = i / H, n = i - m * H;
    float acc = row_b1[(size_t)min(k0 + m, K - 1) * H + n];
    for (int j = 0; j < Lp; ++j) acc = fmaf(md.w1_full_t[(size_t)(2 * S + j) * H + n], x1[m * in0p + 2 * S + j], acc);
    a1[i] = tanh_acc(acc);
  }
  __syncthreads();
  gemm_nn<kEpiTanh>(a1, H, md.w2_t, H, H, H, a2, H, false, md.b2);
  __syncthreads();
  gemm_nn<kEpiNone>(a2, H, md.w3_t, N3p, H, N3p, dob, N3p, false, md.b3);
  __syncthreads();
  // ---- ILT + sphere map derivatives: Dx_c = sum_k w_k rho cos(theta + a_k), theta = pi tanh(u_t), rho = tan((pi/2) sigma(2 u_p)) ----
  for (int i = tid; i < R * (N3p / 2); i += kGradThreads) {
    const int m = i / (N3p / 2), pair = i - m * (N3p / 2);
    float* o = dob + m * N3p + 2 * pair;
    if (pair >= nP) { o[0] = 0.0f; o[1] = 0.0f; continue; }
    const int c = pair / S, kk = pair - c * S;
    const bool valid = k0 + m < K;
    const float gc = valid ? gout[(size_t)(k0 + m) * nx + c] : 0.0f;
    const float quarter = (kk & 3) == 0 ? 0.0f : ((kk & 3) == 1 ? 1.57079632679489662f : ((kk & 3) == 2 ? 3.14159265358979f : -1.57079632679489662f));
    const float ph = quarter - (float)kk * rc[m];
    const float wt = rc[R + m] * (kk == 0 ? 0.5f : 1.0f);
    const float ut = o[0], up = o[1];
    // sech^2 u and sigma(2u) sigma(-2u) through e = exp(-2|u|): no cancellation in either tail (DESIGN.md 2.6)
    const float et = exp_acc(-2.0f * fminf(fabsf(ut), 40.0f));
    const float sech2 = 4.0f * et * __frcp_rn((1.0f + et) * (1.0f + et));
    const float ep = exp_acc(-2.0f * fminf(fabsf(up), 40.0f));
    const float ss = ep * __frcp_rn((1.0f + ep) * (1.0f + ep));
    const float rho = sphere_radius(up);
    const float arg = 3.14159265358979f * tanh_acc(ut) + ph;  // |arg| < 2 pi: cos_reduced's range
    const float cs = cos_reduced(arg), sn = cos_reduced(arg - 1.57079632679489662f);
    const float gw = gc * wt;
    o[0] = -gw * rho * sn * 3.14159265358979f * sech2;
    o[1] = gw * cs * 3.14159265358979f * fmaf(rho, rho * ss, ss);  // (1 + rho^2) ss without forming rho^2
  }
  __syncthreads();
  // ---- MLP backward ----
  wgrad(P + g.p_w4, N3p, a2, H, 0, 0, dob, N3p, 0, 0, 1, H, N3p, N3p, 0);
  colsum(P + g.p_b4, dob, N3p, 0, 0, 1, N3p, N3p, 0);
  gemm_nn<kEpiDtanh>(dob, N3p, W3, H, N3p, H, dz2, H, false, nullptr, a2);
  __syncthreads();
  wgrad(P + g.p_w2, H, a1, H, 0, 0, dz2, H, 0, 0, 1, H, H, H, 0);
  colsum(P + g.p_b2, dz2, H, 0, 0, 1, H, H, 0);
  gemm_nn<kEpiDtanh>(dz2, H, W2, H, H, H, dz1, H, false, nullptr, a1);
  __syncthreads();
  wgrad(P + g.p_w0, H, x1, in0p, 0, 0, dz1, H, 0, 0, 1, in0p, H, H, 0);
  colsum(P + g.p_b0, dz1, H, 0, 0, 1, H, H, 0);
  for (int i = tid; i < R * Lp; i += kGradThreads) {  // gradient of [obs_n | p_action]
    const int m = i / Lp, j = i - m * Lp;
    const float* w = md.w1_full_t + (size_t)(2 * S + j) * H;
    float acc = 0.0f;
    for (int n = 0; n < H; ++n) acc = fmaf(dz1[m * H + n], w[n], acc);
    dxt[m * 16 + j] = acc;
  }
  __syncthreads();
}

// From the gradient of [obs_n | p_action] in dxt: grad_obs, linear_out backward and BPTT through both GRU layers over the
// reversed window (the saved cells of tile_encoder_fwd), grad_act, and the GRU weight gradients into the partial P.
template <int H>
__device__ __forceinline__ void tile_encoder_bwd(const GradShape& g, const ModelDev& md, const float* wt, float* P, const TileBufs& t,
                                                 float* grad_obs, float* grad_act, int k0, int K) {
  constexpr int Hg = H / 2, G3 = 3 * Hg, R = kGradRows;
  const int B = g.B, nx = g.nx, gin = g.gin;
  const int tid = threadIdx.x;
  const float* W_hh0 = wt + g.w_hh0;  // [3Hg][Hg]
  const float* W_ih1 = wt + g.w_ih1;
  const float* W_hh1 = wt + g.w_hh1;
  const float* dxt = t.dxt;
  const float* h1last = tile_h(g, t, 1, B - 1);
  if (grad_obs)
    for (int i = tid; i < R * nx; i += kGradThreads) {
      const int m = i / nx, c = i - m * nx;
      if (k0 + m < K) grad_obs[(size_t)(k0 + m) * nx + c] = dxt[m * 16 + c] * md.state_inv_std[c];
    }
  // ---- linear_out backward ----
  for (int i = tid; i < 2 * Hg + 2; i += kGradThreads) {
    float acc = 0.0f;
    if (i < 2 * Hg) {
      const int o = i / Hg, h = i - o * Hg;
      for (int m = 0; m < R; ++m) acc = fmaf(dxt[m * 16 + nx + o], h1last[m * Hg + h], acc);
      P[g.p_wout + i] += acc;
    } else {
      for (int m = 0; m < R; ++m) acc += dxt[m * 16 + nx + (i - 2 * Hg)];
      P[g.p_bout + i - 2 * Hg] += acc;
    }
  }
  float* dh0 = t.dhb;
  float* dh1 = t.dhb + R * Hg;
  float* dh0n = t.dhb + 2 * R * Hg;
  float* dh1n = t.dhb + 3 * R * Hg;
  for (int i = tid; i < R * Hg; i += kGradThreads) {
    const int m = i / Hg, h = i - m * Hg;
    dh1[i] = fmaf(dxt[m * 16 + nx], md.w_out[h], dxt[m * 16 + nx + 1] * md.w_out[Hg + h]);
    dh0[i] = 0.0f;
  }
  __syncthreads();
  // ---- BPTT over the reversed window: step B-1 (oldest entry) first ----
  for (int st = B - 1; st >= 0; --st) {
    gru_cell_bwd(g, dh1, st > 0 ? tile_h(g, t, 1, st - 1) : nullptr, tile_gate(g, t, 1, st), dh1n);
    __syncthreads();
    const float* G1 = tile_gate(g, t, 1, st);
    if (st > 0) {  // dh1_prev += [dr | dz] W_hh1[r,z] + dghn W_hh1[n]
      gemm_nn<kEpiNone>(G1, 4 * Hg, W_hh1, Hg, 2 * Hg, Hg, dh1n, Hg, true);
      gemm_nn<kEpiNone>(G1 + 3 * Hg, 4 * Hg, W_hh1 + 2 * Hg * Hg, Hg, Hg, Hg, dh1n, Hg, true);
    }
    gemm_nn<kEpiNone>(G1, 4 * Hg, W_ih1, Hg, G3, Hg, dh0, Hg, true);  // layer 1's input is layer 0's output
    __syncthreads();
    gru_cell_bwd(g, dh0, st > 0 ? tile_h(g, t, 0, st - 1) : nullptr, tile_gate(g, t, 0, st), dh0n);
    __syncthreads();
    const float* G0 = tile_gate(g, t, 0, st);
    if (st > 0) {
      gemm_nn<kEpiNone>(G0, 4 * Hg, W_hh0, Hg, 2 * Hg, Hg, dh0n, Hg, true);
      gemm_nn<kEpiNone>(G0 + 3 * Hg, 4 * Hg, W_hh0 + 2 * Hg * Hg, Hg, Hg, Hg, dh0n, Hg, true);
    }
    if (grad_act)
      for (int i = tid; i < R * gin; i += kGradThreads) {  // W_ih0^T dg_i, times the input scale
        const int m = i / gin, u = i - m * gin;
        float acc = 0.0f;
        for (int q = 0; q < G3; ++q) acc = fmaf(G0[m * 4 * Hg + q], md.w_ih0[q * gin + u], acc);
        if (k0 + m < K) grad_act[((size_t)(k0 + m) * B + (B - 1 - st)) * gin + u] = acc * md.act_inv_std[u];
      }
    __syncthreads();
    float* t0 = dh0; dh0 = dh0n; dh0n = t0;
    float* t1 = dh1; dh1 = dh1n; dh1n = t1;
  }
  // ---- GRU weight gradients: products over (step, sample) rows ----
  const int sG = R * 4 * Hg, sH = R * Hg;
  wgrad(P + g.p_whh1, G3, tile_h(g, t, 1, 0), Hg, sH, 1, tile_gate(g, t, 1, 0), 4 * Hg, sG, 1, B, Hg, G3, 2 * Hg, Hg);
  wgrad(P + g.p_wih1, G3, tile_h(g, t, 0, 0), Hg, sH, 0, tile_gate(g, t, 1, 0), 4 * Hg, sG, 0, B, Hg, G3, G3, 0);
  wgrad(P + g.p_whh0, G3, tile_h(g, t, 0, 0), Hg, sH, 1, tile_gate(g, t, 0, 0), 4 * Hg, sG, 1, B, Hg, G3, 2 * Hg, Hg);
  colsum(P + g.p_bih1, tile_gate(g, t, 1, 0), 4 * Hg, sG, 0, B, G3, G3, 0);
  colsum(P + g.p_bhh1, tile_gate(g, t, 1, 0), 4 * Hg, sG, 0, B, G3, 2 * Hg, Hg);
  colsum(P + g.p_bih0, tile_gate(g, t, 0, 0), 4 * Hg, sG, 0, B, G3, G3, 0);
  colsum(P + g.p_bhh0, tile_gate(g, t, 0, 0), 4 * Hg, sG, 0, B, G3, 2 * Hg, Hg);
  for (int i = tid; i < G3 * gin; i += kGradThreads) {
    const int q = i / gin, u = i - q * gin;
    float acc = 0.0f;
    for (int st = 0; st < B; ++st)
      for (int m = 0; m < R; ++m) acc = fmaf(tile_gate(g, t, 0, st)[m * 4 * Hg + q], t.xs[(st * R + m) * 4 + u], acc);
    P[g.p_wih0 + i] += acc;
  }
}

template <int H>
__global__ void __launch_bounds__(kGradThreads, 1) model_grad_tile_kernel(GradArgs a) {
  const GradShape& g = a.g;
  const ModelDev& md = a.m;
  constexpr int Hg = H / 2, R = kGradRows;
  const int B = g.B, S = g.S, nx = g.nx, in0p = g.in0p;
  const int tid = threadIdx.x;
  float* P = a.part + (size_t)blockIdx.x * g.p_total;
  const TileBufs t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);

  for (int i = tid; i < g.p_total; i += kGradThreads) P[i] = 0.0f;

  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int k0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch are done
    // ---- inputs: normalised window (w_nl.py:121), first-layer input, per-row Fourier constants ----
    tile_load_window(g, md, a.act, k0, a.K, t.xs);
    for (int i = tid; i < R * in0p; i += kGradThreads) {
      const int m = i / in0p, j = i - m * in0p;
      const int k = min(k0 + m, a.K - 1);
      float v = 0.0f;
      if (j < 2 * S) v = a.row_sph[(size_t)k * 2 * S + j];
      else if (j < 2 * S + nx) v = (a.obs[(size_t)k * nx + (j - 2 * S)] - md.state_mean[j - 2 * S]) * md.state_inv_std[j - 2 * S];
      t.x1[i] = v;  // p_action columns are filled after the encoder
    }
    tile_fourier_consts(a.row_tn, k0, a.K, t.rc);
    __syncthreads();
    tile_encoder_fwd<H>(g, md, t);
    const float* h1last = tile_h(g, t, 1, B - 1);
    for (int i = tid; i < R * 2; i += kGradThreads) {  // linear_out (w_nl.py:29) -> p_action columns of the MLP input
      const int m = i >> 1, o = i & 1;
      float acc = md.b_out[o];
      for (int k = 0; k < Hg; ++k) acc = fmaf(md.w_out[o * Hg + k], h1last[m * Hg + k], acc);
      t.x1[m * in0p + 2 * S + nx + o] = acc;
    }
    __syncthreads();
    tile_mlp_fwd_bwd<H>(g, md, a.wt, P, t, a.row_b1, a.gout, k0, a.K);
    tile_encoder_bwd<H>(g, md, a.wt, P, t, a.grad_obs, a.grad_act, k0, a.K);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Several prediction times per sample (nlc_model_backward_multi): the K n_t rows (sample k, time j) = row k n_t + j share
// sample k's encoder output, so the backward runs in two stages instead of the fused tile kernel:
//   MLP/ILT stage over the rows, chunk by chunk (model_grad_multi_mlp_kernel), then a fixed-order sum of each sample's
//   per-row gradient of [obs_n | p_action] over j (model_grad_multi_rowsum_kernel), then one encoder stage over the K
//   samples (model_grad_multi_enc_kernel).  Both stages accumulate into the same per-CTA partials as the tile kernel.
// ------------------------------------------------------------------------------------------------------------------
struct MultiArgs {
  ModelDev m;
  GradShape g;
  const float* obs;      // [K][nx]
  const float* p;        // [K][2] encoder output
  const float* gout;     // [rows][nx]   this chunk's rows of grad_out
  const float* row_b1;   // [rows][H]
  const float* row_tn;   // [rows]
  const float* row_sph;  // [rows][2S]
  const float* wt;
  float* part;
  float* scratch;
  float* drow;           // [rows][Lp] gradient of [obs_n | p_action] per row
  long long r0;          // global index of the chunk's first row
  int rows, n_t;
};

template <int H>
__global__ void __launch_bounds__(kGradThreads, 1) model_grad_multi_mlp_kernel(MultiArgs a) {
  const GradShape& g = a.g;
  const ModelDev& md = a.m;
  constexpr int R = kGradRows;
  const int S = g.S, nx = g.nx, Lp = g.Lp, in0p = g.in0p;
  const int tid = threadIdx.x;
  float* P = a.part + (size_t)blockIdx.x * g.p_total;
  const TileBufs t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);
  const int n_tiles = (a.rows + R - 1) / R;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int k0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch are done
    for (int i = tid; i < R * in0p; i += kGradThreads) {  // [theta_s | phi_s | obs_n | p_action | 0] of row r, sample (r0 + r) / n_t
      const int m = i / in0p, j = i - m * in0p;
      const int r = min(k0 + m, a.rows - 1);
      const size_t k = (size_t)((a.r0 + r) / a.n_t);
      float v = 0.0f;
      if (j < 2 * S) v = a.row_sph[(size_t)r * 2 * S + j];
      else if (j < 2 * S + nx) v = (a.obs[k * nx + (j - 2 * S)] - md.state_mean[j - 2 * S]) * md.state_inv_std[j - 2 * S];
      else if (j < 2 * S + Lp) v = a.p[k * 2 + (j - 2 * S - nx)];
      t.x1[i] = v;
    }
    tile_fourier_consts(a.row_tn, k0, a.rows, t.rc);
    __syncthreads();
    tile_mlp_fwd_bwd<H>(g, md, a.wt, P, t, a.row_b1, a.gout, k0, a.rows);
    for (int i = tid; i < R * Lp; i += kGradThreads) {
      const int m = i / Lp, j = i - m * Lp;
      if (k0 + m < a.rows) a.drow[(size_t)(k0 + m) * Lp + j] = t.dxt[m * 16 + j];
    }
  }
}

// dsum[k] (+)= sum of drow over sample k's rows in this chunk, j ascending; a sample's first row starts its sum, so the
// chunks in order give every sample the same sequential sum over j = 0 .. n_t - 1 whatever the chunk boundaries.
__global__ void __launch_bounds__(256) model_grad_multi_rowsum_kernel(const float* __restrict__ drow, long long r0, int rows, int n_t,
                                                                      int Lp, float* __restrict__ dsum) {
  const long long k_first = r0 / n_t, k_last = (r0 + rows - 1) / n_t;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (k_last - k_first + 1) * Lp) return;
  const long long k = k_first + i / Lp;
  const int c = (int)(i % Lp);
  const long long j0 = k * n_t > r0 ? k * n_t : r0, j1 = (k + 1) * n_t < r0 + rows ? (k + 1) * n_t : r0 + rows;
  float acc = j0 == k * n_t ? 0.0f : dsum[k * Lp + c];
  for (long long r = j0; r < j1; ++r) acc += drow[(r - r0) * Lp + c];
  dsum[k * Lp + c] = acc;
}

// Encoder stage: tiles of kGradRows samples, the summed gradient of [obs_n | p_action] of each sample from dsum [K][Lp].
template <int H>
__global__ void __launch_bounds__(kGradThreads, 1) model_grad_multi_enc_kernel(GradArgs a, const float* __restrict__ dsum) {
  const GradShape& g = a.g;
  const ModelDev& md = a.m;
  constexpr int R = kGradRows;
  const int Lp = g.Lp;
  const int tid = threadIdx.x;
  float* P = a.part + (size_t)blockIdx.x * g.p_total;
  const TileBufs t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int k0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch are done
    tile_load_window(g, md, a.act, k0, a.K, t.xs);
    for (int i = tid; i < R * Lp; i += kGradThreads) {  // rows past K repeat sample K - 1 in the window: zero gradient
      const int m = i / Lp, j = i - m * Lp;
      t.dxt[m * 16 + j] = k0 + m < a.K ? dsum[(size_t)(k0 + m) * Lp + j] : 0.0f;
    }
    __syncthreads();
    tile_encoder_fwd<H>(g, md, t);
    tile_encoder_bwd<H>(g, md, a.wt, P, t, a.grad_obs, a.grad_act, k0, a.K);
  }
}

// Row-major [out][in] copies of the matrices the backward multiplies by transposed.
__global__ void __launch_bounds__(256) model_grad_wt_kernel(ModelDev m, GradShape g, float* wt) {
  const int Hg = g.Hg, G3 = g.G3, H = g.H;
  const int n1 = G3 * Hg, n2 = H * H, n3 = g.N3p * H;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < 3 * n1 + n2 + n3; i += gridDim.x * blockDim.x) {
    if (i < 3 * n1) {
      const int w = i / n1, r = i - w * n1, q = r / Hg, k = r - q * Hg;  // [gate row q][unit k] <- _t [k][q]
      const float* src = w == 0 ? m.w_hh0_t : (w == 1 ? m.w_ih1_t : m.w_hh1_t);
      wt[(w == 0 ? g.w_hh0 : (w == 1 ? g.w_ih1 : g.w_hh1)) + r] = src[k * G3 + q];
    } else if (i < 3 * n1 + n2) {
      const int r = i - 3 * n1, n = r / H, k = r - n * H;
      wt[g.w_2 + r] = m.w2_t[k * H + n];
    } else {
      const int r = i - 3 * n1 - n2, col = r / H, h = r - col * H;
      wt[g.w_3 + r] = m.w3_t[(size_t)h * g.N3p + col];
    }
  }
}

// Sum of the per-CTA partials in CTA order, written in the state_dict layout (named_parameters() order).
__global__ void __launch_bounds__(256) model_grad_reduce_kernel(GradShape g, const float* __restrict__ part, int n_part, float* out) {
  const int Hg = g.Hg, G3 = g.G3, H = g.H, S = g.S, nx = g.nx;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < g.o_total; i += gridDim.x * blockDim.x) {
    int src;
    if (i < g.o_whh0) src = g.p_wih0 + i;
    else if (i < g.o_bih0) { const int r = i - g.o_whh0; src = g.p_whh0 + (r % Hg) * G3 + r / Hg; }
    else if (i < g.o_bhh0) src = g.p_bih0 + i - g.o_bih0;
    else if (i < g.o_wih1) src = g.p_bhh0 + i - g.o_bhh0;
    else if (i < g.o_whh1) { const int r = i - g.o_wih1; src = g.p_wih1 + (r % Hg) * G3 + r / Hg; }
    else if (i < g.o_bih1) { const int r = i - g.o_whh1; src = g.p_whh1 + (r % Hg) * G3 + r / Hg; }
    else if (i < g.o_bhh1) src = g.p_bih1 + i - g.o_bih1;
    else if (i < g.o_wout) src = g.p_bhh1 + i - g.o_bhh1;
    else if (i < g.o_bout) src = g.p_wout + i - g.o_wout;
    else if (i < g.o_w0) src = g.p_bout + i - g.o_bout;
    else if (i < g.o_b0) { const int r = i - g.o_w0; src = g.p_w0 + (r % g.in0) * H + r / g.in0; }
    else if (i < g.o_w2) src = g.p_b0 + i - g.o_b0;
    else if (i < g.o_b2) { const int r = i - g.o_w2; src = g.p_w2 + (r % H) * H + r / H; }
    else if (i < g.o_w4) src = g.p_b2 + i - g.o_b2;
    else {
      // linear_tanh_stack.4 row ch * S + k, ch = part * nx + c  <-  paired column 2 (c S + k) + part
      const bool bias = i >= g.o_b4;
      const int r = bias ? i - g.o_b4 : i - g.o_w4;
      const int row = bias ? r : r / H, h = bias ? 0 : r - row * H;
      const int ch = row / S, k = row - ch * S, prt = ch / nx, c = ch - prt * nx;
      const int col = 2 * (c * S + k) + prt;
      src = bias ? g.p_b4 + col : g.p_w4 + h * g.N3p + col;
    }
    float acc = 0.0f;
    for (int c = 0; c < n_part; ++c) acc += part[(size_t)c * g.p_total + src];
    out[i] = acc;
  }
}

static GradShape shape_of(const nlc_model_s* m, int B) { return make_shape(m->nx, m->nu, m->gin, m->Hm, m->S, B); }

static int grad_grid(int K) {
  const int n_tiles = (K + kGradRows - 1) / kGradRows;
  return n_tiles < kGradGridCap ? n_tiles : kGradGridCap;
}

// workspace (floats): row_b1 [K][H] | row_tn [K] | row_sph [K][2S] | weight copies | partials [grid] | scratch [grid]
struct GradWs { size_t b1, tn, sph, wt, part, scr, total; };
static GradWs ws_layout(const GradShape& g, int K) {
  GradWs w;
  size_t o = 0;
  w.b1 = o; o += up64((size_t)K * g.H);
  w.tn = o; o += up64(K);
  w.sph = o; o += up64((size_t)K * 2 * g.S);
  w.wt = o; o += g.w_total;
  const int G = grad_grid(K);
  w.part = o; o += (size_t)G * g.p_total;
  w.scr = o; o += (size_t)G * g.s_total;
  w.total = o;
  return w;
}

// Several prediction times per sample: rows are walked in chunks of at most kMultiChunkRows (rollout.cu), so the per-row
// buffers are bounded whatever K n_t is.
// workspace (floats): p [K][2] | dsum [K][Lp] | row_b1 [C][H] | row_tn [C] | row_sph [C][2S] | drow [C][Lp] | weight copies |
// partials [G] | scratch [G], C = min(K n_t, kMultiChunkRows), G = max(grid of C rows, grid of K samples)
struct MultiWs { size_t p, dsum, b1, tn, sph, drow, wt, part, scr, total; int C, Gm, Ge, G; };
static MultiWs multi_ws_layout(const GradShape& g, int K, int n_t) {
  MultiWs w;
  const long long rows = (long long)K * n_t;
  w.C = rows < kMultiChunkRows ? (int)rows : kMultiChunkRows;
  w.Gm = grad_grid(w.C); w.Ge = grad_grid(K); w.G = w.Gm > w.Ge ? w.Gm : w.Ge;
  size_t o = 0;
  w.p = o; o += up64((size_t)K * 2);
  w.dsum = o; o += up64((size_t)K * g.Lp);
  w.b1 = o; o += up64((size_t)w.C * g.H);
  w.tn = o; o += up64(w.C);
  w.sph = o; o += up64((size_t)w.C * 2 * g.S);
  w.drow = o; o += up64((size_t)w.C * g.Lp);
  w.wt = o; o += g.w_total;
  w.part = o; o += (size_t)w.G * g.p_total;
  w.scr = o; o += (size_t)w.G * g.s_total;
  w.total = o;
  return w;
}

}  // namespace nlc

using namespace nlc;

extern "C" int64_t nlc_model_grad_floats(const nlc_model_desc* d) {
  if (!d || d->state_dim < 1 || d->action_dim < 1 || d->hidden_units < 2 || d->hidden_units % 2 || d->s_terms < 1) return NLC_ERR_ARG;
  const int64_t nx = d->state_dim, gin = d->action_dim + (d->encode_obs_time ? 1 : 0), H = d->hidden_units, S = d->s_terms;
  const int64_t Hg = H / 2, G3 = 3 * Hg, in0 = 2 * S + nx + 2, N3 = 2 * nx * S;
  return G3 * gin + 3 * G3 * Hg + 4 * G3 + 2 * Hg + 2 + H * in0 + H + H * H + H + N3 * H + N3;
}

extern "C" int64_t nlc_model_backward_workspace_bytes(nlc_model_t m, int K, int B) {
  if (!m || K < 1 || B < 1 || B > 8) return NLC_ERR_ARG;
  return (int64_t)(ws_layout(shape_of(m, B), K).total * sizeof(float));
}

extern "C" int nlc_model_backward_ts(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K, int B,
                                     const float* grad_out_dev, float* grad_params_dev, float* grad_obs_dev, float* grad_act_dev,
                                     void* workspace_dev, void* stream) {
  NLC_REQUIRE(m && obs_dev && act_dev && ts_dev && grad_out_dev && grad_params_dev && workspace_dev, NLC_ERR_ARG,
              "nlc_model_backward_ts: null pointer");
  NLC_REQUIRE(K >= 1, NLC_ERR_ARG, "nlc_model_backward_ts: K must be positive");
  NLC_REQUIRE(B >= 1 && B <= 8, NLC_ERR_SHAPE, "nlc_model_backward_ts: window length %d outside [1,8]", B);
  NLC_REQUIRE(((uintptr_t)workspace_dev & 15) == 0, NLC_ERR_ARG, "nlc_model_backward_ts: workspace must be 16-byte aligned");
  int rc = check_device_arch(m->device);
  if (rc != NLC_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const GradShape g = shape_of(m, B);
  const GradWs w = ws_layout(g, K);
  float* ws = static_cast<float*>(workspace_dev);
  rc = launch_forward_ts_prep(m, ts_dev, K, ws + w.b1, ws + w.tn, ws + w.sph, s);
  if (rc != NLC_OK) return rc;
  const int n_wt = 3 * g.G3 * g.Hg + g.H * g.H + g.N3p * g.H;
  model_grad_wt_kernel<<<(n_wt + 255) / 256, 256, 0, s>>>(m->d, g, ws + w.wt);
  NLC_LAUNCH_OK("model_grad_wt_kernel");
  GradArgs a;
  a.m = m->d; a.g = g; a.obs = obs_dev; a.act = act_dev; a.gout = grad_out_dev;
  a.row_b1 = ws + w.b1; a.row_tn = ws + w.tn; a.row_sph = ws + w.sph; a.wt = ws + w.wt;
  a.part = ws + w.part; a.scratch = ws + w.scr; a.grad_obs = grad_obs_dev; a.grad_act = grad_act_dev;
  a.K = K; a.n_tiles = (K + kGradRows - 1) / kGradRows;
  const int G = grad_grid(K);
  if (m->Hm == 128) model_grad_tile_kernel<128><<<G, kGradThreads, 0, s>>>(a);
  else model_grad_tile_kernel<64><<<G, kGradThreads, 0, s>>>(a);
  NLC_LAUNCH_OK("model_grad_tile_kernel");
  model_grad_reduce_kernel<<<(g.o_total + 255) / 256, 256, 0, s>>>(g, ws + w.part, G, grad_params_dev);
  NLC_LAUNCH_OK("model_grad_reduce_kernel");
  return NLC_OK;
}

extern "C" int64_t nlc_model_backward_multi_workspace_bytes(nlc_model_t m, int K, int n_t, int B) {
  if (!m || K < 1 || n_t < 1 || B < 1 || B > 8) return NLC_ERR_ARG;
  if ((long long)K * n_t >= (1LL << 31)) return NLC_ERR_SHAPE;
  return (int64_t)(multi_ws_layout(shape_of(m, B), K, n_t).total * sizeof(float));
}

extern "C" int nlc_model_backward_multi(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K, int n_t,
                                        int B, const float* grad_out_dev, float* grad_params_dev, float* grad_obs_dev,
                                        float* grad_act_dev, void* workspace_dev, void* stream) {
  NLC_REQUIRE(m && obs_dev && act_dev && ts_dev && grad_out_dev && grad_params_dev && workspace_dev, NLC_ERR_ARG,
              "nlc_model_backward_multi: null pointer");
  NLC_REQUIRE(K >= 1 && n_t >= 1, NLC_ERR_ARG, "nlc_model_backward_multi: K and n_t must be positive");
  NLC_REQUIRE((long long)K * n_t < (1LL << 31), NLC_ERR_SHAPE, "nlc_model_backward_multi: K n_t = %lld rows, 2^31 or more",
              (long long)K * n_t);
  NLC_REQUIRE(B >= 1 && B <= 8, NLC_ERR_SHAPE, "nlc_model_backward_multi: window length %d outside [1,8]", B);
  NLC_REQUIRE(((uintptr_t)workspace_dev & 15) == 0, NLC_ERR_ARG, "nlc_model_backward_multi: workspace must be 16-byte aligned");
  int rc = check_device_arch(m->device);
  if (rc != NLC_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const GradShape g = shape_of(m, B);
  const MultiWs w = multi_ws_layout(g, K, n_t);
  float* ws = static_cast<float*>(workspace_dev);
  // the encoder output every row of a sample shares, on the fp32 kernel like the rest of the backward
  rc = encode_history_impl(m, act_dev, m->gin, K, 1, B, ws + w.p, NLC_MATH_FP32, s);
  if (rc != NLC_OK) return rc;
  const int n_wt = 3 * g.G3 * g.Hg + g.H * g.H + g.N3p * g.H;
  model_grad_wt_kernel<<<(n_wt + 255) / 256, 256, 0, s>>>(m->d, g, ws + w.wt);
  NLC_LAUNCH_OK("model_grad_wt_kernel");
  NLC_CUDA_OK(cudaMemsetAsync(ws + w.part, 0, (size_t)w.G * g.p_total * sizeof(float), s));
  MultiArgs ma;
  ma.m = m->d; ma.g = g; ma.obs = obs_dev; ma.p = ws + w.p; ma.row_b1 = ws + w.b1; ma.row_tn = ws + w.tn; ma.row_sph = ws + w.sph;
  ma.wt = ws + w.wt; ma.part = ws + w.part; ma.scratch = ws + w.scr; ma.drow = ws + w.drow; ma.n_t = n_t;
  const long long n_rows = (long long)K * n_t;
  for (long long r0 = 0; r0 < n_rows; r0 += w.C) {
    const int rows = (int)(n_rows - r0 < w.C ? n_rows - r0 : w.C);
    rc = launch_forward_ts_prep(m, ts_dev + r0, rows, ws + w.b1, ws + w.tn, ws + w.sph, s);
    if (rc != NLC_OK) return rc;
    ma.gout = grad_out_dev + r0 * g.nx; ma.r0 = r0; ma.rows = rows;
    if (m->Hm == 128) model_grad_multi_mlp_kernel<128><<<w.Gm, kGradThreads, 0, s>>>(ma);
    else model_grad_multi_mlp_kernel<64><<<w.Gm, kGradThreads, 0, s>>>(ma);
    NLC_LAUNCH_OK("model_grad_multi_mlp_kernel");
    const long long n_sum = ((r0 + rows - 1) / n_t - r0 / n_t + 1) * g.Lp;
    model_grad_multi_rowsum_kernel<<<(unsigned)((n_sum + 255) / 256), 256, 0, s>>>(ws + w.drow, r0, rows, n_t, g.Lp, ws + w.dsum);
    NLC_LAUNCH_OK("model_grad_multi_rowsum_kernel");
  }
  GradArgs a;
  a.m = m->d; a.g = g; a.obs = obs_dev; a.act = act_dev; a.gout = nullptr;
  a.row_b1 = nullptr; a.row_tn = nullptr; a.row_sph = nullptr; a.wt = ws + w.wt;
  a.part = ws + w.part; a.scratch = ws + w.scr; a.grad_obs = grad_obs_dev; a.grad_act = grad_act_dev;
  a.K = K; a.n_tiles = (K + kGradRows - 1) / kGradRows;
  if (m->Hm == 128) model_grad_multi_enc_kernel<128><<<w.Ge, kGradThreads, 0, s>>>(a, ws + w.dsum);
  else model_grad_multi_enc_kernel<64><<<w.Ge, kGradThreads, 0, s>>>(a, ws + w.dsum);
  NLC_LAUNCH_OK("model_grad_multi_enc_kernel");
  model_grad_reduce_kernel<<<(g.o_total + 255) / 256, 256, 0, s>>>(g, ws + w.part, w.G, grad_params_dev);
  NLC_LAUNCH_OK("model_grad_reduce_kernel");
  return NLC_OK;
}
