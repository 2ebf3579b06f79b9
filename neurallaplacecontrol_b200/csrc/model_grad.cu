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
//
// fp64 (nlc_model_forward_f64 / nlc_model_backward_f64, the reference's training precision): the tile machinery below is
// templated on the scalar type and instantiated a second time for double.  The weights then come per call from the
// caller's fp64 parameter buffer (state_dict layout), which model_f64_weights_kernel rearranges into the workspace in the
// layouts ModelDev holds (TileW); only shapes, flags, dt and the fp64 normalisation constants are read from the handle.
// The fp64 forward is the recompute half of the tile steps (encoder, linear_out, MLP) followed by the ILT sum; the fp64
// backward runs the two-stage form of nlc_model_backward_multi for every n_t (n_t = 1 included).
//
// The fp64 planner (planner_f64.cu) runs its history encoder and rollout on the same tile steps (at the end); that encoder
// also encodes the fp64 model's windows.
#include <stddef.h>

#include "common.cuh"
#include "env_cost.cuh"

namespace nlc {

template <typename T>
int launch_forward_ts_prep(nlc_model_s* m, const T* b1_raw, const T* w1_full_t, const T* ts, int K, T* row_b1, T* row_tn, T* row_sph,
                           cudaStream_t s, const T* obs = nullptr, const T* p = nullptr, long long r0 = 0, int n_t = 1,
                           T* row_obs = nullptr, T* row_p = nullptr);
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
  // fp64 only: the forward layouts of every weight (TileW), after the transposed copies (offsets from the image's start)
  int f_wih0, f_bih0, f_bhh0, f_hh0t, f_ih1t, f_hh1t, f_bih1, f_bhh1, f_wout, f_bout, f_w1t, f_b1, f_w2t, f_b2, f_w3t, f_b3, f_total;
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
  o = g.w_total;
  g.f_wih0 = take(G3 * gin); g.f_bih0 = take(G3); g.f_bhh0 = take(G3); g.f_hh0t = take(Hg * G3); g.f_ih1t = take(Hg * G3);
  g.f_hh1t = take(Hg * G3); g.f_bih1 = take(G3); g.f_bhh1 = take(G3); g.f_wout = take(2 * Hg); g.f_bout = take(2);
  g.f_w1t = take(g.in0 * H); g.f_b1 = take(H); g.f_w2t = take(H * H); g.f_b2 = take(H); g.f_w3t = take(H * g.N3p); g.f_b3 = take(g.N3p);
  g.f_total = (int)up64(o);
  return g;
}

// The weights the tile steps read, in ModelDev's layouts: the handle's fp32 arena, or (T = double) the image
// model_f64_weights_kernel builds in the workspace from the caller's parameters.
template <typename T>
struct TileW {
  const T *w_ih0, *b_ih0, *b_hh0, *w_hh0_t, *w_ih1_t, *w_hh1_t, *b_ih1, *b_hh1, *w_out, *b_out;
  const T *w1_full_t, *b1_raw, *w2_t, *b2, *w3_t, *b3;
  const T *state_mean, *state_inv_std, *act_mean, *act_inv_std;
};

static TileW<float> tile_w(const ModelDev& d) {
  TileW<float> w;
  w.w_ih0 = d.w_ih0; w.b_ih0 = d.b_ih0; w.b_hh0 = d.b_hh0; w.w_hh0_t = d.w_hh0_t; w.w_ih1_t = d.w_ih1_t; w.w_hh1_t = d.w_hh1_t;
  w.b_ih1 = d.b_ih1; w.b_hh1 = d.b_hh1; w.w_out = d.w_out; w.b_out = d.b_out;
  w.w1_full_t = d.w1_full_t; w.b1_raw = d.b1_raw; w.w2_t = d.w2_t; w.b2 = d.b2; w.w3_t = d.w3_t; w.b3 = d.b3;
  w.state_mean = d.state_mean; w.state_inv_std = d.state_inv_std; w.act_mean = d.act_mean; w.act_inv_std = d.act_inv_std;
  return w;
}

static TileW<double> tile_w_f64(const ModelDev& d, const GradShape& g, const double* img) {
  TileW<double> w;
  w.w_ih0 = img + g.f_wih0; w.b_ih0 = img + g.f_bih0; w.b_hh0 = img + g.f_bhh0; w.w_hh0_t = img + g.f_hh0t; w.w_ih1_t = img + g.f_ih1t;
  w.w_hh1_t = img + g.f_hh1t; w.b_ih1 = img + g.f_bih1; w.b_hh1 = img + g.f_bhh1; w.w_out = img + g.f_wout; w.b_out = img + g.f_bout;
  w.w1_full_t = img + g.f_w1t; w.b1_raw = img + g.f_b1; w.w2_t = img + g.f_w2t; w.b2 = img + g.f_b2; w.w3_t = img + g.f_w3t;
  w.b3 = img + g.f_b3;
  w.state_mean = d.state_mean64; w.state_inv_std = d.state_inv_std64; w.act_mean = d.act_mean64; w.act_inv_std = d.act_inv_std64;
  return w;
}

template <typename T>
struct GradArgs {
  TileW<T> m;
  GradShape g;
  const T* obs;       // [K][nx]
  const T* act;       // [K][B][gin]
  const T* gout;      // [K][nx]
  const T* row_b1;    // [K][H]
  const T* row_tn;    // [K]
  const T* row_sph;   // [K][2S]
  const T* wt;        // transposed weight copies
  T* part;            // [grid][p_total]
  T* scratch;         // [grid][s_total]
  T* grad_obs;        // [K][nx] or null
  T* grad_act;        // [K][B][gin] or null
  int K, n_tiles;
};

// ------------------------------------------------------------------------------------------------------------------
// Tile products.  Rows are the kGradRows samples of the tile; every thread owns fixed 4 x 4 output blocks, so an output
// element is always written by the same thread (repeated accumulating calls on one output need no barrier between them).
// Everything from here to the kernels is templated on the scalar type T (float: the fp32 backward; double: the fp64
// forward and backward).
// ------------------------------------------------------------------------------------------------------------------
enum { kEpiNone = 0, kEpiTanh = 1, kEpiDtanh = 2 };

// C[m][n] (+)= sum_k A[m][k] W[k][n]  (+ bias[n]; kEpiTanh: tanh of it; kEpiDtanh: times 1 - aux[m][n]^2).
// N, Kd, lda, ldw, ldc multiples of 4; W is read-only for the kernel's lifetime.
template <int EPI, typename T>
__device__ __forceinline__ void gemm_nn(const T* A, int lda, const T* __restrict__ W, int ldw, int Kd, int N, T* C, int ldc,
                                        bool accumulate, const T* __restrict__ bias = nullptr, const T* aux = nullptr) {
  const int CG = N / 4, items = (kGradRows / 4) * CG;
  for (int it = threadIdx.x; it < items; it += kGradThreads) {
    const int rg = it / CG, cg = it - rg * CG;
    T c[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (accumulate) rm::ld4(C + (4 * rg + i) * ldc + 4 * cg, c[i]);
      else if (bias) rm::ld4(bias + 4 * cg, c[i]);
      else c[i][0] = c[i][1] = c[i][2] = c[i][3] = T(0);
    }
#pragma unroll 2
    for (int k = 0; k < Kd; k += 4) {
      T a[4][4];
#pragma unroll
      for (int i = 0; i < 4; ++i) rm::ld4(A + (4 * rg + i) * lda + k, a[i]);
#pragma unroll
      for (int kk = 0; kk < 4; ++kk) {
        T w[4];
        rm::ldg4(W + (size_t)(k + kk) * ldw + 4 * cg, w);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const T av = a[i][kk];
          c[i][0] = rm::fma(av, w[0], c[i][0]);
          c[i][1] = rm::fma(av, w[1], c[i][1]);
          c[i][2] = rm::fma(av, w[2], c[i][2]);
          c[i][3] = rm::fma(av, w[3], c[i][3]);
        }
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      T* dst = C + (4 * rg + i) * ldc + 4 * cg;
      if (EPI == kEpiTanh) {
        for (int j = 0; j < 4; ++j) c[i][j] = tanh_acc(c[i][j]);
      } else if (EPI == kEpiDtanh) {
        T y[4];
        rm::ld4(aux + (4 * rg + i) * ldc + 4 * cg, y);
        c[i][0] *= T(1) - y[0] * y[0]; c[i][1] *= T(1) - y[1] * y[1]; c[i][2] *= T(1) - y[2] * y[2]; c[i][3] *= T(1) - y[3] * y[3];
      }
      rm::st4(dst, c[i]);
    }
  }
}

// Weight gradient: P[k][n] += sum_{s in [s0, s1)} sum_m A_s[m][k] D_s[m][col(n)], A_s = A + (s - alag) sA, D_s = D + s sD,
// col(n) = n + (n >= nsplit ? dshift : 0) (skips a gate slot of the saved GRU gradients).  Kd, N, nsplit multiples of 4.
template <typename T>
__device__ __forceinline__ void wgrad(T* P, int ldp, const T* A, int lda, int sA, int alag, const T* D, int ldd, int sD,
                                      int s0, int s1, int Kd, int N, int nsplit, int dshift) {
  const int CG = N / 4, items = (Kd / 4) * CG;
  for (int it = threadIdx.x; it < items; it += kGradThreads) {
    const int kg = it / CG, cg = it - kg * CG;
    const int dc = 4 * cg + (4 * cg >= nsplit ? dshift : 0);
    T c[4][4] = {};
    for (int s = s0; s < s1; ++s) {
      const T* As = A + (s - alag) * sA + 4 * kg;
      const T* Ds = D + s * sD + dc;
#pragma unroll 4
      for (int m = 0; m < kGradRows; ++m) {
        T av[4], dv[4];
        rm::ld4(As + m * lda, av);
        rm::ld4(Ds + m * ldd, dv);
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) c[i][j] = rm::fma(av[i], dv[j], c[i][j]);
      }
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      T* p = P + (4 * kg + i) * ldp + 4 * cg;
      T v[4];
      rm::ld4(p, v);
      v[0] += c[i][0]; v[1] += c[i][1]; v[2] += c[i][2]; v[3] += c[i][3];
      rm::st4(p, v);
    }
  }
}

// Bias gradient: P[n] += sum_{s in [s0, s1)} sum_m D_s[m][col(n)]
template <typename T>
__device__ __forceinline__ void colsum(T* P, const T* D, int ldd, int sD, int s0, int s1, int N, int nsplit, int dshift) {
  for (int n = threadIdx.x; n < N; n += kGradThreads) {
    const int dc = n + (n >= nsplit ? dshift : 0);
    T acc = T(0);
    for (int s = s0; s < s1; ++s)
      for (int m = 0; m < kGradRows; ++m) acc += D[s * sD + m * ldd + dc];
    P[n] += acc;
  }
}

// GRU cell forward (torch.nn.GRU, gate order r, z, n; the same expressions as encode_gru.cu gru_finish).  gi / gh are the
// bias-free products (gh null: zero state); layer 0 (gin inputs) forms gi here from the step's window entry.
template <typename T>
__device__ __forceinline__ void gru_cell_fwd(const GradShape& g, const T* __restrict__ b_i, const T* __restrict__ b_h,
                                             const T* __restrict__ w_ih0, const T* xs, const T* gi, const T* gh,
                                             const T* hprev, T* gate, T* hout) {
  const int Hg = g.Hg, G3 = g.G3;
  for (int i = threadIdx.x; i < kGradRows * Hg; i += kGradThreads) {
    const int m = i / Hg, u = i - m * Hg;
    T gir, giz, gin_;
    if (gi) {
      gir = gi[m * G3 + u]; giz = gi[m * G3 + Hg + u]; gin_ = gi[m * G3 + 2 * Hg + u];
    } else {
      T acc[3];
#pragma unroll
      for (int q = 0; q < 3; ++q) {
        const T* w = w_ih0 + (q * Hg + u) * g.gin;
        T a = T(0);
        for (int v = 0; v < g.gin; ++v) a = rm::fma(w[v], xs[m * 4 + v], a);
        acc[q] = a;
      }
      gir = acc[0]; giz = acc[1]; gin_ = acc[2];
    }
    const T ghr = gh ? gh[m * G3 + u] : T(0), ghz = gh ? gh[m * G3 + Hg + u] : T(0), ghn0 = gh ? gh[m * G3 + 2 * Hg + u] : T(0);
    const T r = sigmoid_acc((gir + b_i[u]) + (ghr + b_h[u]));
    const T z = sigmoid_acc((giz + b_i[Hg + u]) + (ghz + b_h[Hg + u]));
    const T ghn = ghn0 + b_h[2 * Hg + u];
    const T n = tanh_acc((gin_ + b_i[2 * Hg + u]) + r * ghn);
    const T ho = hprev ? hprev[m * Hg + u] : T(0);
    T* gt = gate + m * 4 * Hg;
    gt[u] = r; gt[Hg + u] = z; gt[2 * Hg + u] = n; gt[3 * Hg + u] = ghn;
    hout[m * Hg + u] = rm::fma(z, ho - n, n);
  }
}

// GRU cell backward: dh -> (dr_pre, dz_pre, dn_pre, d(W_hn h + b_hn)) in place of the saved gates, dh_prev's direct part.
template <typename T>
__device__ __forceinline__ void gru_cell_bwd(const GradShape& g, const T* dh, const T* hprev, T* gate, T* dh_prev) {
  const int Hg = g.Hg;
  for (int i = threadIdx.x; i < kGradRows * Hg; i += kGradThreads) {
    const int m = i / Hg, u = i - m * Hg;
    T* gt = gate + m * 4 * Hg;
    const T r = gt[u], z = gt[Hg + u], n = gt[2 * Hg + u], ghn = gt[3 * Hg + u];
    const T d = dh[m * Hg + u], ho = hprev ? hprev[m * Hg + u] : T(0);
    const T dn = d * (T(1) - z) * (T(1) - n * n);
    const T dr = dn * ghn * r * (T(1) - r);
    const T dz = d * (ho - n) * z * (T(1) - z);
    gt[u] = dr; gt[Hg + u] = dz; gt[2 * Hg + u] = dn; gt[3 * Hg + u] = dn * r;
    dh_prev[m * Hg + u] = d * z;
  }
}

// The per-CTA scratch of a tile (GradShape s_* offsets, in elements of T).
template <typename T>
struct TileBufs {
  T *xs, *gate, *hs, *gi, *gh, *x1, *a1, *a2, *dob, *dz2, *dz1, *dhb, *dxt, *rc;
};
template <typename T>
__device__ __forceinline__ TileBufs<T> tile_bufs(const GradShape& g, T* sc) {
  TileBufs<T> t;
  t.xs = sc + g.s_xs; t.gate = sc + g.s_gate; t.hs = sc + g.s_h; t.gi = sc + g.s_gi; t.gh = sc + g.s_gh; t.x1 = sc + g.s_x1;
  t.a1 = sc + g.s_a1; t.a2 = sc + g.s_a2; t.dob = sc + g.s_do; t.dz2 = sc + g.s_dz2; t.dz1 = sc + g.s_dz1; t.dhb = sc + g.s_dh;
  t.dxt = sc + g.s_dxt; t.rc = sc + g.s_rc;
  return t;
}
// gate [l][st] at (l * B + st) * R * 4Hg, h [l][st] at (l * B + st) * R * Hg
template <typename T>
__device__ __forceinline__ T* tile_gate(const GradShape& g, const TileBufs<T>& t, int l, int st) {
  return t.gate + (size_t)(l * g.B + st) * kGradRows * 4 * g.Hg;
}
template <typename T>
__device__ __forceinline__ T* tile_h(const GradShape& g, const TileBufs<T>& t, int l, int st) {
  return t.hs + (size_t)(l * g.B + st) * kGradRows * g.Hg;
}

// Normalised window of samples k0 .. k0 + R - 1 (w_nl.py:121); rows past K repeat sample K - 1.
template <typename T>
__device__ __forceinline__ void tile_load_window(const GradShape& g, const TileW<T>& md, const T* act, int k0, int K, T* xs) {
  const int B = g.B, gin = g.gin, R = kGradRows;
  for (int i = threadIdx.x; i < B * R * 4; i += kGradThreads) {
    const int st = i / (R * 4), m = (i / 4) % R, u = i & 3;
    const int k = min(k0 + m, K - 1), j = B - 1 - st;  // step st reads entry B-1-st (reversed in time, w_nl.py:27)
    xs[i] = u < gin ? (act[((size_t)k * B + j) * gin + u] - md.act_mean[u]) * md.act_inv_std[u] : T(0);
  }
}

// Per-row Fourier constants pi t / T and exp(gamma t) / T of rows k0 .. k0 + R - 1 (rollout.cu rollout_nl_kernel: the same).
template <typename T>
__device__ __forceinline__ void tile_fourier_consts(const T* row_tn, int k0, int K, T* rc) {
  using C = Real<T>;
  const int R = kGradRows;
  for (int m = threadIdx.x; m < R; m += kGradThreads) {
    const T tn = row_tn[min(k0 + m, K - 1)];
    const T Tp = T(2) * (tn + C::eps);
    rc[m] = C::pi * C::eps / Tp;
    rc[R + m] = rm::exp((C::alpha + C::ln_inv_tol / Tp) * tn) / Tp;
  }
}

// Phase k pi t / T (the quarter turns exact, reduced to (-pi, pi] up to k delta) and Fourier weight of term kk of row m.
template <typename T>
__device__ __forceinline__ void ilt_term_consts(int kk, const T* rc, int m, T& ph, T& wt) {
  using C = Real<T>;
  const T quarter = (kk & 3) == 0 ? T(0) : ((kk & 3) == 1 ? C::half_pi : ((kk & 3) == 2 ? C::pi : -C::half_pi));
  ph = quarter - (T)kk * rc[m];
  wt = rc[kGradRows + m] * (kk == 0 ? T(0.5) : T(1));
}

// Encoder forward (w_nl.py:25-29) of the tile's windows, saving every cell.  Ends on a barrier.
template <int H, typename T>
__device__ __forceinline__ void tile_encoder_fwd(const GradShape& g, const TileW<T>& md, const TileBufs<T>& t) {
  constexpr int Hg = H / 2, G3 = 3 * Hg;
  const int B = g.B;
  for (int st = 0; st < B; ++st) {
    if (st > 0) {
      gemm_nn<kEpiNone>(tile_h(g, t, 0, st - 1), Hg, md.w_hh0_t, G3, Hg, G3, t.gh, G3, false);
      __syncthreads();
    }
    gru_cell_fwd(g, md.b_ih0, md.b_hh0, md.w_ih0, t.xs + st * kGradRows * 4, (const T*)nullptr, st > 0 ? t.gh : nullptr,
                 st > 0 ? tile_h(g, t, 0, st - 1) : nullptr, tile_gate(g, t, 0, st), tile_h(g, t, 0, st));
    __syncthreads();
    gemm_nn<kEpiNone>(tile_h(g, t, 0, st), Hg, md.w_ih1_t, G3, Hg, G3, t.gi, G3, false);
    if (st > 0) gemm_nn<kEpiNone>(tile_h(g, t, 1, st - 1), Hg, md.w_hh1_t, G3, Hg, G3, t.gh, G3, false);
    __syncthreads();
    gru_cell_fwd(g, md.b_ih1, md.b_hh1, (const T*)nullptr, (const T*)nullptr, t.gi, st > 0 ? t.gh : nullptr,
                 st > 0 ? tile_h(g, t, 1, st - 1) : nullptr, tile_gate(g, t, 1, st), tile_h(g, t, 1, st));
    __syncthreads();
  }
}

// linear_out (w_nl.py:29) of the tile's last top-layer state -> the p_action columns of the MLP input x1.  No barrier.
template <typename T>
__device__ __forceinline__ void tile_linear_out(const GradShape& g, const TileW<T>& md, const TileBufs<T>& t) {
  const int Hg = g.Hg, base = 2 * g.S + g.nx;
  const T* h1last = tile_h(g, t, 1, g.B - 1);
  for (int i = threadIdx.x; i < kGradRows * 2; i += kGradThreads) {
    const int m = i >> 1, o = i & 1;
    T acc = md.b_out[o];
    for (int k = 0; k < Hg; ++k) acc = rm::fma(md.w_out[o * Hg + k], h1last[m * Hg + k], acc);
    t.x1[m * g.in0p + base + o] = acc;
  }
}

// First-layer input [theta_s | phi_s | obs_n | p_action | 0] of rows k0 .. k0 + R - 1 of a chunk whose row r is (sample
// (r0 + r) / n_t, time (r0 + r) % n_t): sphere coordinates from row_sph [rows][2S], obs [K][nx] and p [K][2] per sample.
template <typename T>
__device__ __forceinline__ void tile_rows_input(const GradShape& g, const TileW<T>& md, const T* row_sph, const T* obs, const T* p,
                                                long long r0, int rows, int n_t, int k0, T* x1) {
  const int S = g.S, nx = g.nx, Lp = g.Lp, in0p = g.in0p;
  for (int i = threadIdx.x; i < kGradRows * in0p; i += kGradThreads) {
    const int m = i / in0p, j = i - m * in0p;
    const int r = min(k0 + m, rows - 1);
    const size_t k = (size_t)((r0 + r) / n_t);
    T v = T(0);
    if (j < 2 * S) v = row_sph[(size_t)r * 2 * S + j];
    else if (j < 2 * S + nx) v = (obs[k * nx + (j - 2 * S)] - md.state_mean[j - 2 * S]) * md.state_inv_std[j - 2 * S];
    else if (j < 2 * S + Lp) v = p[k * 2 + (j - 2 * S - nx)];
    x1[i] = v;
  }
}

// Representation MLP forward (w_nl.py:55-63) from the first-layer input x1: a1, a2 and the last layer's pre-activations
// in dob.  Rows k0 .. k0 + R - 1 of row_b1 [K][H] (the s-columns, forward_ts_prep_kernel).  Ends on a barrier.
template <int H, typename T>
__device__ __forceinline__ void tile_mlp_fwd(const GradShape& g, const TileW<T>& md, const TileBufs<T>& t, const T* row_b1, int k0,
                                             int K) {
  constexpr int R = kGradRows;
  const int S = g.S, Lp = g.Lp, in0p = g.in0p, N3p = g.N3p;
  T *x1 = t.x1, *a1 = t.a1, *a2 = t.a2, *dob = t.dob;
  for (int i = threadIdx.x; i < R * H; i += kGradThreads) {
    const int m = i / H, n = i - m * H;
    T acc = row_b1[(size_t)min(k0 + m, K - 1) * H + n];
    for (int j = 0; j < Lp; ++j) acc = rm::fma(md.w1_full_t[(size_t)(2 * S + j) * H + n], x1[m * in0p + 2 * S + j], acc);
    a1[i] = tanh_acc(acc);
  }
  __syncthreads();
  gemm_nn<kEpiTanh>(a1, H, md.w2_t, H, H, H, a2, H, false, md.b2);
  __syncthreads();
  gemm_nn<kEpiNone>(a2, H, md.w3_t, N3p, H, N3p, dob, N3p, false, md.b3);
  __syncthreads();
}

// The ILT of tile_mlp_fwd's output (w_nl.py:59-62 + the Fourier series, oracle/ilt.py): out[k0 + m][c] =
// sum_k w_k rho_k cos(theta_k + a_k), k ascending, for the rows below K.  No barrier.
template <typename T>
__device__ __forceinline__ void tile_ilt_out(const GradShape& g, const TileBufs<T>& t, int k0, int K, T* out) {
  using C = Real<T>;
  const int S = g.S, nx = g.nx, N3p = g.N3p;
  for (int i = threadIdx.x; i < kGradRows * nx; i += kGradThreads) {
    const int m = i / nx, c = i - m * nx;
    if (k0 + m >= K) continue;
    const T* o = t.dob + m * N3p + 2 * c * S;
    T acc = T(0);
    for (int kk = 0; kk < S; ++kk) {
      T ph, wt;
      ilt_term_consts(kk, t.rc, m, ph, wt);
      acc += wt * sphere_radius(o[2 * kk + 1]) * cos_reduced(C::pi * tanh_acc(o[2 * kk]) + ph);
    }
    out[(size_t)(k0 + m) * nx + c] = acc;
  }
}

// After tile_mlp_fwd: the ILT + sphere map derivatives against gout, the MLP backward into the partial P, and the gradient
// of [obs_n | p_action] into dxt.  Rows k0 .. k0 + R - 1 of gout [K][nx]; rows past K get zero output gradients.  Ends on
// a barrier.
template <int H, typename T>
__device__ __forceinline__ void tile_mlp_bwd(const GradShape& g, const TileW<T>& md, const T* wt, T* P, const TileBufs<T>& t,
                                             const T* gout, int k0, int K) {
  using C = Real<T>;
  constexpr int R = kGradRows;
  const int S = g.S, nx = g.nx, Lp = g.Lp, in0p = g.in0p, N3p = g.N3p, nP = nx * S;
  const int tid = threadIdx.x;
  const T* W2 = wt + g.w_2;  // [H][H]   (out, in)
  const T* W3 = wt + g.w_3;  // [N3p][H] (paired output column, in)
  T *x1 = t.x1, *a1 = t.a1, *a2 = t.a2, *dob = t.dob, *dz2 = t.dz2, *dz1 = t.dz1, *dxt = t.dxt, *rc = t.rc;
  // ---- ILT + sphere map derivatives: Dx_c = sum_k w_k rho cos(theta + a_k), theta = pi tanh(u_t), rho = tan((pi/2) sigma(2 u_p)) ----
  for (int i = tid; i < R * (N3p / 2); i += kGradThreads) {
    const int m = i / (N3p / 2), pair = i - m * (N3p / 2);
    T* o = dob + m * N3p + 2 * pair;
    if (pair >= nP) { o[0] = T(0); o[1] = T(0); continue; }
    const int c = pair / S, kk = pair - c * S;
    const bool valid = k0 + m < K;
    const T gc = valid ? gout[(size_t)(k0 + m) * nx + c] : T(0);
    T ph, wk;
    ilt_term_consts(kk, rc, m, ph, wk);
    const T ut = o[0], up = o[1];
    // sech^2 u and sigma(2u) sigma(-2u) through e = exp(-2|u|): no cancellation in either tail (DESIGN.md 2.6)
    const T et = exp_acc(T(-2) * rm::min(rm::abs(ut), T(40)));
    const T sech2 = T(4) * et * rm::rcp((T(1) + et) * (T(1) + et));
    const T ep = exp_acc(T(-2) * rm::min(rm::abs(up), T(40)));
    const T ss = ep * rm::rcp((T(1) + ep) * (T(1) + ep));
    const T rho = sphere_radius(up);
    const T arg = C::pi * tanh_acc(ut) + ph;  // |arg| < 2 pi: cos_reduced's range
    const T cs = cos_reduced(arg), sn = cos_reduced(arg - C::half_pi);
    const T gw = gc * wk;
    o[0] = -gw * rho * sn * C::pi * sech2;
    o[1] = gw * cs * C::pi * rm::fma(rho, rho * ss, ss);  // (1 + rho^2) ss without forming rho^2
  }
  __syncthreads();
  // ---- MLP backward ----
  wgrad(P + g.p_w4, N3p, a2, H, 0, 0, dob, N3p, 0, 0, 1, H, N3p, N3p, 0);
  colsum(P + g.p_b4, dob, N3p, 0, 0, 1, N3p, N3p, 0);
  gemm_nn<kEpiDtanh>(dob, N3p, W3, H, N3p, H, dz2, H, false, (const T*)nullptr, a2);
  __syncthreads();
  wgrad(P + g.p_w2, H, a1, H, 0, 0, dz2, H, 0, 0, 1, H, H, H, 0);
  colsum(P + g.p_b2, dz2, H, 0, 0, 1, H, H, 0);
  gemm_nn<kEpiDtanh>(dz2, H, W2, H, H, H, dz1, H, false, (const T*)nullptr, a1);
  __syncthreads();
  wgrad(P + g.p_w0, H, x1, in0p, 0, 0, dz1, H, 0, 0, 1, in0p, H, H, 0);
  colsum(P + g.p_b0, dz1, H, 0, 0, 1, H, H, 0);
  for (int i = tid; i < R * Lp; i += kGradThreads) {  // gradient of [obs_n | p_action]
    const int m = i / Lp, j = i - m * Lp;
    const T* w = md.w1_full_t + (size_t)(2 * S + j) * H;
    T acc = T(0);
    for (int n = 0; n < H; ++n) acc = rm::fma(dz1[m * H + n], w[n], acc);
    dxt[m * 16 + j] = acc;
  }
  __syncthreads();
}

// From the gradient of [obs_n | p_action] in dxt: grad_obs, linear_out backward and BPTT through both GRU layers over the
// reversed window (the saved cells of tile_encoder_fwd), grad_act, and the GRU weight gradients into the partial P.
template <int H, typename T>
__device__ __forceinline__ void tile_encoder_bwd(const GradShape& g, const TileW<T>& md, const T* wt, T* P, const TileBufs<T>& t,
                                                 T* grad_obs, T* grad_act, int k0, int K) {
  constexpr int Hg = H / 2, G3 = 3 * Hg, R = kGradRows;
  const int B = g.B, nx = g.nx, gin = g.gin;
  const int tid = threadIdx.x;
  const T* W_hh0 = wt + g.w_hh0;  // [3Hg][Hg]
  const T* W_ih1 = wt + g.w_ih1;
  const T* W_hh1 = wt + g.w_hh1;
  const T* dxt = t.dxt;
  const T* h1last = tile_h(g, t, 1, B - 1);
  if (grad_obs)
    for (int i = tid; i < R * nx; i += kGradThreads) {
      const int m = i / nx, c = i - m * nx;
      if (k0 + m < K) grad_obs[(size_t)(k0 + m) * nx + c] = dxt[m * 16 + c] * md.state_inv_std[c];
    }
  // ---- linear_out backward ----
  for (int i = tid; i < 2 * Hg + 2; i += kGradThreads) {
    T acc = T(0);
    if (i < 2 * Hg) {
      const int o = i / Hg, h = i - o * Hg;
      for (int m = 0; m < R; ++m) acc = rm::fma(dxt[m * 16 + nx + o], h1last[m * Hg + h], acc);
      P[g.p_wout + i] += acc;
    } else {
      for (int m = 0; m < R; ++m) acc += dxt[m * 16 + nx + (i - 2 * Hg)];
      P[g.p_bout + i - 2 * Hg] += acc;
    }
  }
  T* dh0 = t.dhb;
  T* dh1 = t.dhb + R * Hg;
  T* dh0n = t.dhb + 2 * R * Hg;
  T* dh1n = t.dhb + 3 * R * Hg;
  for (int i = tid; i < R * Hg; i += kGradThreads) {
    const int m = i / Hg, h = i - m * Hg;
    dh1[i] = rm::fma(dxt[m * 16 + nx], md.w_out[h], dxt[m * 16 + nx + 1] * md.w_out[Hg + h]);
    dh0[i] = T(0);
  }
  __syncthreads();
  // ---- BPTT over the reversed window: step B-1 (oldest entry) first ----
  for (int st = B - 1; st >= 0; --st) {
    gru_cell_bwd(g, dh1, st > 0 ? tile_h(g, t, 1, st - 1) : nullptr, tile_gate(g, t, 1, st), dh1n);
    __syncthreads();
    const T* G1 = tile_gate(g, t, 1, st);
    if (st > 0) {  // dh1_prev += [dr | dz] W_hh1[r,z] + dghn W_hh1[n]
      gemm_nn<kEpiNone>(G1, 4 * Hg, W_hh1, Hg, 2 * Hg, Hg, dh1n, Hg, true);
      gemm_nn<kEpiNone>(G1 + 3 * Hg, 4 * Hg, W_hh1 + 2 * Hg * Hg, Hg, Hg, Hg, dh1n, Hg, true);
    }
    gemm_nn<kEpiNone>(G1, 4 * Hg, W_ih1, Hg, G3, Hg, dh0, Hg, true);  // layer 1's input is layer 0's output
    __syncthreads();
    gru_cell_bwd(g, dh0, st > 0 ? tile_h(g, t, 0, st - 1) : nullptr, tile_gate(g, t, 0, st), dh0n);
    __syncthreads();
    const T* G0 = tile_gate(g, t, 0, st);
    if (st > 0) {
      gemm_nn<kEpiNone>(G0, 4 * Hg, W_hh0, Hg, 2 * Hg, Hg, dh0n, Hg, true);
      gemm_nn<kEpiNone>(G0 + 3 * Hg, 4 * Hg, W_hh0 + 2 * Hg * Hg, Hg, Hg, Hg, dh0n, Hg, true);
    }
    if (grad_act)
      for (int i = tid; i < R * gin; i += kGradThreads) {  // W_ih0^T dg_i, times the input scale
        const int m = i / gin, u = i - m * gin;
        T acc = T(0);
        for (int q = 0; q < G3; ++q) acc = rm::fma(G0[m * 4 * Hg + q], md.w_ih0[q * gin + u], acc);
        if (k0 + m < K) grad_act[((size_t)(k0 + m) * B + (B - 1 - st)) * gin + u] = acc * md.act_inv_std[u];
      }
    __syncthreads();
    T* t0 = dh0; dh0 = dh0n; dh0n = t0;
    T* t1 = dh1; dh1 = dh1n; dh1n = t1;
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
    T acc = T(0);
    for (int st = 0; st < B; ++st)
      for (int m = 0; m < R; ++m) acc = rm::fma(tile_gate(g, t, 0, st)[m * 4 * Hg + q], t.xs[(st * R + m) * 4 + u], acc);
    P[g.p_wih0 + i] += acc;
  }
}

template <int H>
__global__ void __launch_bounds__(kGradThreads, 1) model_grad_tile_kernel(GradArgs<float> a) {
  const GradShape& g = a.g;
  const TileW<float>& md = a.m;
  constexpr int R = kGradRows;
  const int S = g.S, nx = g.nx, in0p = g.in0p;
  const int tid = threadIdx.x;
  float* P = a.part + (size_t)blockIdx.x * g.p_total;
  const TileBufs<float> t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);

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
    tile_linear_out(g, md, t);
    __syncthreads();
    tile_mlp_fwd<H>(g, md, t, a.row_b1, k0, a.K);
    tile_mlp_bwd<H>(g, md, a.wt, P, t, a.gout, k0, a.K);
    tile_encoder_bwd<H>(g, md, a.wt, P, t, a.grad_obs, a.grad_act, k0, a.K);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// Several prediction times per sample (nlc_model_backward_multi, and the fp64 backward for every n_t): the K n_t rows
// (sample k, time j) = row k n_t + j share sample k's encoder output, so the backward runs in two stages instead of the
// fused tile kernel:
//   MLP/ILT stage over the rows, chunk by chunk (model_grad_multi_mlp_kernel), then a fixed-order sum of each sample's
//   per-row gradient of [obs_n | p_action] over j (model_grad_multi_rowsum_kernel), then one encoder stage over the K
//   samples (model_grad_multi_enc_kernel).  Both stages accumulate into the same per-CTA partials as the tile kernel.
// ------------------------------------------------------------------------------------------------------------------
template <typename T>
struct MultiArgs {
  TileW<T> m;
  GradShape g;
  const T* obs;      // [K][nx]
  const T* p;        // [K][2] encoder output
  const T* gout;     // [rows][nx]   this chunk's rows of grad_out (the fp64 forward: its output rows)
  const T* row_b1;   // [rows][H]
  const T* row_tn;   // [rows]
  const T* row_sph;  // [rows][2S]
  const T* wt;
  T* part;
  T* scratch;
  T* drow;           // [rows][Lp] gradient of [obs_n | p_action] per row
  long long r0;      // global index of the chunk's first row
  int rows, n_t;
};

template <int H, typename T>
__global__ void __launch_bounds__(kGradThreads, 1) model_grad_multi_mlp_kernel(MultiArgs<T> a) {
  const GradShape& g = a.g;
  const TileW<T>& md = a.m;
  constexpr int R = kGradRows;
  const int Lp = g.Lp;
  const int tid = threadIdx.x;
  T* P = a.part + (size_t)blockIdx.x * g.p_total;
  const TileBufs<T> t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);
  const int n_tiles = (a.rows + R - 1) / R;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int k0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch are done
    tile_rows_input(g, md, a.row_sph, a.obs, a.p, a.r0, a.rows, a.n_t, k0, t.x1);
    tile_fourier_consts(a.row_tn, k0, a.rows, t.rc);
    __syncthreads();
    tile_mlp_fwd<H>(g, md, t, a.row_b1, k0, a.rows);
    tile_mlp_bwd<H>(g, md, a.wt, P, t, a.gout, k0, a.rows);
    for (int i = tid; i < R * Lp; i += kGradThreads) {
      const int m = i / Lp, j = i - m * Lp;
      if (k0 + m < a.rows) a.drow[(size_t)(k0 + m) * Lp + j] = t.dxt[m * 16 + j];
    }
  }
}

// dsum[k] (+)= sum of drow over sample k's rows in this chunk, j ascending; a sample's first row starts its sum, so the
// chunks in order give every sample the same sequential sum over j = 0 .. n_t - 1 whatever the chunk boundaries.
template <typename T>
__global__ void __launch_bounds__(256) model_grad_multi_rowsum_kernel(const T* __restrict__ drow, long long r0, int rows, int n_t,
                                                                      int Lp, T* __restrict__ dsum) {
  const long long k_first = r0 / n_t, k_last = (r0 + rows - 1) / n_t;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (k_last - k_first + 1) * Lp) return;
  const long long k = k_first + i / Lp;
  const int c = (int)(i % Lp);
  const long long j0 = k * n_t > r0 ? k * n_t : r0, j1 = (k + 1) * n_t < r0 + rows ? (k + 1) * n_t : r0 + rows;
  T acc = j0 == k * n_t ? T(0) : dsum[k * Lp + c];
  for (long long r = j0; r < j1; ++r) acc += drow[(r - r0) * Lp + c];
  dsum[k * Lp + c] = acc;
}

// Encoder stage: tiles of kGradRows samples, the summed gradient of [obs_n | p_action] of each sample from dsum [K][Lp].
template <int H, typename T>
__global__ void __launch_bounds__(kGradThreads, 1) model_grad_multi_enc_kernel(GradArgs<T> a, const T* __restrict__ dsum) {
  const GradShape& g = a.g;
  const TileW<T>& md = a.m;
  constexpr int R = kGradRows;
  const int Lp = g.Lp;
  const int tid = threadIdx.x;
  T* P = a.part + (size_t)blockIdx.x * g.p_total;
  const TileBufs<T> t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);
  for (int tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const int k0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch are done
    tile_load_window(g, md, a.act, k0, a.K, t.xs);
    for (int i = tid; i < R * Lp; i += kGradThreads) {  // rows past K repeat sample K - 1 in the window: zero gradient
      const int m = i / Lp, j = i - m * Lp;
      t.dxt[m * 16 + j] = k0 + m < a.K ? dsum[(size_t)(k0 + m) * Lp + j] : T(0);
    }
    __syncthreads();
    tile_encoder_fwd<H>(g, md, t);
    tile_encoder_bwd<H>(g, md, a.wt, P, t, a.grad_obs, a.grad_act, k0, a.K);
  }
}

// ------------------------------------------------------------------------------------------------------------------
// fp64 forward: the recompute half of the tile steps.  f64_encode_kernel (below, shared with the fp64 planner) encodes the
// K windows into linear_out's p [K][2]; model_f64_rows_kernel runs the MLP and the ILT sum over a chunk's rows.
// ------------------------------------------------------------------------------------------------------------------
// a.gout is unused; out: this chunk's rows [rows][nx]
template <int H>
__global__ void __launch_bounds__(kGradThreads, 1) model_f64_rows_kernel(MultiArgs<double> a, double* __restrict__ out) {
  const GradShape& g = a.g;
  const TileW<double>& md = a.m;
  constexpr int R = kGradRows;
  const TileBufs<double> t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);
  const int n_tiles = (a.rows + R - 1) / R;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int k0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch are done
    tile_rows_input(g, md, a.row_sph, a.obs, a.p, a.r0, a.rows, a.n_t, k0, t.x1);
    tile_fourier_consts(a.row_tn, k0, a.rows, t.rc);
    __syncthreads();
    tile_mlp_fwd<H>(g, md, t, a.row_b1, k0, a.rows);
    tile_ilt_out(g, t, k0, a.rows, out);
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

// fp64: the weight image of one call from the caller's parameters prm (state_dict layout, GradShape o_* offsets) - the
// row-major copies of model_grad_wt_kernel at w_*, and every weight in ModelDev's layout at f_* (TileW): the mirror
// image of nlc_model_create's packing, without the fp32 rounding.
__global__ void __launch_bounds__(256) model_f64_weights_kernel(GradShape g, const double* __restrict__ prm, double* __restrict__ img) {
  const int Hg = g.Hg, G3 = g.G3, H = g.H, S = g.S, nx = g.nx, gin = g.gin, in0 = g.in0, N3 = g.N3, N3p = g.N3p;
  const int i0 = blockIdx.x * blockDim.x + threadIdx.x, step = gridDim.x * blockDim.x;
  // paired column col = 2 (c S + k) + part of the last layer <- state_dict row (part nx + c) S + k; -1: padding
  auto w4_row = [&](int col) { return col < N3 ? ((col & 1) * nx + (col >> 1) / S) * S + (col >> 1) % S : -1; };
  for (int i = i0; i < G3 * Hg; i += step) {  // [gate row q][unit k]: state_dict; _t [k][q]
    const int q = i / Hg, k = i - q * Hg;
    img[g.w_hh0 + i] = prm[g.o_whh0 + i]; img[g.w_ih1 + i] = prm[g.o_wih1 + i]; img[g.w_hh1 + i] = prm[g.o_whh1 + i];
    img[g.f_hh0t + k * G3 + q] = prm[g.o_whh0 + i]; img[g.f_ih1t + k * G3 + q] = prm[g.o_wih1 + i];
    img[g.f_hh1t + k * G3 + q] = prm[g.o_whh1 + i];
  }
  for (int i = i0; i < H * H; i += step) {  // W2 [out n][in k]
    const int n = i / H, k = i - n * H;
    img[g.w_2 + i] = prm[g.o_w2 + i];
    img[g.f_w2t + k * H + n] = prm[g.o_w2 + i];
  }
  for (int i = i0; i < N3p * H; i += step) {  // W3 paired: [col][h] and [h][col]
    const int col = i / H, h = i - col * H, src = w4_row(col);
    const double v = src >= 0 ? prm[g.o_w4 + (size_t)src * H + h] : 0.0;
    img[g.w_3 + i] = v;
    img[g.f_w3t + (size_t)h * N3p + col] = v;
  }
  for (int i = i0; i < in0 * H; i += step) {  // W1 [n][in] -> [in][n]
    const int n = i / in0, j = i - n * in0;
    img[g.f_w1t + (size_t)j * H + n] = prm[g.o_w0 + i];
  }
  for (int i = i0; i < N3p; i += step) {
    const int src = w4_row(i);
    img[g.f_b3 + i] = src >= 0 ? prm[g.o_b4 + src] : 0.0;
  }
  for (int i = i0; i < G3 * gin; i += step) img[g.f_wih0 + i] = prm[g.o_wih0 + i];
  for (int i = i0; i < G3; i += step) {
    img[g.f_bih0 + i] = prm[g.o_bih0 + i]; img[g.f_bhh0 + i] = prm[g.o_bhh0 + i];
    img[g.f_bih1 + i] = prm[g.o_bih1 + i]; img[g.f_bhh1 + i] = prm[g.o_bhh1 + i];
  }
  for (int i = i0; i < 2 * Hg + 2; i += step) {
    if (i < 2 * Hg) img[g.f_wout + i] = prm[g.o_wout + i];
    else img[g.f_bout + i - 2 * Hg] = prm[g.o_bout + i - 2 * Hg];
  }
  for (int i = i0; i < H; i += step) { img[g.f_b1 + i] = prm[g.o_b0 + i]; img[g.f_b2 + i] = prm[g.o_b2 + i]; }
}

// Sum of the per-CTA partials in CTA order, written in the state_dict layout (named_parameters() order).
template <typename T>
__global__ void __launch_bounds__(256) model_grad_reduce_kernel(GradShape g, const T* __restrict__ part, int n_part, T* out) {
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
    T acc = T(0);
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
// workspace (elements of the scalar type): p [K][2] | dsum [K][Lp] | row_b1 [C][H] | row_tn [C] | row_sph [C][2S] |
// drow [C][Lp] | weight copies | partials [G] | scratch [G], C = min(K n_t, kMultiChunkRows), G = max(grid of C rows, grid of
// K samples).  fp64: the weight copies are followed by the forward layouts (f_total), and the forward (bwd = false) has no
// dsum, drow or partials.
struct MultiWs { size_t p, dsum, b1, tn, sph, drow, wt, part, scr, total; int C, Gm, Ge, G; };
static MultiWs multi_ws_layout(const GradShape& g, int K, int n_t, bool f64 = false, bool bwd = true) {
  MultiWs w;
  const long long rows = (long long)K * n_t;
  w.C = rows < kMultiChunkRows ? (int)rows : kMultiChunkRows;
  w.Gm = grad_grid(w.C); w.Ge = grad_grid(K); w.G = w.Gm > w.Ge ? w.Gm : w.Ge;
  size_t o = 0;
  w.p = o; o += up64((size_t)K * 2);
  w.dsum = o; o += bwd ? up64((size_t)K * g.Lp) : 0;
  w.b1 = o; o += up64((size_t)w.C * g.H);
  w.tn = o; o += up64(w.C);
  w.sph = o; o += up64((size_t)w.C * 2 * g.S);
  w.drow = o; o += bwd ? up64((size_t)w.C * g.Lp) : 0;
  w.wt = o; o += f64 ? g.f_total : g.w_total;
  w.part = o; o += bwd ? (size_t)w.G * g.p_total : 0;
  w.scr = o; o += (size_t)w.G * g.s_total;
  w.total = o;
  return w;
}

// The argument checks of the (K, n_t) entry points, fn naming the entry point in the messages.
static int multi_check(const char* fn, nlc_model_t m, int K, int n_t, int B, const void* workspace_dev) {
  NLC_REQUIRE(K >= 1 && n_t >= 1, NLC_ERR_ARG, "%s: K and n_t must be positive", fn);
  NLC_REQUIRE((long long)K * n_t < (1LL << 31), NLC_ERR_SHAPE, "%s: K n_t = %lld rows, 2^31 or more", fn, (long long)K * n_t);
  NLC_REQUIRE(B >= 1 && B <= 8, NLC_ERR_SHAPE, "%s: window length %d outside [1,8]", fn, B);
  NLC_REQUIRE(((uintptr_t)workspace_dev & 15) == 0, NLC_ERR_ARG, "%s: workspace must be 16-byte aligned", fn);
  return check_device_arch(m->device);
}

// Bytes of multi_ws_layout, or the error code of arguments the entry point would reject.
static int64_t multi_ws_bytes(nlc_model_t m, int K, int n_t, int B, bool f64, bool bwd) {
  if (!m || K < 1 || n_t < 1 || B < 1 || B > 8) return NLC_ERR_ARG;
  if ((long long)K * n_t >= (1LL << 31)) return NLC_ERR_SHAPE;
  return (int64_t)(multi_ws_layout(shape_of(m, B), K, n_t, f64, bwd).total * (f64 ? sizeof(double) : sizeof(float)));
}

// fp64: the weight image img (GradShape w_* and f_* offsets) of the caller's parameters params_dev.
static int f64_weight_image(const GradShape& g, const double* params_dev, double* img, cudaStream_t s) {
  const int n_img = g.N3p * g.H > g.in0 * g.H ? g.N3p * g.H : g.in0 * g.H;
  model_f64_weights_kernel<<<(n_img + 255) / 256, 256, 0, s>>>(g, params_dev, img);
  NLC_LAUNCH_OK("model_f64_weights_kernel");
  return NLC_OK;
}

// with the fp64 planner's stages at the end of this file
int encode_windows_f64(nlc_model_t m, int B, const double* img, const double* hist, int hist_ch, int K, int T, double* p_out,
                       double* scratch, cudaStream_t s);

// The two stages of the backward and the reduction, once the workspace holds p [K][2] at w.p and the weight copies at w.wt
// (tw: the weights the tile steps read).
template <typename T>
static int backward_two_stage(nlc_model_t m, const GradShape& g, const MultiWs& w, const TileW<T>& tw, T* ws, const T* obs_dev,
                              const T* act_dev, const T* ts_dev, int K, int n_t, const T* grad_out_dev, T* grad_params_dev,
                              T* grad_obs_dev, T* grad_act_dev, cudaStream_t s) {
  NLC_CUDA_OK(cudaMemsetAsync(ws + w.part, 0, (size_t)w.G * g.p_total * sizeof(T), s));
  MultiArgs<T> ma = {};
  ma.m = tw; ma.g = g; ma.obs = obs_dev; ma.p = ws + w.p; ma.row_b1 = ws + w.b1; ma.row_tn = ws + w.tn; ma.row_sph = ws + w.sph;
  ma.wt = ws + w.wt; ma.part = ws + w.part; ma.scratch = ws + w.scr; ma.drow = ws + w.drow; ma.n_t = n_t;
  const long long n_rows = (long long)K * n_t;
  for (long long r0 = 0; r0 < n_rows; r0 += w.C) {
    const int rows = (int)(n_rows - r0 < w.C ? n_rows - r0 : w.C);
    const int rc = launch_forward_ts_prep(m, tw.b1_raw, tw.w1_full_t, ts_dev + r0, rows, ws + w.b1, ws + w.tn, ws + w.sph, s);
    if (rc != NLC_OK) return rc;
    ma.gout = grad_out_dev + r0 * g.nx; ma.r0 = r0; ma.rows = rows;
    if (m->Hm == 128) model_grad_multi_mlp_kernel<128, T><<<w.Gm, kGradThreads, 0, s>>>(ma);
    else model_grad_multi_mlp_kernel<64, T><<<w.Gm, kGradThreads, 0, s>>>(ma);
    NLC_LAUNCH_OK("model_grad_multi_mlp_kernel");
    const long long n_sum = ((r0 + rows - 1) / n_t - r0 / n_t + 1) * g.Lp;
    model_grad_multi_rowsum_kernel<T><<<(unsigned)((n_sum + 255) / 256), 256, 0, s>>>(ws + w.drow, r0, rows, n_t, g.Lp, ws + w.dsum);
    NLC_LAUNCH_OK("model_grad_multi_rowsum_kernel");
  }
  GradArgs<T> a = {};
  a.m = tw; a.g = g; a.obs = obs_dev; a.act = act_dev; a.wt = ws + w.wt; a.part = ws + w.part; a.scratch = ws + w.scr;
  a.grad_obs = grad_obs_dev; a.grad_act = grad_act_dev; a.K = K; a.n_tiles = (K + kGradRows - 1) / kGradRows;
  if (m->Hm == 128) model_grad_multi_enc_kernel<128, T><<<w.Ge, kGradThreads, 0, s>>>(a, ws + w.dsum);
  else model_grad_multi_enc_kernel<64, T><<<w.Ge, kGradThreads, 0, s>>>(a, ws + w.dsum);
  NLC_LAUNCH_OK("model_grad_multi_enc_kernel");
  model_grad_reduce_kernel<T><<<(g.o_total + 255) / 256, 256, 0, s>>>(g, ws + w.part, w.G, grad_params_dev);
  NLC_LAUNCH_OK("model_grad_reduce_kernel");
  return NLC_OK;
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
  rc = launch_forward_ts_prep(m, m->d.b1_raw, m->d.w1_full_t, ts_dev, K, ws + w.b1, ws + w.tn, ws + w.sph, s);
  if (rc != NLC_OK) return rc;
  const int n_wt = 3 * g.G3 * g.Hg + g.H * g.H + g.N3p * g.H;
  model_grad_wt_kernel<<<(n_wt + 255) / 256, 256, 0, s>>>(m->d, g, ws + w.wt);
  NLC_LAUNCH_OK("model_grad_wt_kernel");
  GradArgs<float> a;
  a.m = tile_w(m->d); a.g = g; a.obs = obs_dev; a.act = act_dev; a.gout = grad_out_dev;
  a.row_b1 = ws + w.b1; a.row_tn = ws + w.tn; a.row_sph = ws + w.sph; a.wt = ws + w.wt;
  a.part = ws + w.part; a.scratch = ws + w.scr; a.grad_obs = grad_obs_dev; a.grad_act = grad_act_dev;
  a.K = K; a.n_tiles = (K + kGradRows - 1) / kGradRows;
  const int G = grad_grid(K);
  if (m->Hm == 128) model_grad_tile_kernel<128><<<G, kGradThreads, 0, s>>>(a);
  else model_grad_tile_kernel<64><<<G, kGradThreads, 0, s>>>(a);
  NLC_LAUNCH_OK("model_grad_tile_kernel");
  model_grad_reduce_kernel<float><<<(g.o_total + 255) / 256, 256, 0, s>>>(g, ws + w.part, G, grad_params_dev);
  NLC_LAUNCH_OK("model_grad_reduce_kernel");
  return NLC_OK;
}

extern "C" int64_t nlc_model_backward_multi_workspace_bytes(nlc_model_t m, int K, int n_t, int B) {
  return multi_ws_bytes(m, K, n_t, B, false, true);
}

extern "C" int nlc_model_backward_multi(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K, int n_t,
                                        int B, const float* grad_out_dev, float* grad_params_dev, float* grad_obs_dev,
                                        float* grad_act_dev, void* workspace_dev, void* stream) {
  NLC_REQUIRE(m && obs_dev && act_dev && ts_dev && grad_out_dev && grad_params_dev && workspace_dev, NLC_ERR_ARG,
              "nlc_model_backward_multi: null pointer");
  int rc = multi_check("nlc_model_backward_multi", m, K, n_t, B, workspace_dev);
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
  return backward_two_stage(m, g, w, tile_w(m->d), ws, obs_dev, act_dev, ts_dev, K, n_t, grad_out_dev, grad_params_dev, grad_obs_dev,
                            grad_act_dev, s);
}

// ---------------------------------------------------------------------------------------------------------------------
// fp64 forward and backward (NeuralLaplaceModel math_mode="fp64"): the weights are the caller's fp64 parameters params_dev
// (nlc_model_grad_floats entries, the layout of grad_params_dev), rearranged per call into the workspace.  The K windows
// are encoded by the fp64 planner's encoder at T = 1 (a window per sample, hist = act).
// ---------------------------------------------------------------------------------------------------------------------
extern "C" int64_t nlc_model_forward_f64_workspace_bytes(nlc_model_t m, int K, int n_t, int B) {
  return multi_ws_bytes(m, K, n_t, B, true, false);
}

extern "C" int nlc_model_forward_f64(nlc_model_t m, const double* params_dev, const double* obs_dev, const double* act_dev,
                                     const double* ts_dev, int K, int n_t, int B, double* out_dev, double* p_action_dev,
                                     void* workspace_dev, void* stream) {
  NLC_REQUIRE(m && params_dev && obs_dev && act_dev && ts_dev && out_dev && workspace_dev, NLC_ERR_ARG,
              "nlc_model_forward_f64: null pointer");
  int rc = multi_check("nlc_model_forward_f64", m, K, n_t, B, workspace_dev);
  if (rc != NLC_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const GradShape g = shape_of(m, B);
  const MultiWs w = multi_ws_layout(g, K, n_t, true, false);
  double* ws = static_cast<double*>(workspace_dev);
  double* p = p_action_dev ? p_action_dev : ws + w.p;
  rc = f64_weight_image(g, params_dev, ws + w.wt, s);
  if (rc != NLC_OK) return rc;
  rc = encode_windows_f64(m, B, ws + w.wt, act_dev, g.gin, K, 1, p, ws + w.scr, s);
  if (rc != NLC_OK) return rc;
  MultiArgs<double> ma = {};
  ma.m = tile_w_f64(m->d, g, ws + w.wt); ma.g = g; ma.obs = obs_dev; ma.p = p; ma.row_b1 = ws + w.b1; ma.row_tn = ws + w.tn;
  ma.row_sph = ws + w.sph; ma.wt = ws + w.wt; ma.scratch = ws + w.scr; ma.n_t = n_t;
  const long long n_rows = (long long)K * n_t;
  for (long long r0 = 0; r0 < n_rows; r0 += w.C) {
    const int rows = (int)(n_rows - r0 < w.C ? n_rows - r0 : w.C);
    rc = launch_forward_ts_prep(m, ma.m.b1_raw, ma.m.w1_full_t, ts_dev + r0, rows, ws + w.b1, ws + w.tn, ws + w.sph, s);
    if (rc != NLC_OK) return rc;
    ma.r0 = r0; ma.rows = rows;
    const int G = grad_grid(rows);
    if (m->Hm == 128) model_f64_rows_kernel<128><<<G, kGradThreads, 0, s>>>(ma, out_dev + r0 * g.nx);
    else model_f64_rows_kernel<64><<<G, kGradThreads, 0, s>>>(ma, out_dev + r0 * g.nx);
    NLC_LAUNCH_OK("model_f64_rows_kernel");
  }
  return NLC_OK;
}

extern "C" int64_t nlc_model_backward_f64_workspace_bytes(nlc_model_t m, int K, int n_t, int B) {
  return multi_ws_bytes(m, K, n_t, B, true, true);
}

extern "C" int nlc_model_backward_f64(nlc_model_t m, const double* params_dev, const double* obs_dev, const double* act_dev,
                                      const double* ts_dev, int K, int n_t, int B, const double* grad_out_dev,
                                      double* grad_params_dev, double* grad_obs_dev, double* grad_act_dev, void* workspace_dev,
                                      void* stream) {
  NLC_REQUIRE(m && params_dev && obs_dev && act_dev && ts_dev && grad_out_dev && grad_params_dev && workspace_dev, NLC_ERR_ARG,
              "nlc_model_backward_f64: null pointer");
  int rc = multi_check("nlc_model_backward_f64", m, K, n_t, B, workspace_dev);
  if (rc != NLC_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const GradShape g = shape_of(m, B);
  const MultiWs w = multi_ws_layout(g, K, n_t, true, true);
  double* ws = static_cast<double*>(workspace_dev);
  rc = f64_weight_image(g, params_dev, ws + w.wt, s);
  if (rc != NLC_OK) return rc;
  rc = encode_windows_f64(m, B, ws + w.wt, act_dev, g.gin, K, 1, ws + w.p, ws + w.scr, s);
  if (rc != NLC_OK) return rc;
  return backward_two_stage(m, g, w, tile_w_f64(m->d, g, ws + w.wt), ws, obs_dev, act_dev, ts_dev, K, n_t, grad_out_dev,
                            grad_params_dev, grad_obs_dev, grad_act_dev, s);
}

// ---------------------------------------------------------------------------------------------------------------------
// The fp64 planner's model stages (nlc_planner_f64_*, planner_f64.cu): the tile steps above over a control step's K T
// history windows (f64_encode_kernel, which also encodes the fp64 model's windows) and its K rollouts
// (plan_f64_rollout_kernel).  The weights are the image
// model_f64_weights_kernel builds from the caller's parameters, the s-point columns of the first layer are folded at the
// planner's dt by forward_ts_prep_kernel<double> - the arithmetic of nlc_model_forward_f64 at a uniform time, so a step of
// the rollout equals that forward bit for bit.
// ---------------------------------------------------------------------------------------------------------------------
namespace nlc {

struct PlanF64Args {
  TileW<double> m;
  GradShape g;
  const double* hist;       // [K][L][hist_ch] env units, L = B - 1 + T
  int hist_ch;              // channels stored per entry: an encode_obs_time model's time channel is synthesised
  const double* p;          // [K][T][2] encoder outputs
  const double* state0;     // [nx] (sps = 0) or [K][nx] (sps = 1)
  int sps;
  const double* row_b1;     // [H] first-layer bias with the s-point columns folded at dt
  const double* row_tn;     // [1] the (normalised) prediction time
  const double* pert_cost;  // [K]
  int env, state_constraint;
  double goal_x;
  double* p_out;            // [K][T][2]
  double* cost;             // [K]
  double* states;           // [K][T][nx] or null
  double* scratch;          // [grid][s_total]
  int K, T;
};

// Window w = k T + t is hist[k][t : t + B] (mppi_delay.py:261-288), read in the order of tile_load_window.  With T = 1,
// hist = act and hist_ch = gin these are the model's windows act [K][B][gin], read as tile_load_window reads them.
template <int H>
__global__ void __launch_bounds__(kGradThreads, 1) f64_encode_kernel(PlanF64Args a) {
  const GradShape& g = a.g;
  const TileW<double>& md = a.m;
  constexpr int R = kGradRows;
  const TileBufs<double> t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);
  const long long n_win = (long long)a.K * a.T;
  const long long n_tiles = (n_win + R - 1) / R;
  const int B = g.B, gin = g.gin, L = B - 1 + a.T;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long w0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch are done
    for (int i = threadIdx.x; i < B * R * 4; i += kGradThreads) {
      const int st = i / (R * 4), m = (i / 4) % R, u = i & 3;
      const long long w = w0 + m < n_win ? w0 + m : n_win - 1;
      const long long k = w / a.T;
      const int tt = (int)(w - k * a.T), j = B - 1 - st;
      double v = 0.0;
      if (u < gin) {
        const double x = u < a.hist_ch ? a.hist[((size_t)k * L + tt + j) * a.hist_ch + u] : (double)(B - 1 - j);
        v = (x - md.act_mean[u]) * md.act_inv_std[u];
      }
      t.xs[i] = v;
    }
    __syncthreads();
    tile_encoder_fwd<H>(g, md, t);
    tile_linear_out(g, md, t);
    __syncthreads();
    for (int i = threadIdx.x; i < R * 2; i += kGradThreads) {
      const int m = i >> 1, o = i & 1;
      if (w0 + m < n_win) a.p_out[(size_t)(w0 + m) * 2 + o] = t.x1[m * g.in0p + 2 * g.S + g.nx + o];
    }
  }
}

// A tile of kGradRows samples through the whole horizon: per step the model (tile_rows_input's first-layer input,
// tile_mlp_fwd, tile_ilt_out's sum), state += delta, and the running cost (mppi_delay.py:232-313).
template <int H>
__global__ void __launch_bounds__(kGradThreads, 1) plan_f64_rollout_kernel(PlanF64Args a) {
  using C = Real<double>;
  const GradShape& g = a.g;
  const TileW<double>& md = a.m;
  constexpr int R = kGradRows;
  const int S = g.S, nx = g.nx, nu = g.nu, Lp = g.Lp, in0p = g.in0p, N3p = g.N3p, T = a.T, B = g.B, L = B - 1 + T;
  __shared__ double st[R][kMaxNx], dl[R][kMaxNx], acc[R];
  const TileBufs<double> t = tile_bufs(g, a.scratch + (size_t)blockIdx.x * g.s_total);
  const int n_tiles = (a.K + R - 1) / R;
  for (int tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const int k0 = tile * R;
    __syncthreads();  // the previous tile's last reads of the scratch and of st / acc are done
    for (int i = threadIdx.x; i < R * nx; i += kGradThreads) {
      const int m = i / nx, c = i - m * nx, k = min(k0 + m, a.K - 1);
      st[m][c] = a.state0[(size_t)(a.sps ? k : 0) * nx + c];
    }
    for (int m = threadIdx.x; m < R; m += kGradThreads) acc[m] = 0.0;
    tile_fourier_consts(a.row_tn, 0, 1, t.rc);
    __syncthreads();
    for (int tt = 0; tt < T; ++tt) {
      for (int i = threadIdx.x; i < R * Lp; i += kGradThreads) {
        const int m = i / Lp, j = i - m * Lp;
        const size_t k = (size_t)min(k0 + m, a.K - 1);
        t.x1[m * in0p + 2 * S + j] = j < nx ? (st[m][j] - md.state_mean[j]) * md.state_inv_std[j] : a.p[(k * T + tt) * 2 + (j - nx)];
      }
      __syncthreads();
      tile_mlp_fwd<H>(g, md, t, a.row_b1, 0, 1);
      for (int i = threadIdx.x; i < R * nx; i += kGradThreads) {
        const int m = i / nx, c = i - m * nx;
        const double* o = t.dob + m * N3p + 2 * c * S;
        double d = 0.0;
        for (int kk = 0; kk < S; ++kk) {
          double ph, wt;
          ilt_term_consts(kk, t.rc, m, ph, wt);
          d += wt * sphere_radius(o[2 * kk + 1]) * cos_reduced(C::pi * tanh_acc(o[2 * kk]) + ph);
        }
        dl[m][c] = d;
      }
      __syncthreads();
      for (int m = threadIdx.x; m < R; m += kGradThreads) {
        const int k = min(k0 + m, a.K - 1);
        for (int c = 0; c < nx; ++c) st[m][c] = st[m][c] + dl[m][c];
        acc[m] = acc[m] + env_running_cost(a.env, a.state_constraint, a.goal_x, st[m], a.hist + ((size_t)k * L + tt + B - 1) * nu, nu);
        if (a.states && k0 + m < a.K)
          for (int c = 0; c < nx; ++c) a.states[((size_t)k * T + tt) * nx + c] = st[m][c];
      }
      __syncthreads();
    }
    for (int m = threadIdx.x; m < R; m += kGradThreads)
      if (k0 + m < a.K) a.cost[k0 + m] = acc[m] + a.pert_cost[k0 + m];
  }
}

static int plan_f64_grid(long long rows) { return rows >= (long long)kGradGridCap * kGradRows ? kGradGridCap : (int)((rows + kGradRows - 1) / kGradRows); }

// Doubles of the weight image (model_f64_weights_kernel's layout) and of the per-CTA tile scratch of the two kernels.
size_t plan_f64_image_doubles(nlc_model_t m) { return shape_of(m, 1).f_total; }
size_t plan_f64_scratch_doubles(nlc_model_t m, int B, int K, int T) {
  return (size_t)plan_f64_grid((long long)K * T) * shape_of(m, B).s_total;  // the encoder's grid: at least the rollout's
}

// The weight image of params_dev and the first-layer bias row_b1 [H] / time row_tn [1] at the prediction time ts_dev [1].
int plan_f64_set_params(nlc_model_t m, const double* params_dev, const double* ts_dev, double* img, double* row_b1, double* row_tn,
                        cudaStream_t s) {
  const GradShape g = shape_of(m, 1);
  const int rc = f64_weight_image(g, params_dev, img, s);
  if (rc != NLC_OK) return rc;
  const TileW<double> w = tile_w_f64(m->d, g, img);
  return launch_forward_ts_prep<double>(m, w.b1_raw, w.w1_full_t, ts_dev, 1, row_b1, row_tn, nullptr, s);
}

int encode_windows_f64(nlc_model_t m, int B, const double* img, const double* hist, int hist_ch, int K, int T, double* p_out,
                       double* scratch, cudaStream_t s) {
  PlanF64Args a = {};
  a.g = shape_of(m, B); a.m = tile_w_f64(m->d, a.g, img);
  a.hist = hist; a.hist_ch = hist_ch; a.p_out = p_out; a.scratch = scratch; a.K = K; a.T = T;
  const int G = plan_f64_grid((long long)K * T);
  if (m->Hm == 128) f64_encode_kernel<128><<<G, kGradThreads, 0, s>>>(a);
  else f64_encode_kernel<64><<<G, kGradThreads, 0, s>>>(a);
  NLC_LAUNCH_OK("f64_encode_kernel");
  return NLC_OK;
}

int plan_f64_rollout(nlc_model_t m, int B, const double* img, const double* row_b1, const double* row_tn, const double* state0, int sps,
                     const double* hist, const double* p, const double* pert_cost, int K, int T, int env, int state_constraint,
                     double goal_x, double* cost, double* states, double* scratch, cudaStream_t s) {
  PlanF64Args a = {};
  a.g = shape_of(m, B); a.m = tile_w_f64(m->d, a.g, img);
  a.hist = hist; a.p = p; a.state0 = state0; a.sps = sps; a.row_b1 = row_b1; a.row_tn = row_tn; a.pert_cost = pert_cost;
  a.env = env; a.state_constraint = state_constraint; a.goal_x = goal_x; a.cost = cost; a.states = states; a.scratch = scratch;
  a.K = K; a.T = T;
  const int G = plan_f64_grid(K);
  if (m->Hm == 128) plan_f64_rollout_kernel<128><<<G, kGradThreads, 0, s>>>(a);
  else plan_f64_rollout_kernel<64><<<G, kGradThreads, 0, s>>>(a);
  NLC_LAUNCH_OK("plan_f64_rollout_kernel");
  return NLC_OK;
}

}  // namespace nlc
