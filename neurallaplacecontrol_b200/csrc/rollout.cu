// Stages 2+3 of MPPIDelay.command for the Neural Laplace dynamics: the sequential rollout
//   state <- state + ILT(rep_mlp([s-points | (state-mean)/std | p_action]))      (w_nl.py:117-145)
//   cost  += running_cost(state, u_t)                                            (mppi_delay.py:271-296)
// in ONE launch for the whole horizon.  The encoder outputs p_action[k][t] were produced up front by
// nlc_encode_history (they do not depend on the state).
//
// fp32 CUDA-core (FFMA) form - the 1e-4 parity anchor.  One CTA owns R <= 64 samples for all T steps;
// W2^T, the pair-permuted W3^T and all folded constants stay in shared memory, activations are
// row-major [sample][128] so that the A operand is a warp-wide broadcast and W reads are 512 B rows.
// Per step: L1 (fold of the 2S constant s-columns into the bias leaves an (nx+2)->128 layer), L2
// 128->128, L3 128->2*nx*S with the sphere->complex map and the Fourier weights applied in the epilogue
// (term = w_k * tan(phi/2+pi/4) * cos(theta + k*pi*t/T)), a deterministic fixed-order sum over k, the
// residual state update and the env cost.
#include <stdlib.h>

#include "common.cuh"
#include "env_cost.cuh"

namespace nlc {

constexpr int kH = 128;
constexpr int kRT = 8;  // rows per register tile

struct RollArgs {
  ModelDev m;
  int nx, S, N3p, nu;
  nlc_rollout_opts o;
  const float* state0; int state_per_sample;
  const float* p;     // [K][T][2]
  const float* hist;  // [K][L][nu]
  const float* pert_cost;
  int K, T, B, L, R;
  float* cost_total;
  float* states;
  float* delta_out;  // forward-only mode (nlc_model_forward): write the model output, skip the cost
  // per-sample prediction times (nlc_model_forward_ts): first-layer bias with that sample's s-points folded in, and
  // the sample's normalised time; null on the planner path (one folded time for every sample)
  const float* row_b1;  // [K][128]
  const float* row_tn;  // [K]
  int termRows;  // rows of the a1/term buffer
  int w3_smem;   // 0: W3 (128 x N3p floats) does not fit shared memory next to W2 (S = 33 with nx >= 5) and is read from L2
};

template <int H>
__device__ __forceinline__ void tile_gemm_128(const float* __restrict__ act, const float* __restrict__ WT, int ldw,
                                              int row0, int col0, float acc[kRT][4]) {
#pragma unroll 2
  for (int k4 = 0; k4 < H / 4; ++k4) {
    float4 a[kRT];
#pragma unroll
    for (int i = 0; i < kRT; ++i) a[i] = *reinterpret_cast<const float4*>(act + (row0 + i) * H + 4 * k4);
#pragma unroll
    for (int kk = 0; kk < 4; ++kk) {
      const float4 w = *reinterpret_cast<const float4*>(WT + (4 * k4 + kk) * ldw + col0);
#pragma unroll
      for (int i = 0; i < kRT; ++i) {
        const float av = kk == 0 ? a[i].x : (kk == 1 ? a[i].y : (kk == 2 ? a[i].z : a[i].w));
        acc[i][0] = fmaf(av, w.x, acc[i][0]);
        acc[i][1] = fmaf(av, w.y, acc[i][1]);
        acc[i][2] = fmaf(av, w.z, acc[i][2]);
        acc[i][3] = fmaf(av, w.w, acc[i][3]);
      }
    }
  }
}

// H = hidden_units: 128 (config.py:37) or 64 (the reference class default, w_nl.py:71)
template <int H>
__global__ void __launch_bounds__(256, 1) rollout_nl_kernel(RollArgs a) {
  constexpr int kH = H;  // shadows the file-scope width of the default configuration
  extern __shared__ __align__(16) float smem[];
  const int nx = a.nx, S = a.S, N3p = a.N3p, R = a.R, Lp = nx + 2, nP = nx * S;
  float* w2 = smem;                       // [128][128]
  float* w3 = w2 + kH * kH;               // [128][N3p]
  float* a1 = w3 + (a.w3_smem ? kH * N3p : 0);  // [R][128]; reused as term[R][nP] after L2 (nP may exceed 128)
  const float* w3r = a.w3_smem ? w3 : a.m.w3_t;
  float* a2 = a1 + R * (a.termRows);      // [R][128]
  float* w1x = a2 + R * kH;               // [Lp][128]
  float* b1 = w1x + Lp * kH;              // [128]
  float* b2 = b1 + kH;                    // [128]
  float* b3 = b2 + kH;                    // [N3p]
  float* phase = b3 + N3p;                // [S]
  float* weight = phase + S;              // [S]
  float* in = weight + S;                 // [R][Lp]   normalised [obs | p_action]
  float* st = in + R * Lp;                // [R][nx]   state, env units
  float* smean = st + R * nx;             // [nx]
  float* sinv = smean + nx;               // [nx]
  float* rdelta = sinv + nx;              // [R] per-row pi/2 - pi t/T   (per-sample-time mode)
  float* rscale = rdelta + R;             // [R] per-row exp(gamma t)/T
  const int ldt = a.termRows;             // row stride of a1 / term

  const int tid = threadIdx.x;
  const int k0 = blockIdx.x * R;

  for (int i = tid; i < kH * kH / 4; i += 256) reinterpret_cast<float4*>(w2)[i] = __ldg(reinterpret_cast<const float4*>(a.m.w2_t) + i);
  if (a.w3_smem)
    for (int i = tid; i < kH * N3p / 4; i += 256) reinterpret_cast<float4*>(w3)[i] = __ldg(reinterpret_cast<const float4*>(a.m.w3_t) + i);
  for (int i = tid; i < Lp * kH; i += 256) w1x[i] = a.m.w1x_t[i];
  for (int i = tid; i < kH; i += 256) { b1[i] = a.m.b1_fold[i]; b2[i] = a.m.b2[i]; }
  for (int i = tid; i < N3p; i += 256) b3[i] = a.m.b3[i];
  for (int i = tid; i < S; i += 256) { phase[i] = a.m.ilt_phase[i]; weight[i] = a.m.ilt_weight[i]; }
  if (tid < nx) { smean[tid] = a.m.state_mean[tid]; sinv[tid] = a.m.state_inv_std[tid]; }
  __syncthreads();
  for (int i = tid; i < R * nx; i += 256) {
    const int r = i / nx, c = i - r * nx;
    const int k = min(k0 + r, a.K - 1);
    const float v = a.state0[(size_t)(a.state_per_sample ? k / a.state_per_sample : 0) * nx + c];
    st[i] = v;
    in[r * Lp + c] = (v - smean[c]) * sinv[c];
  }
  for (int i = tid; i < R * 2; i += 256) {
    const int r = i >> 1, o = i & 1;
    const int k = min(k0 + r, a.K - 1);
    in[r * Lp + nx + o] = a.p[((size_t)k * a.T) * 2 + o];
  }
  if (a.row_tn)
    for (int r = tid; r < R; r += 256) {  // torchlaplace Fourier constants of this sample's time (oracle/ilt.py)
      const float tn = a.row_tn[min(k0 + r, a.K - 1)];
      const float T = 2.0f * (tn + 1.0e-6f);
      rdelta[r] = 3.14159265358979f * 1.0e-6f / T;
      rscale[r] = expf((1.0e-3f + 4.605170185988091f / T) * tn) / T;
    }
  __syncthreads();

  float cost_acc = 0.0f;
  const int RG = R / kRT;
  for (int t = 0; t < a.T; ++t) {
    // ---- cost of the previous step's state (mppi_delay.py:288-290), by the row-owner threads ----
    if (t > 0 && tid < R && a.cost_total) {
      const int k = min(k0 + tid, a.K - 1);
      cost_acc += env_running_cost(a.o, st + tid * nx, a.hist + ((size_t)k * a.L + (t - 1) + a.B - 1) * a.nu, a.nu);
    }
    // ---- L1: a1 = tanh(b1' + W1x . in) ----
    for (int i = tid; i < R * kH; i += 256) {
      const int r = i / kH, n = i & (kH - 1);
      float acc = a.row_b1 ? a.row_b1[(size_t)min(k0 + r, a.K - 1) * kH + n] : b1[n];
      for (int j = 0; j < Lp; ++j) acc = fmaf(w1x[j * kH + n], in[r * Lp + j], acc);
      a1[r * ldt + n] = tanh_acc(acc);
    }
    __syncthreads();
    // ---- L2: a2 = tanh(b2 + a1 . W2^T) ----
    for (int it = tid; it < RG * (kH / 4); it += 256) {
      const int rg = it / (kH / 4), cg = it & (kH / 4 - 1);
      float acc[kRT][4];
#pragma unroll
      for (int i = 0; i < kRT; ++i) { acc[i][0] = b2[4 * cg]; acc[i][1] = b2[4 * cg + 1]; acc[i][2] = b2[4 * cg + 2]; acc[i][3] = b2[4 * cg + 3]; }
      // a1 rows have stride ldt
      {
        const float* act = a1;
#pragma unroll 2
        for (int k4 = 0; k4 < kH / 4; ++k4) {
          float4 av4[kRT];
#pragma unroll
          for (int i = 0; i < kRT; ++i) av4[i] = *reinterpret_cast<const float4*>(act + (rg * kRT + i) * ldt + 4 * k4);
#pragma unroll
          for (int kk = 0; kk < 4; ++kk) {
            const float4 w = *reinterpret_cast<const float4*>(w2 + (4 * k4 + kk) * kH + 4 * cg);
#pragma unroll
            for (int i = 0; i < kRT; ++i) {
              const float av = kk == 0 ? av4[i].x : (kk == 1 ? av4[i].y : (kk == 2 ? av4[i].z : av4[i].w));
              acc[i][0] = fmaf(av, w.x, acc[i][0]);
              acc[i][1] = fmaf(av, w.y, acc[i][1]);
              acc[i][2] = fmaf(av, w.z, acc[i][2]);
              acc[i][3] = fmaf(av, w.w, acc[i][3]);
            }
          }
        }
      }
#pragma unroll
      for (int i = 0; i < kRT; ++i)
        *reinterpret_cast<float4*>(a2 + (rg * kRT + i) * kH + 4 * cg) =
            make_float4(tanh_acc(acc[i][0]), tanh_acc(acc[i][1]), tanh_acc(acc[i][2]), tanh_acc(acc[i][3]));
    }
    __syncthreads();
    // ---- L3 + sphere->complex + Fourier weights: term[r][c*S+k] ----
    const int CG = N3p / 4;
    for (int it = tid; it < RG * CG; it += 256) {
      const int rg = it / CG, cg = it - rg * CG;
      float acc[kRT][4];
#pragma unroll
      for (int i = 0; i < kRT; ++i) { acc[i][0] = b3[4 * cg]; acc[i][1] = b3[4 * cg + 1]; acc[i][2] = b3[4 * cg + 2]; acc[i][3] = b3[4 * cg + 3]; }
      tile_gemm_128<H>(a2, w3r, N3p, rg * kRT, 4 * cg, acc);
      const int pair0 = 2 * cg;  // pairs pair0, pair0+1 ; pair = c*S + k
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int pair = pair0 + h;
        if (pair < nP) {
          const int kk = pair % S;
          float ph = phase[kk], wt = weight[kk];
          // k pi t/T = k (pi/2 - delta): the quarter turns are exact, reduced to (-pi, pi]
          const float quarter = (kk & 3) == 0 ? 0.0f : ((kk & 3) == 1 ? 1.57079632679489662f : ((kk & 3) == 2 ? 3.14159265358979f : -1.57079632679489662f));
#pragma unroll
          for (int i = 0; i < kRT; ++i) {
            if (a.row_tn) {
              ph = quarter - (float)kk * rdelta[rg * kRT + i];
              wt = rscale[rg * kRT + i] * (kk == 0 ? 0.5f : 1.0f);
            }
            const float theta = 3.14159265358979f * tanh_acc(acc[i][2 * h]);  // w_nl.py:59
            const float rad = sphere_radius(acc[i][2 * h + 1]);               // w_nl.py:60-62 + sphere_to_complex
            a1[(rg * kRT + i) * ldt + pair] = wt * rad * cos_reduced(theta + ph);
          }
        }
      }
    }
    __syncthreads();
    // ---- fixed-order sum over k, residual update (mppi_with_model.py:121), next step's inputs ----
    for (int i = tid; i < R * nx; i += 256) {
      const int r = i / nx, c = i - r * nx;
      const float* tp = a1 + r * ldt + c * S;
      float d = 0.0f;
      for (int kk = 0; kk < S; ++kk) d += tp[kk];
      const float v = st[i] + d;
      st[i] = v;
      in[r * Lp + c] = (v - smean[c]) * sinv[c];
      if (a.states && k0 + r < a.K) a.states[((size_t)(k0 + r) * a.T + t) * nx + c] = v;
      if (a.delta_out && k0 + r < a.K) a.delta_out[(size_t)(k0 + r) * nx + c] = d;
    }
    if (t + 1 < a.T)
      for (int i = tid; i < R * 2; i += 256) {
        const int r = i >> 1, o = i & 1;
        const int k = min(k0 + r, a.K - 1);
        in[r * Lp + nx + o] = a.p[((size_t)k * a.T + t + 1) * 2 + o];
      }
    __syncthreads();
  }
  if (a.cost_total && tid < R && k0 + tid < a.K) {
    const int k = k0 + tid;
    cost_acc += env_running_cost(a.o, st + tid * nx, a.hist + ((size_t)k * a.L + (a.T - 1) + a.B - 1) * a.nu, a.nu);
    a.cost_total[k] = cost_acc + (a.pert_cost ? a.pert_cost[k] : 0.0f);
  }
}

static size_t rollout_smem_floats(int kH, int nx, int S, int N3p, int R, int termRows, bool w3_smem = true) {
  const int Lp = nx + 2;
  return (size_t)kH * kH + (w3_smem ? (size_t)kH * N3p : 0) + (size_t)R * termRows + (size_t)R * kH + (size_t)Lp * kH + 2 * kH + N3p +
         2 * S + (size_t)R * Lp + (size_t)R * nx + 2 * nx + 2 * (size_t)R + 8;
}

int launch_rollout_fp32(nlc_model_s* m, const nlc_rollout_opts* o, const float* state, int sps, const float* p,
                        const float* hist, const float* pert_cost, int K, int T, int B, int nu, float* cost,
                        float* states, float* delta_out, cudaStream_t stream, const float* row_b1 = nullptr,
                        const float* row_tn = nullptr) {
  RollArgs a;
  a.delta_out = delta_out; a.row_b1 = row_b1; a.row_tn = row_tn;
  a.m = m->d; a.nx = m->nx; a.S = m->S; a.N3p = m->N3p; a.nu = nu; a.o = *o;
  a.state0 = state; a.state_per_sample = sps; a.p = p; a.hist = hist; a.pert_cost = pert_cost;
  a.K = K; a.T = T; a.B = B; a.L = B - 1 + T; a.cost_total = cost; a.states = states;
  const int nP = m->nx * m->S;
  a.termRows = ((nP > m->Hm ? nP : m->Hm) + 3) / 4 * 4;
  const size_t max_bytes = 227 * 1024;
  int R = 64;
  // W3 stays in shared memory when at least 16 rows fit beside it; else (S = 33 with nx >= 5) it is read through L2
  bool w3s = rollout_smem_floats(m->Hm, m->nx, m->S, m->N3p, 16, a.termRows, true) * sizeof(float) <= max_bytes;
  a.w3_smem = w3s ? 1 : 0;
  while (R > 8 && rollout_smem_floats(m->Hm, m->nx, m->S, m->N3p, R, a.termRows, w3s) * sizeof(float) > max_bytes) R -= 8;
  NLC_REQUIRE(rollout_smem_floats(m->Hm, m->nx, m->S, m->N3p, R, a.termRows, w3s) * sizeof(float) <= max_bytes, NLC_ERR_SHAPE,
              "rollout: model (nx=%d, S=%d) does not fit shared memory", m->nx, m->S);
  // spread small K over the SMs: the horizon is sequential, so latency is set by the rows one CTA owns
  int want = (K + 147) / 148;
  want = (want + 7) / 8 * 8;
  if (want < R) R = want;
  a.R = R;
  const size_t smem = rollout_smem_floats(m->Hm, m->nx, m->S, m->N3p, R, a.termRows, w3s) * sizeof(float);
  auto kern = m->Hm == 128 ? rollout_nl_kernel<128> : rollout_nl_kernel<64>;
  NLC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)max_bytes));
  const int grid = (K + R - 1) / R;
  kern<<<grid, 256, smem, stream>>>(a);
  NLC_LAUNCH_OK("rollout_nl_kernel");
  return NLC_OK;
}

int encode_history_impl(nlc_model_t m, const float* hist_dev, int hist_ch, int K, int T, int B, float* p_dev, int math_mode,
                        cudaStream_t s);
int launch_rollout_tc2(nlc_model_s* m, const nlc_rollout_opts* o, const float* state, int sps, const float* p,
                       const float* hist, const float* pert_cost, int K, int T, int B, int nu, float* cost, float* states,
                       float* delta_out, int split3, int tiles_per_cta, cudaStream_t stream, const unsigned int* ready = nullptr,
                       unsigned int ready_target = 0, unsigned int* status = nullptr, const float* row_b1 = nullptr,
                       const float* row_tn = nullptr);
bool rollout_has_tensor_core_form(const nlc_model_s* m);

// NLC_ROLLOUT_TILES=1 or 3 forces the tensor-core rollout's form (1: one tile per CTA, 3: ping-pong) - the parity tests run
// both; anything else leaves the choice to the plan size.  Read at every call.  A forced form also keeps the planner's plain
// sequence (no rollout beside the encoder).
static int forced_rollout_form() {
  const char* f = getenv("NLC_ROLLOUT_TILES");
  return (f && (f[0] == '1' || f[0] == '3')) ? f[0] - '0' : 0;
}

// planner.cu: can the rollout of this plan run BESIDE its history encoder (the one-tile tcgen05 form on ceil(K/128) SMs or the
// ping-pong form on fewer, polling the encoder's per-step readiness counters)?
bool rollout_can_overlap(const nlc_model_s* m, int K, int T, int math_mode) {
  static const bool off = [] { const char* e = getenv("NLC_NO_OVERLAP"); return e && e[0] == '1'; }();
  // up to 74 tiles the encoder keeps at least half the SMs for the whole step; beyond, the planner runs the first part of the
  // encoder alone and the rest beside the rollout (planner.cu) - worth it while the rollout leaves the encoder >= 8 SMs.
  // Ping-pong plans of two passes per CTA (up to 560 tiles; config 4 on one GPU: 512 tiles = 128 CTAs x 2 passes, 20 SMs to
  // spare) encode the first pass's samples before the fork and only the last steps of the last pass's samples beside the
  // rollout: the last pass starts ~T steps after the fork, which leaves the encoder time for those steps.
  // The schedule and its constants were measured at hidden_units = 128; hidden-64 plans run the encoder, then the rollout.
  const int n_tiles = (K + 127) / 128;
  const bool pp_form = 2 * m->nx * m->S <= 256;  // shapes with a ping-pong instantiation (rollout_tc2.cu launch_one)
  return !off && !forced_rollout_form() && math_mode != NLC_MATH_FP32 && m->Hm == 128 && rollout_has_tensor_core_form(m) && T >= 2 &&
         (pp_form ? (n_tiles <= 140 || (pp_overlap_iters(n_tiles) <= 2 && pp_overlap_grid(n_tiles) <= 140)) : n_tiles <= 140);
}
// The overlapped rollout's form: one tile per CTA on n_tiles SMs (9.5 us per step), or - from 89 tiles - the ping-pong form on
// n_tiles / 2 SMs (13.3 us per step of a tile pair), which leaves the encoder 148 - n_tiles / 2 SMs for the whole rollout.
// Model (12.6 us per encoder tile and SM, T = 50): 128 tiles 0.96 -> 0.83 ms, 100 tiles 0.75 -> 0.66 ms, 75 tiles 0.56 (one tile).
bool rollout_overlap_is_ping_pong(const nlc_model_s* m, int K) {
  const int n_tiles = (K + 127) / 128;
  static const int forced = [] { const char* e = getenv("NLC_OVERLAP_FORM"); return e && e[0] ? e[0] - '0' : 0; }();  // measurements
  if (2 * m->nx * m->S > 256) return false;
  if (forced == 1 && n_tiles <= 140) return false;
  if (forced == 3) return true;
  return n_tiles >= 89;
}
int launch_rollout_overlapped(nlc_model_s* m, const nlc_rollout_opts* o, const float* state, int sps, const float* p, const float* hist,
                              const float* pert_cost, int K, int T, int B, int nu, float* cost, float* states, int math_mode,
                              const unsigned int* ready, unsigned int ready_target, unsigned int* status, cudaStream_t stream) {
  return launch_rollout_tc2(m, o, state, sps, p, hist, pert_cost, K, T, B, nu, cost, states, nullptr, math_mode == NLC_MATH_TC_SPLIT3,
                            rollout_overlap_is_ping_pong(m, K) ? 3 : 1, stream, ready, ready_target, status);
}

// math_mode dispatch: the tensor-core kernel when it has an instantiation for (nx, S), else the FFMA kernel
static int launch_rollout(nlc_model_s* m, const nlc_rollout_opts* o, const float* state, int sps, const float* p,
                          const float* hist, const float* pert_cost, int K, int T, int B, int nu, float* cost, float* states,
                          float* delta_out, int math_mode, cudaStream_t stream) {
  if (math_mode != NLC_MATH_FP32 && rollout_has_tensor_core_form(m)) {
    // rollout_tc2.cu: beyond one wave of 128-sample tiles the ping-pong form (two tiles per CTA, all 16 warps alternating
    // between them: form 3), below that one tile on all 16 warps (form 1: the step latency is then all that matters)
    const int forced = forced_rollout_form();
    const int tiles = forced ? forced : ((K + 127) / 128 > 148 ? 3 : 1);
    int rc = launch_rollout_tc2(m, o, state, sps, p, hist, pert_cost, K, T, B, nu, cost, states, delta_out,
                                math_mode == NLC_MATH_TC_SPLIT3, tiles, stream);
    if (rc != NLC_ERR_UNSUPPORTED) return rc;
  }
  if (math_mode != NLC_MATH_FP32 && (long long)K * T >= 4096)
    warn_once(kWarnRolloutFfma, "rollout: nx = %d with %d Fourier terms (%d output columns) has no tcgen05 instantiation; %lld "
              "rollout-steps run on the fp32 CUDA-core kernel", m->nx, m->S, 2 * m->nx * m->S, (long long)K * T);
  return launch_rollout_fp32(m, o, state, sps, p, hist, pert_cost, K, T, B, nu, cost, states, delta_out, stream);
}

int launch_rollout_analytic(const nlc_rollout_opts* o, int nx, const float* state, int sps, const float* hist,
                            const float* pert_cost, int K, int T, int B, int nu, float* cost, float* states,
                            cudaStream_t stream);

}  // namespace nlc

using namespace nlc;

extern "C" int nlc_rollout_cost(nlc_model_t m, const nlc_rollout_opts* o, const float* state_dev, int state_per_sample,
                                const float* p_dev, const float* hist_dev, const float* pert_cost_dev, int K, int T,
                                int B, int nu, float* cost_total_dev, float* states_dev, int math_mode, void* stream) {
  NLC_REQUIRE(o && state_dev && hist_dev && cost_total_dev, NLC_ERR_ARG, "nlc_rollout_cost: null pointer");
  NLC_REQUIRE(K >= 1 && T >= 1 && B >= 1, NLC_ERR_ARG, "nlc_rollout_cost: K, T, B must be positive");
  NLC_REQUIRE(o->env >= NLC_ENV_PENDULUM && o->env <= NLC_ENV_ACROBOT, NLC_ERR_ARG, "unknown env id %d", o->env);
  const int env_nx[3] = {3, 5, 6}, env_nu[3] = {1, 1, 2};
  NLC_REQUIRE(nu == env_nu[o->env], NLC_ERR_SHAPE, "env %d takes nu=%d actions, got %d", o->env, env_nu[o->env], nu);
  if (o->env != NLC_ENV_CARTPOLE)
    NLC_REQUIRE(!o->state_constraint && o->goal_x == 0.0f, NLC_ERR_UNSUPPORTED,
                "state_constraint / change_goal exist only on the cartpole reward (ctcartpole.py:289-297)");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  if (o->dynamics == NLC_DYN_ANALYTIC_DELAY) {
    NLC_REQUIRE(o->delay >= 0 && o->delay < B, NLC_ERR_ARG, "delay %d outside the %d-entry window", o->delay, B);
    return launch_rollout_analytic(o, env_nx[o->env], state_dev, state_per_sample, hist_dev, pert_cost_dev, K, T, B, nu,
                                   cost_total_dev, states_dev, s);
  }
  NLC_REQUIRE(o->dynamics == NLC_DYN_NEURAL_LAPLACE, NLC_ERR_ARG, "unknown dynamics kind %d", o->dynamics);
  NLC_REQUIRE(m && p_dev, NLC_ERR_ARG, "nlc_rollout_cost: Neural Laplace dynamics need a model and p_dev");
  NLC_REQUIRE(m->nx == env_nx[o->env] && m->nu == nu, NLC_ERR_SHAPE, "model dims (%d,%d) do not match env %d", m->nx, m->nu, o->env);
  NLC_REQUIRE(math_mode == NLC_MATH_FP32 || math_mode == NLC_MATH_TC_SPLIT3 || math_mode == NLC_MATH_TC_FP16, NLC_ERR_ARG,
              "unknown math_mode %d", math_mode);
  return launch_rollout(m, o, state_dev, state_per_sample, p_dev, hist_dev, pert_cost_dev, K, T, B, nu, cost_total_dev,
                        states_dev, nullptr, math_mode, s);
}

// NeuralLaplaceModel.forward (w_nl.py:117-145) at the folded prediction time: encoder over the one
// window per sample, then one representation-MLP + ILT evaluation.
extern "C" int nlc_model_forward(nlc_model_t m, const float* obs_dev, const float* act_dev, int K, int B, float* out_dev,
                                 float* p_action_dev, int math_mode, void* stream) {
  NLC_REQUIRE(m && obs_dev && act_dev && out_dev, NLC_ERR_ARG, "nlc_model_forward: null pointer");
  NLC_REQUIRE(p_action_dev != nullptr, NLC_ERR_ARG, "nlc_model_forward: p_action_dev scratch [K][2] is required");
  NLC_REQUIRE(K >= 1, NLC_ERR_ARG, "nlc_model_forward: K must be positive");
  int rc = encode_history_impl(m, act_dev, m->gin, K, 1, B, p_action_dev, math_mode, static_cast<cudaStream_t>(stream));
  if (rc != NLC_OK) return rc;
  nlc_rollout_opts o;
  o.env = m->nx == 3 ? NLC_ENV_PENDULUM : (m->nx == 5 ? NLC_ENV_CARTPOLE : NLC_ENV_ACROBOT);
  o.state_constraint = 0; o.goal_x = 0.0f; o.dynamics = NLC_DYN_NEURAL_LAPLACE; o.delay = 0; o.dt = (float)m->dt;
  return launch_rollout(m, &o, obs_dev, 1, p_action_dev, act_dev, nullptr, K, 1, B, m->gin, nullptr, nullptr, out_dev,
                        math_mode, static_cast<cudaStream_t>(stream));
}


// ---------------------------------------------------------------------------------------------------------------------
// NeuralLaplaceModel.forward with a per-sample prediction time (the irregular-time form of training / validation,
// train_utils.py:401-404, overlay.py:664-737).  The s-points are then per sample: a prep kernel evaluates their sphere
// coordinates and folds them into a per-sample first-layer bias; the encoder and the MLP/ILT kernel are shared with the
// planner path (fp32 FFMA forms).
// ---------------------------------------------------------------------------------------------------------------------
namespace nlc {

// row_sph (optional, [K][2S]): the sphere coordinates [theta_s | phi_s] themselves - the first-layer input columns the
// backward (model_grad.cu) multiplies into dW1.
// row_obs (optional, [K][nx]) and row_p ([K][2]): row k's copy of obs and p of sample (r0 + k) / n_t, for rows that are
// (sample, time) pairs (nlc_model_forward_multi)
// b1_raw [kH] and w1_full_t [2S+nx+2][kH] are the unfolded first layer; T = double is the fp64 forward / backward's form.
template <typename T>
__global__ void __launch_bounds__(128) forward_ts_prep_kernel(const T* __restrict__ b1_raw, const T* __restrict__ w1_full_t, int kH,
                                                              int S, int Lp, int norm_time, T dt, const T* __restrict__ ts,
                                                              int K, T* __restrict__ row_b1, T* __restrict__ row_tn,
                                                              T* __restrict__ row_sph, const T* __restrict__ obs,
                                                              const T* __restrict__ p, long long r0, int n_t,
                                                              T* __restrict__ row_obs, T* __restrict__ row_p) {
  using C = Real<T>;
  __shared__ T th[kMaxS], ph[kMaxS];
  const int k = blockIdx.x, n = threadIdx.x;
  if (row_obs && n < Lp) {
    const size_t src = (size_t)((r0 + k) / n_t);
    if (n < Lp - 2) row_obs[(size_t)k * (Lp - 2) + n] = obs[src * (Lp - 2) + n];
    else row_p[(size_t)k * 2 + n - (Lp - 2)] = p[src * 2 + n - (Lp - 2)];
  }
  T tn = ts[k];
  if (norm_time) tn = tn / (dt * T(8));  // w_nl.py:123
  const T Tp = T(2) * (tn + C::eps);
  const T gamma = C::alpha + C::ln_inv_tol / Tp;
  for (int j = n; j < S; j += kH) {  // oracle/ilt.py: fourier_s_points + complex_to_sphere
    const T im = C::pi * (T)j / Tp;
    th[j] = rm::atan2(im, gamma);
    // phi = asin((r^2-1)/(r^2+1)) = 2 atan(r) - pi/2 (the asin form cancels for large r)
    ph[j] = T(2) * rm::atan(rm::sqrt(rm::fma(gamma, gamma, im * im))) - C::half_pi;
    if (row_sph) { row_sph[(size_t)k * 2 * S + j] = th[j]; row_sph[(size_t)k * 2 * S + S + j] = ph[j]; }
  }
  __syncthreads();
  T acc = b1_raw[n];
  for (int j = 0; j < S; ++j) acc = rm::fma(w1_full_t[(size_t)j * kH + n], th[j], acc);
  for (int j = 0; j < S; ++j) acc = rm::fma(w1_full_t[(size_t)(S + j) * kH + n], ph[j], acc);
  row_b1[(size_t)k * kH + n] = acc;
  if (n == 0) row_tn[k] = tn;
}

// b1_raw / w1_full_t: the handle's fp32 first layer, or (T = double, model_grad.cu) the one of the caller's fp64 weight image;
// dt and the time normalisation are then in fp64 too.
template <typename T>
int launch_forward_ts_prep(nlc_model_s* m, const T* b1_raw, const T* w1_full_t, const T* ts, int K, T* row_b1, T* row_tn, T* row_sph,
                           cudaStream_t s, const T* obs = nullptr, const T* p = nullptr, long long r0 = 0, int n_t = 1,
                           T* row_obs = nullptr, T* row_p = nullptr) {
  forward_ts_prep_kernel<T><<<K, m->Hm, 0, s>>>(b1_raw, w1_full_t, m->Hm, m->S, m->nx + 2, m->normalize && m->normalize_time, (T)m->dt,
                                                ts, K, row_b1, row_tn, row_sph, obs, p, r0, n_t, row_obs, row_p);
  NLC_LAUNCH_OK("forward_ts_prep_kernel");
  return NLC_OK;
}
template int launch_forward_ts_prep(nlc_model_s*, const float*, const float*, const float*, int, float*, float*, float*, cudaStream_t,
                                    const float*, const float*, long long, int, float*, float*);
template int launch_forward_ts_prep(nlc_model_s*, const double*, const double*, const double*, int, double*, double*, double*,
                                    cudaStream_t, const double*, const double*, long long, int, double*, double*);

// The MLP + Fourier ILT of K rows with per-row obs [K][nx], encoder output p [K][2] and prepared row_b1 / row_tn; mm is
// NLC_MATH_FP32 or NLC_MATH_TC_SPLIT3.
static int forward_rows(nlc_model_s* m, const float* obs, const float* p, const float* act, const float* row_b1, const float* row_tn,
                        int K, int B, float* out, int mm, cudaStream_t s) {
  nlc_rollout_opts o;
  o.env = m->nx == 3 ? NLC_ENV_PENDULUM : (m->nx == 5 ? NLC_ENV_CARTPOLE : NLC_ENV_ACROBOT);
  o.state_constraint = 0; o.goal_x = 0.0f; o.dynamics = NLC_DYN_NEURAL_LAPLACE; o.delay = 0; o.dt = (float)m->dt;
  if (mm == NLC_MATH_TC_SPLIT3 && rollout_has_tensor_core_form(m)) {
    // representation MLP on the tensor cores: per-sample first-layer bias added in the first epilogue, per-sample Fourier phases
    // and weights in the last (rollout_tc2.cu, kPerRow)
    int rc = launch_rollout_tc2(m, &o, obs, 1, p, act, nullptr, K, 1, B, m->gin, nullptr, nullptr, out, 1, 1, s, nullptr, 0, nullptr,
                                row_b1, row_tn);
    if (rc != NLC_ERR_UNSUPPORTED) return rc;
  }
  if (mm != NLC_MATH_FP32 && K >= 4096)
    warn_once(kWarnForwardTsFfma, "nlc_model_forward_ts: nx = %d, S = %d has no tcgen05 instantiation; %d samples run on the fp32 kernel",
              m->nx, m->S, K);
  return launch_rollout_fp32(m, &o, obs, 1, p, act, nullptr, K, 1, B, m->gin, nullptr, nullptr, out, s, row_b1, row_tn);
}

// workspace (floats): p [K][2] | row_b1 [C][H] | row_tn [C] | row_obs [C][nx] | row_p [C][2], C = min(K n_t, kMultiChunkRows)
struct MultiFwdWs { size_t p, b1, tn, obs, rp, total; int C; };
static size_t up64f(size_t n) { return (n + 63) / 64 * 64; }
static MultiFwdWs multi_fwd_ws(const nlc_model_s* m, int K, int n_t) {
  MultiFwdWs w;
  const long long rows = (long long)K * n_t;
  w.C = rows < kMultiChunkRows ? (int)rows : kMultiChunkRows;
  size_t o = 0;
  w.p = o; o += up64f((size_t)K * 2);
  w.b1 = o; o += up64f((size_t)w.C * m->Hm);
  w.tn = o; o += up64f(w.C);
  w.obs = o; o += up64f((size_t)w.C * m->nx);
  w.rp = o; o += up64f((size_t)w.C * 2);
  w.total = o;
  return w;
}

}  // namespace nlc

extern "C" int nlc_model_forward_ts(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K,
                                    int B, float* out_dev, float* scratch_dev, int math_mode, void* stream) {
  NLC_REQUIRE(m && obs_dev && act_dev && ts_dev && out_dev && scratch_dev, NLC_ERR_ARG, "nlc_model_forward_ts: null pointer");
  NLC_REQUIRE(K >= 1, NLC_ERR_ARG, "nlc_model_forward_ts: K must be positive");
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  float* p_action = scratch_dev;                 // [K][2]
  float* row_tn = scratch_dev + 2 * (size_t)K;   // [K]
  float* row_b1 = scratch_dev + 4 * (size_t)K;   // [K][hidden_units]   (offset keeps 16-byte alignment)
  NLC_REQUIRE(math_mode == NLC_MATH_FP32 || math_mode == NLC_MATH_TC_SPLIT3 || math_mode == NLC_MATH_TC_FP16, NLC_ERR_ARG,
              "unknown math_mode %d", math_mode);
  // the single-pass fp16 mode has no per-sample-time rollout instantiation: it takes the fp32-class tensor-core form
  const int mm = math_mode == NLC_MATH_TC_FP16 ? NLC_MATH_TC_SPLIT3 : math_mode;
  int rc = encode_history_impl(m, act_dev, m->gin, K, 1, B, p_action, mm, s);
  if (rc != NLC_OK) return rc;
  rc = launch_forward_ts_prep<float>(m, m->d.b1_raw, m->d.w1_full_t, ts_dev, K, row_b1, row_tn, nullptr, s);
  if (rc != NLC_OK) return rc;
  return forward_rows(m, obs_dev, p_action, act_dev, row_b1, row_tn, K, B, out_dev, mm, s);
}

// NeuralLaplaceModel.forward with ts_pred (K, n_t): the K windows are encoded once; the MLP + ILT then runs over the K n_t rows
// (sample k, time j) = row k n_t + j, chunk by chunk, on the kernels of nlc_model_forward_ts - each row is evaluated exactly as
// nlc_model_forward_ts evaluates a sample at that time.
extern "C" int64_t nlc_model_forward_multi_workspace_bytes(nlc_model_t m, int K, int n_t, int B) {
  if (!m || K < 1 || n_t < 1 || B < 1) return NLC_ERR_ARG;
  if ((long long)K * n_t >= (1LL << 31)) return NLC_ERR_SHAPE;
  return (int64_t)(multi_fwd_ws(m, K, n_t).total * sizeof(float));
}

extern "C" int nlc_model_forward_multi(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K, int n_t,
                                       int B, float* out_dev, float* p_action_dev, void* workspace_dev, int math_mode, void* stream) {
  NLC_REQUIRE(m && obs_dev && act_dev && ts_dev && out_dev && workspace_dev, NLC_ERR_ARG, "nlc_model_forward_multi: null pointer");
  NLC_REQUIRE(K >= 1 && n_t >= 1 && B >= 1, NLC_ERR_ARG, "nlc_model_forward_multi: K, n_t and B must be positive");
  NLC_REQUIRE((long long)K * n_t < (1LL << 31), NLC_ERR_SHAPE, "nlc_model_forward_multi: K n_t = %lld rows, 2^31 or more",
              (long long)K * n_t);
  NLC_REQUIRE(((uintptr_t)workspace_dev & 15) == 0, NLC_ERR_ARG, "nlc_model_forward_multi: workspace must be 16-byte aligned");
  NLC_REQUIRE(math_mode == NLC_MATH_FP32 || math_mode == NLC_MATH_TC_SPLIT3 || math_mode == NLC_MATH_TC_FP16, NLC_ERR_ARG,
              "unknown math_mode %d", math_mode);
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const MultiFwdWs w = multi_fwd_ws(m, K, n_t);
  float* ws = static_cast<float*>(workspace_dev);
  float* p = p_action_dev ? p_action_dev : ws + w.p;
  const int mm = math_mode == NLC_MATH_TC_FP16 ? NLC_MATH_TC_SPLIT3 : math_mode;  // as nlc_model_forward_ts
  int rc = encode_history_impl(m, act_dev, m->gin, K, 1, B, p, mm, s);
  if (rc != NLC_OK) return rc;
  const long long n_rows = (long long)K * n_t;
  for (long long r0 = 0; r0 < n_rows; r0 += w.C) {
    const int rows = (int)(n_rows - r0 < w.C ? n_rows - r0 : w.C);
    rc = launch_forward_ts_prep<float>(m, m->d.b1_raw, m->d.w1_full_t, ts_dev + r0, rows, ws + w.b1, ws + w.tn, nullptr, s, obs_dev, p,
                                       r0, n_t, ws + w.obs, ws + w.rp);
    if (rc != NLC_OK) return rc;
    rc = forward_rows(m, ws + w.obs, ws + w.rp, act_dev, ws + w.b1, ws + w.tn, rows, B, out_dev + r0 * m->nx, mm, s);
    if (rc != NLC_OK) return rc;
  }
  return NLC_OK;
}
