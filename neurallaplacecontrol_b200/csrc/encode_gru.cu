// Delayed-history encoder (ReverseGRUEncoder.forward, w_nl.py:25-29) over every window of the K x L
// action history: the encoder output depends on actions only, never on the state, so all K*T windows
// of a plan are encoded up front in one wide, non-recurrent-in-t pass and the sequential rollout only
// carries the representation MLP.
//
// This file is the fp32 CUDA-core (FFMA) form: the 1e-4 parity anchor.  encode_tc2.cu is the tcgen05 form.
//
// One CTA = 256 threads = a tile of 64 windows.  The three recurrent matrices (k-major, 3 x 48 KB) stay
// in shared memory for the CTA's whole persistent loop.  Thread (ug, rg) owns hidden units 4ug..4ug+3 of
// windows 4rg..4rg+3 for all three gates, so the gate nonlinearity is thread-local.  Hidden state lives
// transposed (hT[unit][window]) and ping-pongs between two buffers: one __syncthreads per GRU cell.
// Work skipped relative to the literal reference: products with the zero initial hidden state
// ("hoisted" FLOP count of SURVEY 8d).
#include <stddef.h>
#include <stdlib.h>

#include "common.cuh"

namespace nlc {

constexpr int kEncRows = 64;

struct EncArgs {
  const float* hist;  // [K][L][gin] env units
  float* p_out;       // [K*T][2]
  int K, T, B, L, gin;
  int hist_ch;  // channels stored in hist: gin, or gin-1 when the time channel of encode_obs_time is synthesised
  long long rows;
  ModelDev m;
};

template <int HG>
struct EncSmem {
  static constexpr int kG3 = 3 * HG;
  float w_hh0[HG * kG3];
  float w_ih1[HG * kG3];
  float w_hh1[HG * kG3];
  float w_ih0[kG3 * kMaxNu];
  float b_ih0[kG3], b_hh0[kG3], b_ih1[kG3], b_hh1[kG3];
  float w_out[2 * HG];
  alignas(16) float h0[2][HG * kEncRows];
  alignas(16) float h1[2][HG * kEncRows];
  alignas(16) float act[kEncRows * 8 * kMaxNu];  // [row][B][gin], B <= 8
  float b_out[2];
  float act_mean[kMaxNu], act_inv_std[kMaxNu];
};
static_assert(offsetof(EncSmem<64>, h0) % 16 == 0 && offsetof(EncSmem<64>, h1) % 16 == 0 && offsetof(EncSmem<64>, w_ih1) % 16 == 0, "float4 alignment");
static_assert(offsetof(EncSmem<32>, h0) % 16 == 0 && offsetof(EncSmem<32>, h1) % 16 == 0 && offsetof(EncSmem<32>, w_ih1) % 16 == 0, "float4 alignment");

// acc[g][i][j] += sum_k aT[k][4rg+i] * WT[k][HG g + 4ug + j]
template <int HG>
__device__ __forceinline__ void gemm3(const float* __restrict__ WT, const float* __restrict__ aT, int rg, int ug,
                                      float acc[3][4][4]) {
#pragma unroll 4
  for (int k = 0; k < HG; ++k) {
    const float4 a = *reinterpret_cast<const float4*>(aT + k * kEncRows + 4 * rg);
    const float av[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
    for (int g = 0; g < 3; ++g) {
      const float4 w = *reinterpret_cast<const float4*>(WT + k * (3 * HG) + HG * g + 4 * ug);
      const float wv[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[g][i][j] = fmaf(av[i], wv[j], acc[g][i][j]);
    }
  }
}

__device__ __forceinline__ void zero3(float acc[3][4][4]) {
#pragma unroll
  for (int g = 0; g < 3; ++g)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) acc[g][i][j] = 0.0f;
}

// GRU gate equations (torch.nn.GRU, gate order r,z,n): gi/gh are the input/hidden pre-activations
// WITHOUT bias for r,z,n; h_old may be null (zero state).
template <int HG>
__device__ __forceinline__ void gru_finish(const float gi[3][4][4], const float gh[3][4][4], const float* b_i,
                                           const float* b_h, const float* hT_old, float* hT_new, int rg, int ug) {
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    const int unit = 4 * ug + j;
    const float bir = b_i[unit], biz = b_i[HG + unit], bin = b_i[2 * HG + unit];
    const float bhr = b_h[unit], bhz = b_h[HG + unit], bhn = b_h[2 * HG + unit];
    float4 ho = make_float4(0.f, 0.f, 0.f, 0.f);
    if (hT_old) ho = *reinterpret_cast<const float4*>(hT_old + unit * kEncRows + 4 * rg);
    const float hov[4] = {ho.x, ho.y, ho.z, ho.w};
    float hn[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float r = sigmoid_acc((gi[0][i][j] + bir) + (gh[0][i][j] + bhr));
      float z = sigmoid_acc((gi[1][i][j] + biz) + (gh[1][i][j] + bhz));
      float n = tanh_acc((gi[2][i][j] + bin) + r * (gh[2][i][j] + bhn));
      hn[i] = fmaf(z, hov[i] - n, n);  // (1-z) n + z h
    }
    *reinterpret_cast<float4*>(hT_new + unit * kEncRows + 4 * rg) = make_float4(hn[0], hn[1], hn[2], hn[3]);
  }
}

// input projection of layer 0 (gin <= 4 inputs): gi[g][i][j] = sum_u w_ih0[HG g+unit][u] * x[row][u]
template <int HG>
__device__ __forceinline__ void layer0_input(const EncSmem<HG>& s, int step_j, int B, int gin, int rg, int ug,
                                             float gi[3][4][4]) {
#pragma unroll
  for (int g = 0; g < 3; ++g)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float* w = s.w_ih0 + (HG * g + 4 * ug + j) * gin;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float* x = s.act + ((4 * rg + i) * B + step_j) * gin;
        float acc = 0.0f;
        for (int u = 0; u < gin; ++u) acc = fmaf(w[u], x[u], acc);
        gi[g][i][j] = acc;
      }
    }
}

// HG = hidden_units / 2: 64 (config.py:37) or 32 (the reference class default hidden_units = 64, w_nl.py:71); 4 HG threads
template <int HG>
__global__ void __launch_bounds__(4 * HG, 1) encode_gru_kernel(EncArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  constexpr int kG3 = 3 * HG, kNT = 4 * HG;
  EncSmem<HG>& s = *reinterpret_cast<EncSmem<HG>*>(smem_raw);
  const int tid = threadIdx.x;
  const int rg = tid & 15, ug = tid >> 4;
  const int B = a.B, gin = a.gin;

  {  // weights: global -> shared, once per CTA
    const float4* src[3] = {reinterpret_cast<const float4*>(a.m.w_hh0_t), reinterpret_cast<const float4*>(a.m.w_ih1_t),
                            reinterpret_cast<const float4*>(a.m.w_hh1_t)};
    float4* dst[3] = {reinterpret_cast<float4*>(s.w_hh0), reinterpret_cast<float4*>(s.w_ih1), reinterpret_cast<float4*>(s.w_hh1)};
    for (int w = 0; w < 3; ++w)
      for (int i = tid; i < HG * kG3 / 4; i += kNT) dst[w][i] = __ldg(src[w] + i);
    for (int i = tid; i < kG3 * gin; i += kNT) s.w_ih0[i] = a.m.w_ih0[i];
    for (int i = tid; i < kG3; i += kNT) {
      s.b_ih0[i] = a.m.b_ih0[i]; s.b_hh0[i] = a.m.b_hh0[i]; s.b_ih1[i] = a.m.b_ih1[i]; s.b_hh1[i] = a.m.b_hh1[i];
    }
    for (int i = tid; i < 2 * HG; i += kNT) s.w_out[i] = a.m.w_out[i];
    if (tid < 2) s.b_out[tid] = a.m.b_out[tid];
    if (tid < gin) { s.act_mean[tid] = a.m.act_mean[tid]; s.act_inv_std[tid] = a.m.act_inv_std[tid]; }
  }
  __syncthreads();

  const long long n_tiles = (a.rows + kEncRows - 1) / kEncRows;
  for (long long tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const long long row0 = tile * kEncRows;
    // normalised action windows of the tile (w_nl.py:121): act[row][j][u], j = 0 oldest
    for (int i = tid; i < kEncRows * B * gin; i += kNT) {
      const int r = i / (B * gin), rem = i - r * (B * gin), j = rem / gin, u = rem - j * gin;
      long long row = row0 + r;
      if (row >= a.rows) row = a.rows - 1;
      const long long k = row / a.T;
      const int t = (int)(row - k * a.T);
      // encode_obs_time: the extra channel is the window position counted from the newest entry, B-1 .. 0
      // (mppi_with_model.py:110-119), not stored in the history
      const float v = u < a.hist_ch ? a.hist[((size_t)k * a.L + t + j) * a.hist_ch + u] : (float)(B - 1 - j);
      s.act[i] = (v - s.act_mean[u]) * s.act_inv_std[u];
    }
    __syncthreads();

    float gi[3][4][4], gh[3][4][4];
    // layer 0, first cell: newest entry (reversed order, w_nl.py:27), zero state
    layer0_input<HG>(s, B - 1, B, gin, rg, ug, gi);
    zero3(gh);
    gru_finish<HG>(gi, gh, s.b_ih0, s.b_hh0, nullptr, s.h0[0], rg, ug);
    __syncthreads();
    for (int st = 0; st < B; ++st) {
      const int cur = st & 1, prv = cur ^ 1;
      // layer 1 cell st: x = h0[cur], h = h1[prv] (zero at st == 0)
      zero3(gi);
      gemm3<HG>(s.w_ih1, s.h0[cur], rg, ug, gi);
      zero3(gh);
      if (st > 0) gemm3<HG>(s.w_hh1, s.h1[prv], rg, ug, gh);
      gru_finish<HG>(gi, gh, s.b_ih1, s.b_hh1, st > 0 ? s.h1[prv] : nullptr, s.h1[cur], rg, ug);
      if (st + 1 < B) {  // layer 0 cell st+1: x = window entry B-2-st, h = h0[cur]
        layer0_input<HG>(s, B - 2 - st, B, gin, rg, ug, gi);
        zero3(gh);
        gemm3<HG>(s.w_hh0, s.h0[cur], rg, ug, gh);
        gru_finish<HG>(gi, gh, s.b_ih0, s.b_hh0, s.h0[cur], s.h0[prv], rg, ug);
      }
      __syncthreads();
    }
    if (tid < 2 * kEncRows) {  // linear_out on the top layer's last state (w_nl.py:29)
      const int r = tid & (kEncRows - 1), o = tid >> 6;  // 2 x 64 outputs: the first 128 threads (4 HG >= 128)
      const float* hT = s.h1[(B - 1) & 1];
      float acc = s.b_out[o];
#pragma unroll 8
      for (int k = 0; k < HG; ++k) acc = fmaf(s.w_out[o * HG + k], hT[k * kEncRows + r], acc);
      if (row0 + r < a.rows) a.p_out[(row0 + r) * 2 + o] = acc;
    }
    // no barrier needed here: the next tile's first writes (act, h0[0]) do not alias what the
    // output phase reads (h1), and h1 is next written only after the barrier that follows A(0).
  }
}

template <int HG>
static int launch_encode_fp32_t(const EncArgs& a, cudaStream_t stream) {
  const int smem = (int)sizeof(EncSmem<HG>);
  // function attributes are per device: set on every launch, like every other kernel of the library
  NLC_CUDA_OK(cudaFuncSetAttribute(encode_gru_kernel<HG>, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  long long n_tiles = (a.rows + kEncRows - 1) / kEncRows;
  int grid = (int)(n_tiles < 148 ? n_tiles : 148);
  encode_gru_kernel<HG><<<grid, 4 * HG, smem, stream>>>(a);
  NLC_LAUNCH_OK("encode_gru_kernel");
  return NLC_OK;
}

int launch_encode_fp32(nlc_model_s* m, const float* hist, int hist_ch, int K, int T, int B, float* p, cudaStream_t stream) {
  EncArgs a;
  a.hist_ch = hist_ch;
  a.hist = hist; a.p_out = p; a.K = K; a.T = T; a.B = B; a.L = B - 1 + T; a.gin = m->gin;
  a.rows = (long long)K * T;
  a.m = m->d;
  return m->Hg == 64 ? launch_encode_fp32_t<64>(a, stream) : launch_encode_fp32_t<32>(a, stream);
}

int launch_encode_tc2(nlc_model_s* m, const float* hist, int hist_ch, int K, int T, int B, float* p, int split3, cudaStream_t stream,
                      unsigned int* ready = nullptr, int max_ctas = 0, long long tile_begin = 0, long long tile_end = -1,
                      int k_sub = 0, bool with_head = false);

// hist_ch: channels stored per history entry (model gin for nlc_model_forward, whose caller supplies the time channel
// like the reference's forward; action_dim on the planner path, where encode_obs_time's channel is synthesised)
int encode_history_impl(nlc_model_t m, const float* hist_dev, int hist_ch, int K, int T, int B, float* p_dev, int math_mode,
                        cudaStream_t s) {
  NLC_REQUIRE(m && hist_dev && p_dev, NLC_ERR_ARG, "nlc_encode_history: null pointer");
  NLC_REQUIRE(K >= 1 && T >= 1, NLC_ERR_ARG, "nlc_encode_history: K and T must be positive");
  NLC_REQUIRE(B >= 1 && B <= 8, NLC_ERR_SHAPE, "nlc_encode_history: window length %d outside [1,8]", B);
  NLC_REQUIRE(m->Hg == 64 || m->Hg == 32, NLC_ERR_SHAPE, "encoder hidden size must be 64 or 32");
  switch (math_mode) {
    case NLC_MATH_FP32: return launch_encode_fp32(m, hist_dev, hist_ch, K, T, B, p_dev, s);
    case NLC_MATH_TC_SPLIT3:
    case NLC_MATH_TC_FP16:
      // shapes without a tensor-core instantiation run on the fp32 kernel
      if (B < 2 || B * m->gin > 8 || m->gin > 2) {
        if ((long long)K * T >= 4096)
          warn_once(kWarnEncoderFfma, "encoder: window length %d x input width %d has no tcgen05 instantiation; %lld windows run on the "
                    "fp32 CUDA-core kernel", B, m->gin, (long long)K * T);
        return launch_encode_fp32(m, hist_dev, hist_ch, K, T, B, p_dev, s);
      }
      return launch_encode_tc2(m, hist_dev, hist_ch, K, T, B, p_dev, math_mode == NLC_MATH_TC_SPLIT3, s);
    default: set_error("nlc_encode_history: unknown math_mode %d", math_mode); return NLC_ERR_ARG;
  }
}

// Does (model, window length, math mode) run on the tcgen05 encoder?  (planner.cu: only then can the encoder publish per-step
// readiness to a rollout kernel running beside it.)
bool encoder_is_tensor_core(nlc_model_t m, int B, int math_mode) {
  return math_mode != NLC_MATH_FP32 && !(B < 2 || B * m->gin > 8 || m->gin > 2);
}

// The planner's overlapped form: step-major tile order over the samples from k_sub on, ready[t] counts finished warps of step t
// (4 per tile), tiles [tile_begin, tile_end) of that order (tile_end < 0: to the end), at most max_ctas CTAs so that the
// rollout kernel keeps its SMs.  with_head: the same launch first encodes samples [0, k_sub) in the plain order.
int encode_history_overlapped(nlc_model_t m, const float* hist_dev, int K, int T, int B, float* p_dev, int math_mode,
                              unsigned int* ready, int max_ctas, long long tile_begin, long long tile_end, int k_sub, bool with_head,
                              cudaStream_t s) {
  return launch_encode_tc2(m, hist_dev, m->nu, K, T, B, p_dev, math_mode == NLC_MATH_TC_SPLIT3, s, ready, max_ctas, tile_begin, tile_end,
                           k_sub, with_head);
}

}  // namespace nlc

using namespace nlc;

extern "C" int nlc_encode_history(nlc_model_t m, const float* hist_dev, int K, int T, int B, float* p_dev,
                                  int math_mode, void* stream) {
  NLC_REQUIRE(m != nullptr, NLC_ERR_ARG, "nlc_encode_history: null model");
  return encode_history_impl(m, hist_dev, m->nu, K, T, B, p_dev, math_mode, static_cast<cudaStream_t>(stream));
}
