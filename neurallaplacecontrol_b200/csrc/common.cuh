// Shared helpers of libnlc_b200: error plumbing, the model handle layout, fp32 math with stated
// error bounds, Philox4x32-10.
#pragma once

#include <cuda_runtime.h>
#include <math.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/nlc_b200.h"

namespace nlc {

void set_error(const char* fmt, ...);
int check_device_arch(int device);
void count_launch(int n = 1);
// one line on stderr, once per process and per `slot` (0..15): a shape that has no tensor-core instantiation runs on the
// fp32 CUDA-core kernels - correct, but an order of magnitude slower, so it must not be silent
void warn_once(int slot, const char* fmt, ...);
enum { kWarnEncoderFfma = 0, kWarnRolloutFfma = 1, kWarnForwardTsFfma = 2 };

#define NLC_CUDA_OK(expr)                                                                      \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      nlc::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return NLC_ERR_CUDA;                                                                     \
    }                                                                                          \
  } while (0)

#define NLC_LAUNCH_OK(name)                                                                    \
  do {                                                                                         \
    cudaError_t _e = cudaGetLastError();                                                       \
    if (_e != cudaSuccess) {                                                                   \
      nlc::set_error("launch of %s failed: %s (%s:%d)", name, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return NLC_ERR_CUDA;                                                                     \
    }                                                                                          \
    nlc::count_launch();                                                                       \
  } while (0)

#define NLC_REQUIRE(cond, code, ...)  \
  do {                                \
    if (!(cond)) {                    \
      nlc::set_error(__VA_ARGS__);    \
      return (code);                  \
    }                                 \
  } while (0)

// publication of the shard's triple from the last block of softmax_sum_kernel (G = 0: none)
struct ExchangePub {
  float* const* mailboxes;
  int G, rank, stride;
  const unsigned long long* step_ctr;
};

// End-of-step housekeeping the planner folds into its combine kernel instead of launching tiny kernels / memsets for it
// (planner.cu): every pointer optional.
struct StepTail {
  const float* U_src;            // the rolled control sequence the update applies to (nullptr: U is updated in place)
  unsigned long long* call_ctr;  // sampler call index += 1: the next control step draws fresh samples
  void* softmax_ws;              // stage 4 workspace header: re-armed for the next step (min = +inf, ticket = 0)
  unsigned int* ready;           // encoder readiness counters of the overlapped step: zeroed for the next step
  int n_ready;
  // host entry point (nlc_planner_command_host): the action and a sequence word go straight into MAPPED pinned host memory -
  // the host spins on the word instead of paying a D2H copy node and a stream synchronisation
  float* host_action;            // [nu] mapped host memory (nullptr: none)
  unsigned int* host_seq;        // mapped host word, incremented after the action is visible system-wide
  const float* action_src;       // the planner's device-resident action (written earlier in the same kernel)
  int nu;
};

constexpr int kMaxNx = 8;
constexpr int kMaxNu = 4;   // GRU input width limit (nu, or nu+1 with encode_obs_time)
// Rows per chunk of nlc_model_forward_multi / nlc_model_backward_multi: the per-row buffers of one chunk (row_b1 is hidden_units
// floats a row) stay at 36 MB at hidden 128, inside the 126 MB L2, and are bounded whatever K n_t is.
constexpr int kMultiChunkRows = 65536;
constexpr int kMaxS = 136;  // s-terms supported by the fused rollout (planner uses 17 or 33)

// Device-resident, packed model.  Everything the kernels read is fp32.
struct ModelDev {
  // ---- encoder (w_nl.py:14-29) -------------------------------------------------------------
  float* w_ih0;   // [3Hg][gin]
  float* b_ih0;   // [3Hg]
  float* b_hh0;   // [3Hg]
  float* w_hh0_t; // [Hg][3Hg]   (k-major: transposed for the FFMA kernels)
  float* w_ih1_t; // [Hg][3Hg]
  float* w_hh1_t; // [Hg][3Hg]
  float* b_ih1;   // [3Hg]
  float* b_hh1;   // [3Hg]
  float* w_out;   // [2][Hg]
  float* b_out;   // [2]
  // encode_tc2.cu: the three recurrent matrices as fp16 hi/lo tcgen05 operand images [3][2 (hi,lo)][3Hg * Hg] (K-major
  // canonical layout, tc_pack.cuh) with -log2(e) (r, z rows) and -2 log2(e) (n rows) folded in so that the gate
  // epilogue feeds ex2 directly, W_ih1 with its rows ordered [n | r | z] (one N=192 product into adjacent accumulator
  // columns); and the matching fp32 constants (biases, layer-0 input weights, output layer), layout kE2* below
  void* enc2_w;
  float* enc2_c;
  // input/bias blocks of the two GRU layers, [2 layers][4 Hg accumulator columns][8 halves] =
  // [W0_hi W0_hi W0_lo | W1_hi W1_hi W1_lo | b_hi b_lo]: all three split-3 terms of W_ih0 x + b in ONE K = 16 MMA against
  // the operand block [x0_hi x0_lo x0_hi | x1_hi x1_lo x1_hi | 1 1 | 0 x 8]   (layer 1: biases only)
  void* enc2_x;
  // rollout_tc2.cu: representation MLP with -2 log2(e) folded into every layer (all three feed tanh-like maps):
  // (Hm = 128 or 64; packed at both widths)
  // mlp2_w1 [2 (hi,lo)][Hm x 16]   first layer on the tensor cores, K = [obs_n | p_action | 1 (folded bias) | 0..]
  //                                 (re-packed by nlc_model_set_prediction_time: the bias depends on the s-points);
  // mlp2_w2 [2][Hm x Hm], mlp2_b2 [Hm] scaled;
  // mlp2_w3 [2 (hi,lo)][N3u x Hm], mlp2_b3 [N3u] scaled, in the GROUP-UNIFORM column order (rollout_tc2.cu: every column
  // group of a tile runs the SAME L3 epilogue code): column = 32 j + 8 cg + 2 i + {theta, phi}; regular unit j < NX (S-1)/16:
  // channel j / upc, term 16 (j % upc) + cg + 4 i (upc = (S-1)/16); last unit: the channels' last terms k = S-1, pair i =
  // channel cg + 4 i (zero columns where that channel does not exist)
  void* mlp2_w1;
  void* mlp2_w2;
  float* mlp2_b2;
  void* mlp2_w3;
  float* mlp2_b3;
  // ---- representation MLP (w_nl.py:32-63) --------------------------------------------------
  float* w1_full_t; // [2S+nx+2][Hm]  unfolded first layer (per-sample-time forward)
  float* b1_raw;    // [Hm]
  float* w1x_t;     // [nx+2][Hm]     columns of [obs_n | p_action]
  float* b1_fold;   // [Hm]           b1 + W1[:, :2S] . [theta_s | phi_s]   (fixed prediction time)
  float* w2_t;      // [Hm][Hm]
  float* b2;        // [Hm]
  float* w3_t;      // [Hm][N3p]      columns permuted: col' = 2*(c*S+k) + {0: theta, 1: phi}
  float* b3;        // [N3p]
  float* ilt_phase; // [S]  a_k = k*pi*t/T reduced to (-pi, pi]
  float* ilt_weight;// [S]  exp(gamma t)/T * (k == 0 ? 0.5 : 1)
  // ---- normalisation (w_nl.py:119-129) -----------------------------------------------------
  float* state_mean; // [nx]
  float* state_inv_std; // [nx]   (1/std; 1 when normalize is off)
  float* act_mean;   // [gin]
  float* act_inv_std;// [gin]
  // the same four in fp64, for the fp64 forward / backward (model_grad.cu), whose weights come per call from the caller
  double* state_mean64;
  double* state_inv_std64;
  double* act_mean64;
  double* act_inv_std64;
};

// float offsets inside ModelDev::enc2_c
constexpr int kE2Brz0 = 0;     // [128] -log2e (b_ih0 + b_hh0)[r, z]
constexpr int kE2Bin0 = 128;   // [64]  -2 log2e b_ih0[n]
constexpr int kE2Bhn0 = 192;   // [64]  -2 log2e b_hh0[n]
constexpr int kE2B1 = 256;     // [256] layer 1 in accumulator order [in | r | z | hn]
constexpr int kE2Wih0 = 512;   // [3][kMaxNu][64] scaled layer-0 input weights, [gate][input][unit]
constexpr int kE2Wout = 512 + 3 * kMaxNu * 64;  // [2][64]
constexpr int kE2Bout = kE2Wout + 128;          // [2]
constexpr int kE2Count = kE2Bout + 8;

// Overlapped planner step, ping-pong rollout (rollout_tc2.cu, planner.cu): CTAs and passes ("iterations" of two tiles per CTA) for
// n_tiles whole 128-sample tiles - as many passes as 148 CTAs would need, on as few CTAs as that number of passes allows;
// the encoder runs on the other SMs for the rollout's duration.
inline int pp_overlap_iters(int n_tiles) { return (n_tiles + 295) / 296; }
inline int pp_overlap_grid(int n_tiles) { const int it = pp_overlap_iters(n_tiles); return (n_tiles + 2 * it - 1) / (2 * it); }
// Pass q of CTA c rolls out samples [(q * grid + c) * 256, + 256): the passes before the last cover the first
// (iters - 1) * grid * 256 samples, and the kernel's pass count ceil(K / (grid * 256)) equals pp_overlap_iters.
inline int pp_overlap_k1(int n_tiles) { return (pp_overlap_iters(n_tiles) - 1) * pp_overlap_grid(n_tiles) * 256; }

struct ModelHost {  // fp64 copies kept for re-folding at another prediction time
  double* w0 = nullptr;  // [Hm][2S+nx+2]
  double* b0 = nullptr;  // [Hm]
};

}  // namespace nlc

struct nlc_model_s {
  int device;
  int nx, nu, gin, Hm, Hg, S, N3, N3p;
  int N3u;  // columns of the group-uniform W3 image (0: none packed)
  int normalize, normalize_time, encode_obs_time;
  double dt, ts_pred, t_norm;
  nlc::ModelDev d;
  nlc::ModelHost h;
  void* arena;  // single device allocation backing every pointer in d
  size_t arena_bytes;
  // planners hold the model by pointer: nlc_planner_create takes a reference, nlc_planner_destroy drops it, and
  // nlc_model_destroy on a model that is still referenced only marks it (freed with the last planner)
  int refs;
  bool destroy_requested;
  // layer 1 of the GRU: max over the (r, z) rows of log2(e) (|W_ih1 row|_1 + |W_hh1 row|_1 + |b_ih1 + b_hh1|) < 60 - both inputs
  // are hidden states in (-1, 1), so the tensor-core encoder's exponent clamps are provably idle for that layer
  bool enc_l1_bounded;
};

namespace nlc {

// ---------------------------------------------------------------------------------------------
// fp32 device math.  Error bounds are relative unless stated; they are what the 1e-4 parity
// budget in DESIGN.md is built from.
// ---------------------------------------------------------------------------------------------
#ifdef __CUDACC__

__device__ __forceinline__ float ex2_approx(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}

// exp(x), ~2 ulp: ex2.approx on the rounded product plus a first-order correction for the
// product's rounding error (the plain __expf error grows with |x|).
__device__ __forceinline__ float exp_acc(float x) {
  const float l2e_hi = 1.44269502162933349609375f;  // float(log2 e)
  const float l2e_lo = 1.925963033500011e-8f;       // log2 e - l2e_hi
  float t = x * l2e_hi;
  float r = fmaf(x, l2e_hi, -t);
  r = fmaf(x, l2e_lo, r);
  float e = ex2_approx(t);
  return fmaf(e, r * 0.693147180559945f, e);
}

__device__ __forceinline__ float rcp_acc(float x) { return __frcp_rn(x); }

// sigmoid(x) = 1/(1+exp(-x)); abs error <= ~2e-7.
__device__ __forceinline__ float sigmoid_acc(float x) {
  float e = exp_acc(-fminf(fmaxf(x, -80.f), 80.f));
  return rcp_acc(1.0f + e);
}

// tanh(x): 1 - 2/(exp(2x)+1) for |x| >= 0.05 (abs error <= ~1.5e-7), odd Taylor polynomial below
// (relative error <= 1e-7), so small pre-activations keep their relative accuracy.
__device__ __forceinline__ float tanh_acc(float x) {
  float ax = fabsf(x);
  float e = exp_acc(2.0f * fminf(ax, 15.0f));
  float big = 1.0f - 2.0f * rcp_acc(e + 1.0f);
  float x2 = x * x;
  float small = ax * fmaf(x2, fmaf(x2, fmaf(x2, -0.053968253968254f, 0.133333333333333f), -0.333333333333333f), 1.0f);
  float r = ax < 0.05f ? small : big;
  return copysignf(r, x);
}

// Riemann-sphere radius of the representation output (oracle/ilt.py sphere_to_complex with
// phi = (pi/2) tanh(u), w_nl.py:60-62):   r = tan(phi/2 + pi/4) = tan((pi/2) * sigmoid(2u)).
// Written through s = sigmoid(-2|u|) in (0, 1/2] so that both tails keep full RELATIVE accuracy
// (the literal 1 + tanh(u) cancels catastrophically for u << 0):  x = (pi/2) s in (0, pi/4],
// r = tan(x) for u <= 0 and cot(x) for u > 0, with sin/cos as Taylor polynomials on (0, pi/4]
// (truncation < 3e-9).  Relative error <= ~4e-7.
__device__ __forceinline__ float sphere_radius(float u) {
  float au = fminf(fabsf(u), 40.0f);
  float e = exp_acc(-2.0f * au);
  float s = e * rcp_acc(1.0f + e);
  float x = 1.57079632679489662f * s;
  float x2 = x * x;
  float sn = x * fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, -2.5052108385e-8f, 2.7557319224e-6f), -1.9841269841e-4f),
                                        8.3333333333e-3f), -1.6666666667e-1f), 1.0f);
  float cs = fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, fmaf(x2, -2.7557319224e-7f, 2.4801587302e-5f), -1.3888888889e-3f),
                                    4.1666666667e-2f), -0.5f), 1.0f);
  return u <= 0.0f ? __fdiv_rn(sn, cs) : __fdiv_rn(cs, sn);
}

// cos(x) for |x| <= 2*pi + small: one conditional 2*pi reduction to [-pi, pi], fold to [0, pi/2]
// and a degree-14 even / degree-13 odd Taylor evaluation.  Abs error <= ~2e-7.
__device__ __forceinline__ float cos_reduced(float x) {
  const float two_pi_hi = 6.28318548202514648f, two_pi_lo = -1.7484555314695172e-7f;
  const float pi_f = 3.14159274101257324f;
  float k = (x > pi_f) ? 1.0f : ((x < -pi_f) ? -1.0f : 0.0f);
  x = fmaf(-k, two_pi_hi, x);
  x = fmaf(-k, two_pi_lo, x);
  float ax = fabsf(x);  // [0, pi]
  // cos(ax) = -cos(pi - ax); evaluate on y in [0, pi/2]
  bool flip = ax > 1.57079632679489662f;
  float y = flip ? ((pi_f - ax) + -8.742278000372485e-8f) : ax;  // pi = pi_f + (-8.74e-8)
  // for y in [0, pi/2]: use cos poly if y <= pi/4 else sin(pi/2 - y)
  bool use_sin = y > 0.78539816339744831f;
  float z = use_sin ? ((1.57079637050628662f - y) + -4.371139000186243e-8f) : y;
  float z2 = z * z;
  float cs = fmaf(z2, fmaf(z2, fmaf(z2, fmaf(z2, fmaf(z2, -2.7557319224e-7f, 2.4801587302e-5f), -1.3888888889e-3f),
                                    4.1666666667e-2f), -0.5f), 1.0f);
  float sn = z * fmaf(z2, fmaf(z2, fmaf(z2, fmaf(z2, fmaf(z2, -2.5052108385e-8f, 2.7557319224e-6f), -1.9841269841e-4f),
                                        8.3333333333e-3f), -1.6666666667e-1f), 1.0f);
  float c = use_sin ? sn : cs;
  return flip ? -c : c;
}

// Philox4x32-10 (Salmon et al. 2011), counter (c0..c3), key (k0,k1).
__device__ __host__ __forceinline__ void philox4x32_10(uint32_t c[4], uint32_t k0, uint32_t k1) {
  const uint32_t M0 = 0xD2511F53u, M1 = 0xCD9E8D57u, W0 = 0x9E3779B9u, W1 = 0xBB67AE85u;
#pragma unroll
  for (int r = 0; r < 10; ++r) {
    uint64_t p0 = (uint64_t)M0 * c[0];
    uint64_t p1 = (uint64_t)M1 * c[2];
    uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k0;
    uint32_t n1 = (uint32_t)p1;
    uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k1;
    uint32_t n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k0 += W0; k1 += W1;
  }
}

// ---------------------------------------------------------------------------------------------
// fp64 counterparts of the fp32 helpers above, for the kernels templated on the scalar type
// (model_grad.cu, the per-sample-time prep of rollout.cu).  They keep the same cancellation-free
// forms on top of CUDA's fp64 libm (exp, tanh, tan, cos: <= 2 ulp).
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ double exp_acc(double x) { return exp(x); }
__device__ __forceinline__ double sigmoid_acc(double x) { return 1.0 / (1.0 + exp(-x)); }
__device__ __forceinline__ double tanh_acc(double x) { return tanh(x); }
// tan((pi/2) sigmoid(2u)) through s = sigmoid(-2|u|) in (0, 1/2]: tan((pi/2) s) for u <= 0, cot((pi/2) s) for u > 0;
// |u| clamped at 40 as in the fp32 form (a NaN stays NaN)
__device__ __forceinline__ double sphere_radius(double u) {
  const double au = fabs(u);
  const double e = exp(-2.0 * (au > 40.0 ? 40.0 : au));
  const double t = tan(1.5707963267948966 * (e / (1.0 + e)));
  return u <= 0.0 ? t : 1.0 / t;
}
__device__ __forceinline__ double cos_reduced(double x) { return cos(x); }

// Scalar-type-generic spellings of the libm calls and constants the templated kernels use: the float forms are exactly the
// calls and literals of the fp32 kernels, so their fp32 instantiations compile to the same arithmetic.
namespace rm {
__device__ __forceinline__ float fma(float a, float b, float c) { return fmaf(a, b, c); }
__device__ __forceinline__ double fma(double a, double b, double c) { return ::fma(a, b, c); }
__device__ __forceinline__ float min(float a, float b) { return fminf(a, b); }
__device__ __forceinline__ double min(double a, double b) { return fmin(a, b); }
__device__ __forceinline__ float abs(float a) { return fabsf(a); }
__device__ __forceinline__ double abs(double a) { return fabs(a); }
__device__ __forceinline__ float rcp(float a) { return __frcp_rn(a); }
__device__ __forceinline__ double rcp(double a) { return 1.0 / a; }
__device__ __forceinline__ float exp(float a) { return expf(a); }
__device__ __forceinline__ double exp(double a) { return ::exp(a); }
__device__ __forceinline__ float atan(float a) { return atanf(a); }
__device__ __forceinline__ double atan(double a) { return ::atan(a); }
__device__ __forceinline__ float atan2(float a, float b) { return atan2f(a, b); }
__device__ __forceinline__ double atan2(double a, double b) { return ::atan2(a, b); }
__device__ __forceinline__ float sqrt(float a) { return sqrtf(a); }
__device__ __forceinline__ double sqrt(double a) { return ::sqrt(a); }
// 4 consecutive elements (16-byte aligned for float, 16-byte aligned pairs for double)
__device__ __forceinline__ void ld4(const float* p, float v[4]) {
  const float4 q = *reinterpret_cast<const float4*>(p);
  v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
__device__ __forceinline__ void ld4(const double* p, double v[4]) {
  const double2 a = *reinterpret_cast<const double2*>(p), b = *reinterpret_cast<const double2*>(p + 2);
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void ldg4(const float* p, float v[4]) {
  const float4 q = __ldg(reinterpret_cast<const float4*>(p));
  v[0] = q.x; v[1] = q.y; v[2] = q.z; v[3] = q.w;
}
__device__ __forceinline__ void ldg4(const double* p, double v[4]) {
  const double2 a = __ldg(reinterpret_cast<const double2*>(p)), b = __ldg(reinterpret_cast<const double2*>(p + 2));
  v[0] = a.x; v[1] = a.y; v[2] = b.x; v[3] = b.y;
}
__device__ __forceinline__ void st4(float* p, const float v[4]) { *reinterpret_cast<float4*>(p) = make_float4(v[0], v[1], v[2], v[3]); }
__device__ __forceinline__ void st4(double* p, const double v[4]) {
  *reinterpret_cast<double2*>(p) = make_double2(v[0], v[1]);
  *reinterpret_cast<double2*>(p + 2) = make_double2(v[2], v[3]);
}
}  // namespace rm

// Constants of the Fourier ILT (torchlaplace defaults, oracle/ilt.py) in either precision: the float members are the
// literals of the fp32 kernels.
template <typename T> struct Real;
template <> struct Real<float> {
  static constexpr float pi = 3.14159265358979f, half_pi = 1.57079632679489662f, eps = 1.0e-6f, alpha = 1.0e-3f,
                         ln_inv_tol = 4.605170185988091f;  // -ln(10 alpha)
};
template <> struct Real<double> {
  static constexpr double pi = 3.141592653589793, half_pi = 1.5707963267948966, eps = 1.0e-6, alpha = 1.0e-3,
                          ln_inv_tol = 4.605170185988091;
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}
__device__ __forceinline__ float warp_min(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fminf(v, __shfl_xor_sync(0xffffffffu, v, o));
  return v;
}

#endif  // __CUDACC__

}  // namespace nlc
