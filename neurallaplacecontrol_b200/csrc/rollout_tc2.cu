// Stages 2+3 for the Neural Laplace dynamics, representation MLP on the 5th-generation tensor cores
// (rollout.cu is the fp32 CUDA-core anchor).  Two forms of one recurrence, chosen by plan size in rollout.cu:
//   rollout_pp_kernel   "ping-pong": two 128-sample tiles per CTA, all 16 epilogue warps on one tile's phase at a time + a
//                       dedicated MMA warp - plans beyond one wave of tiles (documented at the kernel)
//   rollout_tc2_kernel  one tile per CTA on all 16 warps - plans within one wave, where the step latency is what counts, and
//                       every plan of the shapes whose W3 does not fit shared memory (streamed, see the kernel)
//
// Same recurrence as rollout.cu: state <- state + ILT(MLP([s | obs_n | p_action])), cost += running_cost, whole horizon in
// one launch, state in registers.  The recurrence is a strict chain per sample (L1 -> L2 -> L3 -> ILT -> next step), so
// inside ONE tile the tensor pipe and the CUDA cores can only alternate: the one-tile form's first version measured 22.7 k
// clocks per step = MUFU time + issue time + MMA time, nothing overlapping.  It overlaps what it can by splitting products
// (kSplitK, kSplitD below); beyond one wave the ping-pong form covers each tile's products with the other tile's epilogues.
//
//   per step                A1 = [obs_n | p_action | 1] as a K = 16 operand (TMEM)          (one thread per sample)
//     M1  D = A1 W1^T       N = 128, K = 16   the first layer WITH its folded bias on the tensor cores
//     E1  tanh -> A         hidden activations re-written as the fp16 hi/lo A operand in TMEM (tcgen05.st)
//     M2  D = A W2^T        N = 128, K = 128
//     E2  + b2, tanh -> A
//     M3  D = A W3^T        the (theta, phi) pre-activations, in the group-uniform column order (l3_units_gu)
//     E3: sphere -> complex map, Fourier weights, fixed-order sum over the terms; the four column groups of a sample
//     exchange partial sums through shared memory; residual add; running cost (overlapped with M3)
//
//   -2 log2(e) is folded into all three layers on the host (model.cu): tanh(x) = 2 / (1 + 2^x') - 1 with x' = -2 log2e x,
//   the reciprocals are Newton iterations on the FMA pipe in packed fp32x2 (f32x2.cuh); per (channel, term) pair the
//   epilogue needs 2 ex2 + 1 cos + 1 rcp on the MUFU pipe instead of 7.
//   NLC_MATH_TC_SPLIT3: operands split hi+lo in fp16, D += A_hi B_hi + A_lo B_hi + A_hi B_lo (fp32-class);
//   NLC_MATH_TC_FP16  : single pass, tanh.approx (the stated looser bound).
//
//   One-tile form: samples are dealt to the CTAs in contiguous ranges (multiples of 32 rows), each walked in tiles of up
//   to 128 rows: a plan that is not a whole number of waves ends on partially filled tiles instead of an idle wave.
//   Warp w owns TMEM lanes 32 (w & 3).. (its 32 samples) and column group w >> 2.  After a CTA barrier warp 0 issues the
//   MMAs under elect.sync: the tile waits for that product anyway, so the issuing thread being held by the MMA queue costs
//   nothing (unlike in the encoder).
#include <cuda_fp16.h>
#include <stdlib.h>

#include <type_traits>

#include "common.cuh"
#include "env_cost.cuh"
#include "f32x2.cuh"
#include "tc_umma.cuh"

namespace nlc {

using namespace umma;

namespace rt2 {

// Both kernels are templates on the MLP width H: 128 (config.py:37) or 64 (the reference class default, w_nl.py:71).  At H = 64
// every thread owns 16 hidden units instead of 32 (one 16-column chunk), the A operand takes H / 2 TMEM columns per image,
// the accumulator region starts at column H, and W3 (at most 106 KB) always stays resident.  The sizes in the comments are
// those of H = 128.
constexpr int kRows = 128, kMaxH = 128;
constexpr uint32_t kLbo = 128;
template <int H> constexpr uint32_t kSboH = (H / 8) * 128;  // K = H operand images
constexpr uint32_t kSbo16 = (16 / 8) * 128;             // K = 16 (first layer)
constexpr uint32_t kColA = 0, kGroupCols = 256, kTmemCols = 512;  // the accumulator region starts at column H (A: hi | lo)
constexpr int kThreads = 512;

struct Args {
  ModelDev m;
  nlc_rollout_opts o;
  const float* state0; int state_per_sample;
  const float* p;
  const float* hist;
  const float* pert_cost;
  int K, T, B, L, nu;
  float* cost_total;
  float* states;
  float* delta_out;
  long long* trace;  // measurement only: clock64 timeline of CTA 0, [step][warp][8 events]
  // overlapped planner step (planner.cu): the history encoder runs BESIDE this kernel on the other SMs in step-major order
  // and bumps ready[t] as the windows of step t complete; p(., t) may be read once ready[t] >= ready_target.  A poll that
  // does not complete within ~1 s (the encoder is not co-resident: a serialising profiler, a shared GPU) sets *status = 1
  // and lets the step finish on whatever is there instead of hanging the device.
  const unsigned int* ready;
  unsigned int ready_target;
  unsigned int* status;
  // per-sample prediction times (nlc_model_forward_ts, one-tile form with kPerRow): row_b1 [K][128] = first-layer bias with
  // that sample's s-points folded in (natural units), row_tn [K] = its normalised time
  const float* row_b1;
  const float* row_tn;
};

__device__ __forceinline__ unsigned int ld_acquire_gpu(const unsigned int* p) {
  unsigned int v;
  asm volatile("ld.acquire.gpu.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
  return v;
}
// warp-wide: lane 0 polls, the warp continues once the windows of step t are published
__device__ __forceinline__ void wait_windows_ready(const Args& a, int t, int lane) {
  if (lane == 0) {
    const long long t0 = clock64();
    while (ld_acquire_gpu(a.ready + t) < a.ready_target) {
      // give up after ~1 s, and at once if any other warp of the launch already has: a plan that is not being encoded beside
      // this kernel costs one second, not one second per step and CTA
      if (ld_acquire_gpu(a.status) != 0u) break;
      if (clock64() - t0 > (1ll << 31)) { atomicExch(a.status, 1u); break; }
      __nanosleep(100);
    }
  }
  __syncwarp();
}

// W1 (2 x 4 KB), W2 (2 x 32 KB), W3 (2 x N3t x 256 B) -> shared memory; bulk copies of at most 32 KB each.  with_w3 = false:
// W3 is streamed half by half instead (load_w3_rows)
template <int kH>
__device__ __forceinline__ void load_weight_images(const ModelDev& m, unsigned char* w1_img, unsigned char* w2_img, unsigned char* w3_img,
                                                   int N3t, uint64_t* bar, bool with_w3 = true) {
  const uint32_t b1 = 2 * kH * 16 * 2, b2 = 2 * kH * kH * 2, b3 = with_w3 ? 2u * (uint32_t)N3t * kH * 2 : 0u;
  constexpr uint32_t kChunk2 = 2 * kH * kH * 2 < 32768 ? 2 * kH * kH * 2 : 32768;
  mbar_expect_tx(bar, b1 + b2 + b3);
  bulk_g2s(w1_img, m.mlp2_w1, b1, bar);
  for (uint32_t o = 0; o < b2; o += kChunk2) bulk_g2s(w2_img + o, static_cast<const unsigned char*>(m.mlp2_w2) + o, kChunk2, bar);
  for (uint32_t o = 0; o < b3; o += 32768) {
    const uint32_t n = b3 - o < 32768 ? b3 - o : 32768;
    bulk_g2s(w3_img + o, static_cast<const unsigned char*>(m.mlp2_w3) + o, n, bar);
  }
}
// Rows [row0, row0 + nrows) of W3 (output columns of the third layer; multiples of 8, so whole 8-row groups of the K-major
// image = contiguous bytes), hi and lo image, into a buffer that holds n_buf rows of each.  Issued by one thread.
template <int kH>
__device__ __forceinline__ void load_w3_rows(const ModelDev& m, unsigned char* w3_buf, int row0, int nrows, int N3t, int n_buf, uint64_t* bar) {
  const uint32_t bytes = (uint32_t)nrows * kH * 2;
  mbar_expect_tx(bar, 2 * bytes);
  for (int img = 0; img < 2; ++img) {
    const unsigned char* src = static_cast<const unsigned char*>(m.mlp2_w3) + ((size_t)img * N3t + row0) * kH * 2;
    unsigned char* dst = w3_buf + (size_t)img * n_buf * kH * 2;
    for (uint32_t o = 0; o < bytes; o += 32768) bulk_g2s(dst + o, src + o, bytes - o < 32768 ? bytes - o : 32768, bar);
  }
}

constexpr int kMaxN3 = 416;  // (theta, phi) columns of the largest instantiation (nx = 6, S = 33: 396 -> 400)
struct SmemTail {  // after the weight images
  alignas(8) uint64_t bar_w;
  alignas(8) uint64_t bar_w3;   // streamed W3 halves (instantiations whose W3 does not fit shared memory)
  alignas(16) float b2[kMaxH];
  alignas(16) float b3[kMaxN3];
  float phase[kMaxS], weight[kMaxS];
  float smean[kMaxNx], sinv[kMaxNx];
  alignas(16) float exch[4][kRows * kMaxNx];     // [column group] partial ILT sums
  alignas(8) uint64_t done[2];
  uint32_t tmem_base;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ float mufu_tanh(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float mufu_cos(float x) { float y; asm("cos.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

// tanh of two pre-activations that carry the folded scale x' = -2 log2(e) x
template <bool kAccurate, int kRcp>
__device__ __forceinline__ f2_t tanh2_scaled(f2_t xs) {
  float a, b;
  if (kAccurate) {
    upk2(xs, a, b);
    const f2_t d = add2(pk2(mufu_ex2(fminf(a, 120.0f)), mufu_ex2(fminf(b, 120.0f))), pk2(1.0f, 1.0f));
    return fma2(pk2(2.0f, 2.0f), rcp2<kRcp>(d), pk2(-1.0f, -1.0f));
  }
  upk2(mul2(xs, pk2(-0.34657359027997264f, -0.34657359027997264f)), a, b);
  return pk2(mufu_tanh(a), mufu_tanh(b));
}

// tanh of 16 pre-activations (8 packed pairs).  With Newton reciprocals (kRcp > 0) the 16 denominators 1 + 2^x' are inverted
// four packed pairs at a time through ONE reciprocal of their product (Montgomery's trick: 3 products up, 6 back - 15 FMA-pipe
// instructions per four pairs instead of 24; the hidden-layer phases of the ping-pong rollout are bound by that pipe).  The
// exponent is clamped at 30 so that the product of four denominators stays finite: 2 / (1 + 2^30) is below half an ulp of 1,
// so the clamped result is the correctly rounded one.  Accuracy: 3 more roundings than the direct Newton reciprocal (~2e-7).
template <bool kAccurate, int kRcp>
__device__ __forceinline__ void tanh16_scaled(f2_t (&v)[8]) {
  if constexpr (!kAccurate || kRcp == 0) {
#pragma unroll
    for (int i = 0; i < 8; ++i) v[i] = tanh2_scaled<kAccurate, kRcp>(v[i]);
  } else {
    const f2_t one = pk2(1.0f, 1.0f), two = pk2(2.0f, 2.0f), mone = pk2(-1.0f, -1.0f);
#pragma unroll
    for (int g = 0; g < 8; g += 4) {
      f2_t d[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        float a, b;
        upk2(v[g + i], a, b);
        d[i] = add2(pk2(mufu_ex2(fminf(a, 30.0f)), mufu_ex2(fminf(b, 30.0f))), one);
      }
      const f2_t p01 = mul2(d[0], d[1]), p23 = mul2(d[2], d[3]);
      const f2_t inv = rcp2<kRcp>(mul2(p01, p23));
      const f2_t i01 = mul2(inv, p23), i23 = mul2(inv, p01);
      v[g + 0] = fma2(two, mul2(i01, d[1]), mone);
      v[g + 1] = fma2(two, mul2(i01, d[0]), mone);
      v[g + 2] = fma2(two, mul2(i23, d[3]), mone);
      v[g + 3] = fma2(two, mul2(i23, d[2]), mone);
    }
  }
}

// 16 fp32 values (8 packed pairs) -> 8 fp16x2 words (hi) and the fp16 residuals (lo)
template <bool kSplit3>
__device__ __forceinline__ void pack16(const f2_t (&v)[8], uint32_t (&ph)[8], uint32_t (&pl)[8]) {
#pragma unroll
  for (int i = 0; i < 8; ++i) {
    float x0, x1;
    upk2(v[i], x0, x1);
    const __half2 hh = __floats2half2_rn(x0, x1);
    ph[i] = *reinterpret_cast<const uint32_t*>(&hh);
    if (kSplit3) {
      const float2 back = __half22float2(hh);
      float r0, r1;  // the residual is exact in fp32 either way; one packed FMA instead of two subtractions
      upk2(fma2(pk2(back.x, back.y), pk2(-1.0f, -1.0f), v[i]), r0, r1);
      const __half2 ll = __floats2half2_rn(r0, r1);
      pl[i] = *reinterpret_cast<const uint32_t*>(&ll);
    }
  }
}
__device__ __forceinline__ void ldtm16p(uint32_t taddr, f2_t (&v)[8]) {
  uint32_t r[16];
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
#pragma unroll
  for (int i = 0; i < 8; ++i) v[i] = pk2u(r[2 * i], r[2 * i + 1]);
}

// D[128 x N] = A[128 x Kdim] (TMEM, hi at a_tmem, lo at a_tmem + kALo = H / 2) * B[N x Kdim]^T (smem image, K-major)
template <bool kSplit3, int kALo>
__device__ __forceinline__ void issue_gemm_ts(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_hi, uint32_t b_lo, int N, int ksteps, uint32_t sbo) {
  const uint32_t idesc = idesc_f16_f32(kRows, N);
  for (int ks = 0; ks < ksteps; ++ks) {
    const uint32_t boff = ks * 2 * kLbo;
    mma_f16_ts(d_tmem, a_tmem + 8 * ks, smem_desc(b_hi + boff, kLbo, sbo), idesc, ks > 0 ? 1u : 0u);
    if (kSplit3) {
      mma_f16_ts(d_tmem, a_tmem + kALo + 8 * ks, smem_desc(b_hi + boff, kLbo, sbo), idesc, 1u);
      mma_f16_ts(d_tmem, a_tmem + 8 * ks, smem_desc(b_lo + boff, kLbo, sbo), idesc, 1u);
    }
  }
}

// Every second K-step of the same product (kHalf = 0: steps 0, 2, ..; 1: steps 1, 3, ..): the one-tile form issues a layer's
// product in two halves, the first as soon as the first 16 of every thread's 32 activation columns are in TMEM, so that half
// of the product runs under the second half of the epilogue that feeds it (strict chain per sample: nothing else covers it).
// kParts = 1 (H = 64: a thread's 16 columns are one K-step): `half` 0 is the whole product.
template <bool kSplit3, int kALo, int kParts = 2>
__device__ __forceinline__ void issue_gemm_ts_half(uint32_t d_tmem, uint32_t a_tmem, uint32_t b_hi, uint32_t b_lo, int N, int ksteps, uint32_t sbo,
                                                   int half) {
  const uint32_t idesc = idesc_f16_f32(kRows, N);
  for (int ks = half; ks < ksteps; ks += kParts) {
    const uint32_t boff = ks * 2 * kLbo;
    mma_f16_ts(d_tmem, a_tmem + 8 * ks, smem_desc(b_hi + boff, kLbo, sbo), idesc, ks > 0 ? 1u : 0u);
    if (kSplit3) {
      mma_f16_ts(d_tmem, a_tmem + kALo + 8 * ks, smem_desc(b_hi + boff, kLbo, sbo), idesc, 1u);
      mma_f16_ts(d_tmem, a_tmem + 8 * ks, smem_desc(b_lo + boff, kLbo, sbo), idesc, 1u);
    }
  }
}

// The same product for a warp that lives on 32 registers (the ping-pong form's MMA warp after setmaxnreg.dec).  Not
// inlined, so that the compiler cannot hoist the descriptors of every product of the step loop into registers (inlined,
// that spilled 246 words under the small budget); inside, fully unrolled with the descriptors advanced by immediates
// (a rolled loop that rebuilt them issued one MMA per ~130 clocks: the MMAs, not the epilogues, then set the step time).
// Called by the whole (converged) warp; ONE thread chosen by elect.sync issues and commits (tc_umma.cuh: elect_one).
template <int kSteps, bool kSplit3, int kALo>
__device__ __noinline__ void issue_gemm_ts_fn(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_hi_desc, uint64_t b_lo_desc, uint32_t idesc,
                                              uint64_t* done) {
  if (elect_one()) {
    fence_after_sync();
#pragma unroll
    for (int ks = 0; ks < kSteps; ++ks) {
      const uint64_t off = (uint64_t)(ks * 2 * kLbo >> 4);  // the start-address field counts 16-byte units
      mma_f16_ts(d_tmem, a_tmem + 8 * ks, b_hi_desc + off, idesc, ks > 0 ? 1u : 0u);
      if (kSplit3) {
        mma_f16_ts(d_tmem, a_tmem + kALo + 8 * ks, b_hi_desc + off, idesc, 1u);
        mma_f16_ts(d_tmem, a_tmem + 8 * ks, b_lo_desc + off, idesc, 1u);
      }
    }
    mma_commit(done);
  }
  __syncwarp();
}

// Two (channel, term) pairs of the L3 epilogue.  v = (theta', phi') pre-activations (bias added, scale folded):
//   y = tanh(theta_pre) -> theta = pi y (w_nl.py:59);   radius = tan((pi/2) sigmoid(2 phi_pre)) (w_nl.py:60-62 + sphere map,
//   written through s = sigmoid(-2|phi_pre|) in (0, 1/2] so both tails keep relative accuracy, common.cuh:sphere_radius);
//   term = weight_k radius cos(pi y + k pi t/T).      MUFU: 2 ex2 + 1 cos + 1 rcp per pair; the two sigmoids' reciprocals
//   come from ONE Newton reciprocal of the product of their denominators.
template <bool kAccurate, int kRcp>
__device__ __forceinline__ void l3_two_pairs(f2_t th, f2_t ph, float phase0, float phase1, float w0, float w1, float& t0, float& t1) {
  float a0, a1, b0, b1;
  upk2(th, a0, a1);
  upk2(ph, b0, b1);
  const f2_t one = pk2(1.0f, 1.0f);
  f2_t y, sg;
  const f2_t e2 = pk2(mufu_ex2(-fabsf(b0)), mufu_ex2(-fabsf(b1)));  // exp(-2|phi_pre|) in (0, 1]
  if (kAccurate) {
    const f2_t d1 = add2(pk2(mufu_ex2(fminf(a0, 60.0f)), mufu_ex2(fminf(a1, 60.0f))), one);
    const f2_t d2 = add2(e2, one);
    if (kRcp == 0) {  // two independent MUFU reciprocals: shortest dependency chain
      y = fma2(pk2(2.0f, 2.0f), rcp2<0>(d1), pk2(-1.0f, -1.0f));
      sg = mul2(e2, rcp2<0>(d2));
    } else {          // one Newton reciprocal of the product on the FMA pipe: fewest MUFU operations
      const f2_t inv = rcp2<kRcp>(mul2(d1, d2));
      y = fma2(pk2(2.0f, 2.0f), mul2(d2, inv), pk2(-1.0f, -1.0f));
      sg = mul2(e2, mul2(d1, inv));
    }
  } else {
    float c0, c1;
    upk2(mul2(th, pk2(-0.34657359027997264f, -0.34657359027997264f)), c0, c1);
    y = pk2(mufu_tanh(c0), mufu_tanh(c1));
    float d0, d1_;
    upk2(add2(e2, one), d0, d1_);
    sg = mul2(e2, pk2(mufu_rcp(d0), mufu_rcp(d1_)));
  }
  const f2_t x = mul2(sg, pk2(1.57079632679489662f, 1.57079632679489662f));  // (0, pi/4]
  const f2_t x2 = mul2(x, x);
  f2_t sn = fma2(x2, pk2(2.7557319224e-6f, 2.7557319224e-6f), pk2(-1.9841269841e-4f, -1.9841269841e-4f));
  sn = fma2(sn, x2, pk2(8.3333333333e-3f, 8.3333333333e-3f));
  sn = fma2(sn, x2, pk2(-1.6666666667e-1f, -1.6666666667e-1f));
  sn = mul2(x, fma2(sn, x2, one));
  f2_t cs = fma2(x2, pk2(2.4801587302e-5f, 2.4801587302e-5f), pk2(-1.3888888889e-3f, -1.3888888889e-3f));
  cs = fma2(cs, x2, pk2(4.1666666667e-2f, 4.1666666667e-2f));
  cs = fma2(cs, x2, pk2(-0.5f, -0.5f));
  cs = fma2(cs, x2, one);
  float sn0, sn1, cs0, cs1;
  upk2(sn, sn0, sn1);
  upk2(cs, cs0, cs1);
  // phi_pre <= 0 (scaled value >= 0): radius = tan(x) = sn / cs, else cot(x) = cs / sn
  const bool neg0 = b0 >= 0.0f, neg1 = b1 >= 0.0f;
  const float rad0 = (neg0 ? sn0 : cs0) * mufu_rcp(neg0 ? cs0 : sn0);
  const float rad1 = (neg1 ? sn1 : cs1) * mufu_rcp(neg1 ? cs1 : sn1);
  // cos(pi y + a_k), a_k = pi k t/T reduced to (-pi, pi]: the argument stays inside (-2 pi, 2 pi), where cos.approx is
  // good to 5.2e-7 absolute without any further range reduction (tools/cos_err.cu; 3.4e-7 with an exact reduction)
  float y0, y1;
  upk2(y, y0, y1);
  t0 = (w0 * rad0) * mufu_cos(fmaf(3.14159265358979f, y0, phase0));
  t1 = (w1 * rad1) * mufu_cos(fmaf(3.14159265358979f, y1, phase1));
}

// A thread reads its (theta, phi) columns in UNITS of 8 columns (4 pairs), and all of its units of a phase (up to four) are
// loaded before the first is used - one TMEM round trip per phase instead of one per 16-column chunk.
__device__ __forceinline__ void ldtm8q(uint32_t taddr, f2_t (&v)[4]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = pk2u(r[2 * i], r[2 * i + 1]);
}
// GROUP-UNIFORM units (ModelDev::mlp2_w3): unit j = 32 columns, 8 per column group, so that the four column groups of a
// sample run the SAME instructions on different addresses - the four warps of an SM sub-partition are the four column
// groups of one row quarter, and with a code variant per group each sub-partition walked four copies of the unrolled
// epilogue (47 KB; a tenth of the warp stalls were instruction fetches).  Regular unit j < NX upc (upc = (S-1)/16): channel
// j / upc (compile time), terms 16 (j % upc) + cg + 4 i; the last unit holds the terms k = S-1 of channels cg and cg + 4.
// tDcg, b3cg, phasecg, weightcg: the D region / bias / Fourier tables offset by this thread's column group (8 cg, 8 cg, cg, cg).
// kPerRow: the sample has its own prediction time - phase_k = k pi t/T = k (pi/2 - rd) reduced to (-pi, pi] with the quarter
// turns exact, weight_k = rs (k == 0 ? 1/2 : 1), rd = pi eps / T and rs = exp(gamma t) / T of that sample (oracle/ilt.py);
// k & 3 = cg for the regular units (their terms are cg + a multiple of 4), 0 for the last (S - 1 is a multiple of 16).
template <int NX, int S, int kJ0, int kJ1, bool kAccurate, int kRcp, bool kPerRow = false>
__device__ __forceinline__ void l3_units_gu(uint32_t tDcg, const float* __restrict__ b3cg, const float* __restrict__ phasecg,
                                            const float* __restrict__ weightcg, int cg, float (&delta)[NX], float rd = 0.0f,
                                            float rs = 0.0f) {
  constexpr int kUpc = (S - 1) / 16, kJ = NX * kUpc, kCount = kJ1 - kJ0;
  static_assert((S - 1) % 16 == 0 && kCount >= 1 && kCount <= 4 && kJ1 <= kJ + 1, "group-uniform units");
  f2_t v[kCount][4];
#pragma unroll
  for (int u = 0; u < kCount; ++u) ldtm8q(tDcg + 32 * u, v[u]);
  tmem_ld_wait();
#pragma unroll
  for (int u = 0; u < kCount; ++u) {
    const int j = kJ0 + u;
    const float4 ba = *reinterpret_cast<const float4*>(b3cg + 32 * j), bb = *reinterpret_cast<const float4*>(b3cg + 32 * j + 4);
    const f2_t bias[4] = {pk2(ba.x, ba.y), pk2(ba.z, ba.w), pk2(bb.x, bb.y), pk2(bb.z, bb.w)};
#pragma unroll
    for (int i = 0; i < 4; i += 2) {
      if (j == kJ && i == 2) break;  // the last unit: two pairs (channels cg and cg + 4), the other four columns are padding
      const f2_t s0 = add2(v[u][i], bias[i]), s1 = add2(v[u][i + 1], bias[i + 1]);
      float th0, ph0, th1, ph1;
      upk2(s0, th0, ph0);
      upk2(s1, th1, ph1);
      float t0, t1;
      if (j < kJ) {
        const int kb = 16 * (j % kUpc) + 4 * i;  // + cg: in the table pointers
        if constexpr (kPerRow) {
          const float qcg = cg == 0 ? 0.0f : (cg == 1 ? 1.57079632679489662f : (cg == 2 ? 3.14159265358979f : -1.57079632679489662f));
          const float kf = (float)(kb + cg);
          l3_two_pairs<kAccurate, kRcp>(pk2(th0, th1), pk2(ph0, ph1), fmaf(-kf, rd, qcg), fmaf(-(kf + 4.0f), rd, qcg),
                                        (kb == 0 && cg == 0) ? 0.5f * rs : rs, rs, t0, t1);
        } else {
          l3_two_pairs<kAccurate, kRcp>(pk2(th0, th1), pk2(ph0, ph1), phasecg[kb], phasecg[kb + 4], weightcg[kb], weightcg[kb + 4], t0, t1);
        }
        delta[j / kUpc] += t0;
        delta[j / kUpc] += t1;
      } else {
        const float phl = kPerRow ? -(float)(S - 1) * rd : phasecg[S - 1 - cg], wl = kPerRow ? rs : weightcg[S - 1 - cg];
        l3_two_pairs<kAccurate, kRcp>(pk2(th0, th1), pk2(ph0, ph1), phl, phl, wl, wl, t0, t1);
#pragma unroll
        for (int c = 0; c < NX; ++c) delta[c] += (c == cg) ? t0 : ((c == cg + 4) ? t1 : 0.0f);
      }
    }
  }
}

// units kJ0 .. kJ1 - 1, four at a time (32 accumulator registers in flight); kBase = the unit in column 0 of the D region
template <int NX, int S, int kJ0, int kJ1, int kBase, bool kAccurate, int kRcp, bool kPerRow>
struct L3GU {
  static __device__ __forceinline__ void run(uint32_t tDcg, const float* b3cg, const float* phasecg, const float* weightcg, int cg,
                                             float (&delta)[NX], float rd, float rs) {
    if constexpr (kJ0 < kJ1) {
      constexpr int kJm = kJ0 + 4 < kJ1 ? kJ0 + 4 : kJ1;
      l3_units_gu<NX, S, kJ0, kJm, kAccurate, kRcp, kPerRow>(tDcg + 32 * (kJ0 - kBase), b3cg, phasecg, weightcg, cg, delta, rd, rs);
      L3GU<NX, S, kJm, kJ1, kBase, kAccurate, kRcp, kPerRow>::run(tDcg, b3cg, phasecg, weightcg, cg, delta, rd, rs);
    }
  }
};

template <int NX, int S>
struct PPShape {  // columns of the group-uniform W3 image: model.cu packs N3u = 32 (NX (S-1)/16 + 1)
  static constexpr int kUnits = NX * ((S - 1) / 16) + 1, N3u = 32 * kUnits;
};

template <int H, int NX, int S, bool kSplit3, int kRcp, bool kPerRow = false>
__global__ void __launch_bounds__(kThreads, 1) rollout_tc2_kernel(Args a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int Lp = NX + 2;
  constexpr int kH = H, kChunks = H / 64;  // 16-column chunks of hidden units per thread
  constexpr uint32_t kSbo = kSboH<H>, kALo = H / 2, kColD = H;
  // the (theta, phi) columns in the GROUP-UNIFORM order (l3_units_gu: one L3 epilogue code for all four column groups)
  constexpr int kUnits = PPShape<NX, S>::kUnits, N3t = PPShape<NX, S>::N3u;
  // One tile, all 16 warps on it in four column groups of H / 4 hidden units, L3 in one piece (A 128 + D up to 256 columns).
  // kStream (H = 128 with more than 256 (theta, phi) columns: S = 33 with nx >= 5, the reference class default w_nl.py:73): L3
  // in two column halves of at most 256 columns, and W3 - which no longer fits shared memory next to W1 and W2 - streamed: one
  // buffer of N3a rows, reloaded by TMA bulk copies (L2-resident source) as soon as the product that read it has completed,
  // each load hidden under the epilogue that follows.  At H = 64 W3 (<= 106 KB) stays resident and the accumulator region
  // (from column 64) holds all of its up to 416 columns: L3 is then always the two kSplitD products of <= 256 columns.
  constexpr bool kStream = H == 128 && N3t > 256;
  constexpr int kUnitsA = kStream ? (kUnits + 1) / 2 : kUnits;        // units in the first column half
  constexpr int N3a = 32 * kUnitsA, N3b = N3t - N3a;
  constexpr int N3buf = kStream ? N3a : N3t;                          // rows of W3 resident at a time
  // kSplitD (resident W3): the L3 product is issued as TWO products into disjoint column ranges of the accumulator,
  // each with its own completion barrier, so the epilogue of the first half's columns runs while the second half is still
  // on the tensor pipe - in this form nothing else covers the products (strict chain per sample)
  constexpr bool kSplitD = !kStream && N3t >= 128;
  constexpr int kUnitsH = kSplitD ? (kUnits + 1) / 2 : kUnits;        // units of the first product
  constexpr int N3h = 32 * kUnitsH;
  static_assert((kStream ? N3a <= 256 && N3b <= 256 : N3h <= 256 && N3t - N3h <= 256) && N3t <= kMaxN3 && Lp + 1 <= 16,
                "tile shape");
  static_assert(kColD + (kStream ? N3a : N3t) <= kTmemCols, "accumulator columns");
  unsigned char* w1_img = smem_raw;                                   // [hi | lo] 128 x 16 halves = 4 KB each
  unsigned char* w2_img = w1_img + 2 * kH * 16 * 2;                   // [hi | lo] 32 KB each
  unsigned char* w3_img = w2_img + 2 * kH * kH * 2;                   // [hi | lo] N3buf * 256 B each
  SmemTail& s = *reinterpret_cast<SmemTail*>(w3_img + 2 * (size_t)N3buf * kH * 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;

  {
    // weight images by TMA bulk copies (one issuing thread, counted on bar_w): only the MMA-issuing warp waits for them, so the
    // load runs under the TMEM allocation and the first operand's preparation - prologue latency is what small plans pay for
    if (warp == 0 && elect_one()) {  // (elect.sync, not tid == 0: the copies' operands then stay in uniform registers)
      mbar_init(&s.bar_w, 1);
      mbar_init(&s.bar_w3, 1);
      mbar_fence_init();
      load_weight_images<kH>(a.m, w1_img, w2_img, w3_img, N3t, &s.bar_w, !kStream);
      if (kStream) load_w3_rows<kH>(a.m, w3_img, 0, N3a, N3t, N3buf, &s.bar_w3);
    }
    for (int i = tid; i < kH; i += kThreads) s.b2[i] = a.m.mlp2_b2[i];
    for (int i = tid; i < kMaxN3; i += kThreads) s.b3[i] = i < N3t ? a.m.mlp2_b3[i] : 0.0f;
    for (int i = tid; i < S; i += kThreads) { s.phase[i] = a.m.ilt_phase[i]; s.weight[i] = a.m.ilt_weight[i]; }
    if (tid < NX) { s.smean[tid] = a.m.state_mean[tid]; s.sinv[tid] = a.m.state_inv_std[tid]; }
    if (tid == 0) {
      for (int g = 0; g < 2; ++g) mbar_init(&s.done[g], 1);
      mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&s.tmem_base, kTmemCols);
  }
  fence_proxy_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = s.tmem_base;

  // samples of this CTA: a contiguous range, a multiple of 32 rows long (except at the very end of the plan)
  const int n_slots = gridDim.x, slot = blockIdx.x;
  const int per_slot = ((a.K + n_slots - 1) / n_slots + 31) / 32 * 32;
  const long long r_begin_ll = (long long)slot * per_slot;
  const int r_begin = (int)(r_begin_ll < a.K ? r_begin_ll : a.K);
  const int r_end = (r_begin + per_slot < a.K) ? r_begin + per_slot : a.K;
  uint64_t* done = &s.done[0];

  {
    // =====================================  the 16 epilogue warps  =====================================
    const int q = warp & 3, cg = warp >> 2;
    const int row = 32 * q + lane;
    const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
    const uint32_t tA = tlane + kColA, tD = tlane + kColD;
    const uint32_t w1_hi = smem_u32(w1_img), w1_lo = w1_hi + kH * 16 * 2;
    const uint32_t w2_hi = smem_u32(w2_img), w2_lo = w2_hi + kH * kH * 2;
    const uint32_t w3_hi = smem_u32(w3_img), w3_lo = w3_hi + (uint32_t)N3buf * kH * 2;
    uint32_t n = 0, n_w3 = 0, n_b = 0;  // products waited for; W3 halves waited for (issuing warp only); second L3 halves (kSplitD)
    bool active_w = false;              // (hidden_split) this warp has live samples in the current tile
    int tstep = 0;
    auto mark = [&](int ev) {
      if (a.trace && blockIdx.x == 0 && lane == 0 && tstep < 104) a.trace[(tstep * 16 + warp) * 8 + ev] = clock64();
    };
    // hand-off to the tensor pipe: every warp has finished its TMEM stores / loads (CTA barrier), then one thread issues
    // product `ev` of the step (0: M1, 3: the second column half of M3 with W3 streamed).  The tile waits for that product
    // anyway (strict chain per sample), so the issuing warp being held by the MMA queue costs nothing.
    if (warp == 0) mbar_wait(&s.bar_w, 0);  // the issuing warp: weight images landed
    auto issue = [&](int ev) {
      tmem_st_wait();
      fence_before_sync();
      asm volatile("bar.sync %0, %1;" ::"r"(1), "n"(kThreads) : "memory");
      if (kStream && warp == 0 && ev == 3) { mbar_wait(&s.bar_w3, n_w3 & 1); ++n_w3; }  // this half of W3 has landed
      if (warp == 0 && elect_one()) {
        fence_after_sync();
        if (ev == 0) issue_gemm_ts<kSplit3, kALo>(tmem + kColD, tmem + kColA, w1_hi, w1_lo, kH, 1, kSbo16);
        else issue_gemm_ts<kSplit3, kALo>(tmem + kColD, tmem + kColA, w3_hi, w3_lo, N3b, kH / 16, kSbo);  // (the buffer holds that half)
        mma_commit(done);
      }
      __syncwarp();
    };
    // products M2 and M3 in two K-halves (issue_gemm_ts_half).  half 0 = the K-steps fed by every thread's first 16
    // activation columns (even steps: thread columns 32 cg .. 32 cg + 15 are K-step 2 cg), half 1 = the rest and the commit(s).
    // H = 64: one part, issued whole with its commit(s) once every thread's 16 columns are in TMEM.
    auto issue_k = [&](int ev, int half) {
      tmem_st_wait();
      fence_before_sync();
      asm volatile("bar.sync %0, %1;" ::"r"(1), "n"(kThreads) : "memory");
      if (kStream && warp == 0 && ev >= 2 && half == 0) { mbar_wait(&s.bar_w3, n_w3 & 1); ++n_w3; }  // this half of W3 has landed
      if (warp == 0 && elect_one()) {
        fence_after_sync();
        if (ev == 1) issue_gemm_ts_half<kSplit3, kALo, kChunks>(tmem + kColD, tmem + kColA, w2_hi, w2_lo, kH, kH / 16, kSbo, half);
        else if (kSplitD) {
          issue_gemm_ts_half<kSplit3, kALo, kChunks>(tmem + kColD, tmem + kColA, w3_hi, w3_lo, N3h, kH / 16, kSbo, half);
          if (half == kChunks - 1) mma_commit(done);  // first column half: the epilogue starts on it while the second half computes
          issue_gemm_ts_half<kSplit3, kALo, kChunks>(tmem + kColD + N3h, tmem + kColA, w3_hi + (uint32_t)(N3h / 8) * kSbo,
                                                     w3_lo + (uint32_t)(N3h / 8) * kSbo, N3t - N3h, kH / 16, kSbo, half);
          if (half == kChunks - 1) mma_commit(&s.done[1]);
        } else {
          issue_gemm_ts_half<kSplit3, kALo, kChunks>(tmem + kColD, tmem + kColA, w3_hi, w3_lo, N3a, kH / 16, kSbo, half);
        }
        if (half == kChunks - 1 && !(ev == 2 && kSplitD)) mma_commit(done);
      }
      __syncwarp();
    };
    auto wait_mma = [&]() {
      mbar_wait_sleep(done, n & 1); ++n;
      fence_after_sync();
    };
    // hidden-layer epilogue with the K-split hand-off: both 16-column chunks of this thread are read BEFORE the first half of
    // the next product may overwrite the accumulator; bias_kind: 0 none, 1 b2, 2 per-sample first-layer bias
    auto hidden_split = [&](int ev_next, int bias_kind, int kk) {
      f2_t va[8], vb[8];
      const int n0 = 16 * kChunks * cg;
      if (active_w) {
        ldtm16p(tD + n0, va);
        if constexpr (kChunks == 2) ldtm16p(tD + n0 + 16, vb);
        tmem_ld_wait();
      }
#pragma unroll
      for (int c16 = 0; c16 < kChunks; ++c16) {
        if (active_w) {
          f2_t (&v)[8] = c16 == 0 ? va : vb;
          const int nn = n0 + 16 * c16;
          if (bias_kind == 1) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 b = *reinterpret_cast<const float4*>(s.b2 + nn + 4 * i);
              v[2 * i] = add2(v[2 * i], pk2(b.x, b.y));
              v[2 * i + 1] = add2(v[2 * i + 1], pk2(b.z, b.w));
            }
          } else if (bias_kind == 2) {  // + (-2 log2 e) x this sample's first-layer bias (the accumulator carries the folded scale)
            const float4* bp = reinterpret_cast<const float4*>(a.row_b1 + (size_t)kk * kH + nn);
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 b = __ldg(bp + i);
              const f2_t c = pk2(-2.8853900817779268f, -2.8853900817779268f);
              v[2 * i] = fma2(pk2(b.x, b.y), c, v[2 * i]);
              v[2 * i + 1] = fma2(pk2(b.z, b.w), c, v[2 * i + 1]);
            }
          }
          tanh16_scaled<kSplit3, kRcp / 10>(v);
          uint32_t ph[8], pl[8];
          pack16<kSplit3>(v, ph, pl);
          tmem_st8(tA + nn / 2, ph);
          if (kSplit3) tmem_st8(tA + kALo + nn / 2, pl);
        }
        issue_k(ev_next, c16);
      }
    };
    for (int tile0 = r_begin; tile0 < r_end; tile0 += kRows) {
      const int nrows = (r_end - tile0 < kRows) ? r_end - tile0 : kRows;
      const bool active = 32 * q < nrows;           // warp-uniform: this warp has at least one live sample
      const bool live = row < nrows;
      const int kk = live ? tile0 + row : r_end - 1;
      float st[NX], in[Lp];
#pragma unroll
      for (int c = 0; c < NX; ++c) {
        st[c] = a.state0[(size_t)(a.state_per_sample ? kk / a.state_per_sample : 0) * NX + c];
        in[c] = (st[c] - s.smean[c]) * s.sinv[c];
      }
      {
        // (__ldcg: p may be written by the encoder kernel while this kernel runs - never through a stale L1 line)
        if (a.ready) wait_windows_ready(a, 0, lane);
        const float2 pv = __ldcg(reinterpret_cast<const float2*>(a.p + ((size_t)kk * a.T) * 2));
        in[NX] = pv.x; in[NX + 1] = pv.y;
      }
      float cost_acc = 0.0f;
      float rd = 0.0f, rs = 0.0f;  // kPerRow: this sample's pi eps / T and exp(gamma t) / T (torchlaplace Fourier constants)
      if (kPerRow) {
        const float tn = a.row_tn[kk];
        const float Tt = 2.0f * (tn + 1.0e-6f);
        rd = 3.14159265358979f * 1.0e-6f / Tt;
        rs = expf((1.0e-3f + 4.605170185988091f / Tt) * tn) / Tt;
      }

      for (int t = 0; t < a.T; ++t) {
        float2 pnext = make_float2(0.f, 0.f);
        if (!a.ready && t + 1 < a.T) pnext = __ldcg(reinterpret_cast<const float2*>(a.p + ((size_t)kk * a.T + t + 1) * 2));

        // ---------------- A1 = [in | 1 | 0..] as the K = 16 operand (one thread per sample) ----------------
        if (cg == 0 && active) {
          f2_t v[8];
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            // the constant-1 column multiplies the folded first-layer bias; with per-sample times the bias comes in E1 instead
            const float one = kPerRow ? 0.0f : 1.0f;
            const float x0 = (2 * i < Lp) ? in[2 * i < Lp ? 2 * i : 0] : (2 * i == Lp ? one : 0.0f);
            const float x1 = (2 * i + 1 < Lp) ? in[2 * i + 1 < Lp ? 2 * i + 1 : 0] : (2 * i + 1 == Lp ? one : 0.0f);
            v[i] = pk2(x0, x1);
          }
          uint32_t ph[8], pl[8];
          pack16<kSplit3>(v, ph, pl);
          tmem_st8(tA, ph);
          if (kSplit3) tmem_st8(tA + kALo, pl);
        }
        mark(0);
        issue(0);
        // ---------------- E1: tanh -> A ----------------
        wait_mma();
        mark(1);
        active_w = active;
        hidden_split(1, kPerRow ? 2 : 0, kk);
        mark(2);
        // ---------------- E2: + b2, tanh -> A ----------------
        wait_mma();
        mark(3);
        hidden_split(2, 1, kk);
        mark(4);
        // overlapped form: the next step's encoder output, polled for and loaded under the L3 product
        if (a.ready && t + 1 < a.T) {
          wait_windows_ready(a, t + 1, lane);
          pnext = __ldcg(reinterpret_cast<const float2*>(a.p + ((size_t)kk * a.T + t + 1) * 2));
        }
        // cost of the previous step's state while the MMA runs (mppi_delay.py:288-290)
        if (cg == 0 && t > 0 && a.cost_total && live)
          cost_acc += env_running_cost_fast(a.o, st, a.hist + ((size_t)kk * a.L + (t - 1) + a.B - 1) * a.nu, a.nu);
        // ---------------- E3: sphere -> complex, Fourier weights, sum over the terms ----------------
        float delta[NX];
#pragma unroll
        for (int c = 0; c < NX; ++c) delta[c] = 0.0f;
        wait_mma();
        mark(5);
        // the first half's product has read the W3 buffer: the second half streams in under this epilogue
        if (kStream && warp == 0 && elect_one()) load_w3_rows<kH>(a.m, w3_img, N3a, N3b, N3t, N3buf, &s.bar_w3);
        const uint32_t tDcg = tD + 8 * cg;
        const float *b3cg = s.b3 + 8 * cg, *phcg = s.phase + cg, *wtcg = s.weight + cg;
        if constexpr (kSplitD) {
          // this thread's units of the first product, then (after the second product's own barrier) of the second
          if (active) L3GU<NX, S, 0, kUnitsH, 0, kSplit3, kRcp % 10, kPerRow>::run(tDcg, b3cg, phcg, wtcg, cg, delta, rd, rs);
          mbar_wait_sleep(&s.done[1], n_b & 1); ++n_b;
          fence_after_sync();
          if (active) L3GU<NX, S, kUnitsH, kUnits, 0, kSplit3, kRcp % 10, kPerRow>::run(tDcg, b3cg, phcg, wtcg, cg, delta, rd, rs);
        } else {
          if (active) L3GU<NX, S, 0, kUnitsA, 0, kSplit3, kRcp % 10, kPerRow>::run(tDcg, b3cg, phcg, wtcg, cg, delta, rd, rs);
        }
        if constexpr (kStream) {
          mark(6);
          issue(3);
          wait_mma();
          mark(7);
          // ... and the first half again for the next step (or the next tile), under this epilogue and the next step's E1 / E2
          if (warp == 0 && elect_one()) load_w3_rows<kH>(a.m, w3_img, 0, N3a, N3t, N3buf, &s.bar_w3);
          // the second half's units, now in column 0.. of the D region
          if (active) L3GU<NX, S, kUnitsA, kUnits, kUnitsA, kSplit3, kRcp % 10, kPerRow>::run(tDcg, b3cg, phcg, wtcg, cg, delta, rd, rs);
        }
#pragma unroll
        for (int c = 0; c < NX; ++c) s.exch[cg][row * NX + c] = delta[c];
        asm volatile("bar.sync %0, %1;" ::"r"(1), "n"(kThreads) : "memory");
        // every thread of a sample adds the partials in the same order: the replicated state stays bit-identical
#pragma unroll
        for (int c = 0; c < NX; ++c) {
          float d = s.exch[0][row * NX + c];
#pragma unroll
          for (int j = 1; j < 4; ++j) d += s.exch[j][row * NX + c];
          st[c] += d;                                             // mppi_with_model.py:121
          in[c] = (st[c] - s.smean[c]) * s.sinv[c];
          if (cg == 3 && live) {
            if (a.states) a.states[((size_t)kk * a.T + t) * NX + c] = st[c];
            if (a.delta_out) a.delta_out[(size_t)kk * NX + c] = d;
          }
        }
        in[NX] = pnext.x; in[NX + 1] = pnext.y;
        ++tstep;
        // exch is rewritten only after the next step's MMA round trips, which need every warp
      }
      if (cg == 0 && live && a.cost_total) {
        cost_acc += env_running_cost_fast(a.o, st, a.hist + ((size_t)kk * a.L + (a.T - 1) + a.B - 1) * a.nu, a.nu);
        a.cost_total[kk] = cost_acc + (a.pert_cost ? a.pert_cost[kk] : 0.0f);
      }
    }
    // the last streamed half (requested for a step that never comes) must have landed before the CTA's shared memory goes
    if (kStream && warp == 0) mbar_wait(&s.bar_w3, n_w3 & 1);
  }
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kTmemCols);
}

// ======================================  ping-pong form  ======================================
// Two 128-sample tiles per CTA, and ALL 16 warps work on ONE tile's epilogue at a time and alternate between the tiles
// phase by phase:
//     E1x E1y  E2x E2y  E3ax E3ay  E3bx E3by  Ux Uy        (x, y = the two tiles;  U = state update + next A1)
// Every product (M2, M3a, M3b, M1 of the next step) is issued at the end of its tile's phase and has the whole following
// phase of the OTHER tile to complete, so the CUDA cores never wait for the tensor pipe and every SM sub-partition always
// has its four warps in the same instruction mix.  Its predecessor ran the two tiles as two free-running 8-warp groups,
// which left each tile two warps per sub-partition (latency-bound epilogues: 33.5 k clocks per step of a tile pair at
// config 4, issue slots 40 % busy).
//   hand-off   a dedicated MMA warp (warp 16): an epilogue warp arrives on the tile's NAMED barrier (bar.arrive: it does not
//              block) after its TMEM stores and moves on to the other tile's phase; the MMA warp waits for the 16 arrivals
//              (bar.sync), issues the product under elect.sync and commits it to the mbarrier done[tile], which the epilogue
//              warps wait on one phase later.  (tcgen05.mma issue is back-pressured by MMA execution: with one of the
//              epilogue warps issuing - even a different one every time - that warp falls behind by the whole product and
//              the next hand-off waits for it: 43.9 k clocks per step, nothing overlapped.)  The register file cannot hold
//              17 warps at 128 registers, so the CTA is launched with 20 warps at 96 and re-balanced with setmaxnreg: 112
//              for the epilogue warps, 32 for the MMA warp's group (whose issue code is a non-inlined, fully unrolled
//              function so that it fits that budget).
//   threads    warp w: TMEM lanes 32 (w & 3).. (its 32 samples of BOTH tiles), column group w >> 2 (32 of the 128 hidden
//              units; of every 32-column unit of the group-uniform (theta, phi) order, columns 8 cg .. 8 cg + 7).  The state of a sample is replicated in its four
//              threads; partial ILT sums are exchanged through shared memory among the four warps of a row quarter.
//   L3         first half = the first four units (128 columns), second half the rest (<= 128): A 128 + D 128 columns per tile.
//   rows       a CTA owns one contiguous row range and walks it 256 rows (two tiles) per pass (the overlapped step: one
//              256-row block per pass, pass-major over the grid); a tile without rows in a pass keeps its hand-offs (the MMA
//              warp's product sequence is fixed) but skips every epilogue.
template <int NX>
struct SmemTailPP {
  alignas(8) uint64_t bar_w;
  alignas(16) float b2[kMaxH];
  alignas(16) float b3[256];
  float phase[kMaxS], weight[kMaxS];
  float smean[kMaxNx], sinv[kMaxNx];
  alignas(16) float exch[2][4][NX * kRows];  // [tile][column group][channel][row] partial ILT sums
  alignas(8) float stage_p[2][kRows][2];     // cp.async landing slots: p_action of the next step ...
  alignas(8) float stage_u[2][2][kRows][2];  // ... and the action this step applies (running cost): [step parity][tile][sample]
  alignas(8) uint64_t done[2];
  uint32_t tmem_base;
};
constexpr int kThreadsPP = kThreads + 128;    // 16 epilogue warps + the MMA warp's group (setmaxnreg works on groups of 4 warps)

template <int H, int NX, int S, bool kSplit3, int kRcp>
__global__ void __launch_bounds__(kThreadsPP, 1) rollout_pp_kernel(Args a) {
  extern __shared__ __align__(128) unsigned char smem_raw[];
  constexpr int Lp = NX + 2;
  constexpr int kH = H, kChunks = H / 64;  // 16-column chunks of hidden units per thread
  constexpr uint32_t kSbo = kSboH<H>, kALo = H / 2, kColD = H;
  // the (theta, phi) columns in the group-uniform order (l3_units_gu): units of 32 columns, the first four in the first half
  constexpr int kUnits = PPShape<NX, S>::kUnits, N3t = PPShape<NX, S>::N3u;
  constexpr int kUnitsA = kUnits < 4 ? kUnits : 4;
  constexpr int N3a = 32 * kUnitsA, N3b = N3t - N3a;
  static_assert(N3b <= 128 && N3t <= 256 && Lp + 1 <= 16, "tile shape");
  unsigned char* w1_img = smem_raw;                                   // [hi | lo] 128 x 16 halves = 4 KB each
  unsigned char* w2_img = w1_img + 2 * kH * 16 * 2;                   // [hi | lo] 32 KB each
  unsigned char* w3_img = w2_img + 2 * kH * kH * 2;                   // [hi | lo] N3t * 256 B each
  SmemTailPP<NX>& s = *reinterpret_cast<SmemTailPP<NX>*>(w3_img + 2 * (size_t)N3t * kH * 2);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (a.trace && blockIdx.x == 0 && lane == 0 && warp < 16) a.trace[(51 * 16 + warp) * 16 + 0] = clock64();
  const long long cta_t0 = clock64();
  unsigned long long cta_g0;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(cta_g0));

  {
    if (warp == 0 && elect_one()) {  // weight images by TMA bulk copies; only the MMA warp waits for them (see rollout_tc2_kernel)
      mbar_init(&s.bar_w, 1);
      mbar_fence_init();
      load_weight_images<kH>(a.m, w1_img, w2_img, w3_img, N3t, &s.bar_w);
    }
    for (int i = tid; i < kH; i += kThreadsPP) s.b2[i] = a.m.mlp2_b2[i];
    for (int i = tid; i < 256; i += kThreadsPP) s.b3[i] = i < N3t ? a.m.mlp2_b3[i] : 0.0f;
    for (int i = tid; i < S; i += kThreadsPP) { s.phase[i] = a.m.ilt_phase[i]; s.weight[i] = a.m.ilt_weight[i]; }
    if (tid < NX) { s.smean[tid] = a.m.state_mean[tid]; s.sinv[tid] = a.m.state_inv_std[tid]; }
    for (int i = tid; i < 2 * 2 * kRows * 2; i += kThreadsPP) (&s.stage_u[0][0][0][0])[i] = 0.0f;
    if (tid == 0) {
      for (int g = 0; g < 2; ++g) mbar_init(&s.done[g], 1);
      mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&s.tmem_base, kTmemCols);
  }
  fence_proxy_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = s.tmem_base;

  const int q = warp & 3, cg = warp >> 2;
  const int row = 32 * q + lane;
  const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
  const uint32_t w1_hi = smem_u32(w1_img), w1_lo = w1_hi + kH * 16 * 2;
  const uint32_t w2_hi = smem_u32(w2_img), w2_lo = w2_hi + kH * kH * 2;
  const uint32_t w3_hi = smem_u32(w3_img), w3_lo = w3_hi + (uint32_t)N3t * kH * 2;
  const uint32_t w3b_off = (uint32_t)(N3a / 8) * kSbo;

  // samples of this CTA: one contiguous range, a multiple of 32 rows long (except at the end of the plan), walked 256 rows
  // (two tiles) per pass.  A last pass of at most 128 rows has ONE live tile: the other tile's phases are skipped and the pass
  // costs a one-tile chain instead of a full ping-pong pass (config 5's 352-tile groups: 0.80 -> 0.69 ms per rollout).
  // Overlapped step (a.ready): pass-major instead - pass q of CTA c covers samples [(q * grid + c) * 256, + 256), so that every
  // pass but the last reads windows the planner encoded before this launch, and only the last pass (samples from
  // (passes - 1) * grid * 256 on, the encoder's step-major sub-plan) polls the readiness counters.
  const int per_cta = ((a.K + (int)gridDim.x - 1) / (int)gridDim.x + 31) / 32 * 32;
  const int pass_rows = 2 * kRows * (int)gridDim.x;
  const int n_iter = a.ready ? (a.K + pass_rows - 1) / pass_rows : (per_cta + 2 * kRows - 1) / (2 * kRows);
  const long long cta_b = (long long)blockIdx.x * per_cta;
  const int cta_begin = (int)(cta_b < a.K ? cta_b : a.K);
  const int cta_end = (cta_begin + per_cta < a.K) ? cta_begin + per_cta : a.K;

  if (warp >= 16) {
    // =====================================  MMA warp (and the rest of its register group)  =====================================
    asm volatile("setmaxnreg.dec.sync.aligned.u32 32;");
    if (warp == 16) {
      // products in the epilogue warps' hand-off order, the two tiles strictly alternating: (M1x M1y) then per step
      // (M2x M2y M3ax M3ay [M3bx M3by] M1x' M1y').  ONE issuing warp on purpose: with a warp per tile the two M2 products
      // interleave on the tensor pipe and the one needed first completes last.
      mbar_wait(&s.bar_w, 0);    // weight images landed
      int mstep = 0, mprod = 0;  // measurement only: the MMA warp's own timeline, second half of the trace buffer
      auto product = [&](int x, int ev) {
        // named barrier 1 + x: the 16 epilogue warps bar.arrive, this warp bar.sync (as an mbarrier, every one of the 16
        // arrivals woke all warps sleeping in try_wait loops: a quarter of the executed instructions were SYNCS/NANOSLEEP/BRA)
        asm volatile("bar.sync %0, %1;" ::"r"(1 + x), "n"(kThreads + 32) : "memory");
        if (lane == 0 && a.trace && blockIdx.x == 0 && mstep < 51 && mprod < 8) a.trace[52 * 256 + mstep * 256 + 2 * mprod] = clock64();
        __syncwarp();
        const uint32_t tg = tmem + kGroupCols * x;
        uint64_t* done = &s.done[x];
        if (ev == 0) issue_gemm_ts_fn<1, kSplit3, kALo>(tg + kColD, tg + kColA, smem_desc(w1_hi, kLbo, kSbo16), smem_desc(w1_lo, kLbo, kSbo16), idesc_f16_f32(kRows, kH), done);
        else if (ev == 1) issue_gemm_ts_fn<kH / 16, kSplit3, kALo>(tg + kColD, tg + kColA, smem_desc(w2_hi, kLbo, kSbo), smem_desc(w2_lo, kLbo, kSbo), idesc_f16_f32(kRows, kH), done);
        else if (ev == 2) issue_gemm_ts_fn<kH / 16, kSplit3, kALo>(tg + kColD, tg + kColA, smem_desc(w3_hi, kLbo, kSbo), smem_desc(w3_lo, kLbo, kSbo), idesc_f16_f32(kRows, N3a), done);
        else issue_gemm_ts_fn<kH / 16, kSplit3, kALo>(tg + kColD, tg + kColA, smem_desc(w3_hi + w3b_off, kLbo, kSbo), smem_desc(w3_lo + w3b_off, kLbo, kSbo),
                                                      idesc_f16_f32(kRows, N3b > 0 ? N3b : 16), done);
        if (lane == 0 && a.trace && blockIdx.x == 0 && mstep < 51 && mprod < 8) a.trace[52 * 256 + mstep * 256 + 2 * mprod + 1] = clock64();
        ++mprod;
      };
      constexpr int kPerStep = N3b > 0 ? 8 : 6;
#pragma unroll 1
      for (int it = 0; it < n_iter; ++it) {
        const int n_products = kPerStep * a.T;   // 2 + kPerStep T - 2: no M1 pair after the last step
#pragma unroll 1
        for (int i = 0; i < n_products; ++i) {
          const int j = i < 2 ? i : (i - 2) % kPerStep;  // position inside the prologue / the step
          const int ev = i < 2 ? 0 : ((j >> 1) + 1 == kPerStep / 2 ? 0 : (j >> 1) + 1);
          if (i >= 2 && j == 0) { ++mstep; mprod = 0; }
          product(i & 1, ev);
        }
      }
    }
  } else {
  // =====================================  epilogue warps  =====================================
  asm volatile("setmaxnreg.inc.sync.aligned.u32 112;");
  // The tile loops below are NOT unrolled (`x` is a run-time value; per-tile register state is reached through selects):
  // unrolled, the step loop was 166 KB of instructions, more than the SM's instruction cache holds - CTAs then ran
  // 14-20 % slower the further their TPC sits from the GPC's instruction path (tools/trace_rollout_pp.py, per-CTA spans).
  int tstep = 0;
  // measurement only (tools/trace_rollout_pp.py): clock64 timeline of CTA 0, [step < 51][warp][16 events]
  auto mark = [&](int ev) {
    if (a.trace && blockIdx.x == 0 && lane == 0 && tstep < 51) a.trace[(tstep * 16 + warp) * 16 + ev] = clock64();
  };
  if (a.trace && blockIdx.x == 0 && lane == 0) a.trace[(51 * 16 + warp) * 16 + 1] = clock64();
  uint32_t nphase = 0;  // products of each tile waited for so far (the two tiles wait once each per phase)
  // this warp's TMEM stores / loads of the phase are done: the MMA warp issues tile x's next product after all 16 arrivals
  auto handoff = [&](int x) {
    tmem_st_wait();
    fence_before_sync();
    asm volatile("bar.arrive %0, %1;" ::"r"(1 + x), "n"(kThreads + 32) : "memory");
  };
  auto wait_mma = [&](int x) {
    mbar_wait_sleep(&s.done[x], nphase & 1u);
    fence_after_sync();
  };

  for (int it = 0; it < n_iter; ++it) {
    // rows [pass_begin, pass_end) of this pass; `poll`: the encoder may still be writing their windows
    int pass_begin = cta_begin + 2 * it * kRows, pass_end = cta_end;
    if (a.ready) {
      pass_begin = min((it * (int)gridDim.x + (int)blockIdx.x) * (2 * kRows), a.K);
      pass_end = pass_begin + 2 * kRows < a.K ? pass_begin + 2 * kRows : a.K;
    }
    const bool poll = a.ready && it + 1 == n_iter;
    // per-tile state: sample index, liveness bits (bit x), state and cost accumulator of both tiles
    int kk0, kk1, amask = 0, lmask = 0;
    float st0[NX], st1[NX], cost0 = 0.0f, cost1 = 0.0f;
#pragma unroll
    for (int x = 0; x < 2; ++x) {
      const int tile0 = pass_begin + x * kRows;
      int nr = pass_end - tile0;
      nr = nr < 0 ? 0 : (nr > kRows ? kRows : nr);
      if (32 * q < nr) amask |= 1 << x;     // warp-uniform: this warp has at least one live sample of tile x
      if (row < nr) lmask |= 1 << x;
      const int k = row < nr ? tile0 + row : pass_end - 1;
      const float* sp = a.state0 + (size_t)(a.state_per_sample ? k / a.state_per_sample : 0) * NX;
#pragma unroll
      for (int c = 0; c < NX; ++c) { if (x == 0) st0[c] = sp[c]; else st1[c] = sp[c]; }
      if (x == 0) kk0 = k; else kk1 = k;
      if (cg == 2) {
        // (last pass of the overlapped step: p is being written by the encoder beside this kernel - wait for step 0's windows,
        // read through L2)
        if (poll) wait_windows_ready(a, 0, lane);
        *reinterpret_cast<float2*>(&s.stage_p[x][row][0]) = __ldcg(reinterpret_cast<const float2*>(a.p + ((size_t)k * a.T) * 2));
      }
    }
    // A1 = [obs_n | p_action | 1 | 0..] as the K = 16 operand of the first layer (one thread per sample: column group 2);
    // p_action comes from this thread's own stage_p slot
    auto write_a1 = [&](int x, const float (&stx)[NX]) {
      if (cg == 2 && ((amask >> x) & 1)) {
        float in[Lp];
#pragma unroll
        for (int c = 0; c < NX; ++c) in[c] = (stx[c] - s.smean[c]) * s.sinv[c];
        const float2 pc = *reinterpret_cast<const float2*>(&s.stage_p[x][row][0]);
        in[NX] = pc.x; in[NX + 1] = pc.y;
        f2_t v[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float x0 = (2 * i < Lp) ? in[2 * i < Lp ? 2 * i : 0] : (2 * i == Lp ? 1.0f : 0.0f);
          const float x1 = (2 * i + 1 < Lp) ? in[2 * i + 1 < Lp ? 2 * i + 1 : 0] : (2 * i + 1 == Lp ? 1.0f : 0.0f);
          v[i] = pk2(x0, x1);
        }
        uint32_t ph[8], pl[8];
        pack16<kSplit3>(v, ph, pl);
        const uint32_t tA = tlane + kGroupCols * x + kColA;
        tmem_st8(tA, ph);
        if (kSplit3) tmem_st8(tA + kALo, pl);
      }
    };
    // hidden layer epilogue: (+ bias,) tanh, re-written as the fp16 hi/lo A operand of the next layer
    auto hidden = [&](int x, bool with_bias) {
      const uint32_t tA = tlane + kGroupCols * x + kColA, tD = tlane + kGroupCols * x + kColD;
      if ((amask >> x) & 1) {
        f2_t vv[kChunks][8];
        ldtm16p(tD + 16 * kChunks * cg, vv[0]);
        if constexpr (kChunks == 2) ldtm16p(tD + 32 * cg + 16, vv[kChunks - 1]);
        tmem_ld_wait();
#pragma unroll
        for (int c16 = 0; c16 < kChunks; ++c16) {
          const int n0 = 16 * kChunks * cg + 16 * c16;
          f2_t (&v)[8] = vv[c16];
          if (with_bias) {
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const float4 b = *reinterpret_cast<const float4*>(s.b2 + n0 + 4 * i);
              v[2 * i] = add2(v[2 * i], pk2(b.x, b.y));
              v[2 * i + 1] = add2(v[2 * i + 1], pk2(b.z, b.w));
            }
          }
          tanh16_scaled<kSplit3, kRcp / 10>(v);
          uint32_t ph[8], pl[8];
          pack16<kSplit3>(v, ph, pl);
          tmem_st8(tA + n0 / 2, ph);
          if (kSplit3) tmem_st8(tA + kALo + n0 / 2, pl);
        }
      }
    };
    // first (kHalf == 0) or second half of the (theta, phi) columns: this thread's units -> partial sums in shared memory
    auto l3_half = [&](int x, auto half_tag) {
      constexpr int kHalf = decltype(half_tag)::value;
      constexpr int kBeg = kHalf == 0 ? 0 : kUnitsA, kEnd = kHalf == 0 ? kUnitsA : kUnits;
      const uint32_t tD = tlane + kGroupCols * x + kColD;
      float delta[NX];
#pragma unroll
      for (int c = 0; c < NX; ++c) delta[c] = 0.0f;
      if constexpr (kBeg < kEnd) {
        if ((amask >> x) & 1)
          l3_units_gu<NX, S, kBeg, kEnd, kSplit3, kRcp % 10>(tD + 8 * cg, s.b3 + 8 * cg, s.phase + cg, s.weight + cg, cg, delta);
      }
      float* e = &s.exch[x][cg][row];
#pragma unroll
      for (int c = 0; c < NX; ++c) e[c * kRows] = (kHalf == 0) ? delta[c] : e[c * kRows] + delta[c];
    };

    // duties of step tt's END state that nothing waits for - its row of `states` (column group 2) and its running cost
    // (column group 3; mppi_delay.py:288-290: the post-step state with the action just applied) - are carried out one
    // step later, behind these groups' units of the last L3 phase: after the state update they would delay the next step's M1
    // (measured at config 4 with the group-uniform units: here 1.325 ms, before the E2 wait 1.333, before the E1 wait 1.378)
    auto deferred = [&](int x, int tt) {
      const int kx = x ? kk1 : kk0;
      if (!((lmask >> x) & 1)) return;
      if (cg == 2 && a.states) {
#pragma unroll
        for (int c = 0; c < NX; ++c) a.states[((size_t)kx * a.T + tt) * NX + c] = x ? st1[c] : st0[c];
      }
      if (cg == 3 && a.cost_total) {
        const float2 uv = *reinterpret_cast<const float2*>(&s.stage_u[tt & 1][x][row][0]);
        const float uc[2] = {uv.x, uv.y};   // zero-padded for nu == 1: a static count keeps the action in registers
        float stx[NX];
#pragma unroll
        for (int c = 0; c < NX; ++c) stx[c] = x ? st1[c] : st0[c];
        const float c = env_running_cost_fast(a.o, stx, uc, 2);
        if (x) cost1 += c; else cost0 += c;
      }
    };

    write_a1(0, st0); handoff(0);
    write_a1(1, st1); handoff(1);

    for (int t = 0; t < a.T; ++t) {
      // operands of the END of this step - the next step's p_action (column group 2) and the action this step applies, for
      // the running cost (column group 3) - start their way now as cp.async copies into per-sample shared-memory slots:
      // no registers held across the step (held in registers they were spilled right after the load, and the spill
      // store stalled the warp on the load at the top of every step)
      // Last pass of the overlapped step (`poll`: the encoder runs beside this kernel and publishes its windows step by step):
      // the 128-byte line of p(k, t+1) also holds later steps that are not written yet, so it must not pass through L1 -
      // ld.global.cg into two registers per tile once step t+1 is published, stored into the landing slot before the exchange
      // barrier below.  The poll and the load are issued behind the E1 hand-offs, where these warps wait for the M2 products
      // anyway: at the top of the step their two dependent L2 round trips delayed E1 of every step.  Earlier passes read
      // windows encoded before the launch; a pass is a 256-sample block, so none of their lines of p (2048 T bytes per block)
      // holds a window of the polled pass.
      float2 pn0 = make_float2(0.f, 0.f), pn1 = make_float2(0.f, 0.f);
#pragma unroll 1
      for (int x = 0; x < 2; ++x) {
        const int kx = x ? kk1 : kk0;
        if (!poll && cg == 2 && t + 1 < a.T)
          asm volatile("cp.async.ca.shared.global [%0], [%1], 8;" ::"r"(smem_u32(&s.stage_p[x][row][0])), "l"(a.p + ((size_t)kx * a.T + t + 1) * 2) : "memory");
        if (cg == 3 && ((lmask >> x) & 1) && a.cost_total) {
          const float* up = a.hist + ((size_t)kx * a.L + t + a.B - 1) * a.nu;
          asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(&s.stage_u[t & 1][x][row][0])), "l"(up) : "memory");
          if (a.nu > 1) asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(smem_u32(&s.stage_u[t & 1][x][row][1])), "l"(up + 1) : "memory");
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
      mark(11);
#pragma unroll 1
      for (int x = 0; x < 2; ++x) { wait_mma(x); mark(0 + x); hidden(x, false); handoff(x); }   // E1 -> M2
      ++nphase;
      if (poll && cg == 2 && t + 1 < a.T) {
        wait_windows_ready(a, t + 1, lane);
        pn0 = __ldcg(reinterpret_cast<const float2*>(a.p + ((size_t)kk0 * a.T + t + 1) * 2));
        pn1 = __ldcg(reinterpret_cast<const float2*>(a.p + ((size_t)kk1 * a.T + t + 1) * 2));
      }
      mark(12);
#pragma unroll 1
      for (int x = 0; x < 2; ++x) { wait_mma(x); mark(2 + x); hidden(x, true); handoff(x); }    // E2 -> M3a
      ++nphase;
      mark(13);
#pragma unroll 1
      for (int x = 0; x < 2; ++x) {                                                             // E3a (-> M3b)
        wait_mma(x);
        mark(4 + x);
        l3_half(x, std::integral_constant<int, 0>());
        if (N3b > 0) handoff(x);
        else if (t > 0) {
          if (x == 0) asm volatile("cp.async.wait_group 1;" ::: "memory");  // the copies of the previous step (this thread's own)
          deferred(x, t - 1);
        }
      }
      ++nphase;
      if (N3b > 0) {
        mark(14);
#pragma unroll 1
        for (int x = 0; x < 2; ++x) {                                                           // E3b
          wait_mma(x);
          mark(6 + x);
          l3_half(x, std::integral_constant<int, 1>());
          if (t > 0) {
            if (x == 0) asm volatile("cp.async.wait_group 1;" ::: "memory");  // the copies of the previous step (this thread's own)
            deferred(x, t - 1);
          }
        }
        ++nphase;
      }
      mark(15);
      if (poll && cg == 2 && t + 1 < a.T) {
        *reinterpret_cast<float2*>(&s.stage_p[0][row][0]) = pn0;
        *reinterpret_cast<float2*>(&s.stage_p[1][row][0]) = pn1;
      }
      asm volatile("cp.async.wait_group 0;" ::: "memory");  // this thread's own copies: it reads only its own slots
      // ONE barrier among the four warps of a row quarter covers the partial sums of both tiles (tile 1's were written last)
      asm volatile("bar.sync %0, %1;" ::"r"(5 + q), "n"(128) : "memory");
      mark(8);
#pragma unroll 1
      for (int x = 0; x < 2; ++x) {                                                   // U: residual, next A1 -> M1
        // every thread of a sample adds the partials in the same order: the replicated state stays bit-identical
        float stx[NX];
#pragma unroll
        for (int c = 0; c < NX; ++c) {
          const float* e = &s.exch[x][0][c * kRows + row];
          const float d = ((e[0] + e[NX * kRows]) + e[2 * NX * kRows]) + e[3 * NX * kRows];
          stx[c] = (x ? st1[c] : st0[c]) + d;                     // mppi_with_model.py:121
          if (x) st1[c] = stx[c]; else st0[c] = stx[c];
          if (cg == 2 && ((lmask >> x) & 1) && a.delta_out) a.delta_out[(size_t)(x ? kk1 : kk0) * NX + c] = d;
        }
        if (t + 1 < a.T) {
          write_a1(x, stx);
          handoff(x);
        }
        mark(9);
      }
      mark(10);
      ++tstep;
    }
    deferred(0, a.T - 1);   // the last step's state: its copies were waited for in the U phase
    deferred(1, a.T - 1);
    if (cg == 3 && a.cost_total) {
      if (lmask & 1) a.cost_total[kk0] = cost0 + (a.pert_cost ? a.pert_cost[kk0] : 0.0f);
      if (lmask & 2) a.cost_total[kk1] = cost1 + (a.pert_cost ? a.pert_cost[kk1] : 0.0f);
    }
  }
  if (a.trace && blockIdx.x == 0 && lane == 0) a.trace[(51 * 16 + warp) * 16 + 2] = clock64();
  }  // epilogue warps
  fence_before_sync();
  __syncthreads();
  if (a.trace && tid == 0) {  // measurement only: every CTA's own span and SM
    uint32_t smid;
    asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
    unsigned long long g1;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(g1));
    a.trace[2 * 52 * 256 + 4 * blockIdx.x] = clock64() - cta_t0;
    a.trace[2 * 52 * 256 + 4 * blockIdx.x + 1] = smid;
    a.trace[2 * 52 * 256 + 4 * blockIdx.x + 2] = (long long)cta_g0;
    a.trace[2 * 52 * 256 + 4 * blockIdx.x + 3] = (long long)g1;
  }
  if (warp == 0) tmem_dealloc(tmem, kTmemCols);
}

template <int kH, int NX, int S, bool kSplit3, int kRcp>
static int launch_pp(const Args& a, cudaStream_t stream) {
  constexpr int N3t = PPShape<NX, S>::N3u;
  const size_t smem = 2 * (size_t)kH * 16 * 2 + 2 * (size_t)kH * kH * 2 + 2 * (size_t)N3t * kH * 2 + sizeof(SmemTailPP<NX>) + 128;
  NLC_REQUIRE(smem <= 227 * 1024, NLC_ERR_SHAPE, "tcgen05 rollout: %zu bytes of shared memory needed", smem);
  auto kern = rollout_pp_kernel<kH, NX, S, kSplit3, kRcp>;
  NLC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  int grid = (a.K + 63) / 64;   // at least one warp of samples per tile slot, at most one CTA per SM
  if (grid > 148) grid = 148;
  // overlapped planner step: whole 128-sample tiles, two per CTA, on as few SMs as possible - the encoder runs on the others
  if (a.ready) grid = pp_overlap_grid((a.K + kRows - 1) / kRows);
  kern<<<grid, kThreadsPP, smem, stream>>>(a);
  NLC_LAUNCH_OK("rollout_pp_kernel");
  return NLC_OK;
}

template <int kH, int NX, int S, bool kSplit3, int kRcp, bool kPerRow = false>
static int launch_one_t(const Args& a, cudaStream_t stream) {
  constexpr int kUnits = PPShape<NX, S>::kUnits, N3t = PPShape<NX, S>::N3u;
  constexpr int N3buf = kH == 128 && N3t > 256 ? 32 * ((kUnits + 1) / 2) : N3t;  // streamed W3: one half resident
  const size_t smem = 2 * (size_t)kH * 16 * 2 + 2 * (size_t)kH * kH * 2 + 2 * (size_t)N3buf * kH * 2 + sizeof(SmemTail) + 128;
  NLC_REQUIRE(smem <= 227 * 1024, NLC_ERR_SHAPE, "tcgen05 rollout: %zu bytes of shared memory needed", smem);
  auto kern = rollout_tc2_kernel<kH, NX, S, kSplit3, kRcp, kPerRow>;
  NLC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  // one tile per 32..128 samples: enough CTAs to give every tile at least one warp of samples, at most one per SM
  int grid = (a.K + 31) / 32;
  if (grid > 148) grid = 148;
  // overlapped planner step: whole 128-sample tiles on as few SMs as possible - the encoder runs on the others
  if (a.ready) grid = (a.K + kRows - 1) / kRows;
  kern<<<grid, kThreads, smem, stream>>>(a);
  NLC_LAUNCH_OK("rollout_tc2_kernel");
  return NLC_OK;
}

// tiles == 3: the ping-pong form (plans of more than one wave of 128-sample tiles), else one tile on all 16 warps
template <int kH, int NX, int S, bool kSplit3, int kRcp>
static int launch_one(const Args& a, int tiles, cudaStream_t stream) {
  if (a.row_b1) {  // per-sample prediction times: the one-tile form's kPerRow instantiation (fp32-class arithmetic only)
    if constexpr (kSplit3) return launch_one_t<kH, NX, S, true, kRcp, true>(a, stream);
    else return NLC_ERR_UNSUPPORTED;
  }
  if constexpr (2 * NX * S > 256) {
    // more (theta, phi) columns than the ping-pong form's accumulators hold: the one-tile form (with W3 streamed at H = 128),
    // whatever the plan size
    return launch_one_t<kH, NX, S, kSplit3, kRcp>(a, stream);
  } else {
    return tiles == 3 ? launch_pp<kH, NX, S, kSplit3, kRcp>(a, stream) : launch_one_t<kH, NX, S, kSplit3, kRcp>(a, stream);
  }
}

}  // namespace rt2

// both MLP widths the model accepts (128 and 64) have every (nx, S) pair below
bool rollout_has_tensor_core_form(const nlc_model_s* m) {
  return (m->S == 17 || m->S == 33) && (m->nx == 3 || m->nx == 5 || m->nx == 6);
}

// returns NLC_ERR_UNSUPPORTED when the (nx, S) pair has no tensor-core instantiation (caller falls back)
static long long* g_roll_trace = nullptr;
void set_rollout_trace(long long* p) { g_roll_trace = p; }

int launch_rollout_tc2(nlc_model_s* m, const nlc_rollout_opts* o, const float* state, int sps, const float* p,
                       const float* hist, const float* pert_cost, int K, int T, int B, int nu, float* cost, float* states,
                       float* delta_out, int split3, int tiles_per_cta, cudaStream_t stream, const unsigned int* ready,
                       unsigned int ready_target, unsigned int* status, const float* row_b1, const float* row_tn) {
  rt2::Args a;
  a.ready = ready; a.ready_target = ready_target; a.status = status;
  a.row_b1 = row_b1; a.row_tn = row_tn;
  NLC_REQUIRE(!row_b1 || (row_tn && split3 && !ready), NLC_ERR_ARG, "rollout: per-sample times need row_tn and the fp32-class tensor-core mode");
  if (2 * m->nx * m->S > 256) tiles_per_cta = 1;
  NLC_REQUIRE(m->N3u == 32 * (m->nx * ((m->S - 1) / 16) + 1), NLC_ERR_SHAPE,
              "tcgen05 rollout: the model holds no group-uniform W3 image for nx=%d S=%d", m->nx, m->S);
  NLC_REQUIRE(!ready || (status && ((tiles_per_cta == 1 && (K + 127) / 128 <= 148) || tiles_per_cta == 3)), NLC_ERR_ARG,
              "rollout: the overlapped forms are the one-tile form of plans within one wave and the ping-pong form");
  a.m = m->d; a.o = *o; a.state0 = state; a.state_per_sample = sps; a.p = p; a.hist = hist; a.pert_cost = pert_cost;
  a.K = K; a.T = T; a.B = B; a.L = B - 1 + T; a.nu = nu; a.cost_total = cost; a.states = states; a.delta_out = delta_out;
  a.trace = g_roll_trace;
  // reciprocal flavour of the fp32-class epilogues: Newton on the FMA pipe for both the MLP tanh and the L3 pair ("33").
  // Ping-pong form at config 4: 1.412 ms; MUFU for the L3 pair ("30") 1.447, for the tanh ("03") 1.427, for both ("00") 1.466
  // (round 2; round 1 measured 1.71 vs 1.85 ms with the ping-pong form's two-group predecessor, profiles/r1_rollout_sweep.md)
#define NLC_RT2_CASE(NX_, S_)                                                                   \
  if (m->nx == NX_ && m->S == S_) {                                                             \
    if (m->Hm == 64) {                                                                          \
      if (!split3) return rt2::launch_one<64, NX_, S_, false, 0>(a, tiles_per_cta, stream);     \
      return rt2::launch_one<64, NX_, S_, true, 33>(a, tiles_per_cta, stream);                  \
    }                                                                                           \
    if (!split3) return rt2::launch_one<128, NX_, S_, false, 0>(a, tiles_per_cta, stream);      \
    return rt2::launch_one<128, NX_, S_, true, 33>(a, tiles_per_cta, stream);                   \
  }
  NLC_RT2_CASE(3, 17)
  NLC_RT2_CASE(5, 17)
  NLC_RT2_CASE(6, 17)
  NLC_RT2_CASE(3, 33)
  NLC_RT2_CASE(5, 33)
  NLC_RT2_CASE(6, 33)
#undef NLC_RT2_CASE
  set_error("tcgen05 rollout has no instantiation for nx=%d S=%d", m->nx, m->S);
  return NLC_ERR_UNSUPPORTED;
}

}  // namespace nlc

// measurement hook (tools/trace_rollout.py): device buffer of 32*16*8 int64 receiving CTA 0's clock64 timeline
extern "C" void nlc_debug_set_rollout_trace(void* dev_ptr) { nlc::set_rollout_trace(static_cast<long long*>(dev_ptr)); }
