// Delayed-history encoder (ReverseGRUEncoder.forward, w_nl.py:25-29) on the 5th-generation tensor cores: the default
// form (encode_gru.cu is the fp32 CUDA-core anchor; umma_selftest.cu checks the operand layouts in isolation).
//
// Dataflow as in encode_gru.cu: all K*T windows of a plan in one wide pass, M = 128 windows per tile, persistent CTAs,
// zero-state products skipped; the recurrent products of a window are tcgen05.mma (kind::f16) with fp32 accumulators in
// TMEM, the gate nonlinearities run on the CUDA cores.  What this form does differently, each item from a measurement
// (profiles/r1_encoder_*.md, r1_mma_rate.md):
//   * a dedicated MMA warp.  tcgen05.mma issue is back-pressured by MMA execution (~95 clk per instruction measured
//     with tools/trace_encoder.py), so an epilogue thread that also issues loses the whole MMA time every cell and the
//     other warps end up waiting for it: a third of every step went into those waits.  16 epilogue warps + 1 MMA warp,
//     coupled only by mbarriers (one arrival per warp); no CTA-wide barrier in the steady state;
//   * the epilogue does gates and nothing else.  Layer 0's input projection W_ih0 x and the biases of BOTH layers ride
//     on the tensor cores as one extra K block of the layer-0 state operand, [x_hi x_lo x_hi .. | 1 1] against
//     [W_hi W_hi W_lo .. | b_hi b_lo]: one K = 16 MMA with accumulate = 0 initialises an accumulator tile with all three
//     split-3 terms of W x + b, the hidden products accumulate on top.  No input FMAs, no bias loads, no re-arming of
//     accumulators, no special case for the zero-state cell (3.06 -> 2.35 ms at config 4);
//   * -log2(e) / -2 log2(e) folded into every operand image on the host (model.cu): pre-activations feed ex2 directly;
//   * gate arithmetic in packed fp32x2 (FFMA2/FADD2/FMUL2: half the issue slots, f32x2.cuh);
//   * the (r, z) reciprocal is a Newton iteration on the FMA pipe instead of a MUFU.RCP: 4 MUFU per hidden unit
//     instead of 5 (tools/pipe_bench.cu: 34 vs 41.5 clk per warp-unit on the bare gate);
//   * W_ih1 rows ordered [n | r | z] and accumulator columns [in | r | z | hn]: a layer-1 cell is two N=192 products;
//   * the threads that feed the [x | 1] block prefetch their window entry one cell ahead straight from global memory.
//
//   operands   fp16 hi (+ lo) images, K-major no-swizzle canonical layout; NLC_MATH_TC_SPLIT3: A_hi B_hi + A_lo B_hi +
//              A_hi B_lo, fp32 accumulate (fp32-class);  NLC_MATH_TC_FP16: A_hi B_hi only.
//   widths     a template on the GRU width HG: 64 (hidden_units = 128) or 32 (hidden_units = 64, the reference class
//              default).  Every product and image below scales with HG; the thread layout and the schedule do not.
//   TMEM       D0[4 HG] = [r | z | hn | in] of layer 0;  D1[4 HG] = [in | r | z | hn] of layer 1: 512 columns at HG = 64,
//              256 at HG = 32.
//   schedule   layer 0 runs one cell ahead of layer 1, so every MMA burst runs under the other layer's gate epilogue:
//                 epi A(s+1) || MMA B(s)   ->   epi B(s) || MMA A(s+2)   ->   ...        (tiles software-pipelined)
//   barriers   bar_a / bar_b: MMA A / B complete (tcgen05.commit);  h0_ready / h1_ready: all 16 epilogue warps stored
//              their operand slice and finished reading their accumulator columns.
//   threads    epilogue warp w < 16: TMEM lanes 32 (w & 3).. (its 32 windows), hidden units HG/4 (w >> 2).. + HG/4 - 1
//              of both layers (16 at HG = 64, 8 at HG = 32); warp 16: MMA issue.  544 threads -> 96 registers per thread
//              (the register file is allocated in units of 4 warps: 104 would not launch).
#include <cuda_fp16.h>

#include "common.cuh"
#include "f32x2.cuh"
#include "tc_umma.cuh"

namespace nlc {

using namespace umma;

namespace enc2 {

constexpr int kRows = 128, kThreads = 512;
constexpr uint32_t kLbo = 128;
// shapes of the GRU width HG (64 or 32); the sizes in the comments are those of HG = 64
template <int HG>
struct Geo {
  static constexpr int kHg = HG, kG3 = 3 * HG;
  static constexpr int kUnits = HG / 4;                          // hidden units per thread and layer
  static constexpr uint32_t kOpBytes = kRows * kHg * 2;          // one fp16 A-operand image (16 KB)
  static constexpr uint32_t kWBytes = kG3 * kHg * 2;             // one fp16 weight image (24 KB)
  static constexpr uint32_t kSbo = (kHg / 8) * 128;
  static constexpr uint32_t kColD0 = 0, kColD1 = 4 * HG, kTmemCols = 8 * HG;  // D0 = [r | z | hn | in], D1 = [in | r | z | hn]
  // layer 0's [x | 1] block: one extra K block of the layer-0 state image (see below)
  static constexpr int kKx = kHg + 16;
  static constexpr uint32_t kSboX = (kKx / 8) * 128;             // 8-row-group stride of the K = 80 image
  static constexpr uint32_t kH0HiBytes = kRows * kKx * 2;        // 20 KB
  static constexpr uint32_t kWxBytes = 4 * HG * 8 * 2;           // B side of the block: [4 HG][8] halves (4 KB)
};

struct Args {
  const float* hist;
  float* p_out;
  int K, T, B, L, hist_ch;
  long long rows;
  // step-major tile order for the overlapped planner step (planner.cu): tile = t * tiles_per_t + sample block, so that all
  // windows of rollout step t are encoded before any of step t + 1; every finished tile bumps ready[t] (4 warps x 1) after
  // its outputs are visible device-wide - the rollout kernel, running beside this one, polls it.  tiles_per_t == 0: the
  // plain sample-major order (window index = k * T + t).
  int tiles_per_t;
  unsigned int* ready;
  long long tile_begin;  // first tile of this launch (step-major order only: the planner may split the encoder in two launches)
  // plans of two rollout passes: the step-major order covers only the samples from k_off on (the pass that runs beside the
  // encoder), and the first head_tiles tiles of the launch encode samples [0, k_off) in the plain order, without readiness
  // counters.  Step-major tile j of the sub-plan is tile head_tiles + j of the launch.
  int head_tiles;
  int k_off;
  long long* trace;  // measurement only: clock64 timeline of CTA 0, [step][warp][8 events]
  ModelDev m;
};

__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}

__device__ __forceinline__ void ldtm8p(uint32_t taddr, f2_t (&v)[4]) {
  uint32_t r[8];
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(taddr)
               : "memory");
#pragma unroll
  for (int i = 0; i < 4; ++i) v[i] = pk2u(r[2 * i], r[2 * i + 1]);
}
// GRU cell update of two hidden units from pre-activations that already carry the exponent scales:
//   pr, pz = -log2e (W_r. + b_r), -log2e (W_z. + b_z);   gi, gh = -2 log2e (W_in x + b_in), -2 log2e (W_hn h + b_hn)
//   r = 1/(1 + 2^pr), z = 1/(1 + 2^pz) through ONE reciprocal of the product;  n = 2/(1 + 2^(gi + r gh)) - 1;
//   h' = n + z (h - n).   Arguments of ex2 are clamped so that the shared-reciprocal product stays finite.
//   kAccurate (fp32-class mode): the (r, z) reciprocal by Newton (rcp2<3>), the n reciprocal by Newton when kNewtonN, else MUFU.
//   !kAccurate: the single-pass fp16 mode's accuracy class - three tanh.approx (|error| <= 2^-10.99) per unit and
//   almost no arithmetic: sigmoid(x) = 0.5 tanh(x/2) + 0.5, with x/2 = -pr / (2 log2e) recovered from the folded scale.
__device__ __forceinline__ float mufu_tanh(float x) { float y; asm("tanh.approx.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }

//   kClampRZ: clamp the (r, z) exponents at 60 so that the shared-reciprocal product (1 + 2^pr)(1 + 2^pz) stays finite.  Not
//   needed (and compiled out) when the pre-activations are provably inside +-60 - layer 1, whose inputs are hidden states in
//   (-1, 1): the bound is the L1 norm of the weight rows, checked when the model is packed (model.cu: enc_l1_bounded).
//   The n exponent needs no clamp with the MUFU reciprocal: 2^x = inf gives rcp = 0, n = -1, h - n = h + 1, all exact limits.
template <bool kAccurate, bool kNewtonN, bool kClampRZ>
__device__ __forceinline__ f2_t gru_pair(f2_t pr, f2_t pz, f2_t gi, f2_t gh, f2_t h_old) {
  if (!kAccurate) {
    const f2_t c = pk2(-0.34657359027997264f, -0.34657359027997264f);  // -1 / (2 log2 e)
    const f2_t half = pk2(0.5f, 0.5f);
    float a0, a1, b0, b1, x0, x1;
    upk2(mul2(pr, c), a0, a1);
    upk2(mul2(pz, c), b0, b1);
    const f2_t r = fma2(pk2(mufu_tanh(a0), mufu_tanh(a1)), half, half);
    const f2_t z = fma2(pk2(mufu_tanh(b0), mufu_tanh(b1)), half, half);
    upk2(mul2(fma2(r, gh, gi), c), x0, x1);
    const f2_t n = pk2(mufu_tanh(x0), mufu_tanh(x1));
    return fma2(z, fma2(n, pk2(-1.0f, -1.0f), h_old), n);
  }
  float a0, a1, b0, b1;
  upk2(pr, a0, a1);
  upk2(pz, b0, b1);
  const f2_t one = pk2(1.0f, 1.0f);
  if (kClampRZ) { a0 = fminf(a0, 60.0f); a1 = fminf(a1, 60.0f); b0 = fminf(b0, 60.0f); b1 = fminf(b1, 60.0f); }
  const f2_t da = add2(pk2(mufu_ex2(a0), mufu_ex2(a1)), one);
  const f2_t db = add2(pk2(mufu_ex2(b0), mufu_ex2(b1)), one);
  const f2_t inv = rcp2<3>(mul2(da, db));
  const f2_t r = mul2(db, inv), z = mul2(da, inv);
  float x0, x1;
  upk2(fma2(r, gh, gi), x0, x1);
  if (kNewtonN) { x0 = fminf(x0, 120.0f); x1 = fminf(x1, 120.0f); }  // the Newton reciprocal needs a finite argument
  const f2_t dn = add2(pk2(mufu_ex2(x0), mufu_ex2(x1)), one);
  const f2_t invn = rcp2<kNewtonN ? 3 : 0>(dn);
  const f2_t n = fma2(pk2(2.0f, 2.0f), invn, pk2(-1.0f, -1.0f));
  const f2_t hm = fma2(pk2(-2.0f, -2.0f), invn, add2(h_old, one));  // h - n = (h + 1) - 2 invn
  return fma2(z, hm, n);
}

// 8 hidden values of this thread's row -> one 16-byte slice of the fp16 hi (+ lo) A-operand image
template <bool kSplit3>
__device__ __forceinline__ void store_operand8(unsigned char* img_hi, uint32_t sbo_hi, unsigned char* img_lo, uint32_t sbo_lo, int row, int u0,
                                               const f2_t (&h)[4]) {
  uint32_t ph[4], pl[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    float x0, x1;
    upk2(h[i], x0, x1);
    const __half2 hh = __floats2half2_rn(x0, x1);
    ph[i] = *reinterpret_cast<const uint32_t*>(&hh);
    if (kSplit3) {
      const float2 back = __half22float2(hh);
      float r0, r1;  // the residual is exact in fp32 either way; one packed FMA instead of two subtractions
      upk2(fma2(pk2(back.x, back.y), pk2(-1.0f, -1.0f), h[i]), r0, r1);
      const __half2 ll = __floats2half2_rn(r0, r1);
      pl[i] = *reinterpret_cast<const uint32_t*>(&ll);
    }
  }
  const uint32_t in_group = (uint32_t)(u0 >> 3) * kLbo + (uint32_t)(row & 7) * 16;
  *reinterpret_cast<uint4*>(img_hi + (uint32_t)(row >> 3) * sbo_hi + in_group) = make_uint4(ph[0], ph[1], ph[2], ph[3]);
  if (kSplit3) *reinterpret_cast<uint4*>(img_lo + (uint32_t)(row >> 3) * sbo_lo + in_group) = make_uint4(pl[0], pl[1], pl[2], pl[3]);
}

// D[128 x 3 HG] += A[128 x HG] * B[3 HG x HG]^T : HG / 16 (x3) MMA instructions (N = 192 at HG = 64, 96 at HG = 32).  The hi
// and lo images of A may have different 8-row-group strides (the layer-0 state image carries an extra K block, see Smem)
template <int HG, bool kSplit3>
__device__ __forceinline__ void issue_gemm_g3(uint32_t d_tmem, uint32_t a_hi, uint32_t a_hi_sbo, uint32_t a_lo, uint32_t a_lo_sbo,
                                              uint32_t b_hi, uint32_t b_lo) {
  using G = Geo<HG>;
  const uint32_t idesc = idesc_f16_f32(kRows, G::kG3);
#pragma unroll
  for (int ks = 0; ks < G::kHg / 16; ++ks) {
    const uint32_t off = ks * 2 * kLbo;  // 16 K-elements = two core matrices
    mma_f16_ss(d_tmem, smem_desc(a_hi + off, kLbo, a_hi_sbo), smem_desc(b_hi + off, kLbo, G::kSbo), idesc, 1u);
    if (kSplit3) {
      mma_f16_ss(d_tmem, smem_desc(a_lo + off, kLbo, a_lo_sbo), smem_desc(b_hi + off, kLbo, G::kSbo), idesc, 1u);
      mma_f16_ss(d_tmem, smem_desc(a_hi + off, kLbo, a_hi_sbo), smem_desc(b_lo + off, kLbo, G::kSbo), idesc, 1u);
    }
  }
}

constexpr int kThreadsAll = kThreads + 32;        // 16 epilogue warps + the MMA warp: the participants of the named barriers
// (Tried and dropped: launching the MMA warp's whole register group - 20 warps at 96 registers - and re-balancing with
// setmaxnreg to 104 / 64 or 112 / 32 registers for the epilogue / MMA warps.  2.37 / 2.41 ms against 2.23 ms at config 4:
// the epilogue does not use the extra registers and the MMA warp issues more slowly on 32.  setmaxnreg.inc draws only on
// what setmaxnreg.dec released inside the CTA - releasing less than the increase needs blocks the CTA for ever.)
constexpr int kBarH0 = 2, kBarH1 = 3;             // named barriers: layer-0 / layer-1 operands published (1: output exchange)
// Layer 0's input projection and biases ride on the tensor cores as one extra K block of the layer-0 state operand:
//   A block (per window)  [x0_hi x0_lo x0_hi | x1_hi x1_lo x1_hi | 1 1 | 0 ...]      (16 halves)
//   B block (per column)  [W0_hi W0_hi W0_lo | W1_hi W1_hi W1_lo | b_hi b_lo | 0 ...]
// so one K = 16 MMA with accumulate = 0 writes  W_ih0 x + b  (all three split terms at once) into D0 = [r | z | hn | in]
// and the hidden products accumulate on top: no input FMAs, no bias loads, no accumulator re-arm in the layer-0 epilogue.
// The B side of that block stores only its first 8 K-elements ([4 HG][8] halves, Geo::kWxBytes): the A side's second 8 are
// zeros for ever, so the descriptor lets the second core matrix alias the next row group's (finite) data - 0 x finite = 0.
constexpr int kC2Wout = 0, kC2Bout = 128, kC2Count = 136;  // shared-memory constants: the output layer ([2][HG] weights, bias)

template <int HG>
struct Smem {
  using G = Geo<HG>;
  alignas(128) unsigned char w[3][2][G::kWBytes];   // [W_hh0, W_ih1 (n|r|z), W_hh1][hi, lo]
  alignas(128) unsigned char wx[2][G::kWxBytes + 128];  // input/bias blocks: layer 0 rows in D0 order, layer 1 in D1 order; + zero pad
  alignas(128) unsigned char h0_hi[G::kH0HiBytes];  // layer-0 state, K = HG + the [x | 1] block
  alignas(128) unsigned char h0_lo[G::kOpBytes];
  alignas(128) unsigned char h1[2][G::kOpBytes];
  alignas(16) float c[kC2Count];
  alignas(16) float pout[3][kRows * 2];
  alignas(8) uint64_t bar_w;                 // weight images landed (TMA bulk copies)
  alignas(8) uint64_t bar_a, bar_b, bar_h0;  // MMA A / MMA B complete; the part of MMA B that reads the layer-0 state image complete
  uint32_t tmem_base;
};

// kSplit3: the fp32-class mode (split-3 products, Newton (r, z) reciprocals, Newton for one n-pair in four); else the
// single-pass fp16 mode with tanh.approx gates
template <int HG, bool kSplit3, int GIN, bool kClamp1, bool kTrace = false>
__global__ void __launch_bounds__(kThreadsAll, 1) encode_tc2_kernel(Args a) {
  using G = Geo<HG>;
  constexpr int kHg = G::kHg, kU = G::kUnits;
  constexpr uint32_t kSbo = G::kSbo, kSboX = G::kSboX, kColD0 = G::kColD0, kColD1 = G::kColD1, kTmemCols = G::kTmemCols;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  Smem<HG>& s = *reinterpret_cast<Smem<HG>*>(smem_raw);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int q = warp & 3, grp = warp >> 2;
  const int row = 32 * q + lane;   // window within the tile == TMEM lane
  const int ubase = kU * grp;      // first of the kU hidden units (per layer) this thread owns
  const int B = a.B;
  int tstep = 0;
  auto mark = [&](int ev) {  // compiled in for tools/trace_encoder.py only: the tests cost instructions in the hot loop
    if (kTrace && a.trace && blockIdx.x == 0 && lane == 0 && tstep < 32) a.trace[(tstep * 16 + warp) * 8 + ev] = clock64();
  };

  {
    // The weight images (144 KB at HG = 64, 36 KB at HG = 32, + the two input/bias blocks) come in by TMA bulk copies issued by ONE thread and counted on
    // an mbarrier that only the MMA warp waits for - no other thread ever reads them - so the load runs under the TMEM
    // allocation, the zero fills and the first window fetch instead of in front of them.
    if (warp == 0 && elect_one()) {  // (elect.sync, not tid == 0: the copies' operands then stay in uniform registers)
      mbar_init(&s.bar_w, 1);
      mbar_fence_init();
      mbar_expect_tx(&s.bar_w, (uint32_t)(3 * 2 * G::kWBytes + 2 * G::kWxBytes));
      const unsigned char* src = reinterpret_cast<const unsigned char*>(a.m.enc2_w);
      for (int i = 0; i < 6; ++i) bulk_g2s(&s.w[0][0][0] + (size_t)i * G::kWBytes, src + (size_t)i * G::kWBytes, G::kWBytes, &s.bar_w);
      const unsigned char* sx = reinterpret_cast<const unsigned char*>(a.m.enc2_x);
      for (int l = 0; l < 2; ++l) bulk_g2s(s.wx[l], sx + (size_t)l * G::kWxBytes, G::kWxBytes, &s.bar_w);
    }
    for (int i = tid; i < 2 * 8; i += blockDim.x)  // the zero pad behind each input/bias block
      reinterpret_cast<uint4*>(s.wx[i >> 3] + G::kWxBytes)[i & 7] = make_uint4(0u, 0u, 0u, 0u);
    uint4* dz = reinterpret_cast<uint4*>(s.h0_hi);  // the second half of the [x | 1] block stays zero for ever
    for (int i = tid; i < (int)(G::kH0HiBytes / 16); i += blockDim.x) dz[i] = make_uint4(0u, 0u, 0u, 0u);
    for (int i = tid; i < 2 * kHg; i += blockDim.x) s.c[kC2Wout + i] = a.m.enc2_c[kE2Wout + i];
    if (tid < 2) s.c[kC2Bout + tid] = a.m.enc2_c[kE2Bout + tid];
    if (tid == 0) {
      mbar_init(&s.bar_a, 1); mbar_init(&s.bar_b, 1); mbar_init(&s.bar_h0, 1);
      mbar_fence_init();
    }
    if (warp == 0) tmem_alloc(&s.tmem_base, kTmemCols);
  }
  fence_proxy_async_smem();
  fence_before_sync();
  __syncthreads();
  fence_after_sync();
  const uint32_t tmem = s.tmem_base;
  const uint32_t tlane = tmem + ((uint32_t)(32 * q) << 16);
  const float* cst = s.c;

  const uint32_t a_h0_hi = smem_u32(s.h0_hi), a_h0_lo = smem_u32(s.h0_lo);
  const uint32_t a_h1_hi = smem_u32(s.h1[0]), a_h1_lo = smem_u32(s.h1[1]);
  const uint32_t w_hh0_hi = smem_u32(s.w[0][0]), w_hh0_lo = smem_u32(s.w[0][1]);
  const uint32_t w_ih1_hi = smem_u32(s.w[1][0]), w_ih1_lo = smem_u32(s.w[1][1]);
  const uint32_t w_hh1_hi = smem_u32(s.w[2][0]), w_hh1_lo = smem_u32(s.w[2][1]);
  const uint32_t w_x0 = smem_u32(s.wx[0]), w_x1 = smem_u32(s.wx[1]);
  const long long n_tiles = (a.rows + kRows - 1) / kRows;   // one past the last tile of this launch
  const long long tile_first = a.tile_begin + blockIdx.x;

  if (warp == 16) {
    // =====================================  MMA warp  =====================================
    // mirrors the epilogue warps' publication order: h0 + the next cell's [x | 1] block (-> layer-0 product of the next
    // cell), then h1 / D1 re-armed (-> layer-1 product of the next cell: input part from h0, hidden part from h1)
    // "operand published" hand-offs are NAMED barriers (epilogue warps bar.arrive, this warp bar.sync): as mbarriers, each of
    // the 16 arrivals woke every warp sleeping in a try_wait loop (this one, and epilogue warps waiting for a commit) for
    // another SYNCS / NANOSLEEP / BRA round - 12 % of all executed instructions in the ncu source view.  An epilogue warp
    // cannot arrive twice in one generation: its next arrival on the same barrier lies behind a wait for a product that
    // this warp issues only after the generation has completed.
    auto wait_ready = [&](int id) {
      asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(kThreadsAll) : "memory");
    };
    auto issue_a = [&](bool with_hidden) {
      if (elect_one()) {
        fence_after_sync();
        mma_f16_ss(tmem + kColD0, smem_desc(a_h0_hi + (kHg / 8) * kLbo, kLbo, kSboX), smem_desc(w_x0, kLbo, 128), idesc_f16_f32(kRows, 4 * kHg), 0u);
        if (with_hidden) issue_gemm_g3<HG, kSplit3>(tmem + kColD0, a_h0_hi, kSboX, a_h0_lo, kSbo, w_hh0_hi, w_hh0_lo);
        mma_commit(&s.bar_a);
      }
      __syncwarp();
    };
    auto issue_b = [&](bool with_h1) {
      if (elect_one()) {
        fence_after_sync();
        // biases first (accumulate = 0 over all of D1 = [in | r | z | hn]): the 1-columns of the [x | 1] block
        mma_f16_ss(tmem + kColD1, smem_desc(a_h0_hi + (kHg / 8) * kLbo, kLbo, kSboX), smem_desc(w_x1, kLbo, 128), idesc_f16_f32(kRows, 4 * kHg), 0u);
        issue_gemm_g3<HG, kSplit3>(tmem + kColD1, a_h0_hi, kSboX, a_h0_lo, kSbo, w_ih1_hi, w_ih1_lo);
        // everything that reads the layer-0 state image is issued: the layer-0 epilogue may overwrite it as soon as THIS much
        // has completed (half a product earlier than bar_b), so its operand stores interleave with its gate math
        mma_commit(&s.bar_h0);
        if (with_h1) issue_gemm_g3<HG, kSplit3>(tmem + kColD1 + kHg, a_h1_hi, kSbo, a_h1_lo, kSbo, w_hh1_hi, w_hh1_lo);
        mma_commit(&s.bar_b);
      }
      __syncwarp();
    };
    if (tile_first < n_tiles) {
      mbar_wait(&s.bar_w, 0);
      wait_ready(kBarH0);  // [x(0) | 1]
      issue_a(false);
      wait_ready(kBarH0);  // h0(0), [x(1) | 1]
      issue_a(true);
      wait_ready(kBarH1);
      issue_b(false);
    }
    for (long long tile = tile_first; tile < n_tiles; tile += gridDim.x) {
      const bool has_next = tile + gridDim.x < n_tiles;
      for (int st = 0; st < B; ++st) {
        if (st + 1 < B || has_next) {
          wait_ready(kBarH0);
          if (st + 2 < B || st + 1 == B) issue_a(true);   // next cell of this tile, or cell 1 of the next tile
          else if (has_next) issue_a(false);              // st + 2 == B: cell 0 of the next tile (zero state)
        }
        wait_ready(kBarH1);
        if (st + 1 < B) issue_b(true);
        else if (has_next) issue_b(false);
      }
    }
  } else {
  // =====================================  epilogue warps  =====================================
  float amean[GIN], ainv[GIN];
#pragma unroll
  for (int v = 0; v < GIN; ++v) { amean[v] = a.m.act_mean[v]; ainv[v] = a.m.act_inv_std[v]; }

  uint32_t n_a = 0, n_b = 0, n_h0 = 0;  // waits completed on bar_a / bar_b / bar_h0
  f2_t h0r[kU / 2], h1r[kU / 2];
  // raw window entry of the FOLLOWING layer-0 cell (threads with grp == 0 feed the operand).  It is normalised only when it is
  // written into the operand, a whole gate epilogue after the load was issued: nothing waits for global memory
  float xraw[GIN] = {};

  // hist offset of this thread's window in a tile (one integer division per tile, not per cell)
  auto window_base = [&](long long tile_) -> size_t {
    if (a.tiles_per_t > 0 && (int)tile_ >= a.head_tiles) {  // step-major: one step t per tile, 128 consecutive samples
      const int ts = (int)tile_ - a.head_tiles;
      const int t = (int)((unsigned)ts / (unsigned)a.tiles_per_t);
      int k = a.k_off + (ts - t * a.tiles_per_t) * kRows + row;
      if (k >= a.K) k = a.K - 1;
      return ((size_t)k * a.L + t) * a.hist_ch;
    }
    long long grow = tile_ * kRows + row;
    if (grow >= a.rows) grow = a.rows - 1;
    long long k;
    if (a.rows <= 0x7fffffffLL) k = (long long)((unsigned)grow / (unsigned)a.T); else k = grow / a.T;
    const int t = (int)(grow - k * a.T);
    return ((size_t)k * a.L + t) * a.hist_ch;
  };
  size_t base_cur = 0, base_next = 0;
  // window entry of layer-0 cell `cell_`: reversed order, cell c consumes entry B-1-c (w_nl.py:27)
  auto fetch_x = [&](bool next_tile_, int cell_) {
    if (grp != 0) return;
    const int j = B - 1 - cell_;
    const float* src = a.hist + (next_tile_ ? base_next : base_cur) + (size_t)j * a.hist_ch;
#pragma unroll
    for (int v = 0; v < GIN; ++v) {
      // channels beyond hist_ch: the time channel of encode_obs_time (mppi_with_model.py:110-119)
      xraw[v] = v < a.hist_ch ? __ldg(src + v) : (float)(B - 1 - j);
    }
  };
  // [x_hi x_lo x_hi | ... | 1 1] -> the extra K block of this window's row in the layer-0 state image
  auto write_x = [&]() {
    if (grp != 0) return;
    __half hv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) hv[i] = __float2half_rn(0.0f);
#pragma unroll
    for (int v = 0; v < GIN; ++v) {
      const float xn = (xraw[v] - amean[v]) * ainv[v];  // w_nl.py:121
      const __half hi = __float2half_rn(xn);
      const __half lo = __float2half_rn(xn - __half2float(hi));
      hv[3 * v] = hi; hv[3 * v + 1] = lo; hv[3 * v + 2] = hi;
    }
    hv[6] = __float2half_rn(1.0f); hv[7] = __float2half_rn(1.0f);
    uint32_t w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) { const __half2 p2 = __halves2half2(hv[2 * i], hv[2 * i + 1]); w[i] = *reinterpret_cast<const uint32_t*>(&p2); }
    *reinterpret_cast<uint4*>(s.h0_hi + (uint32_t)(row >> 3) * kSboX + (kHg / 8) * kLbo + (uint32_t)(row & 7) * 16) = make_uint4(w[0], w[1], w[2], w[3]);
  };
  // layer-0 cell: complete pre-activations come out of D0 = [r | z | hn | in]; with `store` the new state goes into the layer-0
  // state image (after `wait_h0`: see below).
  auto cell_a = [&](bool from_zero, bool store, bool wait_h0) {
    if (from_zero) {  // cell 0 of a window: h = 0 (one uniform branch instead of a select per use)
#pragma unroll
      for (int i = 0; i < kU / 2; ++i) h0r[i] = 0ull;
    }
#pragma unroll
    for (int c = 0; c < kU / 8; ++c) {
      const int u0 = ubase + 8 * c;
      f2_t gr[4], gz[4], gh[4], gn[4];
      ldtm8p(tlane + kColD0 + u0, gr);
      ldtm8p(tlane + kColD0 + kHg + u0, gz);
      ldtm8p(tlane + kColD0 + 2 * kHg + u0, gh);
      ldtm8p(tlane + kColD0 + 3 * kHg + u0, gn);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        // fp32-class: the n-gate reciprocal by Newton for the first of the four pairs of a chunk, MUFU for the others.  The
        // MUFU pipe (70 % busy) and the FMA pipe / issue slots are balanced at one in four: 2.18 ms at config 4 against 2.23
        // (none), 2.21 (two) and 2.29 ms (all four by Newton)
        if (kSplit3 && i == 0) h0r[4 * c + i] = gru_pair<kSplit3, true, true>(gr[i], gz[i], gn[i], gh[i], h0r[4 * c + i]);
        else h0r[4 * c + i] = gru_pair<kSplit3, false, true>(gr[i], gz[i], gn[i], gh[i], h0r[4 * c + i]);
      }
    }
    if (store) {
      // The state image is free once the part of the previous MMA B that reads it has completed (bar_h0: half a product
      // earlier than bar_b).  Waited for AFTER both chunks' gate math: that part completes ~1.8 k clocks after it was
      // issued, later than one chunk's math (waiting after the first chunk showed up as 8.8 % of all stall samples).
      if (wait_h0) { mbar_wait_sleep(&s.bar_h0, n_h0 & 1); ++n_h0; }
#pragma unroll
      for (int c = 0; c < kU / 8; ++c) {
        const f2_t (&hc)[4] = *reinterpret_cast<const f2_t(*)[4]>(&h0r[4 * c]);
        store_operand8<kSplit3>(s.h0_hi, kSboX, s.h0_lo, kSbo, row, ubase + 8 * c, hc);
      }
    }
  };
  // the A operand of the next products is in shared memory (and, for grp 0, the following cell's [x | 1] block is added
  // here): make it visible to the tensor core's proxy and tell the MMA warp
  auto publish_h0 = [&](bool with_x) {
    if (with_x) write_x();
    fence_proxy_async_smem();
    fence_before_sync();
    asm volatile("bar.arrive %0, %1;" ::"r"(kBarH0), "n"(kThreadsAll) : "memory");
  };
  // after the layer-1 epilogue: D1 read (and h1 stored when `with_h1`)
  auto publish_h1 = [&](bool with_h1) {
    if (with_h1) fence_proxy_async_smem();
    fence_before_sync();
    asm volatile("bar.arrive %0, %1;" ::"r"(kBarH1), "n"(kThreadsAll) : "memory");
  };

  // ---- head of the first tile: layer-0 cell 0 (zero state: the [x | 1] product alone), then A(1) and the input part of B(0) ----
  if (tile_first < n_tiles) {
    base_cur = window_base(tile_first);
    fetch_x(false, 0);
    publish_h0(true);
    fetch_x(false, 1);
    mbar_wait_sleep(&s.bar_a, n_a & 1); ++n_a;
    fence_after_sync();
    cell_a(true, true, false);  // nothing has read the state image yet
    publish_h0(true);
    publish_h1(false);  // nothing of layer 1 exists yet: the input part of B(0) can go
  }
  for (long long tile = tile_first; tile < n_tiles; tile += gridDim.x) {
    const long long row0 = tile * kRows;
    const long long next_tile = tile + gridDim.x;
    const bool has_next = next_tile < n_tiles;
    if (has_next) base_next = window_base(next_tile);
    for (int st = 0; st < B; ++st) {
      // ======== layer-0 epilogue: cell st+1 of this tile, or cell 0 of the next one  ||  MMA B(st) ========
      const bool a_slot = st + 1 < B || has_next;
      // the cell after that one: its window entry is fetched now and joins the operand at the publication below
      const bool following = st + 2 < B || st + 1 == B || (st + 2 == B && has_next);
      if (a_slot) {
        // the load is consumed at the publication below, after this cell's gate math
        if (st + 2 < B) fetch_x(false, st + 2);
        else if (st + 1 == B) fetch_x(true, 1);
        else if (has_next) fetch_x(true, 0);
        mark(0);
        mbar_wait_sleep(&s.bar_a, n_a & 1); ++n_a;
        fence_after_sync();
        mark(1);
        // MMA B(st) reads the state image this cell overwrites: cell_a waits for that part of it (bar_h0) before its first store
        cell_a(st + 1 == B, true, true);
        mark(2);
        publish_h0(following);
        mark(3);
      }
      // ======== layer-1 epilogue B(st)  ||  MMA A ========
      if (st == 0) {
#pragma unroll
        for (int i = 0; i < kU / 2; ++i) h1r[i] = 0ull;
      }
      mbar_wait_sleep(&s.bar_b, n_b & 1); ++n_b;
      fence_after_sync();
      mark(4);
#pragma unroll
      for (int c = 0; c < kU / 8; ++c) {
        const int u0 = ubase + 8 * c;
        f2_t gn[4], gr[4], gz[4], gh[4];
        ldtm8p(tlane + kColD1 + u0, gn);
        ldtm8p(tlane + kColD1 + kHg + u0, gr);
        ldtm8p(tlane + kColD1 + 2 * kHg + u0, gz);
        ldtm8p(tlane + kColD1 + 3 * kHg + u0, gh);
        tmem_ld_wait();
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (kSplit3 && i == 0) h1r[4 * c + i] = gru_pair<kSplit3, true, kClamp1>(gr[i], gz[i], gn[i], gh[i], h1r[4 * c + i]);
          else h1r[4 * c + i] = gru_pair<kSplit3, false, kClamp1>(gr[i], gz[i], gn[i], gh[i], h1r[4 * c + i]);
        }
        if (st + 1 < B) {  // MMA B(st), the last reader of the h1 image, has completed (bar_b above): store chunk by chunk
          const f2_t (&hc)[4] = *reinterpret_cast<const f2_t(*)[4]>(&h1r[4 * c]);
          store_operand8<kSplit3>(s.h1[0], kSbo, s.h1[1], kSbo, row, u0, hc);
        }
      }
      mark(5);
      if (st + 1 < B) {
        publish_h1(true);
        mark(6);
        ++tstep;
      } else {
        // ---------------- linear_out on the top layer's last state (w_nl.py:29) ----------------
        float o0 = 0.f, o1 = 0.f;
#pragma unroll
        for (int i = 0; i < kU / 2; ++i) {
          float x0, x1;
          upk2(h1r[i], x0, x1);
          const float2 wa = *reinterpret_cast<const float2*>(cst + kC2Wout + ubase + 2 * i);
          const float2 wb = *reinterpret_cast<const float2*>(cst + kC2Wout + kHg + ubase + 2 * i);
          o0 = fmaf(wa.y, x1, fmaf(wa.x, x0, o0));
          o1 = fmaf(wb.y, x1, fmaf(wb.x, x0, o1));
        }
        if (grp > 0) {
          *reinterpret_cast<float2*>(&s.pout[grp - 1][row * 2]) = make_float2(o0, o1);
          asm volatile("bar.arrive 1, 512;" ::: "memory");
        } else {
          asm volatile("bar.sync 1, 512;" ::: "memory");
          const float2 p0 = *reinterpret_cast<const float2*>(&s.pout[0][row * 2]);
          const float2 p1 = *reinterpret_cast<const float2*>(&s.pout[1][row * 2]);
          const float2 p2 = *reinterpret_cast<const float2*>(&s.pout[2][row * 2]);
          const float2 pv = make_float2(((o0 + p0.x) + p1.x) + p2.x + cst[kC2Bout], ((o1 + p0.y) + p1.y) + p2.y + cst[kC2Bout + 1]);
          if (a.tiles_per_t > 0 && (int)tile >= a.head_tiles) {
            const int ts = (int)tile - a.head_tiles;
            const int t = (int)((unsigned)ts / (unsigned)a.tiles_per_t);
            const int k = a.k_off + (ts - t * a.tiles_per_t) * kRows + row;
            if (k < a.K) *reinterpret_cast<float2*>(a.p_out + ((size_t)k * a.T + t) * 2) = pv;
            // publish: the warp's 32 outputs are ordered before lane 0's device-scope fence and counter bump
            __syncwarp();
            if (lane == 0) { __threadfence(); atomicAdd(a.ready + t, 1u); }
          } else if (row0 + row < a.rows) {
            *reinterpret_cast<float2*>(a.p_out + (row0 + row) * 2) = pv;
          }
        }
        // D1 is read: the input part of the next tile's B(0) can go (its h0 image was published above)
        publish_h1(false);
        mark(6);
        ++tstep;
      }
    }
    base_cur = base_next;
  }
  }  // epilogue warps
  fence_before_sync();
  __syncthreads();
  if (warp == 0) tmem_dealloc(tmem, kTmemCols);
}

}  // namespace enc2

// measurement hooks (tools/trace_encoder.py, tools/bench_encoder.py)
static long long* g_enc_trace = nullptr;
void set_encoder_trace(long long* p) { g_enc_trace = p; }

int launch_encode_tc2(nlc_model_s* m, const float* hist, int hist_ch, int K, int T, int B, float* p, int split3, cudaStream_t stream,
                      unsigned int* ready, int max_ctas, long long tile_begin, long long tile_end, int k_sub, bool with_head) {
  using namespace enc2;
  NLC_REQUIRE(B * m->gin <= 8, NLC_ERR_SHAPE, "tcgen05 encoder: window_length * input_width = %d exceeds 8", B * m->gin);
  NLC_REQUIRE(B >= 2, NLC_ERR_SHAPE, "tcgen05 encoder: window_length must be >= 2");
  NLC_REQUIRE(m->gin == 1 || m->gin == 2, NLC_ERR_SHAPE, "tcgen05 encoder: GRU input width %d has no instantiation", m->gin);
  NLC_REQUIRE(m->Hg == 64 || m->Hg == 32, NLC_ERR_SHAPE, "tcgen05 encoder: GRU width %d has no instantiation", m->Hg);
  NLC_REQUIRE(!ready || (k_sub >= 0 && k_sub < K && ((long long)k_sub * T) % kRows == 0 && (!with_head || tile_begin == 0)), NLC_ERR_ARG,
              "tcgen05 encoder: bad step-major sub-plan (first sample %d of %d)", k_sub, K);
  Args a;
  a.hist = hist; a.p_out = p; a.K = K; a.T = T; a.B = B; a.L = B - 1 + T; a.hist_ch = hist_ch;
  a.rows = (long long)K * T;
  a.tiles_per_t = ready ? (K - k_sub + kRows - 1) / kRows : 0;
  a.ready = ready;
  a.tile_begin = 0;
  a.k_off = ready ? k_sub : 0;
  a.head_tiles = ready && with_head ? (int)((long long)k_sub * T / kRows) : 0;
  a.m = m->d;
  a.trace = g_enc_trace;
  const int smem = (int)(m->Hg == 32 ? sizeof(Smem<32>) : sizeof(Smem<64>)) + 128;
  // fp32-class mode: Newton (3 steps) for the (r, z) reciprocal; for n, Newton for one pair in four and MUFU for the rest;
  // single-pass fp16 mode: three tanh.approx per unit (that mode's accuracy class, 2e-2 bound).
  void (*kern)(Args);
  // layer-1 (r, z) clamps are compiled out when the packed weights prove |pre-activation| * log2(e) < 60 (model.cu)
  const bool c1 = !m->enc_l1_bounded;
#define NLC_ENC_PICK(HG, TR) \
  (m->gin == 1 ? (c1 ? encode_tc2_kernel<HG, true, 1, true, TR> : encode_tc2_kernel<HG, true, 1, false, TR>) \
               : (c1 ? encode_tc2_kernel<HG, true, 2, true, TR> : encode_tc2_kernel<HG, true, 2, false, TR>))
  if (m->Hg == 32) {  // hidden_units = 64 (the clock64 timeline is measured at the 128 width only)
    if (!split3) kern = m->gin == 1 ? encode_tc2_kernel<32, false, 1, true> : encode_tc2_kernel<32, false, 2, true>;
    else kern = NLC_ENC_PICK(32, false);
  } else if (!split3) {
    kern = m->gin == 1 ? encode_tc2_kernel<64, false, 1, true> : encode_tc2_kernel<64, false, 2, true>;
  } else {
    kern = a.trace ? NLC_ENC_PICK(64, true) : NLC_ENC_PICK(64, false);
  }
#undef NLC_ENC_PICK
  NLC_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  long long n_tiles = ready ? (long long)a.tiles_per_t * T : (a.rows + kRows - 1) / kRows;
  if (ready) {
    // step-major: every tile is walked (rows beyond K are masked at the output); [tile_begin, tile_end) of them in this launch,
    // after the head if there is one
    if (tile_end >= 0 && tile_end < n_tiles) n_tiles = tile_end;
    n_tiles += a.head_tiles;
    a.tile_begin = with_head ? 0 : (tile_begin > 0 ? tile_begin : 0);
    a.rows = n_tiles * kRows;
    if (a.tile_begin >= n_tiles) return NLC_OK;
  }
  const int cap = max_ctas > 0 && max_ctas < 148 ? max_ctas : 148;
  const long long mine = n_tiles - a.tile_begin;
  const int grid = (int)(mine < cap ? mine : cap);
  kern<<<grid, kThreadsAll, smem, stream>>>(a);
  NLC_LAUNCH_OK("encode_tc2_kernel");
  return NLC_OK;
}

}  // namespace nlc

// measurement hook (tools/trace_encoder.py): device buffer of 32*16*8 int64 receiving CTA 0's clock64 timeline
extern "C" void nlc_debug_set_encoder_trace(void* dev_ptr) { nlc::set_encoder_trace(static_cast<long long*>(dev_ptr)); }
