// Stage 4 of MPPIDelay.command (planners/mppi_delay.py:210-224): the exponential-weight update as a
// two-pass max-then-sum reduction (here: min of the cost, then the sums), split into the shard-local
// part and a combine over G shards so that K can be sharded over GPUs with ONE small exchange of the
// (beta, eta, W[T][nu]) triple per control step.
//
//   pass 1  softmax_min_kernel : beta_g = min_k c_k                         (reads 4K bytes)
//   pass 2  softmax_sum_kernel : w_k = exp(-(c_k - beta_g)/lambda), eta_g = sum w_k,
//                                W_g[t][u] = sum_k w_k noise[k][t][u]       (reads 4K + 4*K*T*nu bytes)
//           per-block partials, the last block to finish adds them in block order (deterministic).
//   combine softmax_combine_kernel : beta = min beta_g, rescale by exp(-(beta_g-beta)/lambda),
//                                U += W/eta, action = U[0]*u_scale.
// HBM-bound streaming kernels: rows of noise are read as contiguous T*nu-float rows, 32 rows per warp pass.
#include "common.cuh"

namespace nlc {

__device__ __forceinline__ unsigned f2ord(float f) {
  unsigned u = __float_as_uint(f);
  return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}
__device__ __forceinline__ float ord2f(unsigned u) {
  return __uint_as_float((u & 0x80000000u) ? (u & 0x7fffffffu) : ~u);
}

// Weight exp(-inv_lambda (c - beta)) of cost c against the minimum beta, as torch.exp gives it (mppi_delay.py:210-211): 0 for
// a +inf cost - also when beta is +inf, i.e. every cost of a shard overflowed - and for an argument below the fp32 range of
// exp (exp_acc's rounding-error FMA is NaN once x * log2(e) overflows, x < -2.4e38); a NaN cost stays NaN.  Every other
// argument goes through exp_acc, which is 0 anyway below -104: the result is exp_acc's wherever that is finite.
__device__ __forceinline__ float exp_weight(float c, float beta, float inv_lambda) {
  const float x = -inv_lambda * (c - beta);
  return (c == INFINITY || x < -104.0f) ? 0.0f : exp_acc(x);
}

struct SoftWs {           // workspace header (device)
  unsigned min_ord;       // ordered-uint encoding of the running min
  unsigned ticket;        // blocks finished in pass 2
};

__global__ void softmax_init_kernel(SoftWs* ws) {
  ws->min_ord = 0xffffffffu;
  ws->ticket = 0u;
}

__global__ void __launch_bounds__(256) softmax_min_kernel(const float* __restrict__ cost, int K, SoftWs* ws) {
  float m = INFINITY;
  const int n4 = K >> 2;
  const float4* c4 = reinterpret_cast<const float4*>(cost);
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += gridDim.x * blockDim.x) {
    const float4 v = __ldg(c4 + i);
    m = fminf(fminf(m, fminf(v.x, v.y)), fminf(v.z, v.w));
  }
  for (int i = (n4 << 2) + blockIdx.x * blockDim.x + threadIdx.x; i < K; i += gridDim.x * blockDim.x) m = fminf(m, cost[i]);
  m = warp_min(m);
  __shared__ float sm[8];
  if ((threadIdx.x & 31) == 0) sm[threadIdx.x >> 5] = m;
  __syncthreads();
  if (threadIdx.x < 32) {
    m = threadIdx.x < (blockDim.x >> 5) ? sm[threadIdx.x] : INFINITY;
    m = warp_min(m);
    if (threadIdx.x == 0) atomicMin(&ws->min_ord, f2ord(m));
  }
}

// One block = 8 warps over a contiguous range of samples.  A warp takes 32 samples at a time: lane r computes the weight of
// sample r (one exp per sample, not per element), then the 32 noise rows stream through with the weight broadcast by
// shuffle; lane l owns columns l, l+32, ... of W (<= 8 accumulators), so every load is a contiguous 128-byte line and
// 16 loads per lane are in flight (rows unrolled by four).  Partial sums: warps in warp order through shared memory,
// blocks in block order by the last block to finish - run-to-run identical.
__global__ void __launch_bounds__(256) softmax_sum_kernel(const float* __restrict__ cost, const float* __restrict__ noise,
                                                          int K, int TN, float inv_lambda, SoftWs* ws,
                                                          float* partials /*[grid][1+TN]*/, float* triple,
                                                          float* weights, int rows_per_block, ExchangePub pub) {
  __shared__ float red[8][257];
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const float beta = ord2f(ws->min_ord);
  const int kb = blockIdx.x * rows_per_block;
  const int ke = min(K, kb + rows_per_block);
  const int nci = (TN + 31) >> 5;  // column chunks of 32 (<= 8)
  float acc[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) acc[i] = 0.0f;
  float eta = 0.0f;
  for (int k0 = kb + 32 * warp; k0 < ke; k0 += 32 * 8) {
    const int k = k0 + lane;
    float w = 0.0f;
    if (k < ke) {
      w = exp_weight(__ldg(cost + k), beta, inv_lambda);  // _ensure_non_zero, mppi_delay.py:12-13
      if (weights) weights[k] = w;
    }
    eta += w;
    const int nr = min(32, ke - k0);
    const float* base = noise + (size_t)k0 * TN + lane;
    int r = 0;
    for (; r + 4 <= nr; r += 4) {
      float v[4][8];
#pragma unroll
      for (int rr = 0; rr < 4; ++rr)
#pragma unroll
        for (int i = 0; i < 8; ++i)
          v[rr][i] = (i < nci && lane + 32 * i < TN) ? __ldg(base + (size_t)(r + rr) * TN + 32 * i) : 0.0f;
#pragma unroll
      for (int rr = 0; rr < 4; ++rr) {
        const float wr = __shfl_sync(0xffffffffu, w, r + rr);
#pragma unroll
        for (int i = 0; i < 8; ++i) acc[i] = fmaf(wr, v[rr][i], acc[i]);
      }
    }
    for (; r < nr; ++r) {
      const float wr = __shfl_sync(0xffffffffu, w, r);
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (i < nci && lane + 32 * i < TN) acc[i] = fmaf(wr, __ldg(base + (size_t)r * TN + 32 * i), acc[i]);
    }
  }
  eta = warp_sum(eta);
#pragma unroll
  for (int i = 0; i < 8; ++i) red[warp][lane + 32 * i] = acc[i];
  if (lane == 0) red[warp][256] = eta;
  __syncthreads();
  float* my = partials + (size_t)blockIdx.x * (1 + TN);
  if (threadIdx.x < TN) {
    float sacc = 0.0f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) sacc += red[wv][threadIdx.x];
    my[1 + threadIdx.x] = sacc;
  }
  if (threadIdx.x == 0) {
    float sacc = 0.0f;
#pragma unroll
    for (int wv = 0; wv < 8; ++wv) sacc += red[wv][256];
    my[0] = sacc;
  }
  __threadfence();
  __shared__ bool last;
  __syncthreads();
  if (threadIdx.x == 0) last = (atomicAdd(&ws->ticket, 1u) == gridDim.x - 1);
  __syncthreads();
  if (last) {  // fixed block order => run-to-run identical sums
    __threadfence();
    const unsigned long long step = pub.G ? *pub.step_ctr : 0ull;
    const int par = (int)(step & 1ull);
    for (int c = threadIdx.x; c < 1 + TN; c += blockDim.x) {
      float sacc = 0.0f;
      for (unsigned bb = 0; bb < gridDim.x; ++bb) sacc += partials[(size_t)bb * (1 + TN) + c];
      triple[1 + c] = sacc;
      // connected shards (see the exchange notes below): the triple goes straight into every shard's mailbox over NVLink
      for (int g = 0; g < pub.G; ++g) pub.mailboxes[g][((size_t)par * pub.G + pub.rank) * pub.stride + 1 + c] = sacc;
    }
    if (threadIdx.x == 0) {
      triple[0] = beta;
      for (int g = 0; g < pub.G; ++g) pub.mailboxes[g][((size_t)par * pub.G + pub.rank) * pub.stride] = beta;
    }
    if (pub.G) {
      __threadfence_system();
      __syncthreads();
      if ((int)threadIdx.x < pub.G) {
        unsigned int* seq = reinterpret_cast<unsigned int*>(pub.mailboxes[threadIdx.x] + (size_t)2 * pub.G * pub.stride) + par * pub.G + pub.rank;
        const unsigned int id = (unsigned int)(step + 1ull);
        asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(seq), "r"(id) : "memory");
      }
    }
  }
}

__device__ __forceinline__ void step_tail(const StepTail& tl) {
  // called after the combine's last use of the step's data by every thread of the (single) block
  __syncthreads();
  if (tl.ready) for (int i = threadIdx.x; i < tl.n_ready; i += blockDim.x) tl.ready[i] = 0u;
  if (threadIdx.x == 0) {
    if (tl.call_ctr) *tl.call_ctr += 1ull;
    if (tl.softmax_ws) { SoftWs* ws = static_cast<SoftWs*>(tl.softmax_ws); ws->min_ord = 0xffffffffu; ws->ticket = 0u; }
    if (tl.host_seq) {  // everything of the step is done: hand the action to the spinning host thread
      for (int i = 0; i < tl.nu; ++i) tl.host_action[i] = tl.action_src[i];
      __threadfence_system();
      const unsigned int v = *reinterpret_cast<volatile unsigned int*>(tl.host_seq) + 1u;
      asm volatile("st.release.sys.global.u32 [%0], %1;" ::"l"(tl.host_seq), "r"(v) : "memory");
    }
  }
}

// host entry point: state [nx] and action buffer [nb] from mapped pinned host memory into the planner's device buffers (one
// tiny kernel node instead of two H2D copy nodes)
__global__ void ingest_kernel(const float* __restrict__ h_in, float* __restrict__ state_in, float* __restrict__ abuf_in, int nx, int nb) {
  const int i = threadIdx.x;
  if (i < nx) state_in[i] = h_in[i];
  else if (i < nx + nb) abuf_in[i - nx] = h_in[i];
}
int launch_ingest(const float* h_in, float* state_in, float* abuf_in, int nx, int nb, cudaStream_t s) {
  ingest_kernel<<<1, 64, 0, s>>>(h_in, state_in, abuf_in, nx, nb);
  NLC_LAUNCH_OK("ingest_kernel");
  return NLC_OK;
}

__global__ void softmax_combine_kernel(const float* __restrict__ triples, int G, int TN, int nu, float inv_lambda,
                                       float u_scale, float* U, float* action, float* stats, StepTail tl) {
  const int stride = 2 + TN;
  float beta = INFINITY;
  for (int g = 0; g < G; ++g) beta = fminf(beta, triples[g * stride]);
  float eta = 0.0f;
  for (int g = 0; g < G; ++g) eta = fmaf(triples[g * stride + 1], exp_weight(triples[g * stride], beta, inv_lambda), eta);
  for (int c = threadIdx.x; c < TN; c += blockDim.x) {
    float W = 0.0f;
    for (int g = 0; g < G; ++g) W = fmaf(triples[g * stride + 2 + c], exp_weight(triples[g * stride], beta, inv_lambda), W);
    const float u = (tl.U_src ? tl.U_src[c] : U[c]) + W / eta;  // mppi_delay.py:214-216
    U[c] = u;
    if (c < nu && action) action[c] = u * u_scale;  // :217-224
  }
  if (threadIdx.x == 0 && stats) { stats[0] = beta; stats[1] = eta; }
  step_tail(tl);
}

// ---------------------------------------------------------------------------------------------------------------------
// Exchange of the per-shard triples WITHOUT a collective library (K sharded over the GPUs of one node): every shard owns
// a "mailbox" in its own HBM,  float triples[2][G][stride]  followed by  unsigned seq[2][G];  peers map it through CUDA IPC.
//   publish  the last block of softmax_sum_kernel stores the shard's triple into slot [parity][rank] of EVERY shard's mailbox
//            over NVLink (plain peer stores), fences system-wide, then releases seq[parity][rank] = step id in each mailbox;
//   combine  polls its OWN mailbox until all G seq words carry the step id (acquire), then merges as softmax_combine_kernel.
// Parity = step & 1: a shard can be at most one control step ahead of another (its next combine needs everybody's next
// triple), so two slots are enough.  No host, no NCCL, no extra stream: the sharded control step is one CUDA graph.
// ---------------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) softmax_combine_exchange_kernel(float* mailbox, int G, int stride, int TN, int nu, float inv_lambda,
                                                                       float u_scale, float* U, float* action, float* stats,
                                                                       unsigned long long* step_ctr, unsigned int* status, StepTail tl) {
  const unsigned long long step = *step_ctr;
  const int par = (int)(step & 1ull);
  const unsigned int id = (unsigned int)(step + 1ull);
  if (threadIdx.x < G) {
    const unsigned int* seq = reinterpret_cast<const unsigned int*>(mailbox + (size_t)2 * G * stride) + par * G + threadIdx.x;
    const long long t0 = clock64();
    unsigned int v;
    do {
      asm volatile("ld.acquire.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(seq) : "memory");
      if (v == id) break;
      if (clock64() - t0 > (1ll << 34)) { atomicExch(status, 2u); break; }  // ~8 s: a peer is gone; do not hang the device
      __nanosleep(200);
    } while (true);
  }
  __syncthreads();
  const volatile float* triples = mailbox + (size_t)par * G * stride;
  float beta = INFINITY;
  for (int g = 0; g < G; ++g) beta = fminf(beta, triples[g * stride]);
  float eta = 0.0f;
  for (int g = 0; g < G; ++g) eta = fmaf(triples[g * stride + 1], exp_weight(triples[g * stride], beta, inv_lambda), eta);
  for (int c = threadIdx.x; c < TN; c += blockDim.x) {
    float W = 0.0f;
    for (int g = 0; g < G; ++g) W = fmaf(triples[g * stride + 2 + c], exp_weight(triples[g * stride], beta, inv_lambda), W);
    const float u = (tl.U_src ? tl.U_src[c] : U[c]) + W / eta;  // mppi_delay.py:214-216
    U[c] = u;
    if (c < nu && action) action[c] = u * u_scale;  // :217-224
  }
  if (threadIdx.x == 0 && stats) { stats[0] = beta; stats[1] = eta; }
  __syncthreads();
  if (threadIdx.x == 0) *step_ctr = step + 1ull;
  step_tail(tl);
}

int launch_combine_exchange(float* mailbox, int G, int stride, int T, int nu, float lambda_, float u_scale, float* U, float* action,
                            float* stats, unsigned long long* step_ctr, unsigned int* status, const StepTail& tl, cudaStream_t s) {
  softmax_combine_exchange_kernel<<<1, 128, 0, s>>>(mailbox, G, stride, T * nu, nu, 1.0f / lambda_, u_scale, U, action, stats, step_ctr,
                                                    status, tl);
  NLC_LAUNCH_OK("softmax_combine_exchange_kernel");
  return NLC_OK;
}

static int sum_grid(int K) {
  int g = (K + 255) / 256;  // >= 256 rows per block
  if (g > 148 * 4) g = 148 * 4;
  if (g < 1) g = 1;
  return g;
}

}  // namespace nlc

using namespace nlc;

extern "C" int64_t nlc_softmax_workspace_bytes(int K, int TN) {
  return 256 + (int64_t)sum_grid(K) * (1 + TN) * (int64_t)sizeof(float);
}

namespace nlc {
// planner.cu: stage 4's shard-local half.  with_init = false: the workspace header was re-armed by the previous step's
// combine kernel (StepTail); pub: publish the triple to connected shards from the sum kernel's last block.
int softmax_partial_impl(const float* cost_dev, const float* noise_dev, int K, int T, int nu, float lambda_, float* triple_dev,
                         float* weights_dev, void* workspace_dev, bool with_init, const ExchangePub& pub, cudaStream_t s);
int launch_combine(const float* triples_dev, int G, int T, int nu, float lambda_, float u_scale, float* U_dev, float* action_dev,
                   float* stats_dev, const StepTail& tl, cudaStream_t s) {
  softmax_combine_kernel<<<1, 128, 0, s>>>(triples_dev, G, T * nu, nu, 1.0f / lambda_, u_scale, U_dev, action_dev, stats_dev, tl);
  NLC_LAUNCH_OK("softmax_combine_kernel");
  return NLC_OK;
}
}  // namespace nlc

extern "C" int nlc_softmax_partial(const float* cost_dev, const float* noise_dev, int K, int T, int nu, float lambda_,
                                   float* triple_dev, float* weights_dev, void* workspace_dev, void* stream) {
  return softmax_partial_impl(cost_dev, noise_dev, K, T, nu, lambda_, triple_dev, weights_dev, workspace_dev, true,
                              ExchangePub{nullptr, 0, 0, 0, nullptr}, static_cast<cudaStream_t>(stream));
}

int nlc::softmax_partial_impl(const float* cost_dev, const float* noise_dev, int K, int T, int nu, float lambda_, float* triple_dev,
                              float* weights_dev, void* workspace_dev, bool with_init, const ExchangePub& pub, cudaStream_t s) {
  NLC_REQUIRE(cost_dev && noise_dev && triple_dev && workspace_dev, NLC_ERR_ARG, "nlc_softmax_partial: null pointer");
  NLC_REQUIRE(K >= 1 && T >= 1 && nu >= 1, NLC_ERR_ARG, "nlc_softmax_partial: K, T, nu must be positive");
  const int TN = T * nu;
  NLC_REQUIRE(TN <= 256, NLC_ERR_SHAPE, "nlc_softmax_partial: T*nu = %d exceeds 256", TN);
  NLC_REQUIRE(lambda_ > 0.0f, NLC_ERR_ARG, "lambda must be positive");
  NLC_REQUIRE((reinterpret_cast<uintptr_t>(cost_dev) & 15) == 0, NLC_ERR_ARG, "cost_dev must be 16-byte aligned");
  SoftWs* ws = static_cast<SoftWs*>(workspace_dev);
  float* partials = reinterpret_cast<float*>(static_cast<char*>(workspace_dev) + 256);
  if (with_init) {
    softmax_init_kernel<<<1, 1, 0, s>>>(ws);
    NLC_LAUNCH_OK("softmax_init_kernel");
  }
  int gmin = (K / 4 + 255) / 256;
  if (gmin > 148 * 2) gmin = 148 * 2;
  if (gmin < 1) gmin = 1;
  softmax_min_kernel<<<gmin, 256, 0, s>>>(cost_dev, K, ws);
  NLC_LAUNCH_OK("softmax_min_kernel");
  const int grid = sum_grid(K);
  const int rows_per_block = (K + grid - 1) / grid;
  softmax_sum_kernel<<<grid, 256, 0, s>>>(cost_dev, noise_dev, K, TN, 1.0f / lambda_, ws, partials, triple_dev, weights_dev,
                                          rows_per_block, pub);
  NLC_LAUNCH_OK("softmax_sum_kernel");
  return NLC_OK;
}

extern "C" int nlc_softmax_combine(const float* triples_dev, int G, int T, int nu, float lambda_, float u_scale,
                                   float* U_dev, float* action_dev, float* stats_dev, void* stream) {
  NLC_REQUIRE(triples_dev && U_dev, NLC_ERR_ARG, "nlc_softmax_combine: null pointer");
  NLC_REQUIRE(G >= 1 && T >= 1 && nu >= 1 && lambda_ > 0.0f, NLC_ERR_ARG, "nlc_softmax_combine: bad sizes");
  softmax_combine_kernel<<<1, 128, 0, static_cast<cudaStream_t>(stream)>>>(triples_dev, G, T * nu, nu, 1.0f / lambda_,
                                                                           u_scale, U_dev, action_dev, stats_dev,
                                                                           StepTail{nullptr, nullptr, nullptr, nullptr, 0, nullptr, nullptr, nullptr, 0});
  NLC_LAUNCH_OK("softmax_combine_kernel");
  return NLC_OK;
}
