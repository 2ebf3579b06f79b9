// fp64 planner (nlc_planner_f64_*): MPPIDelay.command (mppi_delay.py:193-224) in fp64 throughout, the precision the reference
// plans in.  A handle of its own beside nlc_planner_t: no tensor cores, no encoder beside the rollout, no device exchange, no
// graphs and no mapped staging - one fixed sequence of direct launches per control step:
//   plan_f64_perturb_kernel           stage 1 (warp per sample, lanes over the horizon, as perturb_kernel)
//   f64_encode_kernel                 the K T history windows through the fp64 encoder     } model_grad.cu (the tile steps
//   plan_f64_rollout_kernel           tiles of 32 samples through the whole horizon         }  of the fp64 model)
//   (plan_f64_rollout_analytic_kernel instead of both for the analytic dynamics)
//   plan_f64_softmax_kernel           beta, w = exp(-(1/lambda)(c - beta)), eta              } stage 4: fixed-order sums,
//   plan_f64_update_partial_kernel    per-block sums of (w_k / eta) noise[k] over a k-range  }  bit-identical from call
//   plan_f64_update_finish_kernel     U = rolled U + the partials in block order, action     }  to call
#include <math.h>
#include <string.h>

#include "common.cuh"
#include "env_cost.cuh"

namespace nlc {

// model_grad.cu
size_t plan_f64_image_doubles(nlc_model_t m);
size_t plan_f64_scratch_doubles(nlc_model_t m, int B, int K, int T);
int plan_f64_set_params(nlc_model_t m, const double* params_dev, const double* ts_dev, double* img, double* row_b1, double* row_tn,
                        cudaStream_t s);
int encode_windows_f64(nlc_model_t m, int B, const double* img, const double* hist, int hist_ch, int K, int T, double* p_out,
                       double* scratch, cudaStream_t s);
int plan_f64_rollout(nlc_model_t m, int B, const double* img, const double* row_b1, const double* row_tn, const double* state0, int sps,
                     const double* hist, const double* p, const double* pert_cost, int K, int T, int env, int state_constraint,
                     double goal_x, double* cost, double* states, double* scratch, cudaStream_t s);

constexpr int kF64UpdateBlocks = 148;  // stage 4's k-range blocks at most: fixed, so the summation order depends on K only

}  // namespace nlc

struct nlc_planner_f64_s {
  int device;
  nlc_model_t model;
  nlc_planner_f64_desc d;
  uint64_t calls;      // control steps taken: the sampler's call index
  bool params_set;
  int n_blocks;        // stage 4's k-range blocks
  void* arena;
  double *U, *U_roll, *noise, *perturbed, *hist, *actions, *pert_cost, *p, *cost_total, *weights, *states, *action, *stats,
      *state_in, *abuf_in, *part, *ts, *img, *row_b1, *row_tn, *scratch;
};

namespace nlc {

struct PerturbF64Args {
  int K, T, nu, B, sample_null_action, noise_abs_cost, has_bounds;
  double lambda_, u_scale, u_min[4], u_max[4], sigma_inv[16], sigma_chol[16], noise_mu[4], u_init[4];
  uint32_t seed_lo, seed_hi, call_lo, call_hi;
  const double *U, *noise_in, *action_buffer;
  double *U_roll, *perturbed, *noise, *hist, *actions, *pert_cost;
};

// The standard normals of (sample k, step t): the transform stated in include/nlc_b200.h.
__device__ __forceinline__ double philox_uniform53(uint32_t hi, uint32_t lo) {
  const uint64_t m = ((uint64_t)(hi >> 6) << 26) | (lo >> 6);  // 52 bits
  return (double)(2 * m + 1) * 0x1p-53;                      // odd multiple of 2^-53: in (0, 1), exact
}

__device__ __forceinline__ void philox_normals_f64(const PerturbF64Args& a, uint64_t idx, double z[4]) {
  for (int b = 0; b < (a.nu > 2 ? 2 : 1); ++b) {
    uint32_t c[4] = {(uint32_t)idx, (uint32_t)(idx >> 32), a.call_lo, b ? a.call_hi ^ 0x80000000u : a.call_hi};
    philox4x32_10(c, a.seed_lo, a.seed_hi);
    const double u1 = philox_uniform53(c[0], c[1]), u2 = philox_uniform53(c[2], c[3]);
    const double r = sqrt(-2.0 * log(u1));
    double s, co;
    sincospi(2.0 * u2, &s, &co);
    z[2 * b] = r * co;
    z[2 * b + 1] = r * s;
  }
}

__device__ __forceinline__ double warp_sum_f64(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Stage 1 (mppi_delay.py:199-200, 255-260, 319-343, 347-356); the elementwise chain with explicit round-to-nearest operations
// (no contraction), so perturbed, noise, hist and actions are the reference's fp64 values bit for bit.
template <int NU>
__global__ void __launch_bounds__(256) plan_f64_perturb_kernel(PerturbF64Args a) {
  const int T = a.T, B = a.B, L = B - 1 + T;
  const int lane = threadIdx.x & 31;
  const int warp_in_grid = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  const double u_scale = a.u_scale;
  if (blockIdx.x == 0)  // the rolled U stage 4 updates (mppi_delay.py:199-200)
    for (int i = threadIdx.x; i < T * NU; i += blockDim.x) a.U_roll[i] = i < (T - 1) * NU ? a.U[i + NU] : a.u_init[i - (T - 1) * NU];
  for (int k = warp_in_grid; k < a.K; k += n_warps) {
    double pc = 0.0;
    for (int t = lane; t < T; t += 32) {
      double Ut[NU], nz[NU];
#pragma unroll
      for (int u = 0; u < NU; ++u) Ut[u] = t < T - 1 ? a.U[(t + 1) * NU + u] : a.u_init[u];
      const size_t e = ((size_t)k * T + t) * NU;
      if (a.noise_in) {
#pragma unroll
        for (int u = 0; u < NU; ++u) nz[u] = a.noise_in[e + u];
      } else {
        double z[4];
        philox_normals_f64(a, (uint64_t)k * (uint64_t)T + (uint64_t)t, z);
#pragma unroll
        for (int u = 0; u < NU; ++u) {
          double acc = a.noise_mu[u];
#pragma unroll
          for (int v = 0; v <= u; ++v) acc = fma(a.sigma_chol[u * NU + v], z[v], acc);
          nz[u] = acc;
        }
      }
      double nb[NU];
#pragma unroll
      for (int u = 0; u < NU; ++u) {
        double pa = __dadd_rn(Ut[u], nz[u]);                                  // :321
        if (a.sample_null_action && k == a.K - 1) pa = 0.0;                  // :322-323
        double x = __dmul_rn(pa, u_scale);                                    // :325
        if (a.has_bounds) x = fmax(fmin(x, a.u_max[u]), a.u_min[u]);          // :347-353
        const double pert = __ddiv_rn(x, u_scale);                            // :326
        nb[u] = __dsub_rn(pert, Ut[u]);                                       // :328
        a.perturbed[e + u] = pert;
        a.noise[e + u] = nb[u];
        const double h = __dmul_rn(u_scale, pert);                            // :258 u_scale * perturbed
        a.hist[((size_t)k * L + (B - 1) + t) * NU + u] = h;
        a.actions[e + u] = __ddiv_rn(h, u_scale);                             // :340
      }
#pragma unroll
      for (int v = 0; v < NU; ++v) {  // action_cost = lambda * noise @ Sigma^-1 (:329-335), then sum(U * action_cost) (:343)
        double ac = 0.0;
#pragma unroll
        for (int u = 0; u < NU; ++u) ac = fma(a.lambda_ * (a.noise_abs_cost ? fabs(nb[u]) : nb[u]), a.sigma_inv[u * NU + v], ac);
        pc = fma(Ut[v], ac, pc);
      }
    }
    for (int j = lane; j < (B - 1) * NU; j += 32) a.hist[(size_t)k * L * NU + j] = a.action_buffer[NU + j];  // :255-257
    pc = warp_sum_f64(pc);
    if (lane == 0) a.pert_cost[k] = pc;
  }
}

// Stages 2+3 with the analytic delayed dynamics (oracle.py:11-224): one thread per sample, as rollout_analytic_kernel.
template <int NX>
__global__ void __launch_bounds__(128, 1) plan_f64_rollout_analytic_kernel(int env, int state_constraint, double goal_x, int delay, double dt,
                                                                        const double* __restrict__ state0, int sps,
                                                                        const double* __restrict__ hist, const double* __restrict__ pert_cost,
                                                                        int K, int T, int B, int nu, double* __restrict__ cost,
                                                                        double* __restrict__ states) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const int L = B - 1 + T;
  double s[NX];
#pragma unroll
  for (int c = 0; c < NX; ++c) s[c] = state0[(size_t)(sps ? k : 0) * NX + c];
  double acc = 0.0;
  const double* h = hist + (size_t)k * L * nu;
  for (int t = 0; t < T; ++t) {
    env_analytic_step(env, dt, s, h + (size_t)(t + B - 1 - delay) * nu);
    acc = acc + env_running_cost(env, state_constraint, goal_x, s, h + (size_t)(t + B - 1) * nu, nu);
    if (states) {
#pragma unroll
      for (int c = 0; c < NX; ++c) states[((size_t)k * T + t) * NX + c] = s[c];
    }
  }
  cost[k] = acc + pert_cost[k];
}

// Stage 4 (mppi_delay.py:210-216), first part: beta = min c; w = exp(-(1/lambda)(c - beta)); eta = sum w.  One block; thread
// i takes k = i, i + 1024, ... in order, then a fixed tree.
__global__ void __launch_bounds__(1024) plan_f64_softmax_kernel(const double* __restrict__ cost, int K, double inv_lambda,
                                                                double* __restrict__ w, double* __restrict__ stats) {
  __shared__ double red[1024];
  const int tid = threadIdx.x;
  double mn = INFINITY;
  for (int k = tid; k < K; k += 1024) mn = fmin(mn, cost[k]);
  red[tid] = mn;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if (tid < s) red[tid] = fmin(red[tid], red[tid + s]);
    __syncthreads();
  }
  const double beta = red[0];
  __syncthreads();
  double sum = 0.0;
  for (int k = tid; k < K; k += 1024) {
    const double v = exp(-(inv_lambda * (cost[k] - beta)));
    w[k] = v;
    sum += v;
  }
  red[tid] = sum;
  __syncthreads();
  for (int s = 512; s > 0; s >>= 1) {
    if (tid < s) red[tid] = red[tid] + red[tid + s];
    __syncthreads();
  }
  if (tid == 0) { stats[0] = beta; stats[1] = red[0]; }
}

// part[b][j] = sum over k in block b's range, ascending, of omega_k noise[k][j], omega = (1/eta) w (mppi_delay.py:212-216).
__global__ void __launch_bounds__(256) plan_f64_update_partial_kernel(const double* __restrict__ w, const double* __restrict__ stats,
                                                                      const double* __restrict__ noise, int K, int TN, int chunk,
                                                                      double* __restrict__ part) {
  const int k0 = blockIdx.x * chunk, k1 = min(K, k0 + chunk);
  const double inv_eta = 1.0 / stats[1];
  for (int j = threadIdx.x; j < TN; j += blockDim.x) {
    double acc = 0.0;
    for (int k = k0; k < k1; ++k) acc += (inv_eta * w[k]) * noise[(size_t)k * TN + j];
    part[(size_t)blockIdx.x * TN + j] = acc;
  }
}

__global__ void __launch_bounds__(256) plan_f64_update_finish_kernel(const double* __restrict__ part, int n_blocks, int TN, int nu,
                                                                     double u_scale, const double* __restrict__ U_roll,
                                                                     double* __restrict__ U, double* __restrict__ action) {
  for (int j = threadIdx.x; j < TN; j += blockDim.x) {
    double acc = 0.0;
    for (int b = 0; b < n_blocks; ++b) acc += part[(size_t)b * TN + j];
    const double u = U_roll[j] + acc;
    U[j] = u;
    if (j < nu) action[j] = u * u_scale;  // mppi_delay.py:217-224
  }
}

static void model_release(nlc_model_t m) {
  if (!m) return;
  if (--m->refs <= 0 && m->destroy_requested) { m->refs = 0; nlc_model_destroy(m); }
}

static int perturb_f64(nlc_planner_f64_t p, const double* noise_in, const double* action_buffer, cudaStream_t s) {
  const nlc_planner_f64_desc& d = p->d;
  const nlc_mppi_params& mp = d.base.mppi;
  PerturbF64Args a;
  a.K = mp.K; a.T = mp.T; a.nu = mp.nu; a.B = mp.B;
  a.sample_null_action = mp.sample_null_action; a.noise_abs_cost = mp.noise_abs_cost; a.has_bounds = mp.has_bounds;
  a.lambda_ = d.lambda_; a.u_scale = d.u_scale;
  memcpy(a.u_min, d.u_min, sizeof(a.u_min)); memcpy(a.u_max, d.u_max, sizeof(a.u_max));
  memcpy(a.sigma_inv, d.sigma_inv, sizeof(a.sigma_inv)); memcpy(a.sigma_chol, d.sigma_chol, sizeof(a.sigma_chol));
  memcpy(a.noise_mu, d.noise_mu, sizeof(a.noise_mu)); memcpy(a.u_init, d.u_init, sizeof(a.u_init));
  a.seed_lo = (uint32_t)d.base.seed; a.seed_hi = (uint32_t)(d.base.seed >> 32);
  a.call_lo = (uint32_t)p->calls; a.call_hi = (uint32_t)(p->calls >> 32);
  a.U = p->U; a.noise_in = noise_in; a.action_buffer = action_buffer;
  a.U_roll = p->U_roll; a.perturbed = p->perturbed; a.noise = p->noise; a.hist = p->hist; a.actions = p->actions;
  a.pert_cost = p->pert_cost;
  int blocks = (mp.K + 7) / 8;  // 8 warps per block, one sample per warp
  if (blocks > 148 * 32) blocks = 148 * 32;
  switch (mp.nu) {
    case 1: plan_f64_perturb_kernel<1><<<blocks, 256, 0, s>>>(a); break;
    case 2: plan_f64_perturb_kernel<2><<<blocks, 256, 0, s>>>(a); break;
    case 3: plan_f64_perturb_kernel<3><<<blocks, 256, 0, s>>>(a); break;
    default: plan_f64_perturb_kernel<4><<<blocks, 256, 0, s>>>(a); break;
  }
  NLC_LAUNCH_OK("plan_f64_perturb_kernel");
  return NLC_OK;
}

}  // namespace nlc

using namespace nlc;

extern "C" int nlc_planner_f64_create(nlc_planner_f64_t* out, nlc_model_t model, const nlc_planner_f64_desc* d, int device) {
  NLC_REQUIRE(out && d, NLC_ERR_ARG, "nlc_planner_f64_create: null argument");
  *out = nullptr;
  int rc = check_device_arch(device);
  if (rc != NLC_OK) return rc;
  const nlc_planner_desc& b = d->base;
  const nlc_mppi_params& mp = b.mppi;
  NLC_REQUIRE(b.n_shards == 1, NLC_ERR_UNSUPPORTED, "fp64 planner: n_shards = %d; the fp64 planner is single-shard", b.n_shards);
  NLC_REQUIRE(mp.K >= 1 && mp.T >= 1 && mp.B >= 1 && mp.B <= 8, NLC_ERR_SHAPE, "fp64 planner: K, T >= 1 and 1 <= B <= 8 required");
  NLC_REQUIRE(mp.nu >= 1 && mp.nu <= 4 && b.nx >= 1 && b.nx <= kMaxNx, NLC_ERR_SHAPE, "fp64 planner: nu/nx out of range");
  NLC_REQUIRE(mp.T * mp.nu <= 256, NLC_ERR_SHAPE, "fp64 planner: T*nu exceeds 256");
  NLC_REQUIRE(d->lambda_ > 0.0 && d->u_scale != 0.0, NLC_ERR_ARG, "fp64 planner: lambda must be positive and u_scale non-zero");
  const nlc_rollout_opts& o = b.rollout;
  NLC_REQUIRE(o.env >= NLC_ENV_PENDULUM && o.env <= NLC_ENV_ACROBOT, NLC_ERR_ARG, "fp64 planner: unknown env id %d", o.env);
  const int env_nx[3] = {3, 5, 6}, env_nu[3] = {1, 1, 2};
  NLC_REQUIRE(b.nx == env_nx[o.env] && mp.nu == env_nu[o.env], NLC_ERR_SHAPE, "fp64 planner: env %d has nx=%d, nu=%d", o.env,
              env_nx[o.env], env_nu[o.env]);
  if (o.dynamics == NLC_DYN_NEURAL_LAPLACE) {
    NLC_REQUIRE(model != nullptr, NLC_ERR_ARG, "fp64 planner: Neural Laplace dynamics need a model handle");
    NLC_REQUIRE(model->device == device, NLC_ERR_ARG, "fp64 planner: model lives on device %d, planner on %d", model->device, device);
    NLC_REQUIRE(model->nx == b.nx && model->nu == mp.nu, NLC_ERR_SHAPE, "fp64 planner: model dims do not match");
    NLC_REQUIRE(!model->destroy_requested, NLC_ERR_ARG, "fp64 planner: the model handle has been destroyed");
  } else {
    NLC_REQUIRE(o.dynamics == NLC_DYN_ANALYTIC_DELAY, NLC_ERR_ARG, "fp64 planner: unknown dynamics kind %d", o.dynamics);
    NLC_REQUIRE(o.delay >= 0 && o.delay < mp.B, NLC_ERR_ARG, "fp64 planner: delay %d outside the %d-entry window", o.delay, mp.B);
    model = nullptr;
  }
  nlc_planner_f64_s* p = new nlc_planner_f64_s();
  memset(p, 0, sizeof(*p));
  p->device = device; p->model = model; p->d = *d;
  const size_t K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, nx = b.nx, L = B - 1 + T, TN = T * nu;
  p->n_blocks = (int)((K + 255) / 256 < (size_t)kF64UpdateBlocks ? (K + 255) / 256 : kF64UpdateBlocks);
  const bool nl = model != nullptr;
  const size_t sizes[] = {TN, TN, K * TN, K * TN, K * L * nu, K * TN, K, nl ? K * T * 2 : 0, K, K, b.keep_states ? K * T * nx : 0,
                          4, 2, K * nx, B * nu, (size_t)p->n_blocks * TN, 1, nl ? plan_f64_image_doubles(model) : 0,
                          nl ? (size_t)model->Hm : 0, 1, nl ? plan_f64_scratch_doubles(model, (int)B, (int)K, (int)T) : 0};
  double** slots[] = {&p->U, &p->U_roll, &p->noise, &p->perturbed, &p->hist, &p->actions, &p->pert_cost, &p->p, &p->cost_total,
                      &p->weights, &p->states, &p->action, &p->stats, &p->state_in, &p->abuf_in, &p->part, &p->ts, &p->img,
                      &p->row_b1, &p->row_tn, &p->scratch};
  const int n_slots = sizeof(slots) / sizeof(slots[0]);
  size_t offs[n_slots], total = 0;
  for (int i = 0; i < n_slots; ++i) { offs[i] = total; total += (sizes[i] + 63) / 64 * 64; }
  auto fail = [&](int code) {
    if (p->arena) cudaFree(p->arena);
    delete p;
    return code;
  };
  if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice failed"); return fail(NLC_ERR_CUDA); }
  if (cudaMalloc(&p->arena, total * sizeof(double)) != cudaSuccess) {
    cudaGetLastError(); p->arena = nullptr;
    set_error("fp64 planner: cudaMalloc(%zu) failed", total * sizeof(double));
    return fail(NLC_ERR_NOMEM);
  }
  if (cudaMemset(p->arena, 0, total * sizeof(double)) != cudaSuccess) { set_error("fp64 planner: memset failed"); return fail(NLC_ERR_CUDA); }
  double* base = static_cast<double*>(p->arena);
  for (int i = 0; i < n_slots; ++i) *slots[i] = sizes[i] ? base + offs[i] : nullptr;
  if (cudaMemcpyAsync(p->ts, &d->dt, sizeof(double), cudaMemcpyHostToDevice, cudaStreamLegacy) != cudaSuccess ||
      cudaStreamSynchronize(cudaStreamLegacy) != cudaSuccess) {
    set_error("fp64 planner: copy of dt failed");
    return fail(NLC_ERR_CUDA);
  }
  if (model) model->refs++;
  *out = p;
  return NLC_OK;
}

extern "C" int nlc_planner_f64_destroy(nlc_planner_f64_t p) {
  if (!p) return NLC_OK;
  cudaSetDevice(p->device);
  cudaDeviceSynchronize();  // no kernel of this planner may still read the model when the last reference goes
  model_release(p->model);
  if (p->arena) cudaFree(p->arena);
  cudaGetLastError();
  delete p;
  return NLC_OK;
}

extern "C" int nlc_planner_f64_set_params(nlc_planner_f64_t p, const double* params_dev, void* stream) {
  NLC_REQUIRE(p && params_dev, NLC_ERR_ARG, "nlc_planner_f64_set_params: null argument");
  NLC_REQUIRE(p->model, NLC_ERR_ARG, "nlc_planner_f64_set_params: the planner has analytic dynamics, no model");
  NLC_REQUIRE(!p->model->destroy_requested, NLC_ERR_ARG, "fp64 planner: its model handle has been destroyed");
  NLC_CUDA_OK(cudaSetDevice(p->device));
  const int rc = plan_f64_set_params(p->model, params_dev, p->ts, p->img, p->row_b1, p->row_tn, static_cast<cudaStream_t>(stream));
  if (rc == NLC_OK) p->params_set = true;
  return rc;
}

extern "C" int nlc_planner_f64_set_U(nlc_planner_f64_t p, const double* U_host) {
  NLC_REQUIRE(p && U_host, NLC_ERR_ARG, "nlc_planner_f64_set_U: null argument");
  NLC_CUDA_OK(cudaSetDevice(p->device));
  const size_t n = (size_t)p->d.base.mppi.T * p->d.base.mppi.nu;
  NLC_CUDA_OK(cudaMemcpyAsync(p->U, U_host, sizeof(double) * n, cudaMemcpyHostToDevice, cudaStreamLegacy));
  NLC_CUDA_OK(cudaStreamSynchronize(cudaStreamLegacy));
  return NLC_OK;
}

extern "C" int nlc_planner_f64_get_U(nlc_planner_f64_t p, double* U_host) {
  NLC_REQUIRE(p && U_host, NLC_ERR_ARG, "nlc_planner_f64_get_U: null argument");
  NLC_CUDA_OK(cudaSetDevice(p->device));
  const size_t n = (size_t)p->d.base.mppi.T * p->d.base.mppi.nu;
  NLC_CUDA_OK(cudaMemcpyAsync(U_host, p->U, sizeof(double) * n, cudaMemcpyDeviceToHost, cudaStreamLegacy));
  NLC_CUDA_OK(cudaStreamSynchronize(cudaStreamLegacy));
  return NLC_OK;
}

extern "C" int nlc_planner_f64_buffer(nlc_planner_f64_t p, int which, void** dev_ptr, int64_t* n_doubles) {
  NLC_REQUIRE(p && dev_ptr && n_doubles, NLC_ERR_ARG, "nlc_planner_f64_buffer: null argument");
  const nlc_mppi_params& mp = p->d.base.mppi;
  const int64_t K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, nx = p->d.base.nx, TN = T * nu;
  double* ptr = nullptr;
  int64_t n = 0;
  switch (which) {
    case NLC_BUF_U: ptr = p->U; n = TN; break;
    case NLC_BUF_NOISE: ptr = p->noise; n = K * TN; break;
    case NLC_BUF_PERTURBED: ptr = p->perturbed; n = K * TN; break;
    case NLC_BUF_COST_TOTAL: ptr = p->cost_total; n = K; break;
    case NLC_BUF_WEIGHTS: ptr = p->weights; n = K; break;
    case NLC_BUF_STATES: ptr = p->states; n = p->states ? K * T * nx : 0; break;
    case NLC_BUF_ACTIONS: ptr = p->actions; n = K * TN; break;
    case NLC_BUF_ACTION: ptr = p->action; n = nu; break;
    case NLC_BUF_STATS: ptr = p->stats; n = 2; break;
    case NLC_BUF_HIST: ptr = p->hist; n = K * (B - 1 + T) * nu; break;
    case NLC_BUF_P: ptr = p->p; n = p->p ? K * T * 2 : 0; break;
    case NLC_BUF_STATE: ptr = p->state_in; n = K * nx; break;
    case NLC_BUF_ACTION_BUFFER: ptr = p->abuf_in; n = B * nu; break;
    default: set_error("nlc_planner_f64_buffer: buffer id %d is not a buffer of the fp64 planner", which); return NLC_ERR_ARG;
  }
  *dev_ptr = ptr;
  *n_doubles = n;
  return NLC_OK;
}

extern "C" int nlc_planner_f64_command(nlc_planner_f64_t p, const double* state_dev, int state_per_sample, const double* action_buffer_dev,
                                       const double* noise_in_dev, void* stream) {
  NLC_REQUIRE(p && state_dev && action_buffer_dev, NLC_ERR_ARG, "nlc_planner_f64_command: null argument");
  NLC_REQUIRE(state_per_sample == 0 || state_per_sample == 1, NLC_ERR_ARG, "nlc_planner_f64_command: state_per_sample must be 0 or 1");
  if (p->model) {
    NLC_REQUIRE(!p->model->destroy_requested, NLC_ERR_ARG, "fp64 planner: its model handle has been destroyed");
    NLC_REQUIRE(p->params_set, NLC_ERR_ARG, "fp64 planner: no parameters yet; call nlc_planner_f64_set_params first");
  }
  NLC_CUDA_OK(cudaSetDevice(p->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const nlc_planner_desc& b = p->d.base;
  const nlc_mppi_params& mp = b.mppi;
  const int K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, TN = T * nu;
  int rc = perturb_f64(p, noise_in_dev, action_buffer_dev, s);
  if (rc != NLC_OK) return rc;
  if (p->model) {
    rc = encode_windows_f64(p->model, B, p->img, p->hist, nu, K, T, p->p, p->scratch, s);
    if (rc != NLC_OK) return rc;
    rc = plan_f64_rollout(p->model, B, p->img, p->row_b1, p->row_tn, state_dev, state_per_sample, p->hist, p->p, p->pert_cost, K, T,
                          b.rollout.env, b.rollout.state_constraint, p->d.goal_x, p->cost_total, p->states, p->scratch, s);
    if (rc != NLC_OK) return rc;
  } else {
    const nlc_rollout_opts& o = b.rollout;
    const int grid = (K + 127) / 128;
    switch (b.nx) {
      case 3: plan_f64_rollout_analytic_kernel<3><<<grid, 128, 0, s>>>(o.env, o.state_constraint, p->d.goal_x, o.delay, p->d.dt, state_dev,
                                                                       state_per_sample, p->hist, p->pert_cost, K, T, B, nu, p->cost_total, p->states); break;
      case 5: plan_f64_rollout_analytic_kernel<5><<<grid, 128, 0, s>>>(o.env, o.state_constraint, p->d.goal_x, o.delay, p->d.dt, state_dev,
                                                                       state_per_sample, p->hist, p->pert_cost, K, T, B, nu, p->cost_total, p->states); break;
      default: plan_f64_rollout_analytic_kernel<6><<<grid, 128, 0, s>>>(o.env, o.state_constraint, p->d.goal_x, o.delay, p->d.dt, state_dev,
                                                                        state_per_sample, p->hist, p->pert_cost, K, T, B, nu, p->cost_total, p->states); break;
    }
    NLC_LAUNCH_OK("plan_f64_rollout_analytic_kernel");
  }
  plan_f64_softmax_kernel<<<1, 1024, 0, s>>>(p->cost_total, K, 1.0 / p->d.lambda_, p->weights, p->stats);
  NLC_LAUNCH_OK("plan_f64_softmax_kernel");
  const int chunk = (K + p->n_blocks - 1) / p->n_blocks;
  plan_f64_update_partial_kernel<<<p->n_blocks, 256, 0, s>>>(p->weights, p->stats, p->noise, K, TN, chunk, p->part);
  NLC_LAUNCH_OK("plan_f64_update_partial_kernel");
  plan_f64_update_finish_kernel<<<1, 256, 0, s>>>(p->part, p->n_blocks, TN, nu, p->d.u_scale, p->U_roll, p->U, p->action);
  NLC_LAUNCH_OK("plan_f64_update_finish_kernel");
  p->calls++;
  return NLC_OK;
}

extern "C" int nlc_planner_f64_command_host(nlc_planner_f64_t p, const double* state_host, const double* action_buffer_host,
                                            double* action_host, void* stream) {
  NLC_REQUIRE(p && state_host && action_buffer_host && action_host, NLC_ERR_ARG, "nlc_planner_f64_command_host: null argument");
  NLC_CUDA_OK(cudaSetDevice(p->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const nlc_mppi_params& mp = p->d.base.mppi;
  NLC_CUDA_OK(cudaMemcpyAsync(p->state_in, state_host, sizeof(double) * p->d.base.nx, cudaMemcpyHostToDevice, s));
  NLC_CUDA_OK(cudaMemcpyAsync(p->abuf_in, action_buffer_host, sizeof(double) * mp.B * mp.nu, cudaMemcpyHostToDevice, s));
  const int rc = nlc_planner_f64_command(p, p->state_in, 0, p->abuf_in, nullptr, stream);
  if (rc != NLC_OK) return rc;
  NLC_CUDA_OK(cudaMemcpyAsync(action_host, p->action, sizeof(double) * mp.nu, cudaMemcpyDeviceToHost, s));
  NLC_CUDA_OK(cudaStreamSynchronize(s));
  return NLC_OK;
}
