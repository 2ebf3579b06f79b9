// Stages 2+3 with the analytic delayed dynamics in the planner's `dynamics` slot
// (oracle.py:11-224 behind mppi_with_model.py:129-143): one thread per sample, the horizon in registers.
#include "common.cuh"
#include "env_cost.cuh"

namespace nlc {

template <int NX>
__global__ void __launch_bounds__(128) rollout_analytic_kernel(nlc_rollout_opts o, const float* __restrict__ state0,
                                                               int sps, const float* __restrict__ hist,
                                                               const float* __restrict__ pert_cost, int K, int T, int B,
                                                               int nu, float* __restrict__ cost, float* __restrict__ states) {
  const int k = blockIdx.x * blockDim.x + threadIdx.x;
  if (k >= K) return;
  const int L = B - 1 + T;
  float s[NX];
#pragma unroll
  for (int c = 0; c < NX; ++c) s[c] = state0[(size_t)(sps ? k / sps : 0) * NX + c];
  float acc = 0.0f;
  const float* h = hist + (size_t)k * L * nu;
  for (int t = 0; t < T; ++t) {
    // window = hist[t : t+B]; delayed action = window[-(delay+1)] (oracle.py:23,99,187)
    env_analytic_step(o, s, h + (size_t)(t + B - 1 - o.delay) * nu);
    acc += env_running_cost(o, s, h + (size_t)(t + B - 1) * nu, nu);  // mppi_delay.py:288-290
    if (states) {
#pragma unroll
      for (int c = 0; c < NX; ++c) states[((size_t)k * T + t) * NX + c] = s[c];
    }
  }
  cost[k] = acc + (pert_cost ? pert_cost[k] : 0.0f);
}

int launch_rollout_analytic(const nlc_rollout_opts* o, int nx, const float* state, int sps, const float* hist,
                            const float* pert_cost, int K, int T, int B, int nu, float* cost, float* states,
                            cudaStream_t stream) {
  const int grid = (K + 127) / 128;
  switch (nx) {
    case 3: rollout_analytic_kernel<3><<<grid, 128, 0, stream>>>(*o, state, sps, hist, pert_cost, K, T, B, nu, cost, states); break;
    case 5: rollout_analytic_kernel<5><<<grid, 128, 0, stream>>>(*o, state, sps, hist, pert_cost, K, T, B, nu, cost, states); break;
    case 6: rollout_analytic_kernel<6><<<grid, 128, 0, stream>>>(*o, state, sps, hist, pert_cost, K, T, B, nu, cost, states); break;
    default: set_error("analytic rollout: unsupported nx %d", nx); return NLC_ERR_SHAPE;
  }
  NLC_LAUNCH_OK("rollout_analytic_kernel");
  return NLC_OK;
}

// One closed-loop environment step for I independent instances (mppi_with_model.py:193-216, step_env): roll the action
// buffer and pick the delayed action (get_action, :25-28), advance the state by one explicit-Euler step of the true
// dynamics (base_env.py:136-173 integrate_system(2, ...) as stated analytically by oracle.py:11-224, observation form),
// reward of the new state with the applied action (base_env.py diff_reward = -running_cost).
// delays (optional, [I]): instance i's own delay instead of o.delay.  An entry outside [0, B) sets *status = 1 and leaves
// that instance's state, buffer and reward untouched.
template <int NX>
__global__ void env_step_kernel(nlc_rollout_opts o, const int32_t* __restrict__ delays, float* __restrict__ state,
                                float* __restrict__ abuf, const float* __restrict__ action, int I, int B, int nu,
                                float* __restrict__ reward, unsigned int* __restrict__ status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= I) return;
  const int delay = delays ? delays[i] : o.delay;
  if (delay < 0 || delay >= B) { if (status) *status = 1u; return; }
  float* b = abuf + (size_t)i * B * nu;
  for (int j = 0; j + 1 < B; ++j)
    for (int u = 0; u < nu; ++u) b[j * nu + u] = b[(j + 1) * nu + u];
  for (int u = 0; u < nu; ++u) b[(B - 1) * nu + u] = action[(size_t)i * nu + u];
  const float* at = b + (size_t)(B - 1 - delay) * nu;
  float s[NX];
#pragma unroll
  for (int c = 0; c < NX; ++c) s[c] = state[(size_t)i * NX + c];
  env_analytic_step(o, s, at);
#pragma unroll
  for (int c = 0; c < NX; ++c) state[(size_t)i * NX + c] = s[c];
  if (reward) reward[i] = -env_running_cost(o, s, at, nu);
}

// env_step_kernel in fp64 (the closed loop around the fp64 planner): the same buffer roll and delayed action, the fp64 Euler
// step and running cost of env_cost.cuh that the fp64 planner's analytic rollout uses, dt in fp64.
template <int NX>
__global__ void env_step_f64_kernel(int env, int delay0, const int32_t* __restrict__ delays, double dt, double* __restrict__ state,
                                    double* __restrict__ abuf, const double* __restrict__ action, int I, int B, int nu,
                                    double* __restrict__ reward, unsigned int* __restrict__ status) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= I) return;
  const int delay = delays ? delays[i] : delay0;
  if (delay < 0 || delay >= B) { if (status) *status = 1u; return; }
  double* b = abuf + (size_t)i * B * nu;
  for (int j = 0; j + 1 < B; ++j)
    for (int u = 0; u < nu; ++u) b[j * nu + u] = b[(j + 1) * nu + u];
  for (int u = 0; u < nu; ++u) b[(B - 1) * nu + u] = action[(size_t)i * nu + u];
  const double* at = b + (size_t)(B - 1 - delay) * nu;
  double s[NX];
#pragma unroll
  for (int c = 0; c < NX; ++c) s[c] = state[(size_t)i * NX + c];
  env_analytic_step(env, dt, s, at);
#pragma unroll
  for (int c = 0; c < NX; ++c) state[(size_t)i * NX + c] = s[c];
  if (reward) reward[i] = -env_running_cost(env, 0, 0.0, s, at, nu);
}

// The argument checks of both precisions, before any CUDA call.  delay_dev == nullptr: the scalar delay, checked here;
// otherwise the per-instance delays, checked on the device (status_dev required).
static int env_step_check(const char* name, int env, int delay, const int32_t* delay_dev, unsigned int* status_dev, const void* state_dev,
                          const void* action_buffer_dev, const void* action_dev, int I, int B, int nu) {
  NLC_REQUIRE(state_dev && action_buffer_dev && action_dev, NLC_ERR_ARG, "%s: null pointer", name);
  NLC_REQUIRE(!delay_dev || status_dev, NLC_ERR_ARG, "%s: per-instance delays need a status word", name);
  NLC_REQUIRE(I >= 1 && B >= 1 && B <= 8, NLC_ERR_ARG, "%s: I >= 1 and 1 <= B <= 8 required", name);
  NLC_REQUIRE(env >= NLC_ENV_PENDULUM && env <= NLC_ENV_ACROBOT, NLC_ERR_ARG, "unknown env id %d", env);
  NLC_REQUIRE(delay_dev || (delay >= 0 && delay < B), NLC_ERR_ARG, "%s: delay %d outside the %d-entry action buffer", name, delay, B);
  const int env_nu[3] = {1, 1, 2};
  NLC_REQUIRE(nu == env_nu[env], NLC_ERR_SHAPE, "env %d takes nu=%d actions, got %d", env, env_nu[env], nu);
  int dev = 0;
  NLC_CUDA_OK(cudaGetDevice(&dev));
  return check_device_arch(dev);
}

static int env_step_launch(const nlc_rollout_opts* o, const int32_t* delay_dev, float* state_dev, float* action_buffer_dev,
                           const float* action_dev, int I, int B, int nu, float* reward_dev, unsigned int* status_dev, void* stream) {
  NLC_REQUIRE(o, NLC_ERR_ARG, "nlc_env_step: null pointer");
  int rc = env_step_check("nlc_env_step", o->env, o->delay, delay_dev, status_dev, state_dev, action_buffer_dev, action_dev, I, B, nu);
  if (rc != NLC_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int grid = (I + 127) / 128;
  if (o->env == NLC_ENV_PENDULUM) env_step_kernel<3><<<grid, 128, 0, s>>>(*o, delay_dev, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev);
  else if (o->env == NLC_ENV_CARTPOLE) env_step_kernel<5><<<grid, 128, 0, s>>>(*o, delay_dev, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev);
  else env_step_kernel<6><<<grid, 128, 0, s>>>(*o, delay_dev, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev);
  NLC_LAUNCH_OK("env_step_kernel");
  return NLC_OK;
}

static int env_step_f64_launch(int env, int delay, const int32_t* delay_dev, double dt, double* state_dev, double* action_buffer_dev,
                               const double* action_dev, int I, int B, int nu, double* reward_dev, unsigned int* status_dev, void* stream) {
  int rc = env_step_check("nlc_env_step_f64", env, delay, delay_dev, status_dev, state_dev, action_buffer_dev, action_dev, I, B, nu);
  if (rc != NLC_OK) return rc;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  const int grid = (I + 127) / 128;
  if (env == NLC_ENV_PENDULUM) env_step_f64_kernel<3><<<grid, 128, 0, s>>>(env, delay, delay_dev, dt, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev);
  else if (env == NLC_ENV_CARTPOLE) env_step_f64_kernel<5><<<grid, 128, 0, s>>>(env, delay, delay_dev, dt, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev);
  else env_step_f64_kernel<6><<<grid, 128, 0, s>>>(env, delay, delay_dev, dt, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev);
  NLC_LAUNCH_OK("env_step_f64_kernel");
  return NLC_OK;
}

}  // namespace nlc

extern "C" int nlc_env_step(const nlc_rollout_opts* o, float* state_dev, float* action_buffer_dev, const float* action_dev,
                            int I, int B, int nu, float* reward_dev, void* stream) {
  return nlc::env_step_launch(o, nullptr, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, nullptr, stream);
}

extern "C" int nlc_env_step_delays(const nlc_rollout_opts* o, const int32_t* delay_dev, float* state_dev, float* action_buffer_dev,
                                   const float* action_dev, int I, int B, int nu, float* reward_dev, unsigned int* status_dev,
                                   void* stream) {
  NLC_REQUIRE(delay_dev, NLC_ERR_ARG, "nlc_env_step_delays: null delays");
  return nlc::env_step_launch(o, delay_dev, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev, stream);
}

extern "C" int nlc_env_step_f64(int env, int delay, double dt, double* state_dev, double* action_buffer_dev, const double* action_dev,
                                int I, int B, int nu, double* reward_dev, void* stream) {
  return nlc::env_step_f64_launch(env, delay, nullptr, dt, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, nullptr, stream);
}

extern "C" int nlc_env_step_f64_delays(int env, const int32_t* delay_dev, double dt, double* state_dev, double* action_buffer_dev,
                                       const double* action_dev, int I, int B, int nu, double* reward_dev, unsigned int* status_dev,
                                       void* stream) {
  NLC_REQUIRE(delay_dev, NLC_ERR_ARG, "nlc_env_step_f64_delays: null delays");
  return nlc::env_step_f64_launch(env, 0, delay_dev, dt, state_dev, action_buffer_dev, action_dev, I, B, nu, reward_dev, status_dev, stream);
}
