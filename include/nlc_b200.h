/*
 * nlc_b200.h - C ABI of libnlc_b200.so: the MPPI planning hot path of
 * samholt/NeuralLaplaceControl as hand-written sm_100a CUDA kernels.
 *
 * The reference has no FFI for this path (it is pure Python/PyTorch); the boundary a maintainer
 * would bind is therefore the set of Python callables below.  Each entry point names the
 * reference interface it replaces (file:line relative to the reference tree).  All pointers are
 * plain C pointers; "dev" pointers are CUDA device addresses on the device the handle was created
 * on, "host" pointers are ordinary host memory.  Every function returns 0 on success or a
 * negative nlc_status; nlc_last_error() returns a thread-local message for the last failure.
 * There is no CPU fallback anywhere: without a compute-capability 10.x device every compute
 * entry point returns NLC_ERR_ARCH.
 *
 * Arithmetic: fp32 on the device (the reference runs fp64 on the CPU, mppi_with_model.py:65,101);
 * host-side constant folding is done in fp64 and rounded once.  The model's fp64 entry points
 * (nlc_model_forward_f64 / nlc_model_backward_f64) and the fp64 planner (nlc_planner_f64_*) compute in fp64 throughout.
 */
#ifndef NLC_B200_H
#define NLC_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define NLC_VERSION 100

typedef enum {
  NLC_OK = 0,
  NLC_ERR_ARG = -1,         /* null pointer / invalid enum / non-positive size                     */
  NLC_ERR_SHAPE = -2,       /* dimension outside what the kernels are built for                    */
  NLC_ERR_ARCH = -3,        /* no CUDA device of compute capability 10.x                           */
  NLC_ERR_CUDA = -4,        /* a CUDA runtime call or kernel launch failed                         */
  NLC_ERR_UNSUPPORTED = -5, /* an option of the reference that this path rejects loudly            */
  NLC_ERR_NOMEM = -6
} nlc_status;

/* Environments whose reward the cost stage implements (mppi_with_model.py:145-171 closure over
 * envs/oderl/envs/ctpendulum.py:139-155, ctcartpole.py:289-346, ctacrobot.py:233-255).           */
typedef enum { NLC_ENV_PENDULUM = 0, NLC_ENV_CARTPOLE = 1, NLC_ENV_ACROBOT = 2 } nlc_env;

/* How the rollout advances the state (the `dynamics` slot of MPPIDelay, mppi_delay.py:66,187).    */
typedef enum {
  NLC_DYN_NEURAL_LAPLACE = 0, /* state + NeuralLaplaceModel(state, window, dt)  mppi_with_model.py:103-122 */
  NLC_DYN_ANALYTIC_DELAY = 1  /* oracle.py:11-224 one Euler step with window[:, -(delay+1)]          */
} nlc_dynamics_kind;

/* GEMM arithmetic of the contractions (encoder GRU and representation MLP).                        */
typedef enum {
  NLC_MATH_FP32 = 0,     /* CUDA-core FFMA, fp32 throughout: the 1e-4 parity anchor                 */
  NLC_MATH_TC_SPLIT3 = 1,/* tcgen05 kind::f16, operands split hi+lo in fp16, 3 MMAs, fp32 accumulate */
  NLC_MATH_TC_FP16 = 2   /* tcgen05 kind::f16 single pass (looser bound, see DESIGN.md)              */
} nlc_math_mode;

const char* nlc_last_error(void);
int nlc_version(void);
/* 0 when `device` exists and is compute capability 10.x; NLC_ERR_ARCH otherwise.                   */
int nlc_device_check(int device);
/* number of kernels this library has launched in this process (bench.py's gpu_launches claim)     */
uint64_t nlc_launch_count(void);

/* ------------------------------------------------------------------------------------------------
 * Neural Laplace model handle.   Replaces w_nl.py:66-145 (NeuralLaplaceModel) with its
 * ReverseGRUEncoder (w_nl.py:14-29) and LaplaceRepresentationFunc (w_nl.py:32-63), built as
 * train_utils.py:29-54 does.  Weights are the reference state_dict tensors, row-major fp64 on the
 * host, in PyTorch's own layouts (Linear: [out][in]; GRU: [3*hidden][in], gate order r,z,n).
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t state_dim;      /* nx                                                                      */
  int32_t action_dim;     /* nu                                                                      */
  int32_t hidden_units;   /* MLP width (reference: 128); GRU hidden = hidden_units/2 (w_nl.py:95)    */
  int32_t s_terms;        /* S, ilt_reconstruction_terms                                             */
  int32_t encode_obs_time;/* GRU input = nu+1 when set (w_nl.py:19-20)                               */
  int32_t normalize;      /* w_nl.py:119-129                                                         */
  int32_t normalize_time;
  int32_t action_std_len; /* 1 or nu (train_utils.py builds a length-1 std that broadcasts)          */
  double dt;
  const double* state_mean;  /* [nx] */
  const double* state_std;   /* [nx] */
  const double* action_mean; /* [nu] */
  const double* action_std;  /* [action_std_len] */
  const double* gru_w_ih_l0; /* [3*Hg][gru_in] */
  const double* gru_w_hh_l0; /* [3*Hg][Hg] */
  const double* gru_b_ih_l0; /* [3*Hg] */
  const double* gru_b_hh_l0; /* [3*Hg] */
  const double* gru_w_ih_l1; /* [3*Hg][Hg] */
  const double* gru_w_hh_l1; /* [3*Hg][Hg] */
  const double* gru_b_ih_l1; /* [3*Hg] */
  const double* gru_b_hh_l1; /* [3*Hg] */
  const double* enc_out_w;   /* [2][Hg] */
  const double* enc_out_b;   /* [2] */
  const double* mlp_w0;      /* [hidden][2S+nx+2]   input order [theta_s | phi_s | obs_n | p_action] */
  const double* mlp_b0;      /* [hidden] */
  const double* mlp_w2;      /* [hidden][hidden] */
  const double* mlp_b2;      /* [hidden] */
  const double* mlp_w4;      /* [2*nx*S][hidden]    output index = channel*S + k (w_nl.py:56-58)    */
  const double* mlp_b4;      /* [2*nx*S] */
} nlc_model_desc;

typedef struct nlc_model_s* nlc_model_t;

int nlc_model_create(nlc_model_t* out, const nlc_model_desc* desc, int device);
int nlc_model_destroy(nlc_model_t m);
/* Fold the constants of a fixed prediction time `ts_pred` (seconds; the planner always passes dt,
 * mppi_with_model.py:74): s-points, their sphere coordinates folded into the first MLP bias, the
 * Fourier phases and the exp(gamma t)/T scale (torchlaplace Fourier ILT; PARITY UNPINNED, see
 * oracle/ilt.py).  Called implicitly with dt by nlc_model_create.                                  */
int nlc_model_set_prediction_time(nlc_model_t m, double ts_pred);

/* NeuralLaplaceModel.forward, w_nl.py:117-145, for one fixed prediction time.
 * obs_dev [K][nx], act_dev [K][B][gru_in] env units oldest first, out_dev [K][nx] (delta state),
 * p_action_dev [K][2] optional (the encoder output, w_nl.py:133).                                  */
int nlc_model_forward(nlc_model_t m, const float* obs_dev, const float* act_dev, int K, int B,
                      float* out_dev, float* p_action_dev, int math_mode, void* stream);

/* Same with a per-sample prediction time ts_dev [K] (seconds), the irregular-time form used by
 * training/validation (train_utils.py:401-404): s-points are computed per sample in the kernel.
 * math_mode as in nlc_model_forward (the single-pass fp16 mode takes the fp32-class tensor-core form here). */
int nlc_model_forward_ts(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev,
                         int K, int B, float* out_dev, float* scratch_dev /* [K][132] floats */, int math_mode, void* stream);

/* Gradients of NeuralLaplaceModel.forward with per-sample prediction times (train_utils.py:388-407 loss.backward()).
 * obs_dev, act_dev, ts_dev, K, B as in nlc_model_forward_ts; grad_out_dev [K][nx] is dLoss/d(out).
 * grad_params_dev: nlc_model_grad_floats(desc) floats, OVERWRITTEN, the 16 parameters in named_parameters() order, each
 * in its state_dict layout, at these float offsets (Hg = hidden/2, G3 = 3 Hg, gin = nu (+1 with encode_obs_time),
 * in0 = 2S+nx+2, N3 = 2 nx S):
 *   gru.weight_ih_l0 [G3][gin] at 0,             gru.weight_hh_l0 [G3][Hg] after it, gru.bias_ih_l0 [G3], gru.bias_hh_l0 [G3],
 *   gru.weight_ih_l1 [G3][Hg], gru.weight_hh_l1 [G3][Hg], gru.bias_ih_l1 [G3], gru.bias_hh_l1 [G3],
 *   linear_out.weight [2][Hg], linear_out.bias [2],
 *   linear_tanh_stack.0.weight [hidden][in0], .0.bias [hidden], .2.weight [hidden][hidden], .2.bias [hidden],
 *   .4.weight [N3][hidden], .4.bias [N3]      (each tensor directly after the previous one, no padding).
 * grad_obs_dev [K][nx] and grad_act_dev [K][B][gin] (every stored input channel) may be NULL.
 * workspace_dev: nlc_model_backward_workspace_bytes(m, K, B) bytes, 16-byte aligned.
 * fp32 CUDA cores whatever math mode the forward used; deterministic (bit-identical results for identical inputs). */
int64_t nlc_model_grad_floats(const nlc_model_desc* desc); /* host only: works without a GPU; < 0 on an invalid desc */
int64_t nlc_model_backward_workspace_bytes(nlc_model_t m, int K, int B);
int nlc_model_backward_ts(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K, int B,
                          const float* grad_out_dev, float* grad_params_dev, float* grad_obs_dev, float* grad_act_dev,
                          void* workspace_dev, void* stream);

/* NeuralLaplaceModel.forward with several prediction times per sample: ts_pred (K, n_t) as the reference passes it to
 * laplace_reconstruct (w_nl.py:137-144), which evaluates every (sample, time) pair (torchlaplace laplace_reconstruct,
 * restated in oracle/ilt.py:83-107).  ts_dev [K][n_t] seconds, any order, per sample; out_dev [K][n_t][nx];
 * p_action_dev [K][2] optional (the encoder output).  The K windows are encoded once; the MLP + ILT then runs over the
 * K n_t rows on the kernels of nlc_model_forward_ts, so out[k][j] equals nlc_model_forward_ts at ts[k][j] bit for bit
 * (math_mode likewise).  K n_t >= 2^31 is NLC_ERR_SHAPE.
 * workspace_dev: nlc_model_forward_multi_workspace_bytes(m, K, n_t, B) bytes, 16-byte aligned:
 * 4 (2 K + C (hidden_units + nx + 3)) bytes plus alignment, C = min(K n_t, 65536) rows per chunk.            */
int64_t nlc_model_forward_multi_workspace_bytes(nlc_model_t m, int K, int n_t, int B);
int nlc_model_forward_multi(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K, int n_t,
                            int B, float* out_dev, float* p_action_dev, void* workspace_dev, int math_mode, void* stream);

/* Gradients of nlc_model_forward_multi (loss.backward() through w_nl.py:117-145 with ts_pred (K, n_t)).
 * grad_out_dev [K][n_t][nx]; grad_params_dev, grad_obs_dev, grad_act_dev as in nlc_model_backward_ts.  An MLP/ILT
 * stage over the K n_t rows, a fixed-order sum over j of each sample's gradient of [obs_n | p_action], then one
 * encoder stage (BPTT) over the K samples; fp32 CUDA cores, deterministic.  K n_t >= 2^31 is NLC_ERR_SHAPE.
 * workspace_dev: nlc_model_backward_multi_workspace_bytes(m, K, n_t, B) bytes, 16-byte aligned: 4 K (nx + 4) bytes,
 * 4 C (hidden_units + 2 S + nx + 3) bytes for C = min(K n_t, 65536) rows per chunk, and the per-CTA partials and
 * scratch of at most 148 CTAs, plus alignment.                                                                   */
int64_t nlc_model_backward_multi_workspace_bytes(nlc_model_t m, int K, int n_t, int B);
int nlc_model_backward_multi(nlc_model_t m, const float* obs_dev, const float* act_dev, const float* ts_dev, int K, int n_t,
                             int B, const float* grad_out_dev, float* grad_params_dev, float* grad_obs_dev, float* grad_act_dev,
                             void* workspace_dev, void* stream);

/* NeuralLaplaceModel.forward (w_nl.py:117-145) and its gradients (train_utils.py:388-407 loss.backward()) in fp64 throughout,
 * the precision the reference trains in (train_utils.py:267 .double()).  Every prediction-time form goes through n_t:
 * ts_dev [K][n_t] seconds (n_t = 1: one time per sample; a uniform time is passed per sample), out_dev [K][n_t][nx],
 * p_action_dev [K][2] optional (the encoder output), grad_out_dev [K][n_t][nx]; obs_dev [K][nx], act_dev [K][B][gru_in] and
 * grad_obs_dev / grad_act_dev (either may be NULL) as in nlc_model_backward_ts, all fp64.
 * params_dev: the 16 parameters, fp64 on the device, nlc_model_grad_floats(desc) entries in the layout of grad_params_dev
 * (named_parameters() order, each tensor in its state_dict layout, no padding).  The kernels read the weights from it on
 * every call, never from the handle's fp32 arena: the handle gives only shapes, flags, dt and the normalisation constants
 * (kept in fp64), so it stays valid across optimizer steps.  Non-finite parameters are not checked; they propagate.
 * grad_params_dev: the same layout, fp64, OVERWRITTEN.
 * The forward encodes the K windows once (tiles of 32 samples), then runs the MLP + ILT over the K n_t rows; the backward is
 * the two-stage form of nlc_model_backward_multi for every n_t.  Deterministic: the grid, the tile-to-CTA assignment and
 * every summation order depend on the shapes only.  K n_t >= 2^31 is NLC_ERR_SHAPE; a null required pointer or a
 * workspace that is not 16-byte aligned is NLC_ERR_ARG; B in [1, 8].
 * workspace_dev: nlc_model_{forward,backward}_f64_workspace_bytes(m, K, n_t, B) bytes, 16-byte aligned, bounded whatever
 * n_t is (rows are walked in chunks of C = min(K n_t, 65536)).  With Hg = hidden/2, in0 = 2S+nx+2, N3 = 2 nx S, G = the
 * CTAs of min(K, C) tiles of 32 (at most 148), up to alignment to 4 and 64 elements, the forward takes
 *   8 (2 K + C (hidden + 1 + 2 S) + W + G Sc) bytes,  W = 3 (6 Hg^2 + 3 Hg) + 3 Hg gin + 2 Hg + 2 + in0 hidden
 *                                                         + 2 hidden^2 + 2 hidden + (2 hidden + 1) N3,
 *   Sc = 32 (4 B + 5 B hidden + 9 hidden + in0 + N3 + 18)   (per-CTA tile scratch),
 * and the backward 8 ((K + C)(nx + 2) + G P) bytes more, P = nlc_model_grad_floats (per-CTA gradient partials).          */
int64_t nlc_model_forward_f64_workspace_bytes(nlc_model_t m, int K, int n_t, int B);
int nlc_model_forward_f64(nlc_model_t m, const double* params_dev, const double* obs_dev, const double* act_dev,
                          const double* ts_dev, int K, int n_t, int B, double* out_dev, double* p_action_dev,
                          void* workspace_dev, void* stream);
int64_t nlc_model_backward_f64_workspace_bytes(nlc_model_t m, int K, int n_t, int B);
int nlc_model_backward_f64(nlc_model_t m, const double* params_dev, const double* obs_dev, const double* act_dev,
                           const double* ts_dev, int K, int n_t, int B, const double* grad_out_dev,
                           double* grad_params_dev, double* grad_obs_dev, double* grad_act_dev,
                           void* workspace_dev, void* stream);

/* ReverseGRUEncoder.forward (w_nl.py:25-29) over every window of a K x L action history:
 * hist_dev [K][L][gru_in] env units, windows [t, t+B) for t in [0, T), L = B-1+T.
 * p_dev [K][T][2].                                                                                 */
int nlc_encode_history(nlc_model_t m, const float* hist_dev, int K, int T, int B, float* p_dev,
                       int math_mode, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Stage kernels of MPPIDelay.command (planners/mppi_delay.py:193-356).  Tensors are C-contiguous fp32.
 * ------------------------------------------------------------------------------------------------ */
typedef struct {
  int32_t K;            /* samples on this shard                                                     */
  int32_t T;            /* horizon                                                                   */
  int32_t nu;
  int32_t B;            /* action history window length (action_buffer rows)                         */
  int64_t k_offset;     /* global index of this shard's first sample (bit-exact sample indexing)     */
  int64_t k_total;      /* global K (for sample_null_action and the RNG counter)                     */
  float lambda_;
  float u_scale;
  int32_t has_bounds;                            /* bounds per action dimension (mppi_delay.py:143-150,347-356; the   */
  float u_min[4], u_max[4];                      /* reference's callers pass scalars, mppi_with_model.py:227-228)     */
  int32_t sample_null_action;                    /* mppi_delay.py:322-323                            */
  int32_t noise_abs_cost;                        /* mppi_delay.py:329-333                            */
  float sigma_inv[16];  /* [nu][nu] row-major                                                        */
  float sigma_chol[16]; /* lower Cholesky factor of the covariance, for the on-device sampler        */
  float noise_mu[4];
  float u_init[4];
} nlc_mppi_params;

/* Stage 1: mppi_delay.py:199-200 (roll U), :319-335 (+ :347-356 _bound_action).
 * U_prev_dev [T][nu] is the planner's U before the roll; U_dev receives the rolled U.
 * noise_in_dev [K][T][nu] is the injected sample tensor; when NULL the kernel draws it itself with
 * Philox4x32-10 keyed on (seed, call_index, global sample, t) so results do not depend on sharding.
 * Outputs: perturbed_dev, noise_dev (bounded noise), hist_dev [K][B-1+T][nu] (env units: the rows of
 * action_buffer_dev[1:] then u_scale*perturbed, :255-260), actions_dev = hist/u_scale (:340, optional),
 * pert_cost_dev [K] = sum_t,u U*action_cost (:343).                                                */
int nlc_perturb(const nlc_mppi_params* p, const float* U_prev_dev, float* U_dev, int roll,
                const float* noise_in_dev, uint64_t seed, uint64_t call_index,
                const float* action_buffer_dev, float* perturbed_dev, float* noise_dev, float* hist_dev,
                float* actions_dev, float* pert_cost_dev, void* stream);

typedef struct {
  int32_t env;              /* nlc_env                                                               */
  int32_t state_constraint; /* cartpole only (ctcartpole.py:320-332)                                 */
  float goal_x;             /* cartpole only: 0, -2 or +2 (ctcartpole.py:312-319)                    */
  int32_t dynamics;         /* nlc_dynamics_kind                                                     */
  int32_t delay;            /* NLC_DYN_ANALYTIC_DELAY only                                           */
  float dt;
} nlc_rollout_opts;

/* Stages 2+3: mppi_delay.py:232-313 with the closures of mppi_with_model.py:103-122,145-171.
 * state_dev [nx] (state_per_sample = 0), [K][nx] (= 1) or [ceil(K/n)][nx] (= n > 1: sample k starts from
 * state k / n, the instance-batched form), p_dev [K][T][2] from nlc_encode_history (NULL for
 * analytic dynamics), hist_dev as written by nlc_perturb, pert_cost_dev [K] added to the result
 * (may be NULL).  cost_total_dev [K]; states_dev [K][T][nx] optional.                              */
int nlc_rollout_cost(nlc_model_t m, const nlc_rollout_opts* o, const float* state_dev, int state_per_sample,
                     const float* p_dev, const float* hist_dev, const float* pert_cost_dev, int K, int T, int B,
                     int nu, float* cost_total_dev, float* states_dev, int math_mode, void* stream);

/* Stage 4, shard-local part (mppi_delay.py:210-216): two passes, min then sums.
 * triple_dev [2+T*nu] = (beta, eta, W[t][u] = sum_k exp(-(c_k-beta)/lambda) noise[k][t][u]);
 * weights_dev [K] optional = exp(-(c-beta)/lambda) with the SHARD-local beta.
 * workspace_dev: at least nlc_softmax_workspace_bytes(K, T*nu) bytes.                              */
int64_t nlc_softmax_workspace_bytes(int K, int TN);
int nlc_softmax_partial(const float* cost_dev, const float* noise_dev, int K, int T, int nu, float lambda_,
                        float* triple_dev, float* weights_dev, void* workspace_dev, void* stream);
/* Stage 4, combine: merge G triples [G][2+T*nu] (one per shard, log-sum-exp rescale), apply
 * U[t] += W/eta (mppi_delay.py:215-216) in place, write action_dev [nu] = U[0]*u_scale (:217-224)
 * and stats_dev [2] = (beta, eta) (optional).                                                      */
int nlc_softmax_combine(const float* triples_dev, int G, int T, int nu, float lambda_, float u_scale,
                        float* U_dev, float* action_dev, float* stats_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Planner handle: the whole MPPIDelay object (mppi_delay.py:64-230) with device-resident state.
 * ------------------------------------------------------------------------------------------------ */
typedef struct nlc_planner_s* nlc_planner_t;

typedef struct {
  nlc_mppi_params mppi;
  nlc_rollout_opts rollout;
  int32_t nx;
  int32_t n_shards;     /* G: how many triples nlc_planner_finish will combine                       */
  int32_t shard_index;
  int32_t math_mode;
  int32_t keep_states;  /* write states [K][T][nx] (the reference always does, :295-301)             */
  uint64_t seed;
} nlc_planner_desc;

int nlc_planner_create(nlc_planner_t* out, nlc_model_t model /* may be NULL for analytic dynamics */,
                       const nlc_planner_desc* desc, int device);
int nlc_planner_destroy(nlc_planner_t p);
/* Set the control sequence (U_init, mppi_delay.py:160 / reset :226-230).  host fp64 [T][nu].       */
int nlc_planner_set_U(nlc_planner_t p, const double* U_host);
int nlc_planner_get_U(nlc_planner_t p, double* U_host);

/* Named device buffers of the planner (the attributes the reference leaves on the object,
 * mppi_delay.py:179-184,319-339), for zero-copy views.                                             */
typedef enum {
  NLC_BUF_U = 0, NLC_BUF_NOISE = 1, NLC_BUF_PERTURBED = 2, NLC_BUF_COST_TOTAL = 3, NLC_BUF_WEIGHTS = 4,
  NLC_BUF_STATES = 5, NLC_BUF_ACTIONS = 6, NLC_BUF_TRIPLE = 7, NLC_BUF_ALL_TRIPLES = 8, NLC_BUF_ACTION = 9,
  NLC_BUF_STATS = 10, NLC_BUF_HIST = 11, NLC_BUF_P = 12, NLC_BUF_STATE = 13, NLC_BUF_ACTION_BUFFER = 14
} nlc_buffer_id;
int nlc_planner_buffer(nlc_planner_t p, int which, void** dev_ptr, int64_t* n_floats);

/* One control step, phase 1 (stages 1-3 and the shard-local part of 4) on device inputs:
 * state_dev [nx] or [K][nx], action_buffer_dev [B][nu], noise_in_dev as in nlc_perturb (may be NULL).
 * After it the shard's triple is in NLC_BUF_TRIPLE.                                               */
/* (The two phases must alternate: nlc_planner_finish also bumps the sampler's call index and re-arms stage 4's workspace
 * for the next nlc_planner_rollout.)                                                                */
int nlc_planner_rollout(nlc_planner_t p, const float* state_dev, int state_per_sample,
                        const float* action_buffer_dev, const float* noise_in_dev, void* stream);
/* Phase 2: combine the n_shards triples found in NLC_BUF_ALL_TRIPLES (for n_shards == 1 the local
 * triple is used directly) and update U; the action lands in NLC_BUF_ACTION.                       */
int nlc_planner_finish(nlc_planner_t p, void* stream);

/* Both phases in one call for the single-shard planner, on the planner's own input buffers (NLC_BUF_STATE [nx],
 * NLC_BUF_ACTION_BUFFER [B][nu], filled by the caller) with the on-device sampler.  The fixed launch sequence is captured
 * once into a CUDA graph and replayed with one launch per control step (the sampler's call index lives in device memory);
 * NLC_NO_GRAPH=1 in the environment keeps direct launches.                                          */
int nlc_planner_step(nlc_planner_t p, void* stream);

/* Measurement: the same control step as DIRECT launches with CUDA events at the stage boundaries, so that the kernels are
 * timed inside the step (back to back, warm L2) - the bracket the reference puts around command()
 * (mppi_with_model.py:257-259) split by stage.  ms_out[6] = {perturb, history encoder, rollout + cost, softmax update,
 * encoder-and-rollout section, side-by-side flag}: when the planner runs the encoder beside the rollout (flag 1) the two
 * entries are their overlapping spans from the common fork and [4] is the section's wall time.  Single shard;
 * synchronises the stream.                                                                           */
int nlc_planner_step_profile(nlc_planner_t p, float* ms_out, void* stream);

/* Plans whose sequential rollout leaves SMs idle run their history encoder, wholly or in part, BESIDE the rollout kernel:
 * up to 140 tiles of 128 samples, and ping-pong rollouts of one or two passes per CTA on at most 140 SMs (up to 560 tiles;
 * config 4 on one GPU).  *overlapped = 1 if this planner does.  *status = 1 if, in the last control step, the rollout gave
 * up polling for the encoder's output (~1 s: the two kernels were not co-resident - a serialising tool, a shared GPU;
 * NLC_NO_OVERLAP=1 in the environment keeps the plain sequence); the step's results are then invalid.  Synchronises
 * the device.                                                                                       */
int nlc_planner_overlap_status(nlc_planner_t p, int* overlapped, int* status);

/* Host-side arithmetic of that schedule for K samples, horizon T and a tensor-core model of state size nx with S Fourier
 * terms (no device is touched): out8 = {encoder beside the rollout, ping-pong rollout form, SMs of the rollout, rollout
 * passes per CTA, first sample of the last pass (the samples before it are encoded before the fork), step-major encoder
 * tiles of the last pass's samples encoded before the fork, those tiles in all, horizon steps encoded beside the rollout}.
 * The math mode is the fp32-class tensor-core mode, with the NLC_NO_OVERLAP / NLC_OVERLAP_FACTOR overrides applied. */
int nlc_debug_overlap_plan(int K, int T, int nx, int S, long long* out8);

/* K sharded over the GPUs of ONE node (SURVEY 8e): exchange of the per-shard (beta, eta, W) triples on the device, without
 * a collective library.  Every shard owns a mailbox in its HBM; nlc_planner_exchange_export returns its CUDA IPC handle
 * (64 bytes, for peers in other processes) and/or its device pointer (for peers in the same process).  After
 * nlc_planner_exchange_connect - kind 0: `data` = n_shards IPC handles of 64 bytes in shard order, kind 1: n_shards device
 * pointers; the own slot is ignored - nlc_planner_rollout ends by storing the triple into every peer's mailbox over
 * NVLink and nlc_planner_finish polls the own mailbox for the n_shards triples of the step before it combines; nothing
 * crosses the host, and nlc_planner_step replays the whole sharded control step as one CUDA graph.  All shards must take
 * the same number of control steps.  *status = 2 after a poll gave up (~8 s) because a peer never published.       */
int nlc_planner_exchange_export(nlc_planner_t p, void* ipc_handle_64, void** local_ptr);
int nlc_planner_exchange_connect(nlc_planner_t p, int kind, const void* data);
int nlc_planner_exchange_status(nlc_planner_t p, int* connected, int* status);

/* MPPIDelay.command (mppi_delay.py:193-224) end to end with HOST buffers, single shard: copies the
 * state [nx] and action_buffer [B][nu] (fp64, as the reference's callers hold them) to the device,
 * runs both phases and returns with the action [nu] on the host.  The inputs and the action travel through MAPPED pinned
 * host memory: the step's first kernel reads the staged inputs, its last kernel writes the action and bumps a sequence word
 * the host spins on - no copy nodes and no stream synchronisation on the critical path (later work on the stream is ordered
 * after the step as usual).  Without injected noise the whole step is one CUDA-graph launch.          */
int nlc_planner_command_host(nlc_planner_t p, const double* state_host, const double* action_buffer_host,
                             const float* noise_in_dev, double* action_host, void* stream);

/* ------------------------------------------------------------------------------------------------
 * fp64 planner: MPPIDelay.command (mppi_delay.py:193-224) in fp64 throughout, the precision the reference plans in
 * (its model is .double(), train_utils.py:267; its noise_sigma is fp64, mppi_with_model.py:66-70).  A handle of its own,
 * single shard, direct launches on the caller's stream.  All tensors are C-contiguous fp64.
 *   stage 1  roll U, U[-1] = u_init; perturbed = U + noise, the null sample, bound(perturbed u_scale)/u_scale,
 *            noise = perturbed - U, hist and actions: round-to-nearest fp64 operations in the reference's order, so these
 *            tensors are bit-identical to the reference's for the same noise;
 *   model    the K T history windows through the fp64 encoder, then per tile of 32 samples the whole horizon: fp64 MLP,
 *            Fourier ILT at dt (the arithmetic of nlc_model_forward_f64 at a uniform time), state += delta, running cost;
 *            analytic dynamics: one fp64 Euler step (oracle.py:11-224) per step instead;
 *   stage 4  beta = min c, w = exp(-(1/lambda)(c - beta)), eta = sum w, U[t] += sum_k (w_k/eta) noise[k][t]: fixed-order
 *            sums, so two calls on the same inputs give bit-identical results.
 * On-device sampler (noise_in_dev NULL): Philox4x32-10, key = seed, counter = (idx_lo, idx_hi, call_lo, call_hi) with
 * idx = k T + t and the call index counting this planner's control steps (as nlc_perturb).  Of the four output words
 * (x0, x1, x2, x3): u1 = (2 ((x0 >> 6) 2^26 + (x1 >> 6)) + 1) 2^-53 and u2 likewise from (x2, x3) - 53-bit uniforms in
 * (0, 1), never 0 or 1 - and z0 = r cos(2 pi u2), z1 = r sin(2 pi u2), r = sqrt(-2 log u1) (fp64 sincospi).  nu > 2 takes
 * z2, z3 from a second block, counter word 3 = call_hi ^ 0x80000000.  noise[u] = mu[u] + sum_{v <= u} L[u][v] z[v]
 * (fp64 FMAs, v ascending), L = sigma_chol.
 * ------------------------------------------------------------------------------------------------ */
typedef struct nlc_planner_f64_s* nlc_planner_f64_t;

typedef struct {
  /* K, T, nu, B, nx, env, state_constraint, dynamics, delay, keep_states, seed, sample_null_action, noise_abs_cost,
   * has_bounds are read from base; its float values (lambda_, u_scale, bounds, sigma, mu, u_init, goal_x, dt), k_offset,
   * k_total, shard_index and math_mode are ignored; n_shards must be 1 (else NLC_ERR_UNSUPPORTED).                     */
  nlc_planner_desc base;
  double lambda_, u_scale, dt, goal_x;
  double u_min[4], u_max[4];
  double sigma_inv[16], sigma_chol[16], noise_mu[4], u_init[4];  /* [nu][nu] row-major; sigma_chol lower triangular */
} nlc_planner_f64_desc;

/* model: NULL for analytic dynamics.  The model handle supplies shapes, flags and the fp64 normalisation constants; the
 * planner takes a reference on it (as nlc_planner_create).  B in [1, 8], T nu <= 256.                               */
int nlc_planner_f64_create(nlc_planner_f64_t* out, nlc_model_t model, const nlc_planner_f64_desc* d, int device);
int nlc_planner_f64_destroy(nlc_planner_f64_t p);
/* The model's 16 parameters, fp64 on the device, in the layout of nlc_model_backward_f64's params_dev: rearranged into the
 * planner's own weight image (and the first layer folded at dt) on `stream`; later commands use them until the next call.
 * Required before the first command of a Neural Laplace planner.                                                    */
int nlc_planner_f64_set_params(nlc_planner_f64_t p, const double* params_dev, void* stream);
/* host fp64 [T][nu]; synchronous                                                                                     */
int nlc_planner_f64_set_U(nlc_planner_f64_t p, const double* U_host);
int nlc_planner_f64_get_U(nlc_planner_f64_t p, double* U_host);
/* Device buffers as in nlc_planner_buffer (NLC_BUF_U .. NLC_BUF_ACTION_BUFFER, without the triples), sizes in doubles:
 * WEIGHTS holds w = exp(-(1/lambda)(c - beta)) (cost_total_non_zero), STATS (beta, eta).                            */
int nlc_planner_f64_buffer(nlc_planner_f64_t p, int which, void** dev_ptr, int64_t* n_doubles);
/* One control step on device inputs: state_dev [nx] (state_per_sample 0) or [K][nx] (1), action_buffer_dev [B][nu],
 * noise_in_dev [K][T][nu] or NULL (the on-device sampler).  The action [nu] = U[0] u_scale lands in NLC_BUF_ACTION.  */
int nlc_planner_f64_command(nlc_planner_f64_t p, const double* state_dev, int state_per_sample, const double* action_buffer_dev,
                            const double* noise_in_dev, void* stream);
/* The same with host buffers (state [nx], action_buffer [B][nu]) and the on-device sampler: copies in, one control step,
 * the action [nu] copied back to action_host; synchronises the stream.                                              */
int nlc_planner_f64_command_host(nlc_planner_f64_t p, const double* state_host, const double* action_buffer_host,
                                 double* action_host, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Instance-batched planning and the closed loop (BASELINE config 5; the caller side of the path,
 * mppi_with_model.py:193-216,244-317, for many env x seed instances of ONE environment at once).
 * ------------------------------------------------------------------------------------------------ */
typedef struct nlc_batch_planner_s* nlc_batch_planner_t;

/* n_instances independent MPPIDelay objects (desc->mppi.K samples EACH, desc->n_shards must be 1) with
 * their own control sequence, action buffer and sampler seed; seeds_host [n_instances].  Instance i
 * reproduces nlc_planner_create(desc with seed = seeds[i]).                                         */
int nlc_batch_planner_create(nlc_batch_planner_t* out, nlc_model_t model, const nlc_planner_desc* desc, int n_instances,
                             const uint64_t* seeds_host, int device);
int nlc_batch_planner_destroy(nlc_batch_planner_t p);
/* U_host fp64 [n_instances][T][nu]                                                                  */
int nlc_batch_planner_set_U(nlc_batch_planner_t p, const double* U_host);
/* buffers are the single planner's, concatenated over instances (NLC_BUF_U .. NLC_BUF_P)            */
int nlc_batch_planner_buffer(nlc_batch_planner_t p, int which, void** dev_ptr, int64_t* n_floats);
/* MPPIDelay.command for every instance: state_dev [I][nx], action_buffer_dev [I][B][nu],
 * noise_in_dev [I][K][T][nu] or NULL (on-device sampler), action_dev [I][nu] (env units).
 * Stage 1 and 4 run per instance, the encoder and the rollout once over all I*K samples.            */
int nlc_batch_planner_command(nlc_batch_planner_t p, const float* state_dev, const float* action_buffer_dev,
                              const float* noise_in_dev, float* action_dev, void* stream);

/* step_env (mppi_with_model.py:193-216) for I instances: action_buffer <- roll(action_buffer, -1),
 * action_buffer[-1] <- action (get_action, :25-28); the delayed action action_buffer[-(o->delay+1)] drives
 * one explicit-Euler step of the true dynamics (base_env.py:136-173 as stated by oracle.py:11-224,
 * observation form); reward_dev [I] (optional) = reward of the new state with the applied action.
 * state_dev [I][nx] and action_buffer_dev [I][B][nu] are updated in place.                          */
int nlc_env_step(const nlc_rollout_opts* o, float* state_dev, float* action_buffer_dev, const float* action_dev,
                 int I, int B, int nu, float* reward_dev, void* stream);

/* ------------------------------------------------------------------------------------------------
 * Generic Fourier-series inverse Laplace transform (torchlaplace's Fourier ILT as called from
 * w_nl.py:137-144; BASELINE config 2).  F_dev: complex64 interleaved [N][n_t][S]; t_dev [n_t]
 * (shared time grid, t_per_row = 0) or [N][n_t] (t_per_row = 1); out_dev [N][n_t].
 * x(t) = exp(gamma t)/T [ Re F_0 / 2 + sum_{k>=1} Re(F_k e^{i k pi t/T}) ],  T = 2(t+1e-6),
 * gamma = 1e-3 - ln(1e-2)/T.                                                                       */
int nlc_ilt_fourier(const float* F_dev, const float* t_dev, int t_per_row, int64_t N, int n_t, int S,
                    float* out_dev, void* stream);

/* Self-test of the tcgen05 operand layout used by the tensor-core encoder (no reference counterpart):
 * D_dev[128][N] = A_dev[128][64] . B_dev[n_off : n_off+N][64]^T, fp32 in/out, operands split to fp16 hi(+lo) on
 * the device exactly as the encoder does.                                                           */
int nlc_selftest_umma_gemm(const float* A_dev, const float* B_dev, int n_rows_b, int n_off, int N, int split3,
                           float* D_dev, void* stream);

/* Same self-test with the A operand staged in tensor memory (the fused rollout's operand path):
 * D_dev[128][N] = A_dev[128][Kdim] . B_dev[0:N][Kdim]^T, Kdim 64 or 128.                             */
int nlc_selftest_umma_gemm_ts(const float* A_dev, const float* B_dev, int n_rows_b, int N, int Kdim, int split3,
                              float* D_dev, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* NLC_B200_H */
