// Planner handle: the device-resident state of one MPPIDelay object (planners/mppi_delay.py:64-230) and
// the control step as a fixed sequence of kernel launches on one stream:
//   perturb -> encode_history -> rollout_cost -> softmax (init, min, sum) -> [exchange triples] -> combine
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <vector>

#include "common.cuh"

struct nlc_planner_s {
  int device;
  nlc_model_t model;
  nlc_planner_desc d;
  uint64_t calls;
  // device buffers (one arena)
  void* arena;
  size_t arena_bytes;
  float *U, *U_rolled, *noise, *perturbed, *hist, *actions, *pert_cost, *p, *cost_total, *weights, *states;
  float *triple, *all_triples, *action, *stats, *state_in, *abuf_in;
  void* softmax_ws;
  // MAPPED pinned host staging of the host-buffer entry point: the first kernel of the step reads h_in, the last writes the
  // action and bumps a sequence word in h_out; the host spins on that word (no copy nodes, no stream synchronisation)
  float* h_in;   // [nx + B*nu]
  float* h_out;  // [4] action, then the sequence word at float index 4
  bool to_host;  // the control step being issued belongs to nlc_planner_command_host: its combine kernel reports to h_out
  int kernels_per_step;  // kernels one control step launches (counted during the capture warm-up; for nlc_launch_count)
  // sampler call index in device memory (read by the perturb kernel, bumped right after it) so that a whole control step
  // is a fixed sequence of launches with fixed arguments: captured once into CUDA graphs, replayed with one launch
  unsigned long long* call_ctr;
  cudaStream_t cap_stream;
  cudaGraphExec_t graph_core, graph_host;  // [perturb .. combine] on the planner's own input buffers; same + H2D / D2H copies
  bool graph_core_tried, graph_host_tried;
  // Plans within half a wave of 128-sample tiles leave most SMs idle during the sequential rollout: the history encoder
  // then runs BESIDE the rollout kernel (side stream, fork/join on events - also inside the captured graphs) in step-major
  // order, publishing per-step readiness counters the rollout polls (encode_tc2.cu / rollout_tc2.cu).
  bool overlap;
  cudaStream_t side_stream;
  cudaEvent_t ev_fork, ev_join;
  unsigned int* ready;   // [T] finished encoder warps per rollout step, + 1 status word (1 = a poll timed out)
  bool pending;          // nlc_planner_rollout ran and nlc_planner_finish has not yet: the phases must alternate
  // K sharded over the GPUs of one node: device-side exchange of the triples through peer-mapped mailboxes (stage4_update.cu)
  float* mailbox;               // own: [2][G][xstride] floats + [2][G] sequence words
  int xstride;
  bool xchg;                    // peers connected: publish / poll-and-combine replace the host-side all-gather
  void* peer[64];               // mailbox of every shard as mapped into this process (own slot = mailbox)
  bool peer_ipc[64];            // opened with cudaIpcOpenMemHandle (to be closed)
  float** mailboxes_dev;        // the same table in device memory
  unsigned long long* xstep;    // control steps exchanged so far
  unsigned int* xstatus;        // 2 = a poll for a peer's triple timed out
};

namespace nlc {
int perturb_launch(const nlc_mppi_params* p, const float* U_prev_dev, float* U_dev, int roll, const float* noise_in_dev,
                   uint64_t seed, uint64_t call_index, const unsigned long long* call_index_dev, const float* action_buffer_dev,
                   float* perturbed_dev, float* noise_dev, float* hist_dev, float* actions_dev, float* pert_cost_dev, void* stream);
int softmax_partial_impl(const float* cost_dev, const float* noise_dev, int K, int T, int nu, float lambda_, float* triple_dev,
                         float* weights_dev, void* workspace_dev, bool with_init, const ExchangePub& pub, cudaStream_t s);
int launch_combine(const float* triples_dev, int G, int T, int nu, float lambda_, float u_scale, float* U_dev, float* action_dev,
                   float* stats_dev, const StepTail& tl, cudaStream_t s);
int launch_ingest(const float* h_in, float* state_in, float* abuf_in, int nx, int nb, cudaStream_t s);
int launch_combine_exchange(float* mailbox, int G, int stride, int T, int nu, float lambda_, float u_scale, float* U, float* action,
                            float* stats, unsigned long long* step_ctr, unsigned int* status, const StepTail& tl, cudaStream_t s);
bool encoder_is_tensor_core(nlc_model_t m, int B, int math_mode);
int encode_history_overlapped(nlc_model_t m, const float* hist_dev, int K, int T, int B, float* p_dev, int math_mode,
                              unsigned int* ready, int max_ctas, long long tile_begin, long long tile_end, int k_sub, bool with_head,
                              cudaStream_t s);
bool rollout_can_overlap(const nlc_model_s* m, int K, int T, int math_mode);
bool rollout_overlap_is_ping_pong(const nlc_model_s* m, int K);
int launch_rollout_overlapped(nlc_model_s* m, const nlc_rollout_opts* o, const float* state, int sps, const float* p, const float* hist,
                              const float* pert_cost, int K, int T, int B, int nu, float* cost, float* states, int math_mode,
                              const unsigned int* ready, unsigned int ready_target, unsigned int* status, cudaStream_t stream);
}  // namespace nlc

using namespace nlc;

extern "C" int nlc_planner_create(nlc_planner_t* out, nlc_model_t model, const nlc_planner_desc* d, int device) {
  NLC_REQUIRE(out && d, NLC_ERR_ARG, "nlc_planner_create: null argument");
  *out = nullptr;
  int rc = check_device_arch(device);
  if (rc != NLC_OK) return rc;
  const nlc_mppi_params& mp = d->mppi;
  NLC_REQUIRE(mp.K >= 1 && mp.T >= 1 && mp.B >= 1 && mp.B <= 8, NLC_ERR_SHAPE, "planner: K, T >= 1 and 1 <= B <= 8 required");
  NLC_REQUIRE(mp.nu >= 1 && mp.nu <= 4 && d->nx >= 1 && d->nx <= kMaxNx, NLC_ERR_SHAPE, "planner: nu/nx out of range");
  NLC_REQUIRE(mp.T * mp.nu <= 256, NLC_ERR_SHAPE, "planner: T*nu exceeds 256");
  NLC_REQUIRE(d->n_shards >= 1 && d->n_shards <= 64 && d->shard_index >= 0 && d->shard_index < d->n_shards, NLC_ERR_ARG, "planner: bad shard spec");
  NLC_REQUIRE(mp.lambda_ > 0.0f, NLC_ERR_ARG, "planner: lambda must be positive");
  if (d->rollout.dynamics == NLC_DYN_NEURAL_LAPLACE) {
    NLC_REQUIRE(model != nullptr, NLC_ERR_ARG, "planner: Neural Laplace dynamics need a model handle");
    NLC_REQUIRE(model->device == device, NLC_ERR_ARG, "planner: model lives on device %d, planner on %d", model->device, device);
    NLC_REQUIRE(model->nx == d->nx && model->nu == mp.nu, NLC_ERR_SHAPE, "planner: model dims do not match");
  }
  NLC_REQUIRE(model == nullptr || !model->destroy_requested, NLC_ERR_ARG, "planner: the model handle has been destroyed");
  nlc_planner_s* p = new nlc_planner_s();
  p->device = device; p->model = model; p->d = *d; p->calls = 0; p->arena = nullptr; p->h_in = nullptr; p->h_out = nullptr;
  p->call_ctr = nullptr; p->cap_stream = nullptr; p->graph_core = nullptr; p->graph_host = nullptr;
  p->graph_core_tried = p->graph_host_tried = false;
  p->pending = false; p->to_host = false; p->kernels_per_step = 6;
  p->overlap = false; p->side_stream = nullptr; p->ev_fork = p->ev_join = nullptr; p->ready = nullptr;
  p->mailbox = nullptr; p->xstride = 0; p->xchg = false; p->mailboxes_dev = nullptr; p->xstep = nullptr; p->xstatus = nullptr;
  memset(p->peer, 0, sizeof(p->peer)); memset(p->peer_ipc, 0, sizeof(p->peer_ipc));
  const size_t K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, nx = d->nx, L = B - 1 + T, TN = T * nu;
  std::vector<size_t> sizes = {
      TN, TN, K * TN, K * TN, K * L * nu, K * TN, K, K * T * 2, K, K, (d->keep_states ? K * T * nx : 0),
      2 + TN, (size_t)d->n_shards * (2 + TN), 4, 4, K * nx, B * nu, (size_t)(nlc_softmax_workspace_bytes((int)K, (int)TN) / 4 + 1)};
  std::vector<size_t> offs;
  size_t total = 0;
  for (size_t s : sizes) { offs.push_back(total); total += (s + 63) / 64 * 64; }
  p->arena_bytes = total * sizeof(float);
  auto fail = [&](int code) {
    if (p->arena) cudaFree(p->arena);
    if (p->ready) cudaFree(p->ready);
    if (p->side_stream) cudaStreamDestroy(p->side_stream);
    if (p->ev_fork) cudaEventDestroy(p->ev_fork);
    if (p->ev_join) cudaEventDestroy(p->ev_join);
    if (p->call_ctr) cudaFree(p->call_ctr);
    if (p->h_in) cudaFreeHost(p->h_in);
    if (p->h_out) cudaFreeHost(p->h_out);
    delete p;
    return code;
  };
  if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice failed"); return fail(NLC_ERR_CUDA); }
  if (cudaMalloc(&p->arena, p->arena_bytes) != cudaSuccess) { cudaGetLastError(); p->arena = nullptr; set_error("planner: cudaMalloc(%zu) failed", p->arena_bytes); return fail(NLC_ERR_NOMEM); }
  if (cudaMemset(p->arena, 0, p->arena_bytes) != cudaSuccess) { set_error("planner: memset failed"); return fail(NLC_ERR_CUDA); }
  if (cudaMalloc(&p->call_ctr, sizeof(unsigned long long)) != cudaSuccess || cudaMemset(p->call_ctr, 0, sizeof(unsigned long long)) != cudaSuccess) {
    cudaGetLastError(); set_error("planner: counter allocation failed"); return fail(NLC_ERR_NOMEM);
  }
  float* base = static_cast<float*>(p->arena);
  float** slots[] = {&p->U, &p->U_rolled, &p->noise, &p->perturbed, &p->hist, &p->actions, &p->pert_cost, &p->p,
                     &p->cost_total, &p->weights, &p->states, &p->triple, &p->all_triples, &p->action, &p->stats,
                     &p->state_in, &p->abuf_in};
  for (size_t i = 0; i < sizeof(slots) / sizeof(slots[0]); ++i) *slots[i] = base + offs[i];
  if (!d->keep_states) p->states = nullptr;
  p->softmax_ws = base + offs[17];
  // stage 4's workspace header starts armed (min = +inf as all-ones, ticket = 0); every combine kernel re-arms it (StepTail)
  if (cudaMemset(p->softmax_ws, 0xFF, 4) != cudaSuccess) { set_error("planner: memset failed"); return fail(NLC_ERR_CUDA); }
  if (cudaHostAlloc(&p->h_in, sizeof(float) * 64, cudaHostAllocMapped) != cudaSuccess ||
      cudaHostAlloc(&p->h_out, sizeof(float) * 8, cudaHostAllocMapped) != cudaSuccess) {
    cudaGetLastError(); set_error("planner: pinned allocation failed"); return fail(NLC_ERR_NOMEM);
  }
  memset(p->h_in, 0, sizeof(float) * 64);
  memset(p->h_out, 0, sizeof(float) * 8);
  if (d->rollout.dynamics == NLC_DYN_NEURAL_LAPLACE && encoder_is_tensor_core(model, mp.B, d->math_mode) &&
      rollout_can_overlap(model, mp.K, mp.T, d->math_mode) && d->rollout.env >= 0) {
    if (cudaMalloc(&p->ready, sizeof(unsigned int) * (T + 1)) != cudaSuccess || cudaMemset(p->ready, 0, sizeof(unsigned int) * (T + 1)) != cudaSuccess ||
        cudaStreamCreateWithFlags(&p->side_stream, cudaStreamNonBlocking) != cudaSuccess ||
        cudaEventCreateWithFlags(&p->ev_fork, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&p->ev_join, cudaEventDisableTiming) != cudaSuccess) {
      cudaGetLastError(); set_error("planner: overlap resources could not be created"); return fail(NLC_ERR_NOMEM);
    }
    p->overlap = true;
  }
  if (model) model->refs++;
  *out = p;
  return NLC_OK;
}

// drop a planner's reference on its model; frees the model if nlc_model_destroy was called while it was in use
static void model_release(nlc_model_t m) {
  if (!m) return;
  if (--m->refs <= 0 && m->destroy_requested) { m->refs = 0; nlc_model_destroy(m); }
}

// The planner rolls out on constants folded into the model for ONE prediction time.  NeuralLaplaceModel.forward at
// another uniform time re-folds them in place (nlc_model_set_prediction_time): refuse to plan on that silently.
static int planner_check_model(nlc_planner_t p) {
  if (p->d.rollout.dynamics != NLC_DYN_NEURAL_LAPLACE) return NLC_OK;
  NLC_REQUIRE(!p->model->destroy_requested, NLC_ERR_ARG, "planner: its model handle has been destroyed");
  const double want = (double)p->d.rollout.dt;
  NLC_REQUIRE(fabs(p->model->ts_pred - want) <= 1e-6 * fabs(want), NLC_ERR_ARG,
              "planner: the model is folded for prediction time %.9g, the planner steps by dt = %.9g; call "
              "nlc_model_set_prediction_time(model, dt) before the control step", p->model->ts_pred, want);
  return NLC_OK;
}

extern "C" int nlc_planner_destroy(nlc_planner_t p) {
  if (!p) return NLC_OK;
  cudaSetDevice(p->device);
  cudaDeviceSynchronize();  // no kernel of this planner may still read the model when the last reference goes
  model_release(p->model);
  if (p->graph_core) cudaGraphExecDestroy(p->graph_core);
  if (p->graph_host) cudaGraphExecDestroy(p->graph_host);
  if (p->cap_stream) cudaStreamDestroy(p->cap_stream);
  if (p->side_stream) cudaStreamDestroy(p->side_stream);
  if (p->ev_fork) cudaEventDestroy(p->ev_fork);
  if (p->ev_join) cudaEventDestroy(p->ev_join);
  if (p->ready) cudaFree(p->ready);
  for (int g = 0; g < 64; ++g)
    if (p->peer_ipc[g] && p->peer[g]) cudaIpcCloseMemHandle(p->peer[g]);
  if (p->mailbox) cudaFree(p->mailbox);
  if (p->mailboxes_dev) cudaFree(p->mailboxes_dev);
  if (p->xstep) cudaFree(p->xstep);
  if (p->call_ctr) cudaFree(p->call_ctr);
  if (p->arena) cudaFree(p->arena);
  if (p->h_in) cudaFreeHost(p->h_in);
  if (p->h_out) cudaFreeHost(p->h_out);
  cudaGetLastError();
  delete p;
  return NLC_OK;
}

// ---- device-side exchange of the shard triples (no collective library; stage4_update.cu) -----------------------------
static int planner_mailbox(nlc_planner_t p) {
  if (p->mailbox) return NLC_OK;
  const int G = p->d.n_shards, TN = p->d.mppi.T * p->d.mppi.nu;
  p->xstride = (2 + TN + 3) / 4 * 4;
  const size_t bytes = sizeof(float) * 2 * G * p->xstride + sizeof(unsigned int) * 2 * G;
  NLC_CUDA_OK(cudaSetDevice(p->device));
  NLC_CUDA_OK(cudaMalloc(&p->mailbox, bytes));  // its own allocation: CUDA IPC exports whole allocations
  NLC_CUDA_OK(cudaMemset(p->mailbox, 0, bytes));
  NLC_CUDA_OK(cudaMalloc(&p->mailboxes_dev, sizeof(float*) * G));
  NLC_CUDA_OK(cudaMalloc(&p->xstep, sizeof(unsigned long long) + sizeof(unsigned int)));
  NLC_CUDA_OK(cudaMemset(p->xstep, 0, sizeof(unsigned long long) + sizeof(unsigned int)));
  p->xstatus = reinterpret_cast<unsigned int*>(p->xstep + 1);
  return NLC_OK;
}

extern "C" int nlc_planner_exchange_export(nlc_planner_t p, void* ipc_handle_64, void** local_ptr) {
  NLC_REQUIRE(p, NLC_ERR_ARG, "nlc_planner_exchange_export: null planner");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  int rc = planner_mailbox(p);
  if (rc != NLC_OK) return rc;
  if (ipc_handle_64) NLC_CUDA_OK(cudaIpcGetMemHandle(static_cast<cudaIpcMemHandle_t*>(ipc_handle_64), p->mailbox));
  if (local_ptr) *local_ptr = p->mailbox;
  return NLC_OK;
}

extern "C" int nlc_planner_exchange_connect(nlc_planner_t p, int kind, const void* data) {
  NLC_REQUIRE(p && data, NLC_ERR_ARG, "nlc_planner_exchange_connect: null argument");
  NLC_REQUIRE(kind == 0 || kind == 1, NLC_ERR_ARG, "nlc_planner_exchange_connect: kind must be 0 (IPC handles) or 1 (device pointers)");
  NLC_REQUIRE(!p->xchg, NLC_ERR_ARG, "nlc_planner_exchange_connect: already connected");
  int rc = planner_mailbox(p);
  if (rc != NLC_OK) return rc;
  const int G = p->d.n_shards, me = p->d.shard_index;
  NLC_CUDA_OK(cudaSetDevice(p->device));
  for (int g = 0; g < G; ++g) {
    if (g == me) { p->peer[g] = p->mailbox; continue; }
    if (kind == 1) {
      p->peer[g] = static_cast<void* const*>(data)[g];
      NLC_REQUIRE(p->peer[g] != nullptr, NLC_ERR_ARG, "nlc_planner_exchange_connect: null mailbox pointer for shard %d", g);
    } else {
      cudaIpcMemHandle_t h;
      memcpy(&h, static_cast<const char*>(data) + 64 * (size_t)g, 64);
      void* ptr = nullptr;
      const cudaError_t e = cudaIpcOpenMemHandle(&ptr, h, cudaIpcMemLazyEnablePeerAccess);
      if (e != cudaSuccess) {
        cudaGetLastError();
        for (int j = 0; j < g; ++j)
          if (p->peer_ipc[j]) { cudaIpcCloseMemHandle(p->peer[j]); p->peer_ipc[j] = false; p->peer[j] = nullptr; }
        set_error("nlc_planner_exchange_connect: cudaIpcOpenMemHandle for shard %d failed: %s", g, cudaGetErrorString(e));
        return NLC_ERR_CUDA;
      }
      p->peer[g] = ptr; p->peer_ipc[g] = true;
    }
  }
  NLC_CUDA_OK(cudaMemcpy(p->mailboxes_dev, p->peer, sizeof(float*) * G, cudaMemcpyHostToDevice));
  p->xchg = true;
  // captured graphs (if any) predate the exchange: re-capture on next use
  if (p->graph_core) { cudaGraphExecDestroy(p->graph_core); p->graph_core = nullptr; }
  p->graph_core_tried = false;
  return NLC_OK;
}

extern "C" int nlc_planner_exchange_status(nlc_planner_t p, int* connected, int* status) {
  NLC_REQUIRE(p && connected && status, NLC_ERR_ARG, "nlc_planner_exchange_status: null argument");
  *connected = p->xchg ? 1 : 0;
  *status = 0;
  if (p->xchg) {
    unsigned int v = 0;
    NLC_CUDA_OK(cudaSetDevice(p->device));
    NLC_CUDA_OK(cudaDeviceSynchronize());
    NLC_CUDA_OK(cudaMemcpy(&v, p->xstatus, sizeof(v), cudaMemcpyDeviceToHost));
    *status = (int)v;
  }
  return NLC_OK;
}

extern "C" int nlc_planner_set_U(nlc_planner_t p, const double* U_host) {
  NLC_REQUIRE(p && U_host, NLC_ERR_ARG, "nlc_planner_set_U: null argument");
  const int n = p->d.mppi.T * p->d.mppi.nu;
  std::vector<float> tmp(n);
  for (int i = 0; i < n; ++i) tmp[i] = (float)U_host[i];
  NLC_CUDA_OK(cudaSetDevice(p->device));
  NLC_CUDA_OK(cudaMemcpy(p->U, tmp.data(), sizeof(float) * n, cudaMemcpyHostToDevice));
  return NLC_OK;
}

extern "C" int nlc_planner_get_U(nlc_planner_t p, double* U_host) {
  NLC_REQUIRE(p && U_host, NLC_ERR_ARG, "nlc_planner_get_U: null argument");
  const int n = p->d.mppi.T * p->d.mppi.nu;
  std::vector<float> tmp(n);
  NLC_CUDA_OK(cudaSetDevice(p->device));
  NLC_CUDA_OK(cudaMemcpy(tmp.data(), p->U, sizeof(float) * n, cudaMemcpyDeviceToHost));
  for (int i = 0; i < n; ++i) U_host[i] = tmp[i];
  return NLC_OK;
}

extern "C" int nlc_planner_buffer(nlc_planner_t p, int which, void** dev_ptr, int64_t* n_floats) {
  NLC_REQUIRE(p && dev_ptr && n_floats, NLC_ERR_ARG, "nlc_planner_buffer: null argument");
  const nlc_mppi_params& mp = p->d.mppi;
  const int64_t K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, nx = p->d.nx, TN = T * nu;
  float* ptr = nullptr; int64_t n = 0;
  switch (which) {
    case NLC_BUF_U: ptr = p->U; n = TN; break;
    case NLC_BUF_NOISE: ptr = p->noise; n = K * TN; break;
    case NLC_BUF_PERTURBED: ptr = p->perturbed; n = K * TN; break;
    case NLC_BUF_COST_TOTAL: ptr = p->cost_total; n = K; break;
    case NLC_BUF_WEIGHTS: ptr = p->weights; n = K; break;
    case NLC_BUF_STATES: ptr = p->states; n = p->states ? K * T * nx : 0; break;
    case NLC_BUF_ACTIONS: ptr = p->actions; n = K * TN; break;
    case NLC_BUF_TRIPLE: ptr = p->triple; n = 2 + TN; break;
    case NLC_BUF_ALL_TRIPLES: ptr = p->all_triples; n = (int64_t)p->d.n_shards * (2 + TN); break;
    case NLC_BUF_ACTION: ptr = p->action; n = nu; break;
    case NLC_BUF_STATS: ptr = p->stats; n = 2; break;
    case NLC_BUF_HIST: ptr = p->hist; n = K * (B - 1 + T) * nu; break;
    case NLC_BUF_P: ptr = p->p; n = K * T * 2; break;
    case NLC_BUF_STATE: ptr = p->state_in; n = K * nx; break;
    case NLC_BUF_ACTION_BUFFER: ptr = p->abuf_in; n = B * nu; break;
    default: set_error("nlc_planner_buffer: unknown buffer id %d", which); return NLC_ERR_ARG;
  }
  *dev_ptr = ptr; *n_floats = n;
  return NLC_OK;
}

// stages 1-3 + the shard-local half of stage 4; `ev` (optional, 4 events) receives the stage boundaries:
// ev[0] start | perturb | ev[1] | encoder | ev[2] | rollout + cost | ev[3] | (softmax follows)
// Schedule of the overlapped step (see planner_rollout_impl): the rollout's form, SM count and passes; the samples [0, k1) of
// the passes before the last, encoded in full before the fork; and how many of the encoder's step-major tiles of the last
// pass's samples [k1, K) (sub_tiles per step) run on all SMs before the fork.
struct OverlapSchedule { bool pp; int roll_sms, passes, k1, sub_tiles, beside_steps; long long split; };
static OverlapSchedule overlap_schedule(const nlc_model_s* m, int K, int T) {
  const int n_tiles = (K + 127) / 128;
  OverlapSchedule s;
  s.pp = rollout_overlap_is_ping_pong(m, K);
  s.roll_sms = s.pp ? pp_overlap_grid(n_tiles) : n_tiles;
  s.passes = s.pp ? pp_overlap_iters(n_tiles) : 1;
  s.k1 = s.pp ? pp_overlap_k1(n_tiles) : 0;
  s.sub_tiles = (K - s.k1 + 127) / 128;
  static const double factor = [] { const char* e = getenv("NLC_OVERLAP_FACTOR"); return e && e[0] ? atof(e) : 0.9; }();  // measurements
  const int enc_sms = 148 - s.roll_sms;
  const long long total = (long long)T * s.sub_tiles;
  if (s.passes == 1) {
    const double beside_tiles = factor * enc_sms * (T * (s.pp ? 13.3 : 9.5)) / 12.6;
    long long beside_steps = (long long)(beside_tiles / n_tiles);
    if (beside_steps > T) beside_steps = T;
    // (also below half a wave of tiles: 64 tiles, T = 50 - the first 6 steps on all SMs, then 84 SMs beside the rollout:
    // 0.554 -> 0.538 ms per step against everything beside the rollout)
    if (beside_steps < 1) beside_steps = 1;
    s.split = (T - beside_steps) * n_tiles;
  } else {
    // Only the last pass waits for the encoder.  It needs the windows of step t when it begins step t - 1,
    //   deadline(t) = ((passes - 1) T + t - 1) * 13.3 us after the fork.
    // The encoder beside it walks the last m step-major tiles on enc_sms SMs at 12.6 us per tile; it has completed step t
    // once the m - (T - 1 - t) sub_tiles beside tiles up to the end of step t are done:
    //   (m - (T - 1 - t) sub_tiles) 12.6 / enc_sms <= factor * deadline(t)   for every step t,
    // which holds trivially for the steps encoded before the fork.  m is the largest count that satisfies all of them; it
    // need not end on a step boundary (config 4: the last 7.3 of 50 steps of the last pass's samples).
    double m = (double)total;
    for (int t = 0; t < T; ++t) {
      const double bound = (double)(T - 1 - t) * s.sub_tiles + factor * 13.3 * ((s.passes - 1) * (double)T + t - 1) * enc_sms / 12.6;
      if (bound < m) m = bound;
    }
    s.split = total - (m > 0.0 ? (long long)m : 0);
  }
  s.beside_steps = (int)((total - s.split) / s.sub_tiles);
  return s;
}
// host-side arithmetic only (tests/test_abi_cpu.py): out = {ping-pong form, SMs of the rollout, step-major tiles before the
// fork, step-major tiles in all}
extern "C" int nlc_debug_overlap_schedule(int K, int T, int nx, int S, long long* out4) {
  NLC_REQUIRE(out4 && K >= 1 && T >= 1, NLC_ERR_ARG, "nlc_debug_overlap_schedule: bad argument");
  nlc_model_s m{};
  m.nx = nx; m.S = S; m.Hm = 128;
  const OverlapSchedule s = overlap_schedule(&m, K, T);
  out4[0] = s.pp ? 1 : 0; out4[1] = s.roll_sms; out4[2] = s.split; out4[3] = (long long)T * s.sub_tiles;
  return NLC_OK;
}
extern "C" int nlc_debug_overlap_plan(int K, int T, int nx, int S, long long* out8) {
  NLC_REQUIRE(out8 && K >= 1 && T >= 1, NLC_ERR_ARG, "nlc_debug_overlap_plan: bad argument");
  nlc_model_s m{};
  m.nx = nx; m.S = S; m.Hm = 128;
  const bool ov = rollout_can_overlap(&m, K, T, NLC_MATH_TC_SPLIT3);
  const OverlapSchedule s = overlap_schedule(&m, K, T);
  out8[0] = ov ? 1 : 0; out8[1] = s.pp ? 1 : 0; out8[2] = s.roll_sms; out8[3] = s.passes; out8[4] = s.k1;
  out8[5] = s.split; out8[6] = (long long)T * s.sub_tiles; out8[7] = s.beside_steps;
  return NLC_OK;
}

static int planner_rollout_impl(nlc_planner_t p, const float* state_dev, int state_per_sample, const float* action_buffer_dev,
                                const float* noise_in_dev, void* stream, cudaEvent_t* ev) {
  const nlc_mppi_params& mp = p->d.mppi;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  NLC_CUDA_OK(cudaSetDevice(p->device));
  int rc = planner_check_model(p);
  if (rc != NLC_OK) return rc;
  // nlc_planner_finish re-arms stage 4's workspace, the encoder readiness counters and the sampler for the next rollout
  NLC_REQUIRE(!p->pending, NLC_ERR_ARG, "nlc_planner_rollout called twice without nlc_planner_finish in between");
  p->pending = true;
  if (ev) NLC_CUDA_OK(cudaEventRecord(ev[0], s));
  rc = perturb_launch(&mp, p->U, p->U_rolled, 1, noise_in_dev, p->d.seed, 0, p->call_ctr, action_buffer_dev, p->perturbed,
                      p->noise, p->hist, p->actions, p->pert_cost, stream);
  if (rc != NLC_OK) return rc;
  p->calls++;  // (the device-side call index is bumped by the step's combine kernel)
  if (ev) NLC_CUDA_OK(cudaEventRecord(ev[1], s));
  if (p->overlap) {
    // encoder || rollout: fork after stage 1, the encoder on this stream with all SMs but the rollout's, the rollout (one
    // 128-sample tile per CTA) on the side stream, join before stage 4.  The encoder is launched FIRST in host order: a
    // tool that serialises kernels then runs it to completion before the rollout starts polling.
    // (the readiness counters were zeroed by the previous step's combine kernel)
    // The rollout takes n_tiles SMs (one tile per CTA, ~9.5 us per step) or, from 89 tiles, n_tiles / 2 per pass (ping-pong form,
    // ~13.3 us per step): the encoder has the other SMs for the rollout's duration.  What those cannot encode in that time (12.6 us per
    // tile and SM: measured at config 4 / its shards; a wrong estimate only makes the rollout poll a little longer) is encoded
    // on all SMs BEFORE the fork - the windows of the first steps, the encoder walking its tiles in step-major order.
    // A ping-pong rollout of two passes per CTA (config 4 on one GPU: 512 tiles on 128 SMs) needs the windows of its first
    // pass's samples [0, k1) from its first step on: those are encoded in full before the fork, in the same launch as the
    // first steps of the last pass's samples [k1, K), the sub-plan whose step-major readiness the last pass polls ~T steps
    // after the fork.
    const OverlapSchedule sch = overlap_schedule(p->model, mp.K, mp.T);
    const int roll_sms = sch.roll_sms;
    const long long split = sch.split;  // first step-major tile (of the sub-plan) of the part that runs beside the rollout
    if (split > 0 || sch.k1 > 0) {
      rc = encode_history_overlapped(p->model, p->hist, mp.K, mp.T, mp.B, p->p, p->d.math_mode, p->ready, 148, 0, split, sch.k1, true, s);
      if (rc != NLC_OK) return rc;
    }
    NLC_CUDA_OK(cudaEventRecord(p->ev_fork, s));
    NLC_CUDA_OK(cudaStreamWaitEvent(p->side_stream, p->ev_fork, 0));
    rc = encode_history_overlapped(p->model, p->hist, mp.K, mp.T, mp.B, p->p, p->d.math_mode, p->ready, 148 - roll_sms, split, -1, sch.k1,
                                   false, s);
    if (rc != NLC_OK) return rc;
    if (ev) NLC_CUDA_OK(cudaEventRecord(ev[2], s));  // profile: end of the encoder's own span
    rc = launch_rollout_overlapped(p->model, &p->d.rollout, state_dev, state_per_sample, p->p, p->hist, p->pert_cost, mp.K, mp.T, mp.B,
                                   mp.nu, p->cost_total, p->states, p->d.math_mode, p->ready, 4u * (unsigned)sch.sub_tiles, p->ready + mp.T,
                                   p->side_stream);
    if (rc != NLC_OK) return rc;
    if (ev) NLC_CUDA_OK(cudaEventRecord(ev[5], p->side_stream));  // profile: end of the rollout's span (it starts at ev[1])
    NLC_CUDA_OK(cudaEventRecord(p->ev_join, p->side_stream));
    NLC_CUDA_OK(cudaStreamWaitEvent(s, p->ev_join, 0));
  } else {
    if (p->d.rollout.dynamics == NLC_DYN_NEURAL_LAPLACE) {
      rc = nlc_encode_history(p->model, p->hist, mp.K, mp.T, mp.B, p->p, p->d.math_mode, stream);
      if (rc != NLC_OK) return rc;
    }
    if (ev) NLC_CUDA_OK(cudaEventRecord(ev[2], s));
    rc = nlc_rollout_cost(p->model, &p->d.rollout, state_dev, state_per_sample, p->p, p->hist, p->pert_cost, mp.K, mp.T, mp.B,
                          mp.nu, p->cost_total, p->states, p->d.math_mode, stream);
    if (rc != NLC_OK) return rc;
  }
  if (ev) NLC_CUDA_OK(cudaEventRecord(ev[3], s));
  // connected shards: the last block of the sum kernel stores this shard's triple straight into every peer's mailbox over NVLink
  const ExchangePub pub = p->xchg ? ExchangePub{p->mailboxes_dev, p->d.n_shards, p->d.shard_index, p->xstride, p->xstep}
                                  : ExchangePub{nullptr, 0, 0, 0, nullptr};
  return softmax_partial_impl(p->cost_total, p->noise, mp.K, mp.T, mp.nu, mp.lambda_, p->triple, p->weights, p->softmax_ws, false, pub, s);
}

extern "C" int nlc_planner_rollout(nlc_planner_t p, const float* state_dev, int state_per_sample,
                                   const float* action_buffer_dev, const float* noise_in_dev, void* stream) {
  NLC_REQUIRE(p && state_dev && action_buffer_dev, NLC_ERR_ARG, "nlc_planner_rollout: null argument");
  return planner_rollout_impl(p, state_dev, state_per_sample, action_buffer_dev, noise_in_dev, stream, nullptr);
}

// Measurement entry point: one control step on the planner's own input buffers as DIRECT launches (no graph) with CUDA
// events at the stage boundaries, so the kernels are timed inside the step (warm L2, back to back) rather than alone.
// ms_out[0..5] = perturb, history encoder, rollout + cost, softmax update (partial + combine), encoder-and-rollout section,
// 1 if the two ran side by side (then [1] and [2] are their overlapping spans from the fork, [4] the section's wall time;
// otherwise [4] = [1] + [2]).  Synchronises the stream.
extern "C" int nlc_planner_step_profile(nlc_planner_t p, float* ms_out, void* stream) {
  NLC_REQUIRE(p && ms_out, NLC_ERR_ARG, "nlc_planner_step_profile: null argument");
  NLC_REQUIRE(p->d.n_shards == 1, NLC_ERR_UNSUPPORTED, "nlc_planner_step_profile is a single-shard entry point");
  NLC_CUDA_OK(cudaSetDevice(p->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  cudaEvent_t ev[6];
  for (auto& e : ev) NLC_CUDA_OK(cudaEventCreate(&e));
  int rc = planner_rollout_impl(p, p->state_in, 0, p->abuf_in, nullptr, stream, ev);
  if (rc == NLC_OK) rc = nlc_planner_finish(p, stream);
  if (rc == NLC_OK && cudaEventRecord(ev[4], s) != cudaSuccess) rc = NLC_ERR_CUDA;
  if (rc == NLC_OK && cudaEventSynchronize(ev[4]) != cudaSuccess) rc = NLC_ERR_CUDA;
  if (rc == NLC_OK) {
    bool ok = cudaEventElapsedTime(&ms_out[0], ev[0], ev[1]) == cudaSuccess && cudaEventElapsedTime(&ms_out[1], ev[1], ev[2]) == cudaSuccess &&
              cudaEventElapsedTime(&ms_out[3], ev[3], ev[4]) == cudaSuccess && cudaEventElapsedTime(&ms_out[4], ev[1], ev[3]) == cudaSuccess;
    if (p->overlap) ok = ok && cudaEventElapsedTime(&ms_out[2], ev[1], ev[5]) == cudaSuccess;
    else ok = ok && cudaEventElapsedTime(&ms_out[2], ev[2], ev[3]) == cudaSuccess;
    ms_out[5] = p->overlap ? 1.0f : 0.0f;
    if (!ok) rc = NLC_ERR_CUDA;
  }
  for (auto& e : ev) cudaEventDestroy(e);
  if (rc == NLC_ERR_CUDA) { set_error("nlc_planner_step_profile: CUDA event error: %s", cudaGetErrorString(cudaGetLastError())); }
  return rc;
}

extern "C" int nlc_planner_overlap_status(nlc_planner_t p, int* overlapped, int* status) {
  NLC_REQUIRE(p && overlapped && status, NLC_ERR_ARG, "nlc_planner_overlap_status: null argument");
  *overlapped = p->overlap ? 1 : 0;
  *status = 0;
  if (p->overlap) {
    unsigned int v = 0;
    NLC_CUDA_OK(cudaSetDevice(p->device));
    NLC_CUDA_OK(cudaDeviceSynchronize());
    NLC_CUDA_OK(cudaMemcpy(&v, p->ready + p->d.mppi.T, sizeof(v), cudaMemcpyDeviceToHost));
    *status = (int)v;
  }
  return NLC_OK;
}

extern "C" int nlc_planner_finish(nlc_planner_t p, void* stream) {
  NLC_REQUIRE(p, NLC_ERR_ARG, "nlc_planner_finish: null planner");
  const nlc_mppi_params& mp = p->d.mppi;
  NLC_CUDA_OK(cudaSetDevice(p->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  // the update is applied to the rolled sequence (mppi_delay.py:199-216); the same kernel bumps the sampler's call index and
  // re-arms stage 4's workspace and the encoder readiness counters for the next control step
  NLC_REQUIRE(p->pending, NLC_ERR_ARG, "nlc_planner_finish without a preceding nlc_planner_rollout");
  p->pending = false;
  StepTail tl{p->U_rolled, p->call_ctr, p->softmax_ws, p->overlap ? p->ready : nullptr, mp.T, nullptr, nullptr, nullptr, 0};
  if (p->to_host) { tl.host_action = p->h_out; tl.host_seq = reinterpret_cast<unsigned int*>(p->h_out + 4); tl.action_src = p->action; tl.nu = mp.nu; }
  if (p->xchg)  // wait (on the device) for the G triples of this control step in the own mailbox, then combine
    return launch_combine_exchange(p->mailbox, p->d.n_shards, p->xstride, mp.T, mp.nu, mp.lambda_, mp.u_scale, p->U, p->action, p->stats,
                                   p->xstep, p->xstatus, tl, s);
  const float* triples = p->d.n_shards == 1 ? p->triple : p->all_triples;
  return launch_combine(triples, p->d.n_shards, mp.T, mp.nu, mp.lambda_, mp.u_scale, p->U, p->action, p->stats, tl, s);
}

// One whole control step on the planner's own input buffers (state_in [nx], abuf_in [B][nu]), on-device sampler.
static int planner_core_direct(nlc_planner_t p, void* stream) {
  int rc = nlc_planner_rollout(p, p->state_in, 0, p->abuf_in, nullptr, stream);
  if (rc != NLC_OK) return rc;
  return nlc_planner_finish(p, stream);
}

// Capture that sequence (optionally bracketed by the pinned-host copies of the host entry point) once into a CUDA graph.
// Capture runs on a private stream (the caller's may be the legacy default stream, which cannot capture); the executable
// graph is then launched on the caller's stream.  Any failure leaves the planner on direct launches.
static cudaGraphExec_t planner_capture(nlc_planner_t p, bool with_host_copies) {
  static const bool disabled = [] { const char* e = getenv("NLC_NO_GRAPH"); return e && e[0] == '1'; }();
  if (disabled || (p->d.n_shards != 1 && !p->xchg)) return nullptr;
  if (!p->cap_stream && cudaStreamCreateWithFlags(&p->cap_stream, cudaStreamNonBlocking) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  // first use of every kernel outside capture: one-time function attributes and lazy module loading must not be captured
  const uint64_t calls0 = p->calls;
  const uint64_t launches0 = nlc_launch_count();
  if (planner_core_direct(p, p->cap_stream) != NLC_OK || cudaStreamSynchronize(p->cap_stream) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  p->kernels_per_step = (int)(nlc_launch_count() - launches0);
  // undo the warm-up's side effects on the control sequence and the sampler: U <- U before the roll is not recoverable
  // from U_rolled alone, so the warm-up ran on a scratch copy (see caller); the counter is rewound here
  if (cudaMemsetAsync(p->call_ctr, 0, sizeof(unsigned long long), p->cap_stream) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  unsigned long long c0 = calls0;
  if (cudaMemcpyAsync(p->call_ctr, &c0, sizeof(c0), cudaMemcpyHostToDevice, p->cap_stream) != cudaSuccess ||
      cudaStreamSynchronize(p->cap_stream) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  p->calls = calls0;
  const nlc_mppi_params& mp = p->d.mppi;
  const int nx = p->d.nx, nb = mp.B * mp.nu;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t exec = nullptr;
  if (cudaStreamBeginCapture(p->cap_stream, cudaStreamCaptureModeThreadLocal) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  bool ok = true;
  (void)mp;
  if (with_host_copies) ok = ok && launch_ingest(p->h_in, p->state_in, p->abuf_in, nx, nb, p->cap_stream) == NLC_OK;
  p->to_host = with_host_copies;
  ok = ok && planner_core_direct(p, p->cap_stream) == NLC_OK;
  p->to_host = false;
  const cudaError_t ee = cudaStreamEndCapture(p->cap_stream, &graph);
  p->calls = calls0;  // launches recorded during capture did not run
  if (!ok || ee != cudaSuccess || !graph) { cudaGetLastError(); if (graph) cudaGraphDestroy(graph); return nullptr; }
  if (cudaGraphInstantiate(&exec, graph, 0) != cudaSuccess) { cudaGetLastError(); exec = nullptr; }
  cudaGraphDestroy(graph);
  return exec;
}

// The warm-up inside planner_capture runs a real control step; it must not change the planner's state.  U is saved and
// restored around it (T*nu floats).
static cudaGraphExec_t planner_capture_preserving_state(nlc_planner_t p, bool with_host_copies) {
  const size_t n = sizeof(float) * p->d.mppi.T * p->d.mppi.nu;
  std::vector<float> U(p->d.mppi.T * p->d.mppi.nu), st(p->d.nx), ab(p->d.mppi.B * p->d.mppi.nu);
  if (cudaDeviceSynchronize() != cudaSuccess || cudaMemcpy(U.data(), p->U, n, cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(st.data(), p->state_in, sizeof(float) * st.size(), cudaMemcpyDeviceToHost) != cudaSuccess ||
      cudaMemcpy(ab.data(), p->abuf_in, sizeof(float) * ab.size(), cudaMemcpyDeviceToHost) != cudaSuccess) { cudaGetLastError(); return nullptr; }
  cudaGraphExec_t exec = planner_capture(p, with_host_copies);
  cudaDeviceSynchronize();
  cudaMemcpy(p->U, U.data(), n, cudaMemcpyHostToDevice);
  cudaMemcpy(p->state_in, st.data(), sizeof(float) * st.size(), cudaMemcpyHostToDevice);
  cudaMemcpy(p->abuf_in, ab.data(), sizeof(float) * ab.size(), cudaMemcpyHostToDevice);
  cudaGetLastError();
  return exec;
}

extern "C" int nlc_planner_step(nlc_planner_t p, void* stream) {
  NLC_REQUIRE(p, NLC_ERR_ARG, "nlc_planner_step: null planner");
  NLC_REQUIRE(p->d.n_shards == 1 || p->xchg, NLC_ERR_UNSUPPORTED,
              "nlc_planner_step needs a single shard, or shards connected by nlc_planner_exchange_connect");
  NLC_CUDA_OK(cudaSetDevice(p->device));
  { int rc = planner_check_model(p); if (rc != NLC_OK) return rc; }
  if (!p->graph_core_tried) { p->graph_core_tried = true; p->graph_core = planner_capture_preserving_state(p, false); }
  if (p->graph_core) {
    NLC_CUDA_OK(cudaGraphLaunch(p->graph_core, static_cast<cudaStream_t>(stream)));
    p->calls++;
    count_launch(p->kernels_per_step);
    return NLC_OK;
  }
  return planner_core_direct(p, stream);
}

extern "C" int nlc_planner_command_host(nlc_planner_t p, const double* state_host, const double* action_buffer_host,
                                        const float* noise_in_dev, double* action_host, void* stream) {
  NLC_REQUIRE(p && state_host && action_buffer_host && action_host, NLC_ERR_ARG, "nlc_planner_command_host: null argument");
  NLC_REQUIRE(p->d.n_shards == 1 || p->xchg, NLC_ERR_UNSUPPORTED,
              "nlc_planner_command_host needs a single shard, or shards connected by nlc_planner_exchange_connect");
  const nlc_mppi_params& mp = p->d.mppi;
  const int nx = p->d.nx, nb = mp.B * mp.nu;
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  NLC_CUDA_OK(cudaSetDevice(p->device));
  { int rc = planner_check_model(p); if (rc != NLC_OK) return rc; }
  if (!noise_in_dev && !p->graph_host_tried) { p->graph_host_tried = true; p->graph_host = planner_capture_preserving_state(p, true); }
  NLC_REQUIRE(nx + nb <= 64, NLC_ERR_SHAPE, "nlc_planner_command_host: state + action buffer exceed the 64-float staging area");
  for (int i = 0; i < nx; ++i) p->h_in[i] = (float)state_host[i];
  for (int i = 0; i < nb; ++i) p->h_in[nx + i] = (float)action_buffer_host[i];
  volatile unsigned int* seq = reinterpret_cast<volatile unsigned int*>(p->h_out + 4);
  const unsigned int seq0 = *seq;
  __sync_synchronize();  // the staged inputs are in memory before the launch that reads them
  if (!noise_in_dev && p->graph_host) {  // the whole step as one graph launch: ingest kernel, 5-6 kernels, the last reports to h_out
    NLC_CUDA_OK(cudaGraphLaunch(p->graph_host, s));
    p->calls++;
    count_launch(p->kernels_per_step + 1);  // + the ingest kernel
  } else {
    int rc = launch_ingest(p->h_in, p->state_in, p->abuf_in, nx, nb, s);
    if (rc != NLC_OK) return rc;
    rc = nlc_planner_rollout(p, p->state_in, 0, p->abuf_in, noise_in_dev, stream);
    if (rc != NLC_OK) return rc;
    p->to_host = true;
    rc = nlc_planner_finish(p, stream);
    p->to_host = false;
    if (rc != NLC_OK) return rc;
  }
  // Spin on the sequence word the combine kernel bumps after the action is visible system-wide.  Checked against the stream
  // every ~2 ms of spinning, so that a failed launch or a device error surfaces instead of spinning for ever.
  {
    unsigned long long spins = 0;
    while (*seq == seq0) {
      __builtin_ia32_pause();
      if ((++spins & 0xFFFFull) == 0) {
        const cudaError_t q = cudaStreamQuery(s);
        if (q == cudaSuccess) break;  // the step has retired (the word is visible by now, or the step failed before its end)
        if (q != cudaErrorNotReady) { set_error("nlc_planner_command_host: %s", cudaGetErrorString(q)); return NLC_ERR_CUDA; }
      }
    }
    __sync_synchronize();
    if (*seq == seq0) {
      NLC_CUDA_OK(cudaStreamSynchronize(s));
      NLC_REQUIRE(*seq != seq0, NLC_ERR_CUDA, "nlc_planner_command_host: the control step retired without reporting its action");
    }
  }
  for (int i = 0; i < mp.nu; ++i) action_host[i] = p->h_out[i];
  return NLC_OK;
}

// ------------------------------------------------------------------------------------------------------------------
// Instance-batched planner (BASELINE config 5: many env x seed instances planning in the same control step).
// I independent MPPIDelay objects of one environment / model share ONE wide encoder launch and ONE rollout launch over
// the concatenated I*K samples (both kernels are row-independent; the rollout reads each instance's state through the
// rows-per-state form of `state_per_sample`); stage 1 and stage 4 run per instance on the instance's contiguous slices
// with the same kernels - and hence the same arithmetic - as the single planner, so instance i of a batch reproduces a
// stand-alone planner with the same seed.
// ------------------------------------------------------------------------------------------------------------------
struct nlc_batch_planner_s {
  int device, I;
  nlc_model_t model;
  nlc_planner_desc d;          // per instance (mppi.K = samples per instance)
  std::vector<uint64_t> seeds;
  uint64_t calls;
  void* arena;
  float *U, *U_rolled, *noise, *perturbed, *hist, *actions, *pert_cost, *p, *cost_total, *weights, *states, *triple, *stats;
  char* softmax_ws;
  size_t ws_stride;
};

extern "C" int nlc_batch_planner_create(nlc_batch_planner_t* out, nlc_model_t model, const nlc_planner_desc* d, int n_instances,
                                        const uint64_t* seeds, int device) {
  NLC_REQUIRE(out && d && seeds, NLC_ERR_ARG, "nlc_batch_planner_create: null argument");
  *out = nullptr;
  int rc = check_device_arch(device);
  if (rc != NLC_OK) return rc;
  const nlc_mppi_params& mp = d->mppi;
  NLC_REQUIRE(n_instances >= 1 && n_instances <= 4096, NLC_ERR_ARG, "batch planner: 1..4096 instances");
  NLC_REQUIRE(mp.K >= 1 && mp.T >= 1 && mp.B >= 1 && mp.B <= 8, NLC_ERR_SHAPE, "batch planner: K, T >= 1 and 1 <= B <= 8 required");
  NLC_REQUIRE(mp.nu >= 1 && mp.nu <= 4 && d->nx >= 1 && d->nx <= kMaxNx, NLC_ERR_SHAPE, "batch planner: nu/nx out of range");
  NLC_REQUIRE(mp.T * mp.nu <= 256, NLC_ERR_SHAPE, "batch planner: T*nu exceeds 256");
  NLC_REQUIRE(d->n_shards == 1 && d->shard_index == 0, NLC_ERR_UNSUPPORTED, "batch planner: instances are not K-sharded (shard by instance)");
  NLC_REQUIRE(mp.lambda_ > 0.0f, NLC_ERR_ARG, "batch planner: lambda must be positive");
  NLC_REQUIRE((long long)n_instances * mp.K <= 0x7fffffffLL / (mp.T * 4), NLC_ERR_SHAPE, "batch planner: I*K*T too large");
  if (d->rollout.dynamics == NLC_DYN_NEURAL_LAPLACE) {
    NLC_REQUIRE(model != nullptr, NLC_ERR_ARG, "batch planner: Neural Laplace dynamics need a model handle");
    NLC_REQUIRE(model->device == device, NLC_ERR_ARG, "batch planner: model lives on device %d, planner on %d", model->device, device);
    NLC_REQUIRE(model->nx == d->nx && model->nu == mp.nu, NLC_ERR_SHAPE, "batch planner: model dims do not match");
  }
  // stage 4 reads each instance's cost slice 16 bytes wide (nlc_softmax_partial): instance i starts at cost_total + i*K
  NLC_REQUIRE(n_instances == 1 || mp.K % 4 == 0, NLC_ERR_SHAPE, "batch planner: samples per instance (%d) must be a multiple of 4", mp.K);
  NLC_REQUIRE(model == nullptr || !model->destroy_requested, NLC_ERR_ARG, "batch planner: the model handle has been destroyed");
  nlc_batch_planner_s* p = new nlc_batch_planner_s();
  p->device = device; p->I = n_instances; p->model = model; p->d = *d; p->calls = 0; p->arena = nullptr;
  p->seeds.assign(seeds, seeds + n_instances);
  const size_t I = n_instances, K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, nx = d->nx, L = B - 1 + T, TN = T * nu, IK = I * K;
  p->ws_stride = ((size_t)nlc_softmax_workspace_bytes((int)K, (int)TN) + 255) / 256 * 256;
  std::vector<size_t> sizes = {I * TN, I * TN, IK * TN, IK * TN, IK * L * nu, IK * TN, IK, IK * T * 2, IK, IK,
                               (d->keep_states ? IK * T * nx : 0), I * (2 + TN), I * 2, I * p->ws_stride / 4};
  std::vector<size_t> offs;
  size_t total = 0;
  for (size_t s : sizes) { offs.push_back(total); total += (s + 63) / 64 * 64; }
  auto fail = [&](int code) { if (p->arena) cudaFree(p->arena); delete p; return code; };
  if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice failed"); return fail(NLC_ERR_CUDA); }
  if (cudaMalloc(&p->arena, total * sizeof(float)) != cudaSuccess) { cudaGetLastError(); p->arena = nullptr; set_error("batch planner: cudaMalloc(%zu) failed", total * sizeof(float)); return fail(NLC_ERR_NOMEM); }
  if (cudaMemset(p->arena, 0, total * sizeof(float)) != cudaSuccess) { set_error("batch planner: memset failed"); return fail(NLC_ERR_CUDA); }
  float* base = static_cast<float*>(p->arena);
  float** slots[] = {&p->U, &p->U_rolled, &p->noise, &p->perturbed, &p->hist, &p->actions, &p->pert_cost, &p->p,
                     &p->cost_total, &p->weights, &p->states, &p->triple, &p->stats};
  for (size_t i = 0; i < sizeof(slots) / sizeof(slots[0]); ++i) *slots[i] = base + offs[i];
  if (!d->keep_states) p->states = nullptr;
  p->softmax_ws = reinterpret_cast<char*>(base + offs[13]);
  if (model) model->refs++;
  *out = p;
  return NLC_OK;
}

extern "C" int nlc_batch_planner_destroy(nlc_batch_planner_t p) {
  if (!p) return NLC_OK;
  cudaSetDevice(p->device);
  cudaDeviceSynchronize();
  model_release(p->model);
  if (p->arena) cudaFree(p->arena);
  delete p;
  return NLC_OK;
}

extern "C" int nlc_batch_planner_buffer(nlc_batch_planner_t p, int which, void** dev_ptr, int64_t* n_floats) {
  NLC_REQUIRE(p && dev_ptr && n_floats, NLC_ERR_ARG, "nlc_batch_planner_buffer: null argument");
  const nlc_mppi_params& mp = p->d.mppi;
  const int64_t I = p->I, K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, nx = p->d.nx, TN = T * nu, IK = I * K;
  float* ptr = nullptr; int64_t n = 0;
  switch (which) {
    case NLC_BUF_U: ptr = p->U; n = I * TN; break;
    case NLC_BUF_NOISE: ptr = p->noise; n = IK * TN; break;
    case NLC_BUF_PERTURBED: ptr = p->perturbed; n = IK * TN; break;
    case NLC_BUF_COST_TOTAL: ptr = p->cost_total; n = IK; break;
    case NLC_BUF_WEIGHTS: ptr = p->weights; n = IK; break;
    case NLC_BUF_STATES: ptr = p->states; n = p->states ? IK * T * nx : 0; break;
    case NLC_BUF_ACTIONS: ptr = p->actions; n = IK * TN; break;
    case NLC_BUF_TRIPLE: ptr = p->triple; n = I * (2 + TN); break;
    case NLC_BUF_STATS: ptr = p->stats; n = I * 2; break;
    case NLC_BUF_HIST: ptr = p->hist; n = IK * (B - 1 + T) * nu; break;
    case NLC_BUF_P: ptr = p->p; n = IK * T * 2; break;
    default: set_error("nlc_batch_planner_buffer: unknown buffer id %d", which); return NLC_ERR_ARG;
  }
  *dev_ptr = ptr; *n_floats = n;
  return NLC_OK;
}

extern "C" int nlc_batch_planner_command(nlc_batch_planner_t p, const float* state_dev, const float* action_buffer_dev,
                                         const float* noise_in_dev, float* action_dev, void* stream) {
  NLC_REQUIRE(p && state_dev && action_buffer_dev && action_dev, NLC_ERR_ARG, "nlc_batch_planner_command: null argument");
  const nlc_mppi_params& mp = p->d.mppi;
  const size_t K = mp.K, T = mp.T, nu = mp.nu, B = mp.B, L = B - 1 + T, TN = T * nu;
  const int I = p->I;
  NLC_CUDA_OK(cudaSetDevice(p->device));
  cudaStream_t s = static_cast<cudaStream_t>(stream);
  int rc;
  if (p->d.rollout.dynamics == NLC_DYN_NEURAL_LAPLACE) {
    const double want = (double)p->d.rollout.dt;
    NLC_REQUIRE(!p->model->destroy_requested && fabs(p->model->ts_pred - want) <= 1e-6 * fabs(want), NLC_ERR_ARG,
                "batch planner: the model is folded for prediction time %.9g, not dt = %.9g", p->model->ts_pred, want);
  }
  for (int i = 0; i < I; ++i) {  // stage 1 per instance (its own U, action buffer and RNG stream)
    const size_t o = (size_t)i * K;
    rc = nlc_perturb(&mp, p->U + i * TN, p->U_rolled + i * TN, 1, noise_in_dev ? noise_in_dev + o * TN : nullptr, p->seeds[i], p->calls,
                     action_buffer_dev + (size_t)i * B * nu, p->perturbed + o * TN, p->noise + o * TN, p->hist + o * L * nu,
                     p->actions + o * TN, p->pert_cost + o, stream);
    if (rc != NLC_OK) return rc;
  }
  p->calls++;
  const int IK = (int)(I * K);
  if (p->d.rollout.dynamics == NLC_DYN_NEURAL_LAPLACE) {  // stage 2a: every window of every instance in one pass
    rc = nlc_encode_history(p->model, p->hist, IK, (int)T, (int)B, p->p, p->d.math_mode, stream);
    if (rc != NLC_OK) return rc;
  }
  // stages 2b+3: one launch; sample k reads the state of instance k / K
  rc = nlc_rollout_cost(p->model, &p->d.rollout, state_dev, (int)K, p->p, p->hist, p->pert_cost, IK, (int)T, (int)B, (int)nu,
                        p->cost_total, p->states, p->d.math_mode, stream);
  if (rc != NLC_OK) return rc;
  NLC_CUDA_OK(cudaMemcpyAsync(p->U, p->U_rolled, sizeof(float) * I * TN, cudaMemcpyDeviceToDevice, s));
  for (int i = 0; i < I; ++i) {  // stage 4 per instance
    const size_t o = (size_t)i * K;
    float* triple = p->triple + (size_t)i * (2 + TN);
    rc = nlc_softmax_partial(p->cost_total + o, p->noise + o * TN, (int)K, (int)T, (int)nu, mp.lambda_, triple, p->weights + o,
                             p->softmax_ws + (size_t)i * p->ws_stride, stream);
    if (rc != NLC_OK) return rc;
    rc = nlc_softmax_combine(triple, 1, (int)T, (int)nu, mp.lambda_, mp.u_scale, p->U + i * TN, action_dev + (size_t)i * nu,
                             p->stats + 2 * i, stream);
    if (rc != NLC_OK) return rc;
  }
  return NLC_OK;
}

extern "C" int nlc_batch_planner_set_U(nlc_batch_planner_t p, const double* U_host) {
  NLC_REQUIRE(p && U_host, NLC_ERR_ARG, "nlc_batch_planner_set_U: null argument");
  const size_t n = (size_t)p->I * p->d.mppi.T * p->d.mppi.nu;
  std::vector<float> tmp(n);
  for (size_t i = 0; i < n; ++i) tmp[i] = (float)U_host[i];
  NLC_CUDA_OK(cudaSetDevice(p->device));
  NLC_CUDA_OK(cudaMemcpy(p->U, tmp.data(), sizeof(float) * n, cudaMemcpyHostToDevice));
  return NLC_OK;
}
