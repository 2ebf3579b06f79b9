// Model handle: packs a reference NeuralLaplaceModel state_dict (w_nl.py:66-145) into the device
// layouts the kernels read, and folds the constants of a fixed prediction time in fp64.
#include <stdarg.h>
#include <cmath>
#include <string.h>

#include <atomic>
#include <vector>

#include "common.cuh"
#include "tc_pack.cuh"

namespace nlc {

static thread_local char g_err[512] = "";
static std::atomic<uint64_t> g_launches{0};

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}
void count_launch(int n) { g_launches.fetch_add((uint64_t)n, std::memory_order_relaxed); }

void warn_once(int slot, const char* fmt, ...) {
  static std::atomic<unsigned> seen{0};
  const unsigned bit = 1u << (slot & 15);
  if (seen.fetch_or(bit) & bit) return;
  va_list ap;
  va_start(ap, fmt);
  fputs("libnlc_b200: warning: ", stderr);
  vfprintf(stderr, fmt, ap);
  fputc('\n', stderr);
  va_end(ap);
}

int check_device_arch(int device) {
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0) {
    cudaGetLastError();
    set_error("no CUDA device visible: this library has no CPU path");
    return NLC_ERR_ARCH;
  }
  if (device < 0 || device >= n) {
    set_error("device %d out of range (%d visible)", device, n);
    return NLC_ERR_ARCH;
  }
  // the answer cannot change while the process lives; cudaGetDeviceProperties costs milliseconds, so ask once per device
  static std::atomic<int> cached_major[64];
  int major = device < 64 ? cached_major[device].load(std::memory_order_relaxed) : 0, minor = 0;
  if (major == 0) {
    if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, device) != cudaSuccess ||
        cudaDeviceGetAttribute(&minor, cudaDevAttrComputeCapabilityMinor, device) != cudaSuccess) {
      cudaGetLastError();
      set_error("cudaDeviceGetAttribute(%d) failed", device);
      return NLC_ERR_ARCH;
    }
    if (device < 64) cached_major[device].store(major, std::memory_order_relaxed);
  }
  if (major != 10) {
    set_error("device %d is sm_%dx; the kernels are built for sm_100a only", device, major);
    return NLC_ERR_ARCH;
  }
  return NLC_OK;
}

}  // namespace nlc

using namespace nlc;

extern "C" const char* nlc_last_error(void) { return g_err; }
extern "C" int nlc_version(void) { return NLC_VERSION; }
extern "C" int nlc_device_check(int device) { return check_device_arch(device); }
extern "C" uint64_t nlc_launch_count(void) { return g_launches.load(); }

namespace {

struct Arena {  // host-side staging of one contiguous device allocation
  std::vector<float> data;
  size_t add(size_t n) {
    size_t off = (data.size() + 63) / 64 * 64;  // 256-byte aligned sections
    data.resize(off + n, 0.0f);
    return off;
  }
};

const double kAlpha = 1.0e-3, kTol = 1.0e-2, kScale = 2.0, kEps = 1.0e-6;  // torchlaplace Fourier defaults

}  // namespace

// Fold everything that depends on the (normalised) prediction time.  oracle/ilt.py:fourier_s_points,
// complex_to_sphere, fourier_line_integrate are the CPU statement of the same arithmetic.
static int fold_prediction_time(nlc_model_s* m, double ts_pred) {
  const int S = m->S, Hm = m->Hm, L = m->nx + 2, in0 = 2 * S + L;
  double t = ts_pred;
  if (m->normalize && m->normalize_time) t = ts_pred / (m->dt * 8.0);  // w_nl.py:123
  NLC_REQUIRE(t > 0.0, NLC_ERR_ARG, "prediction time must be positive (got %g)", ts_pred);
  const double T = kScale * (t + kEps);
  const double gamma = kAlpha - log(kTol) / T;
  std::vector<double> th(S), ph(S);
  std::vector<float> phase(S), weight(S), b1(Hm);
  const double scale = exp(gamma * t) / T;
  for (int k = 0; k < S; ++k) {
    double re = gamma, im = M_PI * k / T;
    double r2 = re * re + im * im;
    th[k] = atan2(im, re);
    ph[k] = asin((r2 - 1.0) / (r2 + 1.0));
    double a = fmod(k * M_PI * t / T, 2.0 * M_PI);
    if (a > M_PI) a -= 2.0 * M_PI;
    phase[k] = (float)a;
    weight[k] = (float)(scale * (k == 0 ? 0.5 : 1.0));
  }
  for (int n = 0; n < Hm; ++n) {
    double acc = m->h.b0[n];
    const double* row = m->h.w0 + (size_t)n * in0;
    for (int k = 0; k < S; ++k) acc += row[k] * th[k];
    for (int k = 0; k < S; ++k) acc += row[S + k] * ph[k];
    b1[n] = (float)acc;
  }
  // first layer as a K = 16 tensor-core operand (rollout_tc2.cu): columns [obs_n | p_action | folded bias | 0..], -2 log2(e) folded
  std::vector<uint16_t> w1img((size_t)2 * Hm * 16);
  {
    const double cN = -2.0 * 1.4426950408889634;
    std::vector<double> w1((size_t)Hm * 16, 0.0);
    for (int n = 0; n < Hm; ++n) {
      double acc = m->h.b0[n];
      const double* row = m->h.w0 + (size_t)n * in0;
      for (int k = 0; k < S; ++k) acc += row[k] * th[k];
      for (int k = 0; k < S; ++k) acc += row[S + k] * ph[k];
      for (int j = 0; j < L; ++j) w1[(size_t)n * 16 + j] = cN * row[2 * S + j];
      w1[(size_t)n * 16 + L] = cN * acc;
    }
    nlc::tc_pack_weight_split(w1.data(), Hm, 16, w1img.data(), w1img.data() + (size_t)Hm * 16);
  }
  NLC_CUDA_OK(cudaSetDevice(m->device));
  // the folded constants are rewritten in place: kernels of an earlier control step (possibly on a non-blocking
  // stream, which a plain cudaMemcpy does not order against) must have finished reading them
  NLC_CUDA_OK(cudaDeviceSynchronize());
  NLC_CUDA_OK(cudaMemcpy(m->d.mlp2_w1, w1img.data(), w1img.size() * sizeof(uint16_t), cudaMemcpyHostToDevice));
  NLC_CUDA_OK(cudaMemcpy(m->d.b1_fold, b1.data(), sizeof(float) * Hm, cudaMemcpyHostToDevice));
  NLC_CUDA_OK(cudaMemcpy(m->d.ilt_phase, phase.data(), sizeof(float) * S, cudaMemcpyHostToDevice));
  NLC_CUDA_OK(cudaMemcpy(m->d.ilt_weight, weight.data(), sizeof(float) * S, cudaMemcpyHostToDevice));
  m->ts_pred = ts_pred;
  m->t_norm = t;
  return NLC_OK;
}

extern "C" int nlc_model_set_prediction_time(nlc_model_t m, double ts_pred) {
  NLC_REQUIRE(m != nullptr, NLC_ERR_ARG, "null model");
  return fold_prediction_time(m, ts_pred);
}

extern "C" int nlc_model_create(nlc_model_t* out, const nlc_model_desc* d, int device) {
  NLC_REQUIRE(out && d, NLC_ERR_ARG, "null argument");
  *out = nullptr;
  int rc = check_device_arch(device);
  if (rc != NLC_OK) return rc;
  const int nx = d->state_dim, nu = d->action_dim, Hm = d->hidden_units, S = d->s_terms;
  const int gin = nu + (d->encode_obs_time ? 1 : 0);
  NLC_REQUIRE(nx >= 1 && nx <= kMaxNx, NLC_ERR_SHAPE, "state_dim %d outside [1,%d]", nx, kMaxNx);
  NLC_REQUIRE(nu >= 1 && gin <= kMaxNu, NLC_ERR_SHAPE, "GRU input width %d outside [1,%d]", gin, kMaxNu);
  NLC_REQUIRE(Hm == 128 || Hm == 64, NLC_ERR_SHAPE, "hidden_units must be 128 (config.py:37) or 64 (the class default, w_nl.py:71); got %d", Hm);
  NLC_REQUIRE(S >= 2 && S <= kMaxS, NLC_ERR_SHAPE, "s_terms %d outside [2,%d]", S, kMaxS);
  NLC_REQUIRE(d->action_std_len == 1 || d->action_std_len == nu, NLC_ERR_SHAPE, "action_std_len must be 1 or nu");
  const void* ptrs[] = {d->state_mean, d->state_std, d->action_mean, d->action_std, d->gru_w_ih_l0, d->gru_w_hh_l0,
                        d->gru_b_ih_l0, d->gru_b_hh_l0, d->gru_w_ih_l1, d->gru_w_hh_l1, d->gru_b_ih_l1, d->gru_b_hh_l1,
                        d->enc_out_w, d->enc_out_b, d->mlp_w0, d->mlp_b0, d->mlp_w2, d->mlp_b2, d->mlp_w4, d->mlp_b4};
  for (const void* p : ptrs) NLC_REQUIRE(p != nullptr, NLC_ERR_ARG, "null weight pointer in nlc_model_desc");

  const int Hg = Hm / 2, G3 = 3 * Hg, L = nx + 2, in0 = 2 * S + L, N3 = 2 * nx * S, N3p = (N3 + 3) / 4 * 4, N3t = (N3 + 15) / 16 * 16;
  {
    // Every parameter must be finite.  Besides being meaningless otherwise, the tensor-core encoder's [x | 1] operand
    // block lets the zero half of its A side multiply neighbouring (weight) data of the B side (encode_tc2.cu): that
    // product is exactly zero only for finite data.
    const struct { const double* p; size_t n; const char* name; } chk[] = {
        {d->state_mean, (size_t)nx, "state_mean"}, {d->state_std, (size_t)nx, "state_std"}, {d->action_mean, (size_t)nu, "action_mean"},
        {d->action_std, (size_t)d->action_std_len, "action_std"}, {d->gru_w_ih_l0, (size_t)G3 * gin, "gru.weight_ih_l0"},
        {d->gru_w_hh_l0, (size_t)G3 * Hg, "gru.weight_hh_l0"}, {d->gru_b_ih_l0, (size_t)G3, "gru.bias_ih_l0"}, {d->gru_b_hh_l0, (size_t)G3, "gru.bias_hh_l0"},
        {d->gru_w_ih_l1, (size_t)G3 * Hg, "gru.weight_ih_l1"}, {d->gru_w_hh_l1, (size_t)G3 * Hg, "gru.weight_hh_l1"}, {d->gru_b_ih_l1, (size_t)G3, "gru.bias_ih_l1"},
        {d->gru_b_hh_l1, (size_t)G3, "gru.bias_hh_l1"}, {d->enc_out_w, (size_t)2 * Hg, "linear_out.weight"}, {d->enc_out_b, 2, "linear_out.bias"},
        {d->mlp_w0, (size_t)Hm * in0, "mlp.0.weight"}, {d->mlp_b0, (size_t)Hm, "mlp.0.bias"}, {d->mlp_w2, (size_t)Hm * Hm, "mlp.2.weight"},
        {d->mlp_b2, (size_t)Hm, "mlp.2.bias"}, {d->mlp_w4, (size_t)N3 * Hm, "mlp.4.weight"}, {d->mlp_b4, (size_t)N3, "mlp.4.bias"}};
    for (const auto& c : chk)
      for (size_t i = 0; i < c.n; ++i) NLC_REQUIRE(std::isfinite(c.p[i]), NLC_ERR_ARG, "model parameter %s[%zu] is not finite", c.name, i);
  }
  nlc_model_s* m = new nlc_model_s();
  memset(&m->d, 0, sizeof(m->d));
  m->device = device; m->nx = nx; m->nu = nu; m->gin = gin; m->Hm = Hm; m->Hg = Hg; m->S = S; m->N3 = N3; m->N3p = N3p; m->N3t = N3t;
  m->normalize = d->normalize; m->normalize_time = d->normalize_time; m->encode_obs_time = d->encode_obs_time;
  m->dt = d->dt; m->arena = nullptr; m->refs = 0; m->destroy_requested = false;
  {
    double worst = 0.0;
    for (int g = 0; g < 2 * Hg; ++g) {  // PyTorch gate order r, z, n: rows [0, 2 Hg) are r and z
      double acc = fabs(d->gru_b_ih_l1[g] + d->gru_b_hh_l1[g]);
      for (int k = 0; k < Hg; ++k) acc += fabs(d->gru_w_ih_l1[(size_t)g * Hg + k]) + fabs(d->gru_w_hh_l1[(size_t)g * Hg + k]);
      worst = acc > worst ? acc : worst;
    }
    m->enc_l1_bounded = worst * 1.4426950408889634 < 59.0;  // one unit of slack for the fp16 split and fp32 accumulation
  }

  Arena A;
  auto put = [&](size_t off, size_t i, double v) { A.data[off + i] = (float)v; };
  size_t o_w_ih0 = A.add((size_t)G3 * gin), o_b_ih0 = A.add(G3), o_b_hh0 = A.add(G3);
  size_t o_hh0 = A.add((size_t)Hg * G3), o_ih1 = A.add((size_t)Hg * G3), o_hh1 = A.add((size_t)Hg * G3);
  size_t o_b_ih1 = A.add(G3), o_b_hh1 = A.add(G3), o_wout = A.add(2 * Hg), o_bout = A.add(2);
  size_t o_w1full = A.add((size_t)in0 * Hm), o_b1raw = A.add(Hm), o_w1x = A.add((size_t)L * Hm), o_b1f = A.add(Hm);
  size_t o_w2 = A.add((size_t)Hm * Hm), o_b2 = A.add(Hm), o_w3 = A.add((size_t)Hm * N3p), o_b3 = A.add(N3p);
  size_t o_phase = A.add(S), o_weight = A.add(S);
  size_t o_smean = A.add(nx), o_sinv = A.add(nx), o_amean = A.add(gin), o_ainv = A.add(gin);
  // the same constants in fp64 (two floats per double; sections are 256-byte aligned)
  size_t o_smean64 = A.add(2 * nx), o_sinv64 = A.add(2 * nx), o_amean64 = A.add(2 * gin), o_ainv64 = A.add(2 * gin);
  auto put64 = [&](size_t off, size_t i, double v) { memcpy(A.data.data() + off + 2 * i, &v, sizeof(double)); };
  // tensor-core operand image of the three recurrent GRU matrices: fp16 hi/lo, UMMA canonical layout
  const size_t tc_halves = (size_t)3 * 2 * G3 * Hg;
  size_t o_enc2w = A.add(tc_halves / 2), o_enc2c = A.add(nlc::kE2Count), o_enc2x = A.add(2 * 256 * 8 / 2);
  size_t o_m2w1 = A.add((size_t)2 * Hm * 16 / 2), o_m2w2 = A.add((size_t)2 * Hm * Hm / 2), o_m2w3 = A.add((size_t)2 * N3t * Hm / 2);
  size_t o_m2c = A.add(128 + 416);  // b2 | b3 (up to 416 (theta, phi) columns: rollout_tc2.cu kMaxN3)
  // group-uniform W3 image of the ping-pong rollout: 32 columns per unit, NX (S-1)/16 regular units + 1 unit of last terms
  const int gu_upc = (S - 1) % 16 == 0 ? (S - 1) / 16 : 0;
  const int gu_units = gu_upc ? nx * gu_upc + 1 : 0;
  const int N3u = (Hm == 128 && gu_units >= 1 && gu_units <= 13) ? 32 * gu_units : 0;  // <= 416 columns (rollout_tc2.cu kMaxN3)
  m->N3u = N3u;
  size_t o_m2w3u = A.add((size_t)2 * (N3u ? N3u : 16) * Hm / 2), o_m2cu = A.add(N3u ? N3u : 16);

  for (int i = 0; i < G3 * gin; ++i) put(o_w_ih0, i, d->gru_w_ih_l0[i]);
  for (int i = 0; i < G3; ++i) {
    put(o_b_ih0, i, d->gru_b_ih_l0[i]); put(o_b_hh0, i, d->gru_b_hh_l0[i]);
    put(o_b_ih1, i, d->gru_b_ih_l1[i]); put(o_b_hh1, i, d->gru_b_hh_l1[i]);
  }
  for (int g = 0; g < G3; ++g)
    for (int k = 0; k < Hg; ++k) {
      put(o_hh0, (size_t)k * G3 + g, d->gru_w_hh_l0[(size_t)g * Hg + k]);
      put(o_ih1, (size_t)k * G3 + g, d->gru_w_ih_l1[(size_t)g * Hg + k]);
      put(o_hh1, (size_t)k * G3 + g, d->gru_w_hh_l1[(size_t)g * Hg + k]);
    }
  for (int i = 0; i < 2 * Hg; ++i) put(o_wout, i, d->enc_out_w[i]);
  for (int i = 0; i < 2; ++i) put(o_bout, i, d->enc_out_b[i]);
  for (int n = 0; n < Hm; ++n) {
    for (int i = 0; i < in0; ++i) put(o_w1full, (size_t)i * Hm + n, d->mlp_w0[(size_t)n * in0 + i]);
    for (int i = 0; i < L; ++i) put(o_w1x, (size_t)i * Hm + n, d->mlp_w0[(size_t)n * in0 + 2 * S + i]);
    put(o_b1raw, n, d->mlp_b0[n]);
    put(o_b2, n, d->mlp_b2[n]);
    for (int k = 0; k < Hm; ++k) put(o_w2, (size_t)k * Hm + n, d->mlp_w2[(size_t)n * Hm + k]);
  }
  // third layer: pair the theta and phi columns of every (channel, term)
  for (int c = 0; c < nx; ++c)
    for (int k = 0; k < S; ++k)
      for (int part = 0; part < 2; ++part) {
        const int src = (part * nx + c) * S + k;  // w_nl.py:56-62: theta rows [0,nx), phi rows [nx,2nx)
        const int dst = 2 * (c * S + k) + part;
        for (int h = 0; h < Hm; ++h) put(o_w3, (size_t)h * N3p + dst, d->mlp_w4[(size_t)src * Hm + h]);
        put(o_b3, dst, d->mlp_b4[src]);
      }
  for (int i = 0; i < nx; ++i) {
    put(o_smean, i, d->normalize ? d->state_mean[i] : 0.0);
    put(o_sinv, i, d->normalize ? 1.0 / d->state_std[i] : 1.0);
    put64(o_smean64, i, d->normalize ? d->state_mean[i] : 0.0);
    put64(o_sinv64, i, d->normalize ? 1.0 / d->state_std[i] : 1.0);
  }
  for (int i = 0; i < gin; ++i) {
    // w_nl.py:121 (normalised) / :129 (actions / 3.0).  With encode_obs_time the extra channel is
    // normalised like an action, as the reference's broadcast does.
    double mean = 0.0, stdv = 3.0;
    if (d->normalize) {
      mean = d->action_mean[i < nu ? i : nu - 1];
      stdv = d->action_std[d->action_std_len == 1 ? 0 : (i < nu ? i : nu - 1)];
    }
    put(o_amean, i, mean);
    put(o_ainv, i, 1.0 / stdv);
    put64(o_amean64, i, mean);
    put64(o_ainv64, i, 1.0 / stdv);
  }
  if (Hm == 128) {  // (the tensor-core kernels are built for hidden_units = 128: other widths run on the fp32 kernels)
    // encode_tc2.cu operands: exponent scales folded (sigmoid(x) = 1/(1 + 2^(-log2e x)), tanh(x) = 2/(1 + 2^(-2 log2e x)) - 1)
    const double cR = -1.4426950408889634, cN = 2.0 * cR;
    auto gate_scale = [&](int row) { return row < 2 * Hg ? cR : cN; };
    std::vector<double> w((size_t)G3 * Hg);
    uint16_t* tc2 = reinterpret_cast<uint16_t*>(A.data.data() + o_enc2w);
    const double* mats[3] = {d->gru_w_hh_l0, d->gru_w_ih_l1, d->gru_w_hh_l1};
    for (int mi = 0; mi < 3; ++mi) {
      for (int r = 0; r < G3; ++r) {
        // destination row order: natural [r | z | n], except W_ih1 -> [n | r | z]
        const int dst = (mi == 1) ? (r < 2 * Hg ? r + Hg : r - 2 * Hg) : r;
        for (int k = 0; k < Hg; ++k) w[(size_t)dst * Hg + k] = gate_scale(r) * mats[mi][(size_t)r * Hg + k];
      }
      nlc::tc_pack_weight_split(w.data(), G3, Hg, tc2 + (size_t)mi * 2 * G3 * Hg, tc2 + (size_t)mi * 2 * G3 * Hg + (size_t)G3 * Hg);
    }
    for (int i = 0; i < 2 * Hg; ++i) put(o_enc2c, nlc::kE2Brz0 + i, cR * (d->gru_b_ih_l0[i] + d->gru_b_hh_l0[i]));
    for (int u = 0; u < Hg; ++u) {
      put(o_enc2c, nlc::kE2Bin0 + u, cN * d->gru_b_ih_l0[2 * Hg + u]);
      put(o_enc2c, nlc::kE2Bhn0 + u, cN * d->gru_b_hh_l0[2 * Hg + u]);
      put(o_enc2c, nlc::kE2B1 + u, cN * d->gru_b_ih_l1[2 * Hg + u]);
      put(o_enc2c, nlc::kE2B1 + Hg + u, cR * (d->gru_b_ih_l1[u] + d->gru_b_hh_l1[u]));
      put(o_enc2c, nlc::kE2B1 + 2 * Hg + u, cR * (d->gru_b_ih_l1[Hg + u] + d->gru_b_hh_l1[Hg + u]));
      put(o_enc2c, nlc::kE2B1 + 3 * Hg + u, cN * d->gru_b_hh_l1[2 * Hg + u]);
    }
    for (int g = 0; g < 3; ++g)
      for (int v = 0; v < gin; ++v)
        for (int u = 0; u < Hg; ++u)
          put(o_enc2c, nlc::kE2Wih0 + (size_t)(g * nlc::kMaxNu + v) * Hg + u, (g < 2 ? cR : cN) * d->gru_w_ih_l0[(size_t)(g * Hg + u) * gin + v]);
    if (gin <= 2) {  // the [x | 1] blocks of the tensor-core encoder (encode_tc2.cu): [layer][256 rows][8 halves]
      uint16_t* wx = reinterpret_cast<uint16_t*>(A.data.data() + o_enc2x);
      auto split = [](double v, uint16_t& hi, uint16_t& lo) {
        __half h = __float2half_rn((float)v);
        __half l = __float2half_rn((float)(v - (double)__half2float(h)));
        hi = *reinterpret_cast<uint16_t*>(&h); lo = *reinterpret_cast<uint16_t*>(&l);
      };
      for (int row = 0; row < 256; ++row) {
        const int blk = row / Hg, u = row % Hg;
        uint16_t* r0 = wx + (size_t)row * 8;          // layer 0, accumulator order [r | z | hn | in]
        uint16_t* r1 = wx + (size_t)(256 + row) * 8;  // layer 1, accumulator order [in | r | z | hn]: biases only
        for (int k = 0; k < 8; ++k) r0[k] = r1[k] = 0;
        {
          // r, z: W_ih0 x + b_ih + b_hh;  hn: b_hh[n] only;  in: W_ih0[n] x + b_ih[n]
          const int src_row = blk == 0 ? u : blk == 1 ? Hg + u : 2 * Hg + u;
          const double sc = blk < 2 ? cR : cN;
          const double bias = blk < 2 ? d->gru_b_ih_l0[src_row] + d->gru_b_hh_l0[src_row]
                                      : (blk == 2 ? d->gru_b_hh_l0[src_row] : d->gru_b_ih_l0[src_row]);
          if (blk != 2)
            for (int v = 0; v < gin; ++v) {
              uint16_t hi, lo;
              split(sc * d->gru_w_ih_l0[(size_t)src_row * gin + v], hi, lo);
              r0[3 * v] = hi; r0[3 * v + 1] = hi; r0[3 * v + 2] = lo;
            }
          split(sc * bias, r0[6], r0[7]);
        }
        {
          const double bias = blk == 0 ? cN * d->gru_b_ih_l1[2 * Hg + u]
                            : blk == 1 ? cR * (d->gru_b_ih_l1[u] + d->gru_b_hh_l1[u])
                            : blk == 2 ? cR * (d->gru_b_ih_l1[Hg + u] + d->gru_b_hh_l1[Hg + u])
                                       : cN * d->gru_b_hh_l1[2 * Hg + u];
          split(bias, r1[6], r1[7]);
        }
      }
    }
    for (int i = 0; i < 2 * Hg; ++i) put(o_enc2c, nlc::kE2Wout + i, d->enc_out_w[i]);
    for (int i = 0; i < 2; ++i) put(o_enc2c, nlc::kE2Bout + i, d->enc_out_b[i]);
  }

  if (N3t <= 416 && Hm == 128) {  // rollout_tc2.cu operands: -2 log2(e) folded
    const double cN = -2.0 * 1.4426950408889634;
    std::vector<double> w2s((size_t)Hm * Hm);
    for (size_t i = 0; i < w2s.size(); ++i) w2s[i] = cN * d->mlp_w2[i];
    uint16_t* w2i = reinterpret_cast<uint16_t*>(A.data.data() + o_m2w2);
    nlc::tc_pack_weight_split(w2s.data(), Hm, Hm, w2i, w2i + (size_t)Hm * Hm);
    std::vector<double> w3p((size_t)N3t * Hm, 0.0);
    for (int c = 0; c < nx; ++c)
      for (int k = 0; k < S; ++k)
        for (int part = 0; part < 2; ++part) {
          const int src = (part * nx + c) * S + k, dst = 2 * (c * S + k) + part;
          for (int h = 0; h < Hm; ++h) w3p[(size_t)dst * Hm + h] = cN * d->mlp_w4[(size_t)src * Hm + h];
          put(o_m2c, 128 + dst, cN * d->mlp_b4[src]);
        }
    uint16_t* w3i = reinterpret_cast<uint16_t*>(A.data.data() + o_m2w3);
    nlc::tc_pack_weight_split(w3p.data(), N3t, Hm, w3i, w3i + (size_t)N3t * Hm);
    if (N3u) {  // the same rows in the group-uniform order (see ModelDev::mlp2_w3u)
      std::vector<double> w3u((size_t)N3u * Hm, 0.0);
      const int kJ = nx * gu_upc;
      for (int col = 0; col < N3u; ++col) {
        const int j = col / 32, cgp = (col % 32) / 8, i = (col % 8) / 2, part = col % 2;
        int c, k;
        if (j < kJ) { c = j / gu_upc; k = 16 * (j % gu_upc) + cgp + 4 * i; }
        else { c = cgp + 4 * i; k = S - 1; }
        if (c >= nx) continue;  // no such channel: zero weights and bias (its Fourier weight is zeroed in the kernel too)
        const int src = (part * nx + c) * S + k;
        for (int h = 0; h < Hm; ++h) w3u[(size_t)col * Hm + h] = cN * d->mlp_w4[(size_t)src * Hm + h];
        put(o_m2cu, col, cN * d->mlp_b4[src]);
      }
      uint16_t* w3ui = reinterpret_cast<uint16_t*>(A.data.data() + o_m2w3u);
      nlc::tc_pack_weight_split(w3u.data(), N3u, Hm, w3ui, w3ui + (size_t)N3u * Hm);
    }
    for (int n = 0; n < Hm; ++n) put(o_m2c, n, cN * d->mlp_b2[n]);
  }

  m->h.w0 = new double[(size_t)Hm * in0];
  m->h.b0 = new double[Hm];
  memcpy(m->h.w0, d->mlp_w0, sizeof(double) * Hm * in0);
  memcpy(m->h.b0, d->mlp_b0, sizeof(double) * Hm);

  auto fail = [&](int code) {
    if (m->arena) cudaFree(m->arena);
    delete[] m->h.w0; delete[] m->h.b0; delete m;
    return code;
  };
  if (cudaSetDevice(device) != cudaSuccess) { set_error("cudaSetDevice(%d) failed", device); return fail(NLC_ERR_CUDA); }
  m->arena_bytes = A.data.size() * sizeof(float);
  if (cudaMalloc(&m->arena, m->arena_bytes) != cudaSuccess) { set_error("cudaMalloc(%zu) failed", m->arena_bytes); cudaGetLastError(); m->arena = nullptr; return fail(NLC_ERR_NOMEM); }
  if (cudaMemcpy(m->arena, A.data.data(), m->arena_bytes, cudaMemcpyHostToDevice) != cudaSuccess) { set_error("weight upload failed"); return fail(NLC_ERR_CUDA); }
  float* base = static_cast<float*>(m->arena);
  m->d.w_ih0 = base + o_w_ih0; m->d.b_ih0 = base + o_b_ih0; m->d.b_hh0 = base + o_b_hh0;
  m->d.w_hh0_t = base + o_hh0; m->d.w_ih1_t = base + o_ih1; m->d.w_hh1_t = base + o_hh1;
  m->d.b_ih1 = base + o_b_ih1; m->d.b_hh1 = base + o_b_hh1; m->d.w_out = base + o_wout; m->d.b_out = base + o_bout;
  m->d.enc2_w = base + o_enc2w; m->d.enc2_c = base + o_enc2c; m->d.enc2_x = base + o_enc2x;
  m->d.mlp2_w1 = base + o_m2w1; m->d.mlp2_w2 = base + o_m2w2; m->d.mlp2_w3 = base + o_m2w3; m->d.mlp2_c = base + o_m2c;
  m->d.mlp2_w3u = base + o_m2w3u; m->d.mlp2_cu = base + o_m2cu;
  m->d.w1_full_t = base + o_w1full; m->d.b1_raw = base + o_b1raw; m->d.w1x_t = base + o_w1x; m->d.b1_fold = base + o_b1f;
  m->d.w2_t = base + o_w2; m->d.b2 = base + o_b2; m->d.w3_t = base + o_w3; m->d.b3 = base + o_b3;
  m->d.ilt_phase = base + o_phase; m->d.ilt_weight = base + o_weight;
  m->d.state_mean = base + o_smean; m->d.state_inv_std = base + o_sinv; m->d.act_mean = base + o_amean; m->d.act_inv_std = base + o_ainv;
  m->d.state_mean64 = reinterpret_cast<double*>(base + o_smean64); m->d.state_inv_std64 = reinterpret_cast<double*>(base + o_sinv64);
  m->d.act_mean64 = reinterpret_cast<double*>(base + o_amean64); m->d.act_inv_std64 = reinterpret_cast<double*>(base + o_ainv64);
  rc = fold_prediction_time(m, d->dt);
  if (rc != NLC_OK) return fail(rc);
  *out = m;
  return NLC_OK;
}

extern "C" int nlc_model_destroy(nlc_model_t m) {
  if (!m) return NLC_OK;
  if (m->refs > 0) {  // a planner still rolls out on this model: the last nlc_planner_destroy frees it
    m->destroy_requested = true;
    return NLC_OK;
  }
  cudaSetDevice(m->device);
  if (m->arena) cudaFree(m->arena);
  delete[] m->h.w0;
  delete[] m->h.b0;
  delete m;
  return NLC_OK;
}
