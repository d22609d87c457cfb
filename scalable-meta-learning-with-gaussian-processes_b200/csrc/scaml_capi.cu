// extern "C" entry points of libscaml_b200.so (see include/scaml_b200.h).
// No torch types, no allocation: raw device pointers + sizes + stream.
//
// The file is compiled once per PART (-DSCAML_PART=0..3, build.py runs the four nvcc jobs in parallel and links the
// objects) or, with SCAML_PART undefined, as one translation unit (the -DSCAML_EMU test build):
//   part 0  fit kernel (4-warp), limits / version / workspace queries
//   part 1  fit kernel (8-warp)
//   part 2  kernel matrix, prediction, conditioning, values-from-U
//   part 3  cross blocks, target GP, L-BFGS update, candidate gradients, q-point blocks
#ifndef SCAML_PART
#define SCAML_PART (-1)
#endif
#define SCAML_HAS(k) (SCAML_PART == -1 || SCAML_PART == (k))

#if SCAML_HAS(0) || SCAML_HAS(1)
#include "scaml_fit.cuh"
#include "scaml_fit8.cuh"
#endif
#if SCAML_HAS(2)
#include "scaml_kmat.cuh"
#include "scaml_predict.cuh"
#include "scaml_cond.cuh"
#include "scaml_gradval.cuh"
#endif
#if SCAML_HAS(3)
#include "scaml_cross.cuh"
#include "scaml_target.cuh"
#include "scaml_lbfgs.cuh"
#include "scaml_grad.cuh"
#include "scaml_qblock.cuh"
#endif
#include "scaml_device.cuh"

#ifndef SCAML_EMU
#include <cuda_runtime.h>
#endif
#include <cmath>
#include <cstdlib>

namespace {

constexpr size_t kMaxSmem = 227 * 1024;

int g_num_sms[64] = {0};      // SM count of the CURRENT device, cached per device ordinal
long long* g_prof = nullptr;  // SCAML_PROF builds: per-CTA phase cycle counters
int num_sms() {
#ifdef SCAML_EMU
  return 2;
#else
  int dev = 0;
  cudaGetDevice(&dev);
  int& slot = g_num_sms[(dev >= 0 && dev < 64) ? dev : 0];
  if (slot == 0) {
    int n = 0;
    cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev);
    slot = n > 0 ? n : 148;
  }
  return slot;
#endif
}

inline int pad64(int n) { return ((n + 63) / 64) * 64; }

#if SCAML_HAS(0)
// persistent grid of the fit kernels: CTAs per SM allowed by shared memory (<= 3)
int fit_ctas_per_sm(int n_pad, int d) {
  const size_t s = scaml::fit_smem_bytes(n_pad, d) + 1024;
#ifdef SCAML_FIT_PROBE4
  if (4 * s <= 228 * 1024) return 4;
#endif
  if (3 * s <= 228 * 1024) return 3;
  return (2 * s <= 228 * 1024) ? 2 : 1;
}
int fit_grid_slots(int n_pad, int d) {
  int c = fit_ctas_per_sm(n_pad, d);
  if (const char* env = getenv("SCAML_FIT_CTAS_PER_SM")) {  // experiment knob: fewer co-resident CTAs
    const int v = atoi(env);
    if (v >= 1 && v < c) c = v;
  }
  return num_sms() * c;
}

#endif
#if SCAML_HAS(1)
}  // namespace
__attribute__((visibility("hidden"))) int scaml_detail_dispatch_fit8(const scaml::FitParams& p, int grid, size_t smem,
                                                                   void* stream) {
  return scaml::dispatch_kind(p.spec.kernel, [&](auto K) {
    return scaml::launch(scaml::f8::scaml_fit8_kernel<K.value>, grid, scaml::f8::kThreads, smem, stream, p);
  });
}
namespace {

#endif
#if SCAML_HAS(0)
// Two variants of the fit kernel (same algorithm, same results): 4-warp CTAs, three per SM (scaml_fit.cuh), and
// 8-warp CTAs, two per SM (scaml_fit8.cuh).  Measured on B200 (profiles/r1_fit_variants.txt): the 4-warp
// kernel wins up to n = 320 (RBF 722k vs 652k evals/s, Matern-5/2 626k vs 604k at n = 256), the 8-warp kernel
// for larger tasks (118k vs 110k at n = 512, d = 10).  Round 2: with the lower-triangle skipping as a template
// parameter and the split of the diagonal super-tiles' full tile (scaml_fit.cuh) the 4-warp kernel also wins at
// n = 512 (126.9k vs 121.9k evals/s for 2048 x R2 x 512 x 10; a tie at n = 384; 484k vs 424k at n = 320), so the
// 8-warp kernel is left for tasks beyond 512 points.  SCAML_FIT_IMPL=4|8 forces one (A/B runs).
}  // namespace
__attribute__((visibility("hidden"))) int scaml_detail_dispatch_fit8(const scaml::FitParams& p, int grid, size_t smem,
                                                                   void* stream);
namespace {
bool fit8_by_default(int n_pad) { return n_pad > 512; }
bool use_fit8(int n_pad, int kernel) {
  if (const char* env = getenv("SCAML_FIT_IMPL")) {
    const int v = atoi(env);
    if (v == 4) return false;
    if (v == 8) return true;
  }
  (void)kernel;
  return fit8_by_default(n_pad);
}
// shared memory of the fit kernel the default dispatch picks at n_pad
size_t fit_default_smem_bytes(int n_pad, int d) {
  return fit8_by_default(n_pad) ? scaml::f8::smem_bytes(n_pad, d) : scaml::fit_smem_bytes(n_pad, d);
}

int dispatch_fit(const scaml::FitParams& p, int grid, size_t smem, void* stream) {
  return scaml::dispatch_kind(p.spec.kernel, [&](auto K) {
    return scaml::launch(scaml::scaml_fit_kernel<K.value>, grid, scaml::kFitThreads, smem, stream, p);
  });
}

size_t fit_tile_workspace_bytes(int n_max, int d) {
  const int n_pad = pad64(n_max);
  return (size_t)fit_grid_slots(n_pad, d) * (size_t)scaml::fit_ws_doubles_host(n_pad, d) * sizeof(double);
}

int run_fit(scaml::FitParams p, void* workspace, size_t workspace_bytes, void* stream) {
  if (p.M <= 0 || p.R <= 0 || p.n_max <= 0 || p.d <= 0) return SCAML_E_ARG;
  if (p.d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  p.n_pad = pad64(p.n_max);
  const bool f8 = use_fit8(p.n_pad, p.spec.kernel);
  const size_t smem = f8 ? scaml::f8::smem_bytes(p.n_pad, p.d) : scaml::fit_smem_bytes(p.n_pad, p.d);
  if (smem > kMaxSmem) return SCAML_E_SMEM;
  if (workspace_bytes < scaml_fit_workspace_bytes(p.M, p.R, p.n_max, p.d)) return SCAML_E_WORKSPACE;
  p.workspace = static_cast<double*>(workspace);
  p.ws_stride = scaml::fit_ws_doubles_host(p.n_pad, p.d);
  p.prof = g_prof;
  p.sms = num_sms();
  p.kcache = 1;
  if (const char* env = getenv("SCAML_FIT_KCACHE")) p.kcache = atoi(env) != 0;
  // scheduling block behind the tile workspace: [counter, #items, order[M R]]
  const long long E64 = (long long)p.M * p.R;
  if (E64 > (1LL << 30)) return SCAML_E_UNSUPPORTED;
  p.sched = reinterpret_cast<int32_t*>(static_cast<char*>(workspace) + fit_tile_workspace_bytes(p.n_max, p.d));
  p.order = nullptr;
  if (p.skip != nullptr || p.n_valid != nullptr) {  // active rows, largest tasks first
    int32_t* order = p.sched + 2;
    if (scaml::launch(scaml::scaml_fit_schedule_kernel<0>, 1, scaml::kSchedThreads, 0, stream, p.skip, p.n_valid, p.M,
                      p.R, p.n_max, p.sched, order) != 0)
      return SCAML_E_ARG;
    p.order = order;
  } else {
#ifdef SCAML_EMU
    p.sched[0] = 0;
#else
    if (cudaMemsetAsync(p.sched, 0, 2 * sizeof(int32_t), (cudaStream_t)stream) != cudaSuccess) return SCAML_E_ARG;
#endif
  }
  int grid = fit_grid_slots(p.n_pad, p.d);
  if (f8) {  // register-limited to two 256-thread CTAs per SM
    const int per_sm = (2 * (smem + 1024) <= 228 * 1024) ? 2 : 1;
    if (grid > per_sm * p.sms) grid = per_sm * p.sms;
  }
  const long long E = (long long)p.M * p.R;
  if (E < grid) grid = (int)E;
  return f8 ? scaml_detail_dispatch_fit8(p, grid, smem, stream) : dispatch_fit(p, grid, smem, stream);
}

#endif
}  // namespace

extern "C" {

#if SCAML_HAS(0)
#ifdef SCAML_EMU
// tests only: the device exponential evaluated on the host (same source, same FMA semantics)
void scaml_debug_exp_nonpos(const double* x, double* out, int n) {
  for (int i = 0; i < n; ++i) out[i] = scaml::exp_nonpos(x[i]);
}
// tests only: the kernels launched since the last clear, one demangled name per line; returns the length of the
// whole text (written up to cap - 1 characters and NUL-terminated when cap > 0)
size_t scaml_debug_launch_log(char* buf, size_t cap) {
  std::string all;
  for (const std::string& s : cuemu::launch_log()) all += s + "\n";
  if (buf != nullptr && cap > 0) {
    const size_t k = all.size() < cap - 1 ? all.size() : cap - 1;
    std::memcpy(buf, all.data(), k);
    buf[k] = '\0';
  }
  return all.size();
}
void scaml_debug_launch_log_clear(void) { cuemu::launch_log().clear(); }
#endif
#ifdef SCAML_ABLATE
void scaml_debug_set_ablate(int bits) { cudaMemcpyToSymbol(scaml::g_ablate, &bits, sizeof(int)); }
#endif
#ifdef SCAML_PROF
// diagnostics build only: device buffer of [grid][16] long long phase counters
void scaml_debug_set_prof(void* buf) { g_prof = static_cast<long long*>(buf); }
#endif

const char* scaml_version(void) {
#ifdef SCAML_EMU
  return "scaml_b200 0.1.0 cpu-logic-emulation (tests only)";
#else
  return "scaml_b200 0.1.0 sm_100a";
#endif
}

int scaml_fit_limits(int* n_max_limit, int* d_limit) {
  if (d_limit) *d_limit = scaml::kMaxP - 2;
  if (n_max_limit) {
    // the 8-warp kernel (n_pad > 512) stages 3 n_pad doubles, the 4-warp one 2 n_pad: the limit is the 8-warp one's
    int n = 64;
    while (fit_default_smem_bytes(n + 64, 6) <= kMaxSmem) n += 64;
    *n_max_limit = n;
  }
  return 0;
}

size_t scaml_fit_workspace_bytes(int M, int R, int n_max, int d) {
  if (M <= 0 || R <= 0 || n_max <= 0 || d <= 0) return 0;
  // per-CTA tile workspaces + the scheduling block [counter, #items, order[M R]] (int32), rounded up to 16 bytes
  const size_t sched = ((2 + (size_t)M * R) * sizeof(int32_t) + 15) / 16 * 16;
  return fit_tile_workspace_bytes(n_max, d) + sched;
}

int scaml_lml_grad(const double* X, const double* y, const int32_t* n_valid, const double* theta_raw,
                   const double* jitter, const int32_t* skip, double* lml, double* grad, int32_t* info,
                   void* workspace, size_t workspace_bytes, int M, int R, int n_max, int d,
                   const scaml_hyper_spec* spec, void* stream) {
  if (!X || !y || !theta_raw || !lml || !grad || !info || !workspace || !spec) return SCAML_E_ARG;
  scaml::FitParams p{};
  p.X = X, p.y = y, p.n_valid = n_valid, p.theta_raw = theta_raw, p.jitter = jitter, p.skip = skip;
  p.lml = lml, p.grad = grad, p.info = info;
  p.M = M, p.R = R, p.n_max = n_max, p.d = d, p.mode = scaml::kModeLmlGrad;
  p.spec = *spec;
  return run_fit(p, workspace, workspace_bytes, stream);
}

int scaml_lml_grad_ladder(const double* X, const double* y, const int32_t* n_valid, const double* theta_raw,
                          const int32_t* skip, double* lml, double* grad, int32_t* info, void* workspace,
                          size_t workspace_bytes, int M, int R, int n_max, int d, const scaml_hyper_spec* spec,
                          void* stream) {
  if (!X || !y || !theta_raw || !lml || !grad || !info || !workspace || !spec) return SCAML_E_ARG;
  scaml::FitParams p{};
  p.X = X, p.y = y, p.n_valid = n_valid, p.theta_raw = theta_raw, p.jitter = nullptr, p.skip = skip;
  p.lml = lml, p.grad = grad, p.info = info;
  p.M = M, p.R = R, p.n_max = n_max, p.d = d, p.mode = scaml::kModeLmlGrad, p.ladder = 1;
  p.spec = *spec;
  return run_fit(p, workspace, workspace_bytes, stream);
}

int scaml_factorize_ladder(const double* X, const double* y, const int32_t* n_valid, const double* theta_raw,
                           double* linv_packed, double* alpha, double* theta, int32_t* info, void* workspace,
                           size_t workspace_bytes, int M, int n_max, int d, const scaml_hyper_spec* spec,
                           void* stream) {
  if (!X || !y || !theta_raw || !linv_packed || !alpha || !theta || !info || !workspace || !spec) return SCAML_E_ARG;
  scaml::FitParams p{};
  p.X = X, p.y = y, p.n_valid = n_valid, p.theta_raw = theta_raw, p.jitter = nullptr, p.skip = nullptr;
  p.info = info, p.linv_out = linv_packed, p.alpha_out = alpha, p.theta_out = theta;
  p.M = M, p.R = 1, p.n_max = n_max, p.d = d, p.mode = scaml::kModeFactorize, p.ladder = 1;
  p.spec = *spec;
  return run_fit(p, workspace, workspace_bytes, stream);
}

int scaml_factorize(const double* X, const double* y, const int32_t* n_valid, const double* theta_raw,
                    const double* jitter, double* linv_packed, double* alpha, double* theta, int32_t* info,
                    void* workspace, size_t workspace_bytes, int M, int n_max, int d, const scaml_hyper_spec* spec,
                    void* stream) {
  if (!X || !y || !theta_raw || !linv_packed || !alpha || !theta || !info || !workspace || !spec) return SCAML_E_ARG;
  scaml::FitParams p{};
  p.X = X, p.y = y, p.n_valid = n_valid, p.theta_raw = theta_raw, p.jitter = jitter, p.skip = nullptr;
  p.info = info, p.linv_out = linv_packed, p.alpha_out = alpha, p.theta_out = theta;
  p.M = M, p.R = 1, p.n_max = n_max, p.d = d, p.mode = scaml::kModeFactorize;
  p.spec = *spec;
  return run_fit(p, workspace, workspace_bytes, stream);
}

#endif
#if SCAML_HAS(2)
int scaml_kernel_matrix(const double* X, const int32_t* n_valid, const double* theta, double* K, int M, int n_max,
                        int d, int kernel, void* stream) {
  if (!X || !theta || !K || M <= 0 || n_max <= 0 || d <= 0) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  if (kernel < 0 || kernel > 3) return SCAML_E_ARG;
  return scaml::launch_kmat(X, n_valid, theta, K, M, n_max, d, kernel, stream);
}

int scaml_predict_max_points(int d) {
  if (d <= 0 || d > scaml::kMaxP - 2) return 0;
  int n = 0, ct = 0, alias = 0;
  while (scaml::predict_config(n + 64, d, &ct, &alias)) n += 64;
  return n;
}

size_t scaml_predict_workspace_bytes(int M, int n_max, int d, int B) {
  return scaml::predict_workspace_bytes(M, pad64(n_max), d, B, num_sms());
}

int scaml_predict_weighted(const double* X, const int32_t* n_valid, const double* theta, const double* linv_packed,
                           const double* alpha, const double* ybar, const double* ystd, const double* w,
                           const double* Xc, double* mean, double* var, void* workspace, size_t workspace_bytes,
                           int M, int n_max, int d, int B, int kernel, void* stream) {
  if (!X || !theta || !linv_packed || !alpha || !ybar || !ystd || !w || !Xc || !mean || !var) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_predict_workspace_bytes(M, n_max, d, B) || (!workspace && workspace_bytes))
    return SCAML_E_WORKSPACE;
  return scaml::launch_predict_weighted(X, n_valid, theta, linv_packed, alpha, ybar, ystd, w, Xc, mean, var,
                                        static_cast<double*>(workspace), M, n_max, pad64(n_max), d, B, kernel,
                                        num_sms(), stream);
}

#endif
#if SCAML_HAS(3)
int scaml_predict_cross_max_points(int d) {
  if (d <= 0 || d > scaml::kMaxP - 2) return 0;
  int n = 0;
  while (scaml::cross_smem_bytes(n + 64, d) <= (size_t)227 * 1024) n += 64;
  return n;
}

size_t scaml_predict_cross_workspace_bytes(int M, int nA, int nB, int reduce) {
  return scaml::cross_workspace_bytes(M, nA, nB, reduce, num_sms());
}

int scaml_predict_cross(const double* X, const int32_t* n_valid, const double* theta, const double* linv_packed,
                        const double* alpha, const double* ybar, const double* ystd, const double* w, const double* XA,
                        const double* XB, double* mean, double* cov, void* workspace, size_t workspace_bytes, int M,
                        int n_max, int d, int nA, int nB, int kernel, int reduce, void* stream) {
  if (!X || !theta || !linv_packed || !alpha || !ybar || !ystd || !XA || !XB || !mean || !cov) return SCAML_E_ARG;
  if (reduce && !w) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || nA <= 0 || nB <= 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  const size_t need = scaml_predict_cross_workspace_bytes(M, nA, nB, reduce);
  if (workspace_bytes < need || (need && !workspace)) return SCAML_E_WORKSPACE;
  return scaml::launch_predict_cross(X, n_valid, theta, linv_packed, alpha, ybar, ystd, w, XA, XB, mean, cov,
                                     static_cast<double*>(workspace), M, n_max, pad64(n_max), d, nA, nB, kernel,
                                     reduce, num_sms(), stream);
}

size_t scaml_target_workspace_bytes(int n_t, int R) {
  if (n_t <= 0 || R <= 0) return 0;
  return scaml::target_workspace_doubles(n_t, R) * sizeof(double);
}

int scaml_target_max_points(int d) {
  if (d <= 0 || d > scaml::kMaxP - 2) return 0;
  int nt = 0;
  while (scaml::target_smem_bytes(nt + 1, d) <= (size_t)227 * 1024) ++nt;
  return nt;
}

int scaml_target_lml_grad(const double* source_means, const double* source_covs, const double* Xt, const double* yt,
                          const double* w, const double* theta_raw, const double* jitter, double mu_all, double s_all,
                          double* lml, double* grad_w, double* grad_theta, int32_t* info, void* workspace,
                          size_t workspace_bytes, int M, int n_t, int d, int R, const scaml_hyper_spec* spec,
                          int w_prior, double w_p1, double w_p2, void* stream) {
  if (!source_means || !source_covs || !Xt || !yt || !w || !theta_raw || !lml || !grad_w || !grad_theta || !info ||
      !workspace || !spec)
    return SCAML_E_ARG;
  if (M <= 0 || n_t <= 0 || d <= 0 || R <= 0 || !(s_all > 0.0)) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_target_workspace_bytes(n_t, R)) return SCAML_E_WORKSPACE;
  scaml::TargetParams p{};
  p.smeans = source_means, p.scovs = source_covs, p.Xt = Xt, p.yt = yt, p.w = w, p.theta_raw = theta_raw;
  p.jitter = jitter, p.lml = lml, p.grad_w = grad_w, p.grad_theta = grad_theta, p.info = info;
  double* ws = static_cast<double*>(workspace);
  p.covw = ws;
  p.Wmat = ws + (size_t)R * n_t * n_t;
  p.meanw = ws + 2 * (size_t)R * n_t * n_t;
  p.alpha = p.meanw + (size_t)R * n_t;
  p.big = (n_t >= scaml::kTgtBigFrom) ? ws + scaml::target_small_doubles(n_t, R) : nullptr;
  p.mu_all = mu_all, p.s_all = s_all;
  p.M = M, p.nt = n_t, p.d = d, p.R = R, p.w_prior = w_prior, p.w_p1 = w_p1, p.w_p2 = w_p2;
  p.spec = *spec;
  return scaml::launch_target(p, num_sms(), stream);
}

int scaml_target_lml_grad_ladder(const double* source_means, const double* source_covs, const double* Xt,
                                 const double* yt, const double* w, const double* theta_raw, double mu_all,
                                 double s_all, double* lml, double* grad_w, double* grad_theta, int32_t* info,
                                 void* workspace, size_t workspace_bytes, int M, int n_t, int d, int R,
                                 const scaml_hyper_spec* spec, int w_prior, double w_p1, double w_p2, void* stream) {
  if (!source_means || !source_covs || !Xt || !yt || !w || !theta_raw || !lml || !grad_w || !grad_theta || !info ||
      !workspace || !spec)
    return SCAML_E_ARG;
  if (M <= 0 || n_t <= 0 || d <= 0 || R <= 0 || !(s_all > 0.0)) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_target_workspace_bytes(n_t, R)) return SCAML_E_WORKSPACE;
  scaml::TargetParams p{};
  p.smeans = source_means, p.scovs = source_covs, p.Xt = Xt, p.yt = yt, p.w = w, p.theta_raw = theta_raw;
  p.jitter = nullptr, p.jitter_value = 0.0, p.ladder = 1;
  p.lml = lml, p.grad_w = grad_w, p.grad_theta = grad_theta, p.info = info;
  double* ws = static_cast<double*>(workspace);
  p.covw = ws;
  p.Wmat = ws + (size_t)R * n_t * n_t;
  p.meanw = ws + 2 * (size_t)R * n_t * n_t;
  p.alpha = p.meanw + (size_t)R * n_t;
  p.big = (n_t >= scaml::kTgtBigFrom) ? ws + scaml::target_small_doubles(n_t, R) : nullptr;
  p.mu_all = mu_all, p.s_all = s_all;
  p.M = M, p.nt = n_t, p.d = d, p.R = R, p.w_prior = w_prior, p.w_p1 = w_p1, p.w_p2 = w_p2;
  p.spec = *spec;
  return scaml::launch_target(p, num_sms(), stream);
}

int scaml_target_factorize(const double* source_means, const double* source_covs, const double* Xt, const double* yt,
                           const double* w, const double* theta_raw, double jitter_value, double mu_all, double s_all,
                           double* linv_t, double* alpha_t, double* theta, double* lml, int32_t* info, void* workspace,
                           size_t workspace_bytes, int M, int n_t, int d, const scaml_hyper_spec* spec, void* stream) {
  if (!source_means || !source_covs || !Xt || !yt || !w || !theta_raw || !linv_t || !alpha_t || !theta || !lml ||
      !info || !workspace || !spec)
    return SCAML_E_ARG;
  if (M <= 0 || n_t <= 0 || d <= 0 || !(s_all > 0.0)) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_target_workspace_bytes(n_t, 1) + sizeof(double) * (size_t)(d + 2 + 1))
    return SCAML_E_WORKSPACE;
  scaml::TargetParams p{};
  p.smeans = source_means, p.scovs = source_covs, p.Xt = Xt, p.yt = yt, p.w = w, p.theta_raw = theta_raw;
  double* ws = static_cast<double*>(workspace);
  p.covw = ws;
  p.Wmat = ws + (size_t)n_t * n_t;
  p.meanw = ws + 2 * (size_t)n_t * n_t;
  p.alpha = alpha_t;
  p.grad_theta = p.meanw + n_t + n_t;  // scratch: the gradient is not part of this call's contract
  p.big = (n_t >= scaml::kTgtBigFrom) ? ws + scaml::target_small_doubles(n_t, 1) + (d + 3) : nullptr;
  p.jitter = nullptr;
  p.lml = lml, p.grad_w = nullptr, p.info = info;
  p.linv_out = linv_t, p.theta_out = theta;
  p.mu_all = mu_all, p.s_all = s_all;
  p.M = M, p.nt = n_t, p.d = d, p.R = 1, p.w_prior = 0, p.w_p1 = 0, p.w_p2 = 0;
  p.spec = *spec;
  p.jitter_value = jitter_value;
  return scaml::launch_target(p, num_sms(), stream);
}

int scaml_target_posterior(const double* prior_mean, const double* prior_var, const double* cross, const double* Xc,
                           const double* Xt, const double* theta, const double* linv_t, const double* alpha_t,
                           double mu_all, double s_all, double* mean, double* var, int B, int n_t, int d, int kernel,
                           void* stream) {
  if (!prior_mean || !prior_var || !cross || !Xc || !Xt || !theta || !linv_t || !alpha_t || !mean || !var)
    return SCAML_E_ARG;
  if (B <= 0 || n_t <= 0 || d <= 0 || kernel < 0 || kernel > 3 || !(s_all > 0.0)) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2) return SCAML_E_UNSUPPORTED;
  scaml::TargetPostParams p{};
  p.pm = prior_mean, p.pv = prior_var, p.cross = cross, p.Xc = Xc, p.Xt = Xt, p.theta = theta, p.linv = linv_t;
  p.alpha = alpha_t, p.mean = mean, p.var = var, p.mu_all = mu_all, p.s_all = s_all;
  p.B = B, p.nt = n_t, p.d = d, p.kernel = kernel;
  return scaml::launch_target_posterior(p, num_sms(), stream);
}

int scaml_target_posterior_beta(const double* prior_mean, const double* prior_var, const double* cross,
                                const double* Xc, const double* Xt, const double* theta, const double* linv_t,
                                const double* alpha_t, double mu_all, double s_all, double* mean, double* var,
                                double* beta, int B, int n_t, int d, int kernel, void* stream) {
  if (!prior_mean || !prior_var || !cross || !Xc || !Xt || !theta || !linv_t || !alpha_t || !mean || !var || !beta)
    return SCAML_E_ARG;
  if (B <= 0 || n_t <= 0 || d <= 0 || kernel < 0 || kernel > 3 || !(s_all > 0.0)) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128) return SCAML_E_UNSUPPORTED;
  scaml::TargetPostParams p{};
  p.pm = prior_mean, p.pv = prior_var, p.cross = cross, p.Xc = Xc, p.Xt = Xt, p.theta = theta, p.linv = linv_t;
  p.alpha = alpha_t, p.mean = mean, p.var = var, p.beta = beta, p.mu_all = mu_all, p.s_all = s_all;
  p.B = B, p.nt = n_t, p.d = d, p.kernel = kernel, p.n_tp = scaml::cond_ntp(n_t);
  return scaml::launch_target_posterior(p, num_sms(), stream);
}

size_t scaml_posterior_grad_workspace_bytes(int M, int n_max, int d, int B) {
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0) return 0;
  const int ntile = (B + scaml::kGradCT - 1) / scaml::kGradCT;
  return sizeof(double) * ((size_t)scaml::grad_nsplit(M, ntile, num_sms()) * (size_t)B * 2 * (size_t)d +
                           (size_t)M * (size_t)pad64(n_max));
}

int scaml_posterior_grad(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                         const double* ystd, const double* w, const double* Xc, double* U, const double* Xt,
                         const double* A, const double* alpha_t, const double* beta, const double* theta_t,
                         double s_all, double* dmean, double* dvar, void* workspace, size_t workspace_bytes, int M,
                         int n_max, int d, int B, int n_t, int kernel, int kernel_t, void* stream) {
  if (!X || !theta || !alpha || !ystd || !w || !Xc || !U || !dmean || !dvar || !workspace) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || n_t < 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (n_t > 0 && (!Xt || !A || !alpha_t || !beta || !theta_t || !(s_all > 0.0) || kernel_t < -1 || kernel_t > 3))
    return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128 || B > 128) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_posterior_grad_workspace_bytes(M, n_max, d, B)) return SCAML_E_WORKSPACE;
  scaml::GradParams p{};
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.alpha = alpha, p.ystd = ystd, p.w = w, p.Xc = Xc, p.U = U;
  p.Xt = Xt, p.A = A, p.alpha_t = alpha_t, p.beta = beta, p.theta_t = theta_t;
  p.dmean = dmean, p.dvar = dvar;
  p.s_all = n_t > 0 ? s_all : 1.0;
  p.M = M, p.n_max = n_max, p.n_pad = pad64(n_max), p.d = d, p.B = B, p.B_p = scaml::cond_ntp(B);
  p.n_t = n_t, p.n_tp = n_t > 0 ? scaml::cond_ntp(n_t) : 0;
  p.ntile = (B + scaml::kGradCT - 1) / scaml::kGradCT;
  p.nsplit = scaml::grad_nsplit(M, p.ntile, num_sms());
  p.part = static_cast<double*>(workspace);
  p.aal = p.part + (size_t)p.nsplit * (size_t)B * 2 * (size_t)d;
  p.kernel_t = kernel_t;
  return scaml::launch_posterior_grad(p, kernel, num_sms(), stream);
}

size_t scaml_qblock_cov_workspace_bytes(int M, int B, int q) {
  if (M <= 0 || B <= 0 || q <= 0) return 0;
  const int ntile = (B + 31) / 32;
  return sizeof(double) * (size_t)scaml::grad_nsplit(M, ntile, num_sms()) * (size_t)B * (size_t)q;
}

int scaml_qblock_cov(const double* X, const int32_t* n_valid, const double* theta, const double* ystd, const double* w,
                     const double* Xc, const double* U, double* cov, void* workspace, size_t workspace_bytes, int M,
                     int n_max, int d, int B, int q, int kernel, void* stream) {
  if (!X || !theta || !ystd || !w || !Xc || !U || !cov || !workspace) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || q <= 0 || B % q != 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || B > 128 || q > scaml::kQMax) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_qblock_cov_workspace_bytes(M, B, q)) return SCAML_E_WORKSPACE;
  scaml::QBlockCovParams p{};
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.ystd = ystd, p.w = w, p.Xc = Xc, p.U = U, p.cov = cov;
  p.M = M, p.n_max = n_max, p.n_pad = pad64(n_max), p.d = d, p.B = B, p.B_p = scaml::cond_ntp(B), p.q = q;
  p.ntile = (B + 31) / 32;
  p.nsplit = scaml::grad_nsplit(M, p.ntile, num_sms());
  p.part = static_cast<double*>(workspace);
  return scaml::launch_qblock_cov(p, kernel, num_sms(), stream);
}

size_t scaml_qblock_vjp_workspace_bytes(int M, int n_max, int d, int B, int n_t) {
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || n_t < 0) return 0;
  return scaml_posterior_grad_workspace_bytes(M, n_max, d, B) +
         sizeof(double) * ((size_t)2 * B * d + (size_t)B * scaml::cond_ntp(n_t));
}

int scaml_qblock_vjp(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                     const double* ystd, const double* w, const double* Xc, double* U, const double* Xt, const double* A,
                     const double* alpha_t, const double* beta, const double* theta_t, double s_all,
                     const double* g_mean, const double* g_cov, double* dX, void* workspace, size_t workspace_bytes,
                     int M, int n_max, int d, int B, int q, int n_t, int kernel, int kernel_t, void* stream) {
  if (!X || !theta || !alpha || !ystd || !w || !Xc || !U || !theta_t || !g_mean || !g_cov || !dX || !workspace)
    return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || q <= 0 || B % q != 0 || n_t < 0 || kernel < 0 || kernel > 3 ||
      kernel_t < 0 || kernel_t > 3)
    return SCAML_E_ARG;
  if (n_t > 0 && (!Xt || !A || !alpha_t || !beta || !(s_all > 0.0))) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128 || B > 128 || q > scaml::kQMax) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_qblock_vjp_workspace_bytes(M, n_max, d, B, n_t)) return SCAML_E_WORKSPACE;
  const int n_tp = n_t > 0 ? scaml::cond_ntp(n_t) : 0;
  double* ws = static_cast<double*>(workspace);
  double* dmean = ws + scaml_posterior_grad_workspace_bytes(M, n_max, d, B) / sizeof(double);
  double* dvar = dmean + (size_t)B * d;
  double* beta_f = dvar + (size_t)B * d;
  scaml::GradParams g{};
  g.X = X, g.n_valid = n_valid, g.theta = theta, g.alpha = alpha, g.ystd = ystd, g.w = w, g.Xc = Xc, g.U = U;
  g.Xt = Xt, g.A = A, g.alpha_t = alpha_t, g.beta = beta_f, g.theta_t = theta_t;
  g.dmean = dmean, g.dvar = dvar;
  g.s_all = n_t > 0 ? s_all : 1.0;
  g.M = M, g.n_max = n_max, g.n_pad = pad64(n_max), g.d = d, g.B = B, g.B_p = scaml::cond_ntp(B);
  g.n_t = n_t, g.n_tp = n_tp;
  g.ntile = (B + scaml::kGradCT - 1) / scaml::kGradCT;
  g.nsplit = scaml::grad_nsplit(M, g.ntile, num_sms());
  g.part = ws;
  g.aal = g.part + (size_t)g.nsplit * (size_t)B * 2 * (size_t)d;
  g.kernel_t = kernel_t;
  scaml::QBlockVjpParams p{};
  p.n_valid = n_valid, p.X = X, p.theta = theta, p.ystd = ystd, p.w = w, p.Xc = Xc, p.gcov = g_cov, p.gmean = g_mean;
  p.U = U, p.beta = beta, p.beta_f = beta_f, p.theta_t = theta_t, p.dmean = dmean, p.dvar = dvar, p.dX = dX;
  p.s2t = g.s_all * g.s_all;
  p.M = M, p.n_max = n_max, p.n_pad = g.n_pad, p.d = d, p.B = B, p.B_p = g.B_p, p.q = q, p.n_t = n_t, p.n_tp = n_tp;
  p.kernel_t = kernel_t;
  return scaml::launch_qblock_vjp(p, g, kernel, num_sms(), stream);
}

#endif
#if SCAML_HAS(2)
size_t scaml_posterior_values_from_u_workspace_bytes(int M, int B, int n_t) {
  if (M <= 0 || B <= 0 || n_t < 0) return 0;
  const int ntile = (B + scaml::kGvCT - 1) / scaml::kGvCT;
  const size_t ns = (size_t)scaml::gradval_nsplit(M, ntile, num_sms());
  return sizeof(double) * (ns * (size_t)B * ((size_t)scaml::cond_ntp(n_t) + 2) +
                           (n_t > 0 ? scaml::comb_dpart_doubles(M, B, n_t, num_sms()) : 0));
}

int scaml_posterior_values_from_u(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                                  const double* ybar, const double* ystd, const double* w, const double* Xc,
                                  const double* U, const double* Xt, const double* A, double* mean, double* var,
                                  double* cross, void* workspace, size_t workspace_bytes, int M, int n_max, int d,
                                  int B, int n_t, int kernel, void* stream) {
  if (!X || !theta || !alpha || !ybar || !ystd || !w || !Xc || !U || !mean || !var || !workspace) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || n_t < 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (n_t > 0 && (!Xt || !A || !cross)) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128 || B > 128) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_posterior_values_from_u_workspace_bytes(M, B, n_t)) return SCAML_E_WORKSPACE;
  scaml::GradValParams p{};
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.alpha = alpha, p.ybar = ybar, p.ystd = ystd, p.w = w, p.Xc = Xc;
  p.U = U, p.A = A, p.mean = mean, p.var = var;
  p.M = M, p.n_max = n_max, p.n_pad = pad64(n_max), p.d = d, p.B = B, p.B_p = scaml::cond_ntp(B);
  p.n_t = n_t, p.n_tp = n_t > 0 ? scaml::cond_ntp(n_t) : 0;
  p.ntile = (B + scaml::kGvCT - 1) / scaml::kGvCT;
  p.nsplit = scaml::gradval_nsplit(M, p.ntile, num_sms());
  p.cxp = static_cast<double*>(workspace);
  p.mvp = p.cxp + (size_t)p.nsplit * (size_t)B * (size_t)p.n_tp;
  int rc = scaml::launch_grad_values(p, kernel, num_sms(), stream);
  if (rc != 0 || n_t == 0) return rc;
  scaml::CondCombineParams c{};
  c.theta = theta, c.ystd = ystd, c.w = w, c.Xc = Xc, c.Xt = Xt, c.cxp = p.cxp, c.cross = cross;
  c.M = M, c.d = d, c.B = B, c.n_t = n_t, c.n_tp = p.n_tp, c.nsplit = p.nsplit;
  c.ntsplit = scaml::comb_ntsplit(M, B, n_t, num_sms());
  c.dpart = p.mvp + (size_t)p.nsplit * (size_t)B * 2;
  return scaml::launch_cond_combine(c, kernel, stream);
}

#endif
#if SCAML_HAS(3)
int scaml_lbfgs_step(const scaml_lbfgs_state* st, double* xt, const double* ft, const double* gt, const double* lower,
                     int E, int D, int m, int init, double gtol, double ftol, int maxiter, int max_ls, void* stream) {
  if (!st || !xt || !ft || !gt || !st->x || !st->f || !st->g || !st->d || !st->t || !st->S || !st->Y || !st->rho ||
      !st->count || !st->head || !st->iters || !st->ls_count || !st->flags)
    return SCAML_E_ARG;
  scaml::LbfgsParams p;
  p.x = st->x, p.f = st->f, p.g = st->g, p.d = st->d, p.t = st->t, p.S = st->S, p.Y = st->Y, p.rho = st->rho;
  p.count = st->count, p.head = st->head, p.iters = st->iters, p.ls_count = st->ls_count, p.flags = st->flags;
  p.xt = xt, p.ft = ft, p.gt = gt, p.lower = lower;
  p.E = E, p.D = D, p.m = m, p.init = init, p.maxiter = maxiter, p.max_ls = max_ls, p.gtol = gtol, p.ftol = ftol;
  return scaml::launch_lbfgs_step(p, stream);
}

#endif
#if SCAML_HAS(2)
int scaml_cond_prepare(const double* X, const int32_t* n_valid, const double* theta, const double* linv_packed,
                       const double* Xt, double* A, int M, int n_max, int d, int n_t, int kernel, void* stream) {
  if (!X || !theta || !linv_packed || !Xt || !A) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || n_t <= 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128) return SCAML_E_UNSUPPORTED;
  scaml::CondPrepParams p{};
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.linv = linv_packed, p.Xt = Xt, p.A = A;
  p.M = M, p.n_max = n_max, p.n_pad = pad64(n_max), p.d = d, p.n_t = n_t;
  return scaml::launch_cond_prepare(p, kernel, num_sms(), stream);
}

int scaml_cond_prepare_pruned(const double* X, const int32_t* n_valid, const double* theta, const double* linv_packed,
                              const double* Xt, const double* w, double* A, int M, int n_max, int d, int n_t,
                              int kernel, void* stream) {
  if (!X || !theta || !linv_packed || !Xt || !w || !A) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || n_t <= 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128) return SCAML_E_UNSUPPORTED;
  scaml::CondPrepParams p{};
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.linv = linv_packed, p.Xt = Xt, p.skip_w = w, p.A = A;
  p.M = M, p.n_max = n_max, p.n_pad = pad64(n_max), p.d = d, p.n_t = n_t;
  return scaml::launch_cond_prepare(p, kernel, num_sms(), stream);
}

int scaml_cond_caches(const double* X, const int32_t* n_valid, const double* theta, const double* alpha,
                      const double* ybar, const double* ystd, const double* Xt, const double* A, double* mean,
                      double* cov, int M, int n_max, int d, int n_t, int kernel, void* stream) {
  if (!X || !theta || !alpha || !ybar || !ystd || !Xt || !A || !mean || !cov) return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || n_t <= 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128) return SCAML_E_UNSUPPORTED;
  scaml::CondCachesParams p{};
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.alpha = alpha, p.ybar = ybar, p.ystd = ystd, p.Xt = Xt, p.A = A;
  p.mean = mean, p.cov = cov, p.M = M, p.n_max = n_max, p.n_pad = pad64(n_max), p.d = d, p.n_t = n_t;
  return scaml::launch_cond_caches(p, kernel, num_sms(), stream);
}

int scaml_cond_combine_task_splits(int M, int B, int n_t) {
  if (M <= 0 || B <= 0 || n_t <= 0) return 0;
  return scaml::comb_ntsplit(M, B, n_t, num_sms());
}

size_t scaml_predict_conditioned_workspace_bytes(int M, int n_max, int d, int B, int n_t) {
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || n_t <= 0) return 0;
  int ct = 64, alias = 0;
  if (!scaml::predict_config(pad64(n_max), d, &ct, &alias)) return 0;
  const int ns = scaml::predict_nsplit(M, B, num_sms(), ct);
  const size_t pv = ns > 1 ? sizeof(double) * 2 * (size_t)ns * (size_t)B : 0;
  return pv + sizeof(double) * ((size_t)ns * (size_t)B * (size_t)scaml::cond_ntp(n_t) +
                                scaml::comb_dpart_doubles(M, B, n_t, num_sms()));
}

int scaml_predict_conditioned(const double* X, const int32_t* n_valid, const double* theta, const double* linv_packed,
                              const double* alpha, const double* ybar, const double* ystd, const double* w,
                              const double* Xc, const double* Xt, const double* A, double* mean, double* var,
                              double* cross, void* workspace, size_t workspace_bytes, int M, int n_max, int d, int B,
                              int n_t, int kernel, void* stream) {
  if (!X || !theta || !linv_packed || !alpha || !ybar || !ystd || !w || !Xc || !Xt || !A || !mean || !var || !cross ||
      !workspace)
    return SCAML_E_ARG;
  if (M <= 0 || n_max <= 0 || d <= 0 || B <= 0 || n_t <= 0 || kernel < 0 || kernel > 3) return SCAML_E_ARG;
  if (d > scaml::kMaxP - 2 || n_t > 128) return SCAML_E_UNSUPPORTED;
  if (workspace_bytes < scaml_predict_conditioned_workspace_bytes(M, n_max, d, B, n_t)) return SCAML_E_WORKSPACE;
  const int n_tp = scaml::cond_ntp(n_t);
  int ct = 64, alias = 0;
  if (!scaml::predict_config(pad64(n_max), d, &ct, &alias)) return SCAML_E_SMEM;
  const int ns = scaml::predict_nsplit(M, B, num_sms(), ct);
  double* part = static_cast<double*>(workspace);
  double* cxp = part + (ns > 1 ? 2 * (size_t)ns * (size_t)B : 0);
  int rc = scaml::launch_predict_weighted(X, n_valid, theta, linv_packed, alpha, ybar, ystd, w, Xc, mean, var, part, M,
                                          n_max, pad64(n_max), d, B, kernel, num_sms(), stream, A, cxp, n_tp);
  if (rc != 0) return rc;
  scaml::CondCombineParams c{};
  c.theta = theta, c.ystd = ystd, c.w = w, c.Xc = Xc, c.Xt = Xt, c.cxp = cxp, c.cross = cross;
  c.M = M, c.d = d, c.B = B, c.n_t = n_t, c.n_tp = n_tp, c.nsplit = ns;
  c.ntsplit = scaml::comb_ntsplit(M, B, n_t, num_sms());
  c.dpart = cxp + (size_t)ns * (size_t)B * (size_t)n_tp;
  return scaml::launch_cond_combine(c, kernel, stream);
}

#endif
}  // extern "C"
