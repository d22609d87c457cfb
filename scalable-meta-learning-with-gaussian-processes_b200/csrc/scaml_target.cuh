// Target-GP objective of ScaML-GP in training mode (a7): (LML + log priors) / n_t and its
// gradient w.r.t. the M source weights and the raw target-kernel parameters, for R rows
// (restarts) at once.  Reference: ScaMLGP.forward train branch + priors,
// scamlgp/model.py:319-338, 359-363, 376-383; objective as in scamlgp/utils.py:171-177.
//
//   mean = (S w - mu_all) / s_all                    S   = source_means [n_t][M]
//   K    = (sum_i w_i^2 C_i) / s_all^2 + s k(X_t) + (noise + jitter) I     C = source_covs [n_t][n_t][M]
//
// Three kernels: (A) the two weighted contractions over the M tasks -- HBM bound, one warp per
// (a,b) entry streaming M contiguous doubles, fixed-order reduction; (B) one CTA per row for the
// small dense n_t x n_t algebra in shared memory (Cholesky, inverse, alpha, W = alpha alpha^T -
// K^-1, kernel-parameter gradient); (C) one thread per task for dL/dw_i, again a coalesced
// stream over C.  n_t <= 116 (two n_t x (n_t+1) matrices in shared memory).
#pragma once
#include "scaml_device.cuh"

namespace scaml {

constexpr int kTgtThreads = 256;

struct TargetParams {
  const double* smeans;  // [nt][M]
  const double* scovs;   // [nt][nt][M]
  const double* Xt;      // [nt][d]
  const double* yt;      // [nt] standardised with the all-data transform
  const double* w;       // [R][M]
  const double* theta_raw;  // [R][P]
  const double* jitter;     // [R] or null
  double* lml;              // [R]
  double* grad_w;           // [R][M]
  double* grad_theta;       // [R][P]
  int32_t* info;            // [R]
  double* covw;             // ws [R][nt][nt]
  double* meanw;            // ws [R][nt]
  double* Wmat;             // ws [R][nt][nt]
  double* alpha;            // ws [R][nt]
  double* big;              // ws [R][target_big_doubles]: K | L^-1 | scaled inputs of rows too large for shared memory
  double* linv_out;         // factorize: [nt][nt] row-major L^-1 (lower), or null
  double* theta_out;        // factorize: [P] constrained, or null
  double mu_all, s_all;
  double jitter_value;      // used when `jitter` is null
  int ladder;               // 1: psd_safe_cholesky jitter ladder (+1e-8, +1e-7, +1e-6) inside the kernel on failure
  int M, nt, d, R, w_prior;
  double w_p1, w_p2;
  scaml_hyper_spec spec;
};

inline size_t target_small_doubles(int nt, int R) { return (size_t)R * (2 * (size_t)nt * nt + 2 * (size_t)nt); }
inline size_t target_smem_bytes(int nt, int d) {
  return sizeof(double) * (2 * (size_t)nt * (nt + 1) + 4 * (size_t)nt + (size_t)d * nt + 4 * kMaxP + 64 + 2 * kTgtThreads);
}
// n_t x n_t systems that do not fit 227 KB of shared memory (n_t > ~116) keep K, L^-1 and the scaled inputs in a
// per-row global block (L2 resident: 2 x 5 MB at n_t = 800) -- same code, same order of operations, `BIG` variant
constexpr int kTgtBigFrom = 100;   // workspace is sized with the block from here on (any d)
constexpr int kTgtMaxPoints = 1024;
#ifdef SCAML_EMU
inline
#else
__host__ __device__ inline
#endif
size_t target_big_doubles(int nt) { return 2 * (size_t)nt * (nt + 1) + (size_t)kMaxP * nt; }
inline size_t target_big_smem_bytes(int nt) { return sizeof(double) * (4 * (size_t)nt + 4 * kMaxP + 64 + 2 * kTgtThreads); }
inline size_t target_workspace_doubles(int nt, int R) {
  return target_small_doubles(nt, R) + (nt >= kTgtBigFrom ? (size_t)R * target_big_doubles(nt) : 0);
}

// (A) covw[r][a][b] = sum_i w_i^2 C[a][b][i] / s^2 ; meanw[r][a] = (sum_i w_i S[a][i] - mu) / s
__global__ void __launch_bounds__(kTgtThreads) scaml_target_reduce_kernel(const TargetParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r = blockIdx.y;
  const long long items = (long long)p.nt * p.nt + p.nt;
  const double* w = p.w + (size_t)r * p.M;
  for (long long it = (long long)blockIdx.x * (kTgtThreads / 32) + warp; it < items;
       it += (long long)gridDim.x * (kTgtThreads / 32)) {
    const bool is_cov = it < (long long)p.nt * p.nt;
    const double* src = is_cov ? p.scovs + (size_t)it * p.M : p.smeans + (size_t)(it - (long long)p.nt * p.nt) * p.M;
    double acc = 0.0;
    for (int i = lane; i < p.M; i += 32) {
      const double wi = w[i];
      acc = fma(is_cov ? wi * wi : wi, src[i], acc);
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      if (is_cov)
        p.covw[(size_t)r * p.nt * p.nt + it] = acc / (p.s_all * p.s_all);
      else
        p.meanw[(size_t)r * p.nt + (it - (long long)p.nt * p.nt)] = (acc - p.mu_all) / p.s_all;
    }
  }
}

// block-wide fixed-order sum (result valid in every thread)
SCAML_DEVICE double block_sum(double v, double* red) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  v = warp_sum(v);
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  double s = 0.0;
  for (int k = 0; k < kTgtThreads / 32; ++k) s += red[k];
  __syncthreads();
  return s;
}

// (B) dense n_t x n_t part, one CTA per row r
template <int KIND, bool BIG>
__global__ void __launch_bounds__(kTgtThreads) scaml_target_factor_kernel(const TargetParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, nt = p.nt, ld = nt + 1, d = p.d, P = d + 2, r = blockIdx.x;
  double* gbig = BIG ? p.big + (size_t)r * target_big_doubles(nt) : nullptr;
  double* K = BIG ? gbig : sm;        // nt x ld : K_y, then L (lower)
  double* Li = K + (size_t)nt * ld;   // nt x ld : L^-1, then K^-1
  double* rv = BIG ? sm : Li + (size_t)nt * ld;  // residual y - mean
  double* zv = rv + nt;
  double* al = zv + nt;
  double* dg = al + nt;           // 1 / L_kk
  double* xs = BIG ? Li + (size_t)nt * ld : dg + nt;  // [d][nt] scaled inputs
  double* par = BIG ? dg + nt : xs + (size_t)d * nt;  // th | lp | dlp | chain
  double* th = par, *lp = par + kMaxP, *dlp = par + 2 * kMaxP, *chain = par + 3 * kMaxP;
  double* red = par + 4 * kMaxP;  // 64
  int* flag = reinterpret_cast<int*>(red + 32);
  const scaml_hyper_spec& sp = p.spec;
  const double* w = p.w + (size_t)r * p.M;

  if (tid < P) {
    const double raw = p.theta_raw[(size_t)r * P + tid];
    double lo, hi, p1, p2;
    int pk;
    if (tid < d) {
      lo = sp.ls_lo, hi = sp.ls_hi, pk = sp.ls_prior, p1 = sp.ls_p1, p2 = sp.ls_p2;
    } else if (tid == d) {
      lo = sp.os_lo, hi = sp.os_hi, pk = sp.os_prior, p1 = sp.os_p1, p2 = sp.os_p2;
    } else {
      lo = sp.noise_lo, hi = sp.noise_hi, pk = sp.noise_prior, p1 = sp.noise_p1, p2 = sp.noise_p2;
    }
    const double sg = sigmoid(raw), v = lo + (hi - lo) * sg;
    th[tid] = v;
    lp[tid] = log_prior(pk, p1, p2, v);
    dlp[tid] = dlog_prior(pk, p1, p2, v);
    chain[tid] = (hi - lo) * sg * (1.0 - sg);
    if (p.theta_out != nullptr) p.theta_out[(size_t)r * P + tid] = v;
  }
  if (tid == 0) *flag = 0;
  __syncthreads();
  const double os = th[d], base_add = th[d + 1] + (p.jitter ? p.jitter[r] : p.jitter_value);
  for (int i = tid; i < nt * d; i += kTgtThreads) {
    const int a = i / d, k = i - a * d;
    xs[k * nt + a] = p.Xt[i] / th[k];
  }
  for (int i = tid; i < nt; i += kTgtThreads) rv[i] = p.yt[i] - p.meanw[(size_t)r * nt + i];
  __syncthreads();
  // linear_operator's psd_safe_cholesky retries a failed factorisation with jitter 1e-8, 1e-7, 1e-6 (fp64); with
  // p.ladder the retries happen here, so the host never has to read `info` back between L-BFGS rounds
  double logdet = 0.0;
  const int nlev = p.ladder ? 4 : 1;
  for (int lev = 0; lev < nlev; ++lev) {
  const double diag_add = base_add + (lev == 0 ? 0.0 : (lev == 1 ? 1e-8 : (lev == 2 ? 1e-7 : 1e-6)));
  if (lev > 0) {
    __syncthreads();  // every thread has read the flag of the failed attempt
    if (tid == 0) *flag = 0;
    __syncthreads();
  }
  // ---- K_y -------------------------------------------------------------------------- //
  for (int i = tid; i < nt * nt; i += kTgtThreads) {
    const int a = i / nt, b = i - a * nt;
    double r2 = 0.0;
    for (int k = 0; k < d; ++k) {
      const double df = xs[k * nt + a] - xs[k * nt + b];
      r2 = fma(df, df, r2);
    }
    double v = p.covw[(size_t)r * nt * nt + i] + os * kappa_of<KIND>(r2);
    if (a == b) v += diag_add;
    K[a * ld + b] = v;
  }
  __syncthreads();
  // ---- Cholesky (right-looking, in place, lower) -------------------------------------- //
  logdet = 0.0;
  for (int k = 0; k < nt; ++k) {
    const double dkk = K[k * ld + k];
    if (!(dkk > 0.0) || !(dkk < 1e300)) {
      if (tid == 0 && *flag == 0) *flag = k + 1;
      break;  // uniform: every thread reads the same dkk
    }
    const double rs = rsqrt(dkk);
    logdet += log(dkk);
    __syncthreads();
    for (int a = k + tid; a < nt; a += kTgtThreads) K[a * ld + k] *= rs;
    if (tid == 0) dg[k] = rs;
    __syncthreads();
    const int m = nt - k - 1;  // trailing size
    for (int i = tid; i < m * m; i += kTgtThreads) {
      const int a = k + 1 + i / m, b = k + 1 + i % m;
      if (b <= a) K[a * ld + b] = fma(-K[a * ld + k], K[b * ld + k], K[a * ld + b]);
    }
    __syncthreads();
  }
  __syncthreads();
  if (*flag == 0) break;  // uniform
  }  // jitter levels
  if (*flag != 0) {
    if (tid == 0) {
      p.info[r] = *flag;
      p.lml[r] = nan("");
    }
    if (tid < P) p.grad_theta[(size_t)r * P + tid] = nan("");
    for (int i = tid; i < nt; i += kTgtThreads) p.alpha[(size_t)r * nt + i] = nan("");
    for (int i = tid; i < nt * nt; i += kTgtThreads) p.Wmat[(size_t)r * nt * nt + i] = nan("");
    return;
  }
  // ---- L^-1 : thread c solves L x = e_c ------------------------------------------------ //
  for (int c = tid; c < nt; c += kTgtThreads) {
    for (int a = 0; a < c; ++a) Li[a * ld + c] = 0.0;
    for (int a = c; a < nt; ++a) {
      double s = (a == c) ? 1.0 : 0.0;
      for (int k = c; k < a; ++k) s = fma(-K[a * ld + k], Li[k * ld + c], s);
      Li[a * ld + c] = s * dg[a];
    }
  }
  __syncthreads();
  if (p.linv_out != nullptr)
    for (int i = tid; i < nt * nt; i += kTgtThreads) p.linv_out[(size_t)r * nt * nt + i] = Li[(i / nt) * ld + (i % nt)];
  // z = L^-1 r ; alpha = L^-T z
  for (int a = tid; a < nt; a += kTgtThreads) {
    double s = 0.0;
    for (int k = 0; k <= a; ++k) s = fma(Li[a * ld + k], rv[k], s);
    zv[a] = s;
  }
  __syncthreads();
  for (int a = tid; a < nt; a += kTgtThreads) {
    double s = 0.0;
    for (int k = a; k < nt; ++k) s = fma(Li[k * ld + a], zv[k], s);
    al[a] = s;
    p.alpha[(size_t)r * nt + a] = s;
  }
  __syncthreads();
  // ---- W = alpha alpha^T - K^-1 (written to K's storage and to the workspace) ---------- //
  for (int i = tid; i < nt * nt; i += kTgtThreads) {
    const int a = i / nt, b = i - a * nt;
    const int k0 = a > b ? a : b;
    double s = 0.0;
    for (int k = k0; k < nt; ++k) s = fma(Li[k * ld + a], Li[k * ld + b], s);
    const double wv = al[a] * al[b] - s;
    K[a * ld + b] = wv;
    p.Wmat[(size_t)r * nt * nt + i] = wv;
  }
  __syncthreads();
  // ---- kernel-parameter gradient, quad, priors ----------------------------------------- //
  double q = 0.0;
  for (int a = tid; a < nt; a += kTgtThreads) q = fma(zv[a], zv[a], q);
  const double quad = block_sum(q, red);
  double wpr = 0.0;
  for (int i = tid; i < p.M; i += kTgtThreads) wpr += log_prior(p.w_prior, p.w_p1, p.w_p2, w[i]);
  const double wprior = block_sum(wpr, red);
  double gS = 0.0, gT = 0.0;
  for (int i = tid; i < nt * nt; i += kTgtThreads) {
    const int a = i / nt, b = i - a * nt;
    double r2 = 0.0;
    for (int k = 0; k < d; ++k) {
      const double df = xs[k * nt + a] - xs[k * nt + b];
      r2 = fma(df, df, r2);
    }
    gS = fma(K[a * ld + b], kappa_of<KIND>(r2), gS);
    if (a == b) gT += K[a * ld + b];
  }
  gS = block_sum(gS, red);
  gT = block_sum(gT, red);
  for (int k = 0; k < d; ++k) {
    double gl = 0.0;
    for (int i = tid; i < nt * nt; i += kTgtThreads) {
      const int a = i / nt, b = i - a * nt;
      double r2 = 0.0;
      for (int kk = 0; kk < d; ++kk) {
        const double df = xs[kk * nt + a] - xs[kk * nt + b];
        r2 = fma(df, df, r2);
      }
      double kap, kd;
      kappa_pair<KIND>(r2, kap, kd);
      const double df = xs[k * nt + a] - xs[k * nt + b];
      gl = fma(K[a * ld + b] * kd, df * df, gl);
    }
    gl = block_sum(gl, red);
    if (tid == 0) p.grad_theta[(size_t)r * P + k] = (0.5 * os * gl / th[k] + dlp[k]) * chain[k] / (double)nt;
  }
  if (tid == 0) {
    p.grad_theta[(size_t)r * P + d] = (0.5 * gS + dlp[d]) * chain[d] / (double)nt;
    p.grad_theta[(size_t)r * P + d + 1] = (0.5 * gT + dlp[d + 1]) * chain[d + 1] / (double)nt;
    double prior = wprior;
    for (int k = 0; k < P; ++k) prior += lp[k];
    p.lml[r] = (-0.5 * (quad + logdet + (double)nt * kLog2Pi) + prior) / (double)nt;
    p.info[r] = 0;
  }
}

// (C) dL/dw_i = [ alpha^T S[:,i] / s + (w_i / s^2) sum_ab W_ab C[a][b][i] + dlogp(w_i) ] / n_t
__global__ void __launch_bounds__(kTgtThreads) scaml_target_wgrad_kernel(const TargetParams p) {
  const int r = blockIdx.y, nt = p.nt;
  const double* Wm = p.Wmat + (size_t)r * nt * nt;
  const double* al = p.alpha + (size_t)r * nt;
  for (int i = blockIdx.x * kTgtThreads + threadIdx.x; i < p.M; i += gridDim.x * kTgtThreads) {
    const double wi = p.w[(size_t)r * p.M + i];
    double gm = 0.0, gc = 0.0;
    for (int a = 0; a < nt; ++a) gm = fma(__ldg(al + a), p.smeans[(size_t)a * p.M + i], gm);
    for (int ab = 0; ab < nt * nt; ++ab) gc = fma(__ldg(Wm + ab), p.scovs[(size_t)ab * p.M + i], gc);
    const double g = gm / p.s_all + wi * gc / (p.s_all * p.s_all) + dlog_prior(p.w_prior, p.w_p1, p.w_p2, wi);
    p.grad_w[(size_t)r * p.M + i] = g / (double)nt;
  }
}

// ---- conditioning on the target data at B candidates (q = 1) --------------------------------- //
//   k_s[j]  = cross[b][j] / s_all^2 + s k(x_b, X_t[j])
//   mean[b] = mu_all + s_all ( (pm[b] - mu_all)/s_all + k_s . alpha_t )
//   var[b]  = s_all^2 ( pv[b]/s_all^2 + s - || L_t^-1 k_s ||^2 )
// exact-GP conditioning of ExactGP.__call__ in eval mode on top of ScaMLGP.forward
// (reference scamlgp/model.py:364-383); one warp per candidate, L_t^-1 staged in shared memory.
struct TargetPostParams {
  const double* pm;     // [B] weighted source posterior mean (raw-Y units)
  const double* pv;     // [B] weighted source posterior variance
  const double* cross;  // [B][nt] weighted source cross-covariance with the target inputs
  const double* Xc;     // [B][d]
  const double* Xt;     // [nt][d]
  const double* theta;  // [P] constrained target-kernel parameters
  const double* linv;   // [nt][nt] row-major L_t^-1
  const double* alpha;  // [nt]
  double* mean;         // [B]
  double* var;          // [B]
  double* beta;         // optional [B][n_tp]: K_t^-1 k_s (needed by the candidate gradient, scaml_grad.cuh)
  double mu_all, s_all;
  int B, nt, d, kernel, n_tp;
};
constexpr int kPostThreads = 256;
inline size_t target_post_smem_bytes(int nt, int d) {
  const int ld = nt | 1;
  return sizeof(double) * ((size_t)nt * ld + (size_t)nt * d + nt + (kPostThreads / 32) * (size_t)(2 * nt + d) + kMaxP);
}
// BIG (n_t too large for L_t^-1 in shared memory): L_t^-1 is read straight from global memory (L2), row stride n_t
template <bool BIG>
__global__ void __launch_bounds__(kPostThreads) scaml_target_posterior_kernel(const TargetPostParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, nt = p.nt, d = p.d, ld = BIG ? nt : (nt | 1);
  const double* Li = BIG ? p.linv : sm;   // nt x ld
  double* xt = sm + (BIG ? 0 : (size_t)nt * ld);  // [nt][d] scaled
  double* al = xt + (size_t)nt * d;       // nt
  double* wk = al + nt;                   // per warp: k_s [nt] | x_b scaled [d] | L_t^-1 k_s [nt]
  double* th = wk + (kPostThreads / 32) * (size_t)(2 * nt + d);
  if (tid < d + 2) th[tid] = p.theta[tid];
  __syncthreads();
  if (!BIG)
    for (int i = tid; i < nt * nt; i += kPostThreads) sm[(i / nt) * ld + (i % nt)] = p.linv[i];
  for (int i = tid; i < nt * d; i += kPostThreads) xt[i] = p.Xt[i] / th[i % d];
  for (int i = tid; i < nt; i += kPostThreads) al[i] = p.alpha[i];
  __syncthreads();
  const double os = th[d], s2 = p.s_all * p.s_all;
  double* ks = wk + warp * (size_t)(2 * nt + d);
  double* xb = ks + nt;
  double* sv = xb + d;
  const int wpg = kPostThreads / 32;
  for (long long b = (long long)blockIdx.x * wpg + warp; b < p.B; b += (long long)gridDim.x * wpg) {
    __syncwarp();
    for (int k = lane; k < d; k += 32) xb[k] = p.Xc[(size_t)b * d + k] / th[k];
    __syncwarp();
    double dot = 0.0;
    for (int j = lane; j < nt; j += 32) {
      double r2 = 0.0;
      for (int k = 0; k < d; ++k) {
        const double df = xb[k] - xt[j * d + k];
        r2 = fma(df, df, r2);
      }
      const double v = p.cross[(size_t)b * nt + j] / s2 + os * kappa_rt(p.kernel, r2);
      ks[j] = v;
      dot = fma(v, al[j], dot);
    }
    __syncwarp();
    double ssq = 0.0;
    for (int i = lane; i < nt; i += 32) {
      double s = 0.0;
      const double* row = Li + (size_t)i * ld;
      for (int j = 0; j <= i; ++j) s = fma(row[j], ks[j], s);
      ssq = fma(s, s, ssq);
      sv[i] = s;
    }
    if (p.beta != nullptr) {  // beta = L_t^-T (L_t^-1 k_s)
      __syncwarp();
      for (int j = lane; j < p.n_tp; j += 32) {
        double s = 0.0;
        for (int i = j; i < nt; ++i) s = fma(Li[(size_t)i * ld + j], sv[i], s);
        p.beta[(size_t)b * p.n_tp + j] = s;
      }
    }
    dot = warp_sum(dot);
    ssq = warp_sum(ssq);
    if (lane == 0) {
      p.mean[b] = p.mu_all + p.s_all * ((p.pm[b] - p.mu_all) / p.s_all + dot);
      p.var[b] = s2 * (p.pv[b] / s2 + os - ssq);
    }
  }
}
inline int launch_target_posterior(const TargetPostParams& p, int num_sms, void* stream) {
  size_t smem = target_post_smem_bytes(p.nt, p.d);
  const bool big = smem > 227 * 1024;
  if (big) smem -= sizeof(double) * (size_t)p.nt * (p.nt | 1);
  if (smem > 227 * 1024 || p.nt > kTgtMaxPoints) return SCAML_E_SMEM;
  const int grid = stride_grid(((long long)p.B + kPostThreads / 32 - 1) / (kPostThreads / 32), 2LL * num_sms);
  return big ? launch(scaml_target_posterior_kernel<true>, grid, kPostThreads, smem, stream, p)
             : launch(scaml_target_posterior_kernel<false>, grid, kPostThreads, smem, stream, p);
}

inline int launch_target(const TargetParams& p, int num_sms, void* stream) {
  size_t smem = target_smem_bytes(p.nt, p.d);
  const bool big = smem > 227 * 1024;
  if (big) {  // K, L^-1 and the scaled inputs move to the per-row global block
    if (p.nt < kTgtBigFrom || p.nt > kTgtMaxPoints || p.big == nullptr) return SCAML_E_SMEM;
    smem = target_big_smem_bytes(p.nt);
  }
  const long long items = (long long)p.nt * p.nt + p.nt;
  const dim3 reduce_grid(stride_grid((items + 7) / 8, 8LL * num_sms), p.R);
  const dim3 wgrad_grid(stride_grid((p.M + kTgtThreads - 1) / kTgtThreads, 4LL * num_sms), p.R);
  // the dispatch rejects an unknown kernel family before anything is launched
  return dispatch_kind(p.spec.kernel, [&](auto K) {
    int rc = launch(scaml_target_reduce_kernel, reduce_grid, kTgtThreads, 0, stream, p);
    if (rc) return rc;
    rc = big ? launch(scaml_target_factor_kernel<K.value, true>, p.R, kTgtThreads, smem, stream, p)
             : launch(scaml_target_factor_kernel<K.value, false>, p.R, kTgtThreads, smem, stream, p);
    if (rc || p.grad_w == nullptr) return rc;
    return launch(scaml_target_wgrad_kernel, wgrad_grid, kTgtThreads, 0, stream, p);
  });
}

}  // namespace scaml
