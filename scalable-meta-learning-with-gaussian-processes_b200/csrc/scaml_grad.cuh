// Analytic candidate gradients of the ScaML-GP posterior (row f3 of SURVEY 8f: "UCB with d mu/dx, d sigma^2/dx from
// the kernel").  The reference obtains them by autograd through `ScaMLGP.forward` (eval branch,
// scamlgp/model.py:364-375) and gpytorch's exact prediction when botorch's optimize_acqf runs L-BFGS-B on the
// acquisition function (consumer: UpperConfidenceBound, scamlgp/utils.py:215-224).
//
// With  S = s_all,  c_m = w_m^2 ystd_m^2,  u_m(x) = K_m^-1 k*_m(x),  A_m = K_m^-1 K_m(X_m, X_t),
// beta(x) = K_t^-1 k_s(x)  (scaml_target_posterior, beta output)  and the un-standardised posterior
//   mean(x) = sum_m w_m (ybar_m + ystd_m k*_m^T alpha_m) + S k_s^T alpha_t
//   var(x)  = sum_m c_m (s_m - k*_m^T u_m) + S^2 (s_t - k_s^T beta),
//   k_s[j]  = sum_m c_m (K_m(x, x_tj) - k*_m^T A_m[:, j]) / S^2 + s_t kappa_t(x, x_tj)
// every x-dependence sits in a kernel value kappa(x, z), z a training input of task m or a target input, so
//   d mean / dx_k = sum_m sum_{z in [X_m; X_t]} cm_z  d(s_m kappa_m(x, z))/dx_k  +  S s_t sum_j alpha_t[j] d kappa_t(x, x_tj)/dx_k
//   d var  / dx_k = sum_m sum_{z in [X_m; X_t]} cv_z  d(s_m kappa_m(x, z))/dx_k  -  2 S^2 s_t sum_j beta[j] d kappa_t(x, x_tj)/dx_k
// with the coefficients
//   training row i : cm = w_m ystd_m alpha_m[i] - (c_m / S) (A_m alpha_t)[i]      cv = -2 c_m (u_m[i] - (A_m beta)[i])
//   target row j   : cm = (c_m / S) alpha_t[j]                                    cv = -2 c_m beta[j]
// and  d kappa(x, z)/dx_k = -kd (x_k - z_k) / l_k^2,  kd = -2 dkappa/dr^2  (scaml_device.cuh).
//
// u_m for a tile of candidates is exactly what scaml_cond_prepare computes with the candidates in the place of the
// target inputs (U = K_m^-1 K_m(X_m, Xc), both triangular products on DMMA), so the n^2 work is done there; the
// kernels here are the O(n (n_t + d)) contraction per (task, candidate):
//   scaml_grad_mix_kernel      : U <- U - A_m beta and aal <- A_m alpha_t, a [32 x n_t] x [n_t x B] DMMA product per
//                                (task, 32-row chunk) with beta^T | alpha_t resident in shared memory;
//   scaml_grad_contract_kernel : lane <-> candidate (32-candidate tiles), the 8 warps split the rows of a task in
//                                4-row blocks (4 independent exp chains per thread); the sum over the tasks of a
//                                split stays in registers (fixed order), one cross-warp reduction at the end;
//   scaml_grad_finish_kernel   : fixed-order sum of the task splits + the target-kernel terms, one warp per candidate.
#pragma once
#include "scaml_device.cuh"

namespace scaml {

struct GradParams {
  const double* X;         // [M][n_max][d]
  const int32_t* n_valid;  // [M] or null
  const double* theta;     // [M][P] constrained
  const double* alpha;     // [M][n_pad]
  const double* ystd;      // [M]
  const double* w;         // [M] (pruned: 0 -> task skipped)
  const double* Xc;        // [B][d]
  double* U;               // [M][n_pad][B_p]  in: K_m^-1 K_m(X_m, Xc); the mix kernel turns it into U - A beta in place
  double* aal;             // [M][n_pad] workspace: A_m alpha_t (n_t > 0)
  const double* Xt;        // [n_t][d]               (n_t > 0)
  const double* A;         // [M][n_pad][n_tp]       (n_t > 0)
  const double* alpha_t;   // [n_t]                  (n_t > 0)
  const double* beta;      // [B][n_tp]              (n_t > 0)
  const double* theta_t;   // [P] constrained target-kernel parameters (n_t > 0)
  double* part;            // [nsplit][B][2 d]
  double* dmean;           // [B][d]
  double* dvar;            // [B][d]
  double s_all;
  int M, n_max, n_pad, d, B, B_p, n_t, n_tp, nsplit, ntile, kernel_t;
};

constexpr int kGradThreads = 256;
constexpr int kGradWarps = kGradThreads / 32;
constexpr int kGradCT = 32;  // candidates per tile (lane <-> candidate)
#ifndef SCAML_GRAD_ROWS
#define SCAML_GRAD_ROWS 4
#endif
constexpr int kGR = SCAML_GRAD_ROWS;  // rows per thread and step = independent exp chains in flight

// shared memory (doubles): xs [max(n_pad, 512)][d] (aliased by red [warps][2 d][32] at the end) | al [n_pad]
//                          | xts [n_tp][d] | bt [n_tp][32] | at [n_tp] | il2 [kMaxP]
#ifndef SCAML_EMU
__host__ __device__
#endif
inline size_t grad_xs_rows(int n_pad) { return n_pad > 2 * 32 * kGradWarps ? n_pad : 2 * 32 * kGradWarps; }
inline size_t grad_smem_bytes(int n_pad, int d, int n_tp) {
  return sizeof(double) * (grad_xs_rows(n_pad) * d + n_pad + (size_t)n_tp * d + (size_t)n_tp * 32 + n_tp + kMaxP + 8);
}
inline int grad_nsplit(int M, int ntile, int num_sms) {
  int ns = (2 * num_sms + ntile - 1) / ntile;
  if (ns > M) ns = M;
  if (ns < 1) ns = 1;
  return ns;
}

// U <- U - A_m beta (all candidates of the call) and aal <- A_m alpha_t: per (task, 32-row chunk) one
// [32 x n_tp] x [n_tp x (B_p + 8)] product on the FP64 tensor cores (column B_p of the right-hand side is alpha_t).
// Staged operands are padded to a row stride = 4 (mod 8) doubles (conflict-free DMMA fragment loads).
constexpr int kMixMaxCB = 9;  // column blocks per warp: (128 + 8) / 8 = 17 over two warp groups
inline int mix_ldb(int B_p) { return B_p + 8 + 4; }
inline size_t grad_mix_smem_bytes(int n_tp, int B_p) {
  return sizeof(double) * ((size_t)n_tp * mix_ldb(B_p) + 32 * (size_t)(n_tp + 4));
}
__global__ void __launch_bounds__(kGradThreads) scaml_grad_mix_kernel(const GradParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const int ntp = p.n_tp, nt = p.n_t, Bp = p.B_p, ldb = Bp + 12, lda = ntp + 4, n_pad = p.n_pad;
  double* bts = sm;                        // [ntp][ldb]: beta^T | alpha_t | 0
  double* Ach = bts + (size_t)ntp * ldb;   // [32][lda]
  for (int i = tid; i < ntp * (Bp + 8); i += kGradThreads) {
    const int j = i / (Bp + 8), c = i - j * (Bp + 8);
    double v = 0.0;
    if (j < nt) {
      if (c < p.B) v = p.beta[(size_t)c * ntp + j];
      else if (c == Bp) v = p.alpha_t[j];
    }
    bts[(size_t)j * ldb + c] = v;
  }
  const int nchunk = n_pad / 32, ncb = Bp / 8 + 1;  // column blocks incl. the alpha_t block
  const int rb = warp & 3, cb0 = warp >> 2;
  const long long items = (long long)p.M * nchunk;
  for (long long it = blockIdx.x; it < items; it += gridDim.x) {
    const int m = (int)(it / nchunk), ch = (int)(it - (long long)m * nchunk);
    const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
    if (p.w[m] == 0.0 || 32 * ch >= nv) continue;  // uniform over the CTA
    __syncthreads();  // previous chunk consumed (and bts staged)
    const double* src = p.A + ((size_t)m * n_pad + 32 * ch) * ntp;
    for (int i = tid; i < 32 * ntp; i += kGradThreads) Ach[(i / ntp) * lda + (i % ntp)] = src[i];
    // the U entries this thread will update: loaded now, so that their DRAM latency overlaps the A chunk and the DMMAs
    double2 uq[kMixMaxCB];
    {
      const double* ur0 = p.U + ((size_t)m * n_pad + 32 * ch + 8 * rb + g) * Bp;
#pragma unroll
      for (int c = 0; c < kMixMaxCB; ++c)
        uq[c] = (cb0 + 2 * c < ncb - 1) ? *reinterpret_cast<const double2*>(ur0 + 8 * (cb0 + 2 * c) + 2 * t4)
                                        : make_double2(0.0, 0.0);
    }
    __syncthreads();
    double acc[kMixMaxCB][2];
#pragma unroll
    for (int c = 0; c < kMixMaxCB; ++c) acc[c][0] = acc[c][1] = 0.0;
    const double* ar = Ach + (size_t)(8 * rb + g) * lda + t4;
    const double* br = bts + (size_t)t4 * ldb + 8 * cb0 + g;
    for (int s = 0; s < ntp / 4; ++s) {
      const double a = ar[4 * s];
#pragma unroll
      for (int c = 0; c < kMixMaxCB; ++c)
        if (cb0 + 2 * c < ncb) dmma884(acc[c], a, br[(size_t)4 * s * ldb + 16 * c]);
    }
    const int row = 32 * ch + 8 * rb + g;
    double* ur = p.U + ((size_t)m * n_pad + row) * Bp;
#pragma unroll
    for (int c = 0; c < kMixMaxCB; ++c) {
      const int cb = cb0 + 2 * c;
      if (cb < ncb - 1) {
        *reinterpret_cast<double2*>(ur + 8 * cb + 2 * t4) = make_double2(uq[c].x - acc[c][0], uq[c].y - acc[c][1]);
      } else if (cb == ncb - 1 && t4 == 0) {
        p.aal[(size_t)m * n_pad + row] = acc[c][0];
      }
    }
  }
}

template <int KIND, int DMAX>
__global__ void __launch_bounds__(kGradThreads, 1) scaml_grad_contract_kernel(const GradParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int d = p.d, P = d + 2, n_pad = p.n_pad, nt = p.n_t, ntp = p.n_tp;
  double* xs = sm;                               // [n_pad][d] raw inputs of the task
  double* al = xs + grad_xs_rows(n_pad) * d;     // [n_pad] mean coefficient of the training rows
  double* xts = al + n_pad;                      // [ntp][d] raw target inputs
  double* bt = xts + (size_t)ntp * d;            // [ntp][32] beta of this tile, candidate fastest
  double* at = bt + (size_t)ntp * 32;            // [ntp] alpha_t
  double* il2 = at + ntp;                        // [kMaxP] 1 / l_k^2 of the task
  double* red = xs;                              // [warps][2 d][32], after the last task of the item
  const int items = p.nsplit * p.ntile;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int split = it / p.ntile, tile = it - split * p.ntile;
    const int b = tile * kGradCT + lane;
    const bool live = b < p.B;
    const int bc = live ? b : p.B - 1;  // dead lanes shadow the last candidate (results discarded)
    const int m_lo = (int)((long long)p.M * split / p.nsplit), m_hi = (int)((long long)p.M * (split + 1) / p.nsplit);
    __syncthreads();
    for (int i = tid; i < ntp * d; i += kGradThreads) xts[i] = (i / d < nt) ? p.Xt[i] : 0.0;
    for (int i = tid; i < ntp * 32; i += kGradThreads) {
      const int j = i >> 5, l = i & 31;
      const int bb = tile * kGradCT + l < p.B ? tile * kGradCT + l : p.B - 1;
      bt[i] = (j < nt) ? p.beta[(size_t)bb * ntp + j] : 0.0;
    }
    for (int i = tid; i < ntp; i += kGradThreads) at[i] = (i < nt) ? p.alpha_t[i] : 0.0;
    double x[DMAX], accm[DMAX], accv[DMAX];
#pragma unroll
    for (int k = 0; k < DMAX; ++k) {
      x[k] = (k < d) ? p.Xc[(size_t)bc * d + k] : 0.0;
      accm[k] = accv[k] = 0.0;
    }
    for (int m = m_lo; m < m_hi; ++m) {
      const double wm = p.w[m];
      if (wm == 0.0) continue;  // pruned task (uniform over the CTA)
      const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
      const double* th = p.theta + (size_t)m * P;
      const double os = th[d], sy = p.ystd[m];
      const double cmw = wm * sy, c = cmw * cmw, cS = c / p.s_all;
      const double* Xm = p.X + (size_t)m * p.n_max * d;
      const double* Um = p.U + (size_t)m * n_pad * p.B_p;  // already U - A beta when n_t > 0 (mix kernel)
      __syncthreads();  // previous task's xs / al / il2 are no longer read
      for (int i = tid; i < nv * d; i += kGradThreads) xs[i] = Xm[i];
      for (int i = tid; i < nv; i += kGradThreads) {
        const double a = cmw * p.alpha[(size_t)m * n_pad + i];
        al[i] = nt > 0 ? a - cS * p.aal[(size_t)m * n_pad + i] : a;
      }
      if (tid < d) {
        const double l = th[tid];
        il2[tid] = 1.0 / (l * l);
      }
      __syncthreads();
      double un[kGR];  // U of the next row block, in flight under the current block's exponentials
#pragma unroll
      for (int u = 0; u < kGR; ++u) {
        const int i = kGR * warp + u;
        un[u] = Um[(size_t)(i < nv ? i : nv - 1) * p.B_p + bc];
      }
      for (int i0 = kGR * warp; i0 < nv; i0 += kGR * kGradWarps) {  // this warp: rows i0 .. i0 + kGR - 1
        double r2[kGR], kap[kGR], kd[kGR], gm[kGR], gv[kGR];
#pragma unroll
        for (int u = 0; u < kGR; ++u) {
          const int i = i0 + u;
          const bool ok = i < nv;
          const int ic = ok ? i : nv - 1;
          const double uu = un[u];
          const int inx = i + kGR * kGradWarps;
          un[u] = Um[(size_t)(inx < nv ? inx : nv - 1) * p.B_p + bc];
          gm[u] = ok ? al[ic] : 0.0;
          gv[u] = ok ? -2.0 * c * uu : 0.0;
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < DMAX; ++k)
            if (k < d) {
              const double df = x[k] - xs[ic * d + k];
              s = fma(df * il2[k], df, s);
            }
          r2[u] = s;
        }
        kappa_n<KIND, kGR, true>(r2, kap, kd);
#pragma unroll
        for (int u = 0; u < kGR; ++u) {
          const double f = os * kd[u];
          gm[u] *= f;
          gv[u] *= f;
        }
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
          if (k < d) {
            const double xk = x[k], ik = il2[k];
#pragma unroll
            for (int u = 0; u < kGR; ++u) {
              const int ic = (i0 + u < nv) ? i0 + u : nv - 1;
              const double df = (xk - xs[ic * d + k]) * ik;
              accm[k] = fma(gm[u], df, accm[k]);
              accv[k] = fma(gv[u], df, accv[k]);
            }
          }
      }
      // target inputs as extra rows of the task's kernel (the K_m(x, x_tj) terms of k_s)
      for (int j0 = 4 * warp; j0 < nt; j0 += 4 * kGradWarps) {
        double r2[4], kap[4], kd[4], gm[4], gv[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = j0 + u;
          const bool ok = j < nt;
          const int jc = ok ? j : nt - 1;
          gm[u] = ok ? cS * at[jc] : 0.0;
          gv[u] = ok ? -2.0 * c * bt[jc * 32 + lane] : 0.0;
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < DMAX; ++k)
            if (k < d) {
              const double df = x[k] - xts[jc * d + k];
              s = fma(df * il2[k], df, s);
            }
          r2[u] = s;
        }
        kappa_n<KIND, 4, true>(r2, kap, kd);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const double f = os * kd[u];
          gm[u] *= f;
          gv[u] *= f;
        }
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
          if (k < d) {
            const double xk = x[k], ik = il2[k];
#pragma unroll
            for (int u = 0; u < 4; ++u) {
              const int jc = (j0 + u < nt) ? j0 + u : nt - 1;
              const double df = (xk - xts[jc * d + k]) * ik;
              accm[k] = fma(gm[u], df, accm[k]);
              accv[k] = fma(gv[u], df, accv[k]);
            }
          }
      }
    }
    // cross-warp reduction in a fixed order; d kappa/dx_k = -kd (x_k - z_k)/l_k^2 -> the sign goes in here
    __syncthreads();
#pragma unroll
    for (int k = 0; k < DMAX; ++k)
      if (k < d) {
        red[((size_t)warp * 2 * d + k) * 32 + lane] = accm[k];
        red[((size_t)warp * 2 * d + d + k) * 32 + lane] = accv[k];
      }
    __syncthreads();
    for (int i = tid; i < 2 * d * 32; i += kGradThreads) {
      const int k2 = i >> 5, l = i & 31;
      double s = 0.0;
      for (int wv = 0; wv < kGradWarps; ++wv) s += red[((size_t)wv * 2 * d + k2) * 32 + l];
      const int bb = tile * kGradCT + l;
      if (bb < p.B) p.part[((size_t)split * p.B + bb) * 2 * d + k2] = -s;
    }
  }
}

// dmean[b][k] = sum_split part + S s_t sum_j alpha_t[j] dkappa_t/dx_k ;  dvar[b][k] = sum_split part - 2 S^2 s_t sum_j beta[b][j] dkappa_t/dx_k
__global__ void __launch_bounds__(64) scaml_grad_finish_kernel(const GradParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, d = p.d, nt = p.n_t;
  const int wpg = blockDim.x >> 5;
  for (long long b = (long long)blockIdx.x * wpg + warp; b < p.B; b += (long long)gridDim.x * wpg) {
    double gmj[4] = {0.0, 0.0, 0.0, 0.0}, gvj[4] = {0.0, 0.0, 0.0, 0.0};
    const bool tterms = nt > 0 && p.kernel_t >= 0;  // kernel_t < 0: task-sharded partial sums, another rank adds them
    if (tterms) {
      const double os = p.theta_t[d], S = p.s_all;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int j = lane + 32 * u;
        if (j < nt) {
          double r2 = 0.0;
          for (int k = 0; k < d; ++k) {
            const double df = (p.Xc[(size_t)b * d + k] - p.Xt[(size_t)j * d + k]) / p.theta_t[k];
            r2 = fma(df, df, r2);
          }
          double kap, kd;
          switch (p.kernel_t) {
            case SCAML_KERNEL_RBF: kappa_pair<SCAML_KERNEL_RBF>(r2, kap, kd); break;
            case SCAML_KERNEL_MATERN12: kappa_pair<SCAML_KERNEL_MATERN12>(r2, kap, kd); break;
            case SCAML_KERNEL_MATERN32: kappa_pair<SCAML_KERNEL_MATERN32>(r2, kap, kd); break;
            default: kappa_pair<SCAML_KERNEL_MATERN52>(r2, kap, kd); break;
          }
          gmj[u] = S * os * p.alpha_t[j] * kd;
          gvj[u] = -2.0 * S * S * os * p.beta[(size_t)b * p.n_tp + j] * kd;
        }
      }
    }
    for (int k = 0; k < d; ++k) {
      double sm_ = 0.0, sv_ = 0.0;
      if (tterms) {
        const double l = p.theta_t[k], il2 = 1.0 / (l * l);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int j = lane + 32 * u;
          if (j < nt) {
            const double df = (p.Xc[(size_t)b * d + k] - p.Xt[(size_t)j * d + k]) * il2;
            sm_ = fma(gmj[u], df, sm_);
            sv_ = fma(gvj[u], df, sv_);
          }
        }
        sm_ = -warp_sum(sm_);
        sv_ = -warp_sum(sv_);
      }
      double am = 0.0, av = 0.0;  // lanes stride over the task splits, then a fixed-order warp tree
      for (int s = lane; s < p.nsplit; s += 32) {
        am += p.part[((size_t)s * p.B + b) * 2 * d + k];
        av += p.part[((size_t)s * p.B + b) * 2 * d + d + k];
      }
      am = warp_sum(am);
      av = warp_sum(av);
      if (lane == 0) {
        p.dmean[(size_t)b * d + k] = am + sm_;
        p.dvar[(size_t)b * d + k] = av + sv_;
      }
    }
  }
}

inline int launch_posterior_grad(GradParams p, int kernel, int num_sms, void* stream) {
  const size_t smem = grad_smem_bytes(p.n_pad, p.d, p.n_tp);
  if (smem > 227 * 1024) return SCAML_E_SMEM;
  if (p.n_t > 0) {
    const size_t msm = grad_mix_smem_bytes(p.n_tp, p.B_p);
    if (msm > 227 * 1024) return SCAML_E_SMEM;
    int per_sm = (int)((227 * 1024) / (msm + 1024));
    if (per_sm > 4) per_sm = 4;
    if (per_sm < 1) per_sm = 1;
    const long long mitems = (long long)p.M * (p.n_pad / 32);
    const int rc = launch(scaml_grad_mix_kernel, stride_grid(mitems, (long long)per_sm * num_sms), kGradThreads, msm,
                          stream, p);
    if (rc) return rc;
  }
  const int grid = stride_grid(p.nsplit * p.ntile, 2 * num_sms);
  const int rc = dispatch_kind(kernel, [&](auto K) {
    return dispatch_dmax(p.d, [&](auto D) {
      return launch(scaml_grad_contract_kernel<K.value, D.value>, grid, kGradThreads, smem, stream, p);
    });
  });
  if (rc) return rc;
  // one warp per candidate, two warps per CTA
  return launch(scaml_grad_finish_kernel, stride_grid(((long long)p.B + 1) / 2, 4LL * num_sms), 64, 0, stream, p);
}

}  // namespace scaml
