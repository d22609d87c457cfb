// Joint posterior of q-point blocks and its vector-Jacobian product: the quantities a batch acquisition (qUCB, qEI)
// needs when L-BFGS-B optimises q candidates jointly (botorch's optimize_acqf with q > 1 over `ScaMLGP.forward`, eval
// branch, reference scamlgp/model.py:364-375).  Points Xc [B][d] come in blocks of q consecutive points (B = nb q).
//
// With the notation of scaml_grad.cuh (c_m = w_m^2 ystd_m^2, S = s_all, u_m(x) = K_m^-1 k*_m(x), beta(x) = K_t^-1 k_s(x))
// the weighted prior block of block b is
//   Sp_ij = sum_m c_m ( s_m kappa_m(x_i, x_j) - k*_m(x_i)^T u_m(x_j) ),             i, j in the same block,
// and the conditioned block Sigma = Sp + S^2 s_t kappa_t(x_i, x_j) - S^2 k_s(x_i)^T beta(x_j) (Sp + s_t kappa_t for
// n_t = 0).  Given g [B] = da/dmean and G [nb][q][q] = da/dSigma, with Gh = (G + G^T)/2 per block,
//   da/dx_i = g_i dmean_i + 2 sum_j Gh_ij d_1 Sigma(x_i, x_j).
// Every term of d_1 Sigma except the direct kernel terms is the q = 1 dvar formula with the coefficient vectors
// u_i - A beta_i and beta_i replaced by sum_j Gh_ij (u_j - A beta_j) and sum_j Gh_ij beta_j (the factor 2 of dvar =
// 2 d_1 var is the 2 above).  So the VJP is
//   scaml_qblock_fold_kernel       : U <- U Gh (block-diagonal, per task row), beta~ = Gh beta;
//   scaml_grad_{mix,contract,finish}_kernel (unchanged, with U Gh and beta~) : dmean_i and the folded dvar_i;
//   scaml_qblock_direct_kernel     : + 2 sum_{j != i} Gh_ij d_1[ sum_m c_m s_m kappa_m(x_i, x_j) + S^2 s_t kappa_t(x_i, x_j) ]
//                                    and dX_i = g_i dmean_i + folded dvar_i + direct_i.
// The block values run in scaml_qblock_cov_kernel: lane <-> point (32-point tiles), the 8 warps split the rows of a
// task, per row one kernel value and q FMAs against the row of U -- O(n (q + d)) per (task, point), the n^2 work stays
// in scaml_cond_prepare.  Every sum over tasks runs in a fixed order (deterministic).
#pragma once
#include "scaml_grad.cuh"

namespace scaml {

constexpr int kQMax = 16;      // points per block
constexpr int kQbThreads = 256;
constexpr int kQbWarps = kQbThreads / 32;

struct QBlockCovParams {
  const double* X;         // [M][n_max][d]
  const int32_t* n_valid;  // [M] or null
  const double* theta;     // [M][P] constrained
  const double* ystd;      // [M]
  const double* w;         // [M] (0 -> task skipped)
  const double* Xc;        // [B][d]
  const double* U;         // [M][n_pad][B_p]
  double* part;            // [nsplit][B][q]
  double* cov;             // [B / q][q][q]
  int M, n_max, n_pad, d, B, B_p, q, nsplit, ntile;
};

// shared memory (doubles): xs [n_pad][d] (aliased by red [warps][q][32] at the end) | il2 [kMaxP]
inline size_t qblock_cov_smem_bytes(int n_pad, int d) {
  const size_t red = (size_t)kQbWarps * kQMax * 32;
  const size_t xs = (size_t)n_pad * d;
  return sizeof(double) * ((xs > red ? xs : red) + kMaxP);
}

template <int KIND, int DMAX>
__global__ void __launch_bounds__(kQbThreads, 1) scaml_qblock_cov_kernel(const QBlockCovParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int d = p.d, P = d + 2, n_pad = p.n_pad, q = p.q;
  const size_t xs_len = (size_t)n_pad * d > (size_t)kQbWarps * kQMax * 32 ? (size_t)n_pad * d
                                                                           : (size_t)kQbWarps * kQMax * 32;
  double* xs = sm;            // [n_pad][d] raw inputs of the task
  double* il2 = sm + xs_len;  // [kMaxP] 1 / l_k^2 of the task
  double* red = sm;           // [warps][q][32], after the last task of the item
  const int items = p.nsplit * p.ntile;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int split = it / p.ntile, tile = it - split * p.ntile;
    const int b = tile * 32 + lane;
    const bool live = b < p.B;
    const int bc = live ? b : p.B - 1;  // dead lanes shadow the last point (results discarded)
    const int jb = (bc / q) * q;        // first point of this point's block
    const int m_lo = (int)((long long)p.M * split / p.nsplit), m_hi = (int)((long long)p.M * (split + 1) / p.nsplit);
    double x[DMAX], acc[kQMax];
#pragma unroll
    for (int k = 0; k < DMAX; ++k) x[k] = (k < d) ? p.Xc[(size_t)bc * d + k] : 0.0;
#pragma unroll
    for (int j = 0; j < kQMax; ++j) acc[j] = 0.0;
    for (int m = m_lo; m < m_hi; ++m) {
      const double wm = p.w[m];
      if (wm == 0.0) continue;  // pruned task (uniform over the CTA)
      const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
      const double* th = p.theta + (size_t)m * P;
      const double cw = wm * p.ystd[m], cs = cw * cw * th[d];  // c_m s_m
      const double* Xm = p.X + (size_t)m * p.n_max * d;
      const double* Um = p.U + (size_t)m * n_pad * p.B_p + jb;
      __syncthreads();  // previous task's xs / il2 are no longer read
      for (int i = tid; i < nv * d; i += kQbThreads) xs[i] = Xm[i];
      if (tid < d) {
        const double l = th[tid];
        il2[tid] = 1.0 / (l * l);
      }
      __syncthreads();
      // - c_m s_m sum_r kappa(x_i, x_r) U[r][j]  (U = K^-1 k*: k*^T u = s_m kappa^T U)
      for (int r0 = 4 * warp; r0 < nv; r0 += 4 * kQbWarps) {
        double r2[4], kap[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          const int rc = (r0 + u < nv) ? r0 + u : nv - 1;
          double s = 0.0;
#pragma unroll
          for (int k = 0; k < DMAX; ++k)
            if (k < d) {
              const double df = x[k] - xs[rc * d + k];
              s = fma(df * il2[k], df, s);
            }
          r2[u] = s;
        }
        kappa_n<KIND, 4, false>(r2, kap, kap);
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          if (r0 + u >= nv) break;
          const double f = -cs * kap[u];
          const double* ur = Um + (size_t)(r0 + u) * p.B_p;
#pragma unroll
          for (int j = 0; j < kQMax; ++j)
            if (j < q) acc[j] = fma(f, ur[j], acc[j]);
        }
      }
      if (warp == 0) {  // + c_m s_m kappa(x_i, x_j): once per task
#pragma unroll
        for (int j = 0; j < kQMax; ++j)
          if (j < q) {
            double s = 0.0;
#pragma unroll
            for (int k = 0; k < DMAX; ++k)
              if (k < d) {
                const double df = x[k] - p.Xc[(size_t)(jb + j) * d + k];
                s = fma(df * il2[k], df, s);
              }
            acc[j] = fma(cs, kappa_of<KIND>(s), acc[j]);
          }
      }
    }
    // cross-warp reduction in a fixed order
    __syncthreads();
#pragma unroll
    for (int j = 0; j < kQMax; ++j)
      if (j < q) red[((size_t)warp * q + j) * 32 + lane] = acc[j];
    __syncthreads();
    for (int i = tid; i < q * 32; i += kQbThreads) {
      const int j = i >> 5, l = i & 31;
      double s = 0.0;
      for (int wv = 0; wv < kQbWarps; ++wv) s += red[((size_t)wv * q + j) * 32 + l];
      const int bb = tile * 32 + l;
      if (bb < p.B) p.part[((size_t)split * p.B + bb) * q + j] = s;
    }
  }
}

// cov[b][ii][j] = (sum_split part[.][i][j] + sum_split part[.][j'][ii]) / 2 for i = b q + ii, j' = b q + j: the two
// triangles are summed in different orders, the mean makes every block exactly symmetric
__global__ void __launch_bounds__(128) scaml_qblock_cov_finish_kernel(const QBlockCovParams p) {
  const int q = p.q;
  for (long long t = (long long)blockIdx.x * blockDim.x + threadIdx.x; t < (long long)p.B * q;
       t += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(t / q), j = (int)(t - (long long)i * q);
    const int jb = (i / q) * q, ii = i - jb;
    double a = 0.0, c = 0.0;
    for (int s = 0; s < p.nsplit; ++s) {
      a += p.part[((size_t)s * p.B + i) * q + j];
      c += p.part[((size_t)s * p.B + jb + j) * q + ii];
    }
    p.cov[t] = 0.5 * (a + c);
  }
}

struct QBlockVjpParams {
  const int32_t* n_valid;  // [M] or null
  const double* X;         // [M][n_max][d]
  const double* theta;     // [M][P] constrained
  const double* ystd;      // [M]
  const double* w;         // [M]
  const double* Xc;        // [B][d]
  const double* gcov;      // [B / q][q][q] da/dSigma
  const double* gmean;     // [B] da/dmean
  double* U;               // [M][n_pad][B_p], folded in place
  const double* beta;      // [B][n_tp] (n_t > 0)
  double* beta_f;          // [B][n_tp] Gh beta (n_t > 0)
  const double* theta_t;   // [P] constrained target-kernel parameters
  const double* dmean;     // [B][d]  (grad path outputs with the folded inputs)
  const double* dvar;      // [B][d]
  double* dX;              // [B][d]
  double s2t;              // S^2 (1 for n_t = 0): scale of the target kernel in Sigma
  int M, n_max, n_pad, d, B, B_p, q, n_t, n_tp, kernel_t;
};

SCAML_DEVICE double qblock_gsym(const double* gcov, int q, int i, int j) {  // Gh_ij, i and j in the same block
  const int jb = (i / q) * q, ii = i - jb, jj = j - jb;
  const double* g = gcov + (size_t)jb * q;
  return 0.5 * (g[ii * q + jj] + g[jj * q + ii]);
}

// U[r][i] <- sum_j Gh_ij U[r][j] for the rows r < n_valid of the live tasks, one (task, 32-row chunk) per item:
// the chunk is staged in shared memory, thread <-> column
constexpr int kFoldThreads = 128;
inline size_t qblock_fold_smem_bytes(int B_p) { return sizeof(double) * 32 * (size_t)B_p; }
__global__ void __launch_bounds__(kFoldThreads) scaml_qblock_fold_kernel(const QBlockVjpParams p) {
  SCAML_DYN_SMEM(double, sm);  // [32][B_p]
  const int tid = threadIdx.x, q = p.q, Bp = p.B_p;
  const int i = tid < p.B ? tid : p.B - 1;
  const int jb = (i / q) * q;
  double gh[kQMax];
#pragma unroll
  for (int j = 0; j < kQMax; ++j) gh[j] = (j < q) ? qblock_gsym(p.gcov, q, i, jb + j) : 0.0;
  const int nchunk = p.n_pad / 32;
  const long long items = (long long)p.M * nchunk;
  for (long long it = blockIdx.x; it < items; it += gridDim.x) {
    const int m = (int)(it / nchunk), ch = (int)(it - (long long)m * nchunk);
    const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
    if (p.w[m] == 0.0 || 32 * ch >= nv) continue;  // uniform over the CTA
    const int rows = nv - 32 * ch < 32 ? nv - 32 * ch : 32;
    double* src = p.U + ((size_t)m * p.n_pad + 32 * ch) * Bp;
    __syncthreads();  // previous chunk consumed
    for (int e = tid; e < rows * Bp; e += kFoldThreads) sm[e] = src[e];
    __syncthreads();
    if (tid < p.B) {
      for (int r = 0; r < rows; ++r) {
        double s = 0.0;
#pragma unroll
        for (int j = 0; j < kQMax; ++j)
          if (j < q) s = fma(gh[j], sm[r * Bp + jb + j], s);
        src[(size_t)r * Bp + tid] = s;
      }
    }
  }
}

// beta~[i][t] = sum_j Gh_ij beta[j][t]
__global__ void __launch_bounds__(128) scaml_qblock_fold_beta_kernel(const QBlockVjpParams p) {
  const int q = p.q, ntp = p.n_tp;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < (long long)p.B * ntp;
       e += (long long)gridDim.x * blockDim.x) {
    const int i = (int)(e / ntp), t = (int)(e - (long long)i * ntp), jb = (i / q) * q;
    double s = 0.0;
    for (int j = 0; j < q; ++j) s = fma(qblock_gsym(p.gcov, q, i, jb + j), p.beta[(size_t)(jb + j) * ntp + t], s);
    p.beta_f[e] = s;
  }
}

// dX_i = g_i dmean_i + dvar_i + 2 sum_{j != i} Gh_ij d_1[ sum_m c_m s_m kappa_m(x_i, x_j) + S^2 s_t kappa_t(x_i, x_j) ]:
// one warp per point, lane l takes the tasks l, l + 32, ... (fixed order), fixed-order warp tree per dimension
template <int KIND, int DMAX>
__global__ void __launch_bounds__(64) scaml_qblock_direct_kernel(const QBlockVjpParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, d = p.d, P = d + 2, q = p.q;
  const int wpg = blockDim.x >> 5;
  for (long long b = (long long)blockIdx.x * wpg + warp; b < p.B; b += (long long)gridDim.x * wpg) {
    const int i = (int)b, jb = (i / q) * q;
    double x[DMAX], acc[DMAX];
#pragma unroll
    for (int k = 0; k < DMAX; ++k) {
      x[k] = (k < d) ? p.Xc[(size_t)i * d + k] : 0.0;
      acc[k] = 0.0;
    }
    for (int m = lane; m < p.M; m += 32) {
      const double wm = p.w[m];
      if (wm == 0.0) continue;
      const double* th = p.theta + (size_t)m * P;
      const double cw = wm * p.ystd[m], cs = cw * cw * th[d];
      for (int j = jb; j < jb + q; ++j) {
        if (j == i) continue;
        double r2 = 0.0;
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
          if (k < d) {
            const double df = (x[k] - p.Xc[(size_t)j * d + k]) / th[k];
            r2 = fma(df, df, r2);
          }
        double kap, kd;
        kappa_pair<KIND>(r2, kap, kd);
        const double f = qblock_gsym(p.gcov, q, i, j) * cs * kd;
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
          if (k < d) acc[k] = fma(f, (x[k] - p.Xc[(size_t)j * d + k]) / (th[k] * th[k]), acc[k]);
      }
    }
#pragma unroll
    for (int k = 0; k < DMAX; ++k)
      if (k < d) acc[k] = warp_sum(acc[k]);
    if (lane == 0) {
      const double os = p.theta_t[d];
      for (int j = jb; j < jb + q; ++j) {
        if (j == i) continue;
        double r2 = 0.0;
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
          if (k < d) {
            const double df = (x[k] - p.Xc[(size_t)j * d + k]) / p.theta_t[k];
            r2 = fma(df, df, r2);
          }
        double kap, kd;
        switch (p.kernel_t) {
          case SCAML_KERNEL_RBF: kappa_pair<SCAML_KERNEL_RBF>(r2, kap, kd); break;
          case SCAML_KERNEL_MATERN12: kappa_pair<SCAML_KERNEL_MATERN12>(r2, kap, kd); break;
          case SCAML_KERNEL_MATERN32: kappa_pair<SCAML_KERNEL_MATERN32>(r2, kap, kd); break;
          default: kappa_pair<SCAML_KERNEL_MATERN52>(r2, kap, kd); break;
        }
        const double f = qblock_gsym(p.gcov, q, i, j) * p.s2t * os * kd;
#pragma unroll
        for (int k = 0; k < DMAX; ++k)
          if (k < d) acc[k] = fma(f, (x[k] - p.Xc[(size_t)j * d + k]) / (p.theta_t[k] * p.theta_t[k]), acc[k]);
      }
      // d kappa / dx_k = -kd (x_k - z_k) / l_k^2: the sign and the factor 2 go in here
      const double gm = p.gmean[i];
#pragma unroll
      for (int k = 0; k < DMAX; ++k)
        if (k < d)
          p.dX[(size_t)i * d + k] = fma(gm, p.dmean[(size_t)i * d + k], p.dvar[(size_t)i * d + k]) - 2.0 * acc[k];
    }
  }
}

inline int launch_qblock_cov(const QBlockCovParams& p, int kernel, int num_sms, void* stream) {
  const size_t smem = qblock_cov_smem_bytes(p.n_pad, p.d);
  if (smem > 227 * 1024) return SCAML_E_SMEM;
  const int grid = stride_grid(p.nsplit * p.ntile, 2 * num_sms);
  const int rc = dispatch_kind(kernel, [&](auto K) {
    return dispatch_dmax(p.d, [&](auto D) {
      return launch(scaml_qblock_cov_kernel<K.value, D.value>, grid, kQbThreads, smem, stream, p);
    });
  });
  if (rc) return rc;
  return launch(scaml_qblock_cov_finish_kernel, stride_grid(((long long)p.B * p.q + 127) / 128), 128, 0, stream, p);
}

// fold, then the q = 1 gradient path on the folded inputs (g.beta = beta~, g.dmean / g.dvar the intermediate
// outputs), then the direct terms and the combination
inline int launch_qblock_vjp(const QBlockVjpParams& p, GradParams g, int kernel, int num_sms, void* stream) {
  const long long fitems = (long long)p.M * (p.n_pad / 32);
  int rc = launch(scaml_qblock_fold_kernel, stride_grid(fitems, 4LL * num_sms), kFoldThreads,
                  qblock_fold_smem_bytes(p.B_p), stream, p);
  if (rc) return rc;
  if (p.n_t > 0) {
    rc = launch(scaml_qblock_fold_beta_kernel, stride_grid(((long long)p.B * p.n_tp + 127) / 128), 128, 0, stream, p);
    if (rc) return rc;
  }
  rc = launch_posterior_grad(g, kernel, num_sms, stream);
  if (rc) return rc;
  const int grid = stride_grid((p.B + 1) / 2);  // one warp per point, two per CTA
  return dispatch_kind(kernel, [&](auto K) {
    return dispatch_dmax(p.d, [&](auto D) {
      return launch(scaml_qblock_direct_kernel<K.value, D.value>, grid, 64, 0, stream, p);
    });
  });
}

}  // namespace scaml
