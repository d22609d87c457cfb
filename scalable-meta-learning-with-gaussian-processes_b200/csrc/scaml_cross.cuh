// Source-GP posterior cross-covariances (K6/K7 with q > 1):
//   mean_m(A),   Sigma_m(A, B) = ystd_m^2 ( K_m(A,B) - V_m(A)^T V_m(B) ),   V_m(.) = L_m^-1 K_m(X_m, .)
// for point sets A (nA) and B (nB), either per task (reduce = 0: the `source_means` /
// `source_covs` caches of ScaMLGP.__init__, reference scamlgp/model.py:278-289) or reduced over
// the tasks with the ScaML-GP weights (reduce = 1: sum_m w_m mean_m, sum_m w_m^2 Sigma_m -- the
// joint-prior blocks that ScaMLGP.forward builds in eval mode, model.py:364-375, 108-135).
//
// One 128-thread CTA owns a 32 x 32 tile of (A, B) points.  Per task it builds k(X_m, A) and
// k(X_m, B) once in shared memory, streams the packed L^-1 tiles (cp.async, double buffered
// half tiles) through the DMMA micro-kernel of the fit to get V(A), V(B) one 64-row slab at a
// time, and accumulates G = V(A)^T V(B) with DMMA as well.  Reductions are in fixed order.
#pragma once
#include "scaml_device.cuh"
#include "scaml_fit.cuh"

namespace scaml {

constexpr int kCT = 32;  // points per tile side

struct CrossParams {
  const double* X;
  const int32_t* n_valid;
  const double* theta;  // [M][P] constrained
  const double* linv;   // packed C-layout tiles
  const double* alpha;  // [M][n_pad]
  const double* ybar;
  const double* ystd;
  const double* w;  // [M] (reduce = 1) or null
  const double* XA;  // [nA][d]
  const double* XB;  // [nB][d]
  double* mean;      // reduce ? [nA] : [nA][M]
  double* cov;       // reduce ? [nA][nB] : [nA][nB][M]
  double* part;      // reduce && nsplit > 1: [nsplit][nA*nB + nA]
  int M, n_max, n_pad, d, nA, nB, reduce, nsplit, tilesA, tilesB;
};

inline size_t cross_smem_bytes(int n_pad, int d) {
  const int NB = n_pad / kBS;
  return sizeof(double) * ((size_t)2 * NB * kTileS + 4 * kHalfS + 4 * kTileS + (size_t)n_pad + 2 * (size_t)d * kCT +
                           2 * (size_t)d * kCT + 256 + 8);
}
inline int cross_nsplit(int M, int tiles, int num_sms) {
  int ns = (num_sms + tiles - 1) / tiles;
  if (ns < 1) ns = 1;
  if (ns > M) ns = M;
  return ns;
}

// o(16x16 quadrant of a 32x32 product) += sum_kk A[kk][r] * B[kk][c], kk over one padded 32-row tile
SCAML_DEVICE void small_gemm_acc(SAcc& o, const double* A, const double* B, const FThr& t) {
  const double* ar = A + t.t4 * kLd + 16 * (t.warp >> 1) + t.g;
  const double* br = B + t.t4 * kLd + 16 * (t.warp & 1) + t.g;
#pragma unroll 4
  for (int s = 0; s < 8; ++s) {
    const double a0 = ar[0], a1 = ar[8], b0 = br[0], b1 = br[8];
    ar += 4 * kLd;
    br += 4 * kLd;
    dmma884(o[0][0], a0, b0);
    dmma884(o[0][1], a0, b1);
    dmma884(o[1][0], a1, b0);
    dmma884(o[1][1], a1, b1);
  }
}

template <int KIND>
__global__ void __launch_bounds__(kFitThreads, 1) scaml_cross_kernel(const CrossParams p) {
  SCAML_DYN_SMEM(double, sm);
  const FThr t = make_fthr();
  const int d = p.d, P = d + 2, n_pad = p.n_pad, NBmax = n_pad / kBS;
  double* KA = sm;                        // NBmax padded tiles [a][c]
  double* KB = KA + (size_t)NBmax * kTileS;
  double* LS = KB + (size_t)NBmax * kTileS;  // 2 stages x 2 padded half tiles
  double* VA = LS + 4 * kHalfS;           // 2 padded tiles (rows of the slab = kk)
  double* VB = VA + 2 * kTileS;
  double* alp = VB + 2 * kTileS;          // n_pad
  double* xr = alp + n_pad;               // raw points [side][d][32]
  double* xsx = xr + 2 * d * kCT;         // scaled points [side][d][32]
  double* red = xsx + 2 * d * kCT;        // 256
  const long long lstride = (long long)tri(NBmax) * kTile;
  const int tiles = p.tilesA * p.tilesB;
  const int items = p.reduce ? tiles * p.nsplit : tiles * p.M;
  const int mper = (p.M + p.nsplit - 1) / p.nsplit;
  // this thread's element of the 32x32 output: quadrant (warp>>1, warp&1), rows 8i+g, cols 8j+2*t4+e
  const int qr = 16 * (t.warp >> 1) + t.g, qc = 16 * (t.warp & 1) + 2 * t.t4;

  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int tile = it % tiles, rest = it / tiles;
    const int ta = tile / p.tilesB, tb = tile % p.tilesB;
    const int a0 = ta * kCT, b0 = tb * kCT;
    const int m_lo = p.reduce ? rest * mper : rest;
    const int m_hi = p.reduce ? ((m_lo + mper < p.M) ? m_lo + mper : p.M) : rest + 1;
    __syncthreads();
    for (int i = t.tid; i < 2 * d * kCT; i += kFitThreads) {
      const int side = i / (d * kCT), r = i - side * d * kCT, k = r / kCT, c = r - k * kCT;
      const int gp = (side == 0 ? a0 : b0) + c, np = side == 0 ? p.nA : p.nB;
      const double* src = side == 0 ? p.XA : p.XB;
      xr[i] = (gp < np) ? src[(size_t)gp * d + k] : 0.0;
    }
    SAcc csum;
#pragma unroll
    for (int i = 0; i < 2; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j) csum[i][j][0] = csum[i][j][1] = 0.0;
    double msum = 0.0;

    for (int m = m_lo; m < m_hi; ++m) {
      const double wm = p.reduce ? p.w[m] : 1.0;
      if (p.reduce && wm == 0.0) continue;
      const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
      const int NS = (nv + kSB - 1) / kSB, npt = NS * kSB;
      const double* th = p.theta + (size_t)m * P;
      const double os = th[d], ys = p.ystd[m];
      const double* Xm = p.X + (size_t)m * p.n_max * d;
      __syncthreads();
      for (int i = t.tid; i < npt; i += kFitThreads) alp[i] = p.alpha[(size_t)m * n_pad + i];
      for (int i = t.tid; i < 2 * d * kCT; i += kFitThreads) {
        const int k = (i / kCT) % d;
        xsx[i] = xr[i] / th[k];
      }
      __syncthreads();
      // ---- k(X_m, A), k(X_m, B) into shared memory + mean partials ------------------- //
      {
        const int c = t.tid & 31, side = (t.tid >> 5) & 1, aq = t.tid >> 6;
        double* Kd = side == 0 ? KA : KB;
        const double* xp = xsx + side * d * kCT + c;
        double mu = 0.0;
        for (int a = aq; a < npt; a += 2) {
          double r2 = 0.0;
          if (a < nv)
            for (int k = 0; k < d; ++k) {
              const double df = __ldg(Xm + (size_t)a * d + k) / th[k] - xp[k * kCT];
              r2 = fma(df, df, r2);
            }
          const double kv = (a < nv) ? os * kappa_of<KIND>(r2) : 0.0;
          Kd[(a >> 5) * kTileS + (a & 31) * kLd + c] = kv;
          mu = fma(kv, alp[a], mu);
        }
        red[t.tid] = mu;  // [aq][side][c]
      }
      __syncthreads();
      // ---- slabs of V(A), V(B) and G += V(A)^T V(B) ---------------------------------- //
      const double* Lm = p.linv + (size_t)m * lstride;
      SAcc gacc;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j) gacc[i][j][0] = gacc[i][j][1] = 0.0;
      const int side = t.warp >> 1, rb = t.warp & 1;  // this warp: V(side) rows 32*rb.. of the slab
      const double* Ksrc = side == 0 ? KA : KB;
      for (int I = 0; I < NS; ++I) {
        Acc acc;
        facc_zero(acc);
        const int n = 2 * (2 * I + 2);  // sub-chunks (16 deep) over tiles kb = 0 .. 2I+1
        auto issue = [&](int s, double* st) {
          const int kb = s >> 1, off = (s & 1) * kHalfG;
          if (kb <= 2 * I) half_async(st, Lm + (size_t)(tri(2 * I) + kb) * kTile + off, t.tid);
          half_async(st + kHalfS, Lm + (size_t)(tri(2 * I + 1) + kb) * kTile + off, t.tid);
          cp_async_commit();
        };
        issue(0, LS);
        for (int s = 0; s < n; ++s) {
          double* st = LS + (s & 1) * 2 * kHalfS;
          if (s + 1 < n) {
            issue(s + 1, LS + ((s + 1) & 1) * 2 * kHalfS);
            cp_async_wait<1>();
          } else {
            cp_async_wait<0>();
          }
          __syncthreads();
          const int kb = s >> 1;
          if (kb <= 2 * I + rb) {
            // only the first two column tiles (j = 0..3 covers 32 columns): acc[i][j] full 32x32
            fmma<4>(acc, st + rb * kHalfS, Ksrc + (size_t)kb * kTileS + (s & 1) * kHalfS, t, false);
          }
          __syncthreads();
        }
        // slab -> shared (row-major: rows of the slab are the contraction index of G)
        store_tile_R((side == 0 ? VA : VB) + rb * kTileS, kLd, acc, t, 1.0);
        __syncthreads();
        small_gemm_acc(gacc, VA, VB, t);
        small_gemm_acc(gacc, VA + kTileS, VB + kTileS, t);
        __syncthreads();
      }
      // ---- epilogue: Sigma(A,B) quadrant, means ------------------------------------- //
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int ca = qr + 8 * i, cb = qc + 8 * j + e;
            double r2 = 0.0;
            for (int k = 0; k < d; ++k) {
              const double df = xsx[k * kCT + ca] - xsx[d * kCT + k * kCT + cb];
              r2 = fma(df, df, r2);
            }
            const double cv = ys * ys * (os * kappa_of<KIND>(r2) - gacc[i][j][e]);
            if (p.reduce) {
              csum[i][j][e] = fma(wm * wm, cv, csum[i][j][e]);
            } else if (a0 + ca < p.nA && b0 + cb < p.nB) {
              p.cov[((size_t)(a0 + ca) * p.nB + (b0 + cb)) * p.M + m] = cv;
            }
          }
      if (t.tid < kCT && tb == 0) {
        const double mu = red[t.tid] + red[64 + t.tid];  // side 0, both a-halves
        const double mv = p.ybar[m] + ys * mu;
        if (p.reduce)
          msum = fma(wm, mv, msum);
        else if (a0 + t.tid < p.nA)
          p.mean[(size_t)(a0 + t.tid) * p.M + m] = mv;
      }
    }
    if (p.reduce) {
      double* cdst = p.nsplit == 1 ? p.cov : p.part + (size_t)rest * ((size_t)p.nA * p.nB + p.nA);
      double* mdst = p.nsplit == 1 ? p.mean : cdst + (size_t)p.nA * p.nB;
#pragma unroll
      for (int i = 0; i < 2; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int ca = a0 + qr + 8 * i, cb = b0 + qc + 8 * j + e;
            if (ca < p.nA && cb < p.nB) cdst[(size_t)ca * p.nB + cb] = csum[i][j][e];
          }
      if (t.tid < kCT && tb == 0 && a0 + t.tid < p.nA) mdst[a0 + t.tid] = msum;
    }
  }
}

__global__ void scaml_cross_reduce_kernel(const double* part, double* cov, double* mean, int nsplit, long long ncov,
                                          int nA) {
  const long long tot = ncov + nA;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < tot; i += (long long)gridDim.x * blockDim.x) {
    double s = 0.0;
    for (int k = 0; k < nsplit; ++k) s += part[(size_t)k * tot + i];
    if (i < ncov)
      cov[i] = s;
    else
      mean[i - ncov] = s;
  }
}

inline size_t cross_workspace_bytes(int M, int nA, int nB, int reduce, int num_sms) {
  if (!reduce) return 0;
  const int tiles = ((nA + kCT - 1) / kCT) * ((nB + kCT - 1) / kCT);
  const int ns = cross_nsplit(M, tiles, num_sms);
  return ns > 1 ? sizeof(double) * (size_t)ns * ((size_t)nA * nB + nA) : 0;
}

inline int launch_predict_cross(const double* X, const int32_t* n_valid, const double* theta, const double* linv,
                                const double* alpha, const double* ybar, const double* ystd, const double* w,
                                const double* XA, const double* XB, double* mean, double* cov, double* workspace, int M,
                                int n_max, int n_pad, int d, int nA, int nB, int kernel, int reduce, int num_sms,
                                void* stream) {
  CrossParams p;
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.linv = linv, p.alpha = alpha, p.ybar = ybar, p.ystd = ystd, p.w = w;
  p.XA = XA, p.XB = XB, p.mean = mean, p.cov = cov, p.part = workspace;
  p.M = M, p.n_max = n_max, p.n_pad = n_pad, p.d = d, p.nA = nA, p.nB = nB, p.reduce = reduce;
  p.tilesA = (nA + kCT - 1) / kCT, p.tilesB = (nB + kCT - 1) / kCT;
  const int tiles = p.tilesA * p.tilesB;
  p.nsplit = reduce ? cross_nsplit(M, tiles, num_sms) : 1;
  const size_t smem = cross_smem_bytes(n_pad, d);
  if (smem > 227 * 1024) return SCAML_E_SMEM;
  long long items = reduce ? (long long)tiles * p.nsplit : (long long)tiles * M;
  long long cap = 4LL * num_sms;
  int grid = (int)(items < cap ? items : cap);
  const int rc = dispatch_kind(kernel, [&](auto K) {
    return launch(scaml_cross_kernel<K.value>, grid, kFitThreads, smem, stream, p);
  });
  if (rc != 0 || !reduce || p.nsplit == 1) return rc;
  const long long ncov = (long long)nA * nB;
  return launch(scaml_cross_reduce_kernel, stride_grid((ncov + nA + 255) / 256, 1184), 256, 0, stream, workspace, cov,
                mean, p.nsplit, ncov, nA);
}

}  // namespace scaml
