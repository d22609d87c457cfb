// Conditioning of the weighted source prior on the target data, at scale (rows a6/a8 of SURVEY 8a).
//
// The ScaML-GP posterior at a candidate x needs, next to the weighted prior mean / variance, the prior
// cross-covariance with the n_t target inputs (reference scamlgp/model.py:364-375: the eval-branch forward
// evaluates every source posterior at [X_t; x] jointly):
//     cross[x, j] = sum_m w_m^2 s_m^2 ( K_m(x, x_tj) - k*_m(x)^T K_m^-1 K_m(X_m, x_tj) ).
// With  A_m = K_m^-1 K_m(X_m, X_t)  (n x n_t, depends only on the fitted source GPs and X_t, i.e. it is computed
// once per `report`) the second term is  k*_m(x)^T A_m[:, j]  -- a contraction with the very k* tile the
// prediction kernel already holds in shared memory, so it is fused there (scaml_predict.cuh, CROSS = true) as
// extra DMMAs fed from k* (shared) and A_m (L2).  This file holds
//   scaml_cond_prepare_kernel : A_m = L_m^-T (L_m^-1 K_m(X_m, X_t)) for all tasks, both triangular products on
//                               the FP64 tensor cores, V = L^-1 K held in shared memory in place of K;
//   scaml_cond_combine_kernel : cross = sum_m c_m K_m(x, x_tj) - (sum over task splits of the fused partials).
// Before: scaml_predict_cross(reduce = 1) recomputed L^-1 K(X_m, X_t) for every 32-candidate tile and took 9x
// the time of the prior prediction (722 ms vs 80 ms for 4096 tasks x 4096 candidates).
#pragma once
#include <cstdlib>

#include "scaml_predict.cuh"

namespace scaml {

struct CondPrepParams {
  const double* X;
  const int32_t* n_valid;
  const double* theta;  // [M][P] constrained
  const double* linv;   // packed C-layout tiles
  const double* Xt;     // [n_t][d]
  const double* skip_w; // optional [M]: tasks with skip_w[m] == 0 are left untouched (pruned tasks)
  double* A;            // [M][n_pad][n_tp]
  int M, n_max, n_pad, d, n_t, n_tp, pw, npanel;
};

// shared memory (doubles): KV [n_pad][pw+4] | stage kPStages x 2 tiles | xst [d][n_pad] | xts [d][pw] | invl
inline size_t cond_prep_smem_bytes(int n_pad, int d, int pw) {
  return sizeof(double) * ((size_t)n_pad * (pw + 4) + (size_t)kPStages * 2 * kPTile + (size_t)d * n_pad +
                           (size_t)d * pw + kMaxP + 8);
}
// panel width: 8, 16, 32 or 64 columns (the kernel is instantiated per width) -- the narrowest that covers n_tp,
// else the widest that fits shared memory; columns of a panel beyond n_tp are zero columns that are not stored
inline int cond_panel_width(int n_pad, int d, int n_tp) {
  int want = 8;
  while (want < 64 && want < n_tp) want <<= 1;
  for (int pw = want; pw >= 8; pw >>= 1)
    if (cond_prep_smem_bytes(n_pad, d, pw) <= 227 * 1024) return pw;
  return 0;
}

// NJT = 8-column blocks per panel (1 .. 8), a template parameter: the products below issue one DMMA per column
// block, and a predicated-off DMMA (j >= njt at run time) would still hold the warp for its 16 issue cycles -- a
// 32-column panel ran at the speed of a 64-column one.
template <int KIND, int NJT>
__global__ void __launch_bounds__(kPredThreads, 1) scaml_cond_prepare_kernel(const CondPrepParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const int d = p.d, P = d + 2, n_pad = p.n_pad, pw = p.pw, ld = pw + 4;
  double* KV = sm;                                   // [n_pad][ld]: K(X_m, X_t panel), then V = L^-1 K in place
  double* stage = KV + (size_t)n_pad * ld;           // kPStages x 2 padded tiles
  double* xst = stage + kPStages * 2 * kPTile;       // [d][n_pad]
  double* xts = xst + (size_t)d * n_pad;             // [d][pw]
  double* invl = xts + (size_t)d * pw;               // [kMaxP]
  const long long lstride = (long long)tri(n_pad / kBS) * kTile;
  const int items = p.M * p.npanel;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int m = it / p.npanel, pn = it - m * p.npanel;
    if (p.skip_w != nullptr && p.skip_w[m] == 0.0) continue;  // uniform over the CTA
    const int j0 = pn * pw;
    constexpr int njt = NJT;  // 8-column blocks of a panel; the columns of a last, narrower panel beyond n_tp are
                              // zero columns of K (masked below) whose results are not stored
    const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
    const int NS = (nv + kSB - 1) / kSB, npt = NS * kSB, NB = 2 * NS;
    const double* th = p.theta + (size_t)m * P;
    const double os = th[d];
    const double* Lm = p.linv + (size_t)m * lstride;
    const double* Xm = p.X + (size_t)m * p.n_max * d;
    __syncthreads();
    if (tid < d) invl[tid] = 1.0 / th[tid];
    __syncthreads();
    for (int a = tid; a < npt; a += kPredThreads)
      for (int k = 0; k < d; ++k) xst[k * n_pad + a] = (a < nv) ? Xm[(size_t)a * d + k] * invl[k] : 0.0;
    for (int i = tid; i < pw * d; i += kPredThreads) {
      const int k = i / pw, j = i - k * pw;
      xts[i] = (j0 + j < p.n_t) ? p.Xt[(size_t)(j0 + j) * d + k] * invl[k] : 0.0;
    }
    __syncthreads();
    // ---- K(X_m, X_t panel): thread <-> column j of the panel, rows in phases, 8 interleaved exp chains -------- //
    {
      constexpr int PW = 8 * NJT, QN = kPredThreads / PW, U = 8;
      const int j = tid % PW, q = tid / PW;
      const bool jin = (j0 + j < p.n_t);
      for (int a0 = q; a0 < npt; a0 += QN * U) {
        double r2[U];
#pragma unroll
        for (int u = 0; u < U; ++u) r2[u] = 0.0;
        for (int k = 0; k < d; ++k) {
          const double xt = xts[k * pw + j];
          const double* xr = xst + k * n_pad + a0;
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const double df = ((a0 + u * QN < npt) ? xr[u * QN] : 0.0) - xt;  // QN U > 64 for narrow panels
            r2[u] = fma(df, df, r2[u]);
          }
        }
        double kap[U];
        kappa_n<KIND, U, false>(r2, kap, kap);
#pragma unroll
        for (int u = 0; u < U; ++u) {
          const int a = a0 + u * QN;
          if (a < npt) KV[(size_t)a * ld + j] = (a < nv && jin) ? os * kap[u] : 0.0;
        }
      }
    }
    __syncthreads();
    // ---- pass 1: V = L^-1 K, super-rows bottom-up so that V_I can overwrite the rows of K it no longer needs -- //
    {
      const int rb = warp >> 2, ib = warp & 3;  // this warp: rows 32 rb + 8 ib + {0..7} of the super-row
      // flat chunk list: I = NS-1 .. 0, ck = 0 .. 2I+1
      const int L = NS * (NS + 1);
      int iI = NS - 1, ick = 0, issued = 0;
      auto issue_one = [&]() {
        if (issued < L) {
          pred_issue(Lm, PChunk{iI, ick}, stage + (issued % kPStages) * 2 * kPTile, tid);
          if (++ick > 2 * iI + 1) {
            --iI;
            ick = 0;
          }
          ++issued;
        }
        cp_async_commit();
      };
      issue_one();
      issue_one();
      int q = 0;
      for (int I = NS - 1; I >= 0; --I) {
        double acc[8][2];
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j][0] = acc[j][1] = 0.0;
        const int brow = 2 * I + rb;
        for (int ck = 0; ck <= 2 * I + 1; ++ck, ++q) {
          cp_async_wait<1>();
          __syncthreads();
          issue_one();
          if (ck <= brow) {
            const bool dg = (ck == brow);
            const double* ar = stage + ((q % kPStages) * 2 + rb) * kPTile + t4 * kPLd + 8 * ib + g;
            const double* br = KV + (size_t)(32 * ck + t4) * ld + g;
#pragma unroll
            for (int s = 0; s < 8; ++s) {
              if (!dg || s < 2 * ib + 2) {  // diagonal tile: L^-1(r, kk) = 0 for kk > r
                const double a = ar[0];
#pragma unroll
                for (int j = 0; j < 8; ++j)
                  if (j < njt) dmma884(acc[j], a, br[8 * j]);
              }
              ar += 4 * kPLd;
              br += 4 * ld;
            }
          }
        }
        __syncthreads();  // every warp has finished reading the K rows of this super-row
        {
          double* vr = KV + (size_t)(64 * I + 32 * rb + 8 * ib + g) * ld + 2 * t4;
#pragma unroll
          for (int j = 0; j < 8; ++j)
            if (j < njt) *reinterpret_cast<double2*>(vr + 8 * j) = make_double2(acc[j][0], acc[j][1]);
        }
      }
      cp_async_wait<0>();
      __syncthreads();  // V complete
    }
    // ---- pass 2: A = L^-T V, 32-row blocks top-down; tile (rbk, ab) is read transposed from its staged copy -- //
    {
      const int ib = warp & 3, jpar = warp >> 2;  // rows 8 ib + {0..7} of the block, column blocks j = jpar, jpar+2, ..
      const int L2 = (NB * (NB + 1)) / 2;
      int iab = 0, irb = 0, issued = 0;
      auto issue_one = [&]() {
        if (issued < L2) {
          ptile_async(stage + (issued % kPStages) * 2 * kPTile, Lm + (size_t)(tri(irb) + iab) * kTile, tid);
          if (++irb >= NB) {
            ++iab;
            irb = iab;
          }
          ++issued;
        }
        cp_async_commit();
      };
      issue_one();
      issue_one();
      int q = 0;
      for (int ab = 0; ab < NB; ++ab) {
        double acc[4][2];
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[j][0] = acc[j][1] = 0.0;
        for (int rbk = ab; rbk < NB; ++rbk, ++q) {
          cp_async_wait<1>();
          __syncthreads();
          issue_one();
          const bool dg = (rbk == ab);
          // staged tile: row c (= column a of L^-1), entries r: A_op[a][r] = L^-1(r, a) = staged[a * kPLd + r]
          const double* ar = stage + (q % kPStages) * 2 * kPTile + (8 * ib + g) * kPLd + t4;
          const double* br = KV + (size_t)(32 * rbk + t4) * ld + 8 * jpar + g;
#pragma unroll
          for (int s = 0; s < 8; ++s) {
            if (!dg || s >= 2 * ib) {  // diagonal tile: L^-1(r, a) = 0 for r < a
              const double a = ar[4 * s];
#pragma unroll
              for (int j = 0; j < (NJT + 1) / 2; ++j)
                if (NJT % 2 == 0 || jpar + 2 * j < njt) dmma884(acc[j], a, br[16 * j]);
            }
            br += 4 * ld;
          }
        }
        {
          const int a = 32 * ab + 8 * ib + g;
          double* dst = p.A + ((size_t)m * n_pad + a) * p.n_tp + j0 + 2 * t4;
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (jpar + 2 * j < njt && j0 + 8 * (jpar + 2 * j) < p.n_tp)
              *reinterpret_cast<double2*>(dst + 8 * (jpar + 2 * j)) = make_double2(acc[j][0], acc[j][1]);
        }
      }
      cp_async_wait<0>();
    }
  }
}

// cross[b][j] = sum_m c_m os_m kappa_m(x_b, x_tj) - sum_s cxp[s][b][j],  c_m = w_m^2 ystd_m^2 (tasks with w = 0 skipped)
// With few (candidate, target) pairs the sum over the M tasks is split over `ntsplit` CTAs per pair block (partials in
// dpart, summed in a fixed order by scaml_cond_combine_finish_kernel): at 64 candidates x 32 target points the
// unsplit kernel ran on 8 CTAs and took 1.4 ms for 4096 tasks -- half of a small-batch posterior call.
struct CondCombineParams {
  const double* theta;
  const double* ystd;
  const double* w;
  const double* Xc;   // [B][d]
  const double* Xt;   // [n_t][d]
  const double* cxp;  // [nsplit][B][n_tp]
  double* cross;      // [B][n_t]
  double* dpart;      // [ntsplit][B][n_t] (ntsplit > 1)
  int M, d, B, n_t, n_tp, nsplit, ntsplit;
};

constexpr int kCombTasks = 32;
inline int comb_ntsplit(int M, int B, int n_t, int num_sms) {
  const long long nblk = ((long long)B * n_t + 255) / 256;
  long long ns = (2LL * num_sms) / nblk;
  const long long cap = (M + 4 * kCombTasks - 1) / (4 * kCombTasks);  // at least 128 tasks per split
  if (ns > cap) ns = cap;
  if (const char* env = getenv("SCAML_COMB_TSPLIT")) {  // test knob: force the split path at tiny sizes
    const int v = atoi(env);
    if (v >= 1) ns = v < M ? v : M;
  }
  return ns < 1 ? 1 : (int)ns;
}
inline size_t comb_dpart_doubles(int M, int B, int n_t, int num_sms) {
  const int ns = comb_ntsplit(M, B, n_t, num_sms);
  return ns > 1 ? (size_t)ns * (size_t)B * (size_t)n_t : 0;
}

template <int KIND>
__global__ void __launch_bounds__(256) scaml_cond_combine_kernel(const CondCombineParams p) {
  SCAML_DYN_SMEM(double, sm);  // coef [32] | invl [32][d]
  double* coef = sm;
  double* invl = sm + kCombTasks;
  const int d = p.d, P = d + 2;
  const long long pairs = (long long)p.B * p.n_t;
  const long long nblk = (pairs + blockDim.x - 1) / blockDim.x;
  for (long long item = blockIdx.x; item < nblk * p.ntsplit; item += gridDim.x) {
    const int ts = (int)(item / nblk);
    const long long pr = (item - (long long)ts * nblk) * blockDim.x + threadIdx.x;
    const int m_lo = (int)((long long)p.M * ts / p.ntsplit), m_hi = (int)((long long)p.M * (ts + 1) / p.ntsplit);
    const bool live = pr < pairs;
    const int b = live ? (int)(pr / p.n_t) : 0, j = live ? (int)(pr - (long long)b * p.n_t) : 0;
    double dx[kMaxP];
    for (int k = 0; k < d; ++k) dx[k] = p.Xc[(size_t)b * d + k] - p.Xt[(size_t)j * d + k];
    double acc = 0.0;
    for (int m0 = m_lo; m0 < m_hi; m0 += kCombTasks) {
      __syncthreads();
      for (int i = threadIdx.x; i < kCombTasks * (d + 1); i += blockDim.x) {
        const int mm = i / (d + 1), k = i - mm * (d + 1), m = m0 + mm;
        if (m < m_hi) {
          const double* th = p.theta + (size_t)m * P;
          if (k == d) {
            const double wy = p.w[m] * p.ystd[m];
            coef[mm] = wy * wy * th[d];
          } else {
            invl[mm * d + k] = 1.0 / th[k];
          }
        } else if (k == d) {
          coef[mm] = 0.0;
        } else {
          invl[mm * d + k] = 0.0;
        }
      }
      __syncthreads();
      for (int mm = 0; mm < kCombTasks; mm += 4) {
        double r2[4];
#pragma unroll
        for (int u = 0; u < 4; ++u) {
          double s = 0.0;
          for (int k = 0; k < d; ++k) {
            const double v = dx[k] * invl[(mm + u) * d + k];
            s = fma(v, v, s);
          }
          r2[u] = s;
        }
        double kap[4];
        kappa_n<KIND, 4, false>(r2, kap, kap);
#pragma unroll
        for (int u = 0; u < 4; ++u) acc = fma(coef[mm + u], kap[u], acc);  // coef = 0 for pruned / padded tasks
      }
    }
    if (live) {
      if (p.ntsplit > 1) {
        p.dpart[(size_t)ts * pairs + pr] = acc;
      } else {
        double sub = 0.0;
        for (int s = 0; s < p.nsplit; ++s) sub += p.cxp[((size_t)s * p.B + b) * p.n_tp + j];
        p.cross[(size_t)b * p.n_t + j] = acc - sub;
      }
    }
  }
}

// ntsplit > 1: cross = (sum of the task-split partials, fixed order) - (sum of the fused partials, fixed order)
__global__ void __launch_bounds__(256) scaml_cond_combine_finish_kernel(const CondCombineParams p) {
  const long long pairs = (long long)p.B * p.n_t;
  for (long long pr = (long long)blockIdx.x * blockDim.x + threadIdx.x; pr < pairs; pr += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(pr / p.n_t), j = (int)(pr - (long long)b * p.n_t);
    double acc = 0.0, sub = 0.0;
    for (int t = 0; t < p.ntsplit; ++t) acc += p.dpart[(size_t)t * pairs + pr];
    for (int s = 0; s < p.nsplit; ++s) sub += p.cxp[((size_t)s * p.B + b) * p.n_tp + j];
    p.cross[(size_t)b * p.n_t + j] = acc - sub;
  }
}

// Per-task caches of ScaMLGP.__init__ (reference scamlgp/model.py:278-289) from A_m:
//   source_means[t][m]    = ybar_m + ystd_m  K_m(x_t, X_m) alpha_m
//   source_covs[t][t'][m] = ystd_m^2 ( K_m(x_t, x_t') - K_m(x_t, X_m) A_m[:, t'] )
// One CTA per task walks X_m in 32-row chunks: K chunk and A chunk in shared memory, the n_t x n_t accumulator
// tile in shared memory as well (every thread owns its entries: no races, fixed order).
struct CondCachesParams {
  const double* X;
  const int32_t* n_valid;
  const double* theta;
  const double* alpha;  // [M][n_pad]
  const double* ybar;
  const double* ystd;
  const double* Xt;   // [n_t][d]
  const double* A;    // [M][n_pad][n_tp]
  double* mean;       // [n_t][M]
  double* cov;        // [n_t][n_t][M]
  int M, n_max, n_pad, d, n_t, n_tp;
};
// shared memory (doubles): acc [n_t][n_t] | macc [n_t] | Kc [32][n_tp+1] | Ac [32][n_tp] | alc [32] | xts [d][n_tp] | invl
inline size_t cond_caches_smem_bytes(int d, int n_t, int n_tp) {
  return sizeof(double) * ((size_t)n_t * n_t + n_t + 32 * (size_t)(n_tp + 1) + 32 * (size_t)n_tp + 32 +
                           (size_t)d * n_tp + kMaxP + 8);
}

template <int KIND>
__global__ void __launch_bounds__(256) scaml_cond_caches_kernel(const CondCachesParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, d = p.d, P = d + 2, nt = p.n_t, ntp = p.n_tp, ldk = ntp + 1;
  double* acc = sm;                        // [nt][nt]
  double* macc = acc + (size_t)nt * nt;    // [nt]
  double* Kc = macc + nt;                  // [32][ldk]
  double* Ac = Kc + 32 * (size_t)ldk;      // [32][ntp]
  double* alc = Ac + 32 * (size_t)ntp;     // [32]
  double* xts = alc + 32;                  // [d][ntp]
  double* invl = xts + (size_t)d * ntp;    // [kMaxP]
  for (int m = blockIdx.x; m < p.M; m += gridDim.x) {
    const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
    const double* th = p.theta + (size_t)m * P;
    const double os = th[d], ys = p.ystd[m];
    const double* Xm = p.X + (size_t)m * p.n_max * d;
    __syncthreads();
    if (tid < d) invl[tid] = 1.0 / th[tid];
    for (int i = tid; i < nt * nt + nt; i += 256) acc[i] = 0.0;  // acc and macc are contiguous
    __syncthreads();
    for (int i = tid; i < d * ntp; i += 256) {
      const int k = i / ntp, j = i - k * ntp;
      xts[i] = (j < nt) ? p.Xt[(size_t)j * d + k] * invl[k] : 0.0;
    }
    for (int a0 = 0; a0 < nv; a0 += 32) {
      __syncthreads();
      for (int i = tid; i < 32 * ntp; i += 256) {
        const int r = i / ntp, j = i - r * ntp, a = a0 + r;
        double kv = 0.0;
        if (a < nv && j < nt) {
          double r2 = 0.0;
          for (int k = 0; k < d; ++k) {
            const double df = Xm[(size_t)a * d + k] * invl[k] - xts[k * ntp + j];
            r2 = fma(df, df, r2);
          }
          kv = os * kappa_of<KIND>(r2);
        }
        Kc[r * ldk + j] = kv;
        Ac[i] = (a < nv) ? p.A[((size_t)m * p.n_pad + a) * ntp + j] : 0.0;
      }
      if (tid < 32) alc[tid] = (a0 + tid < nv) ? p.alpha[(size_t)m * p.n_pad + a0 + tid] : 0.0;
      __syncthreads();
      for (int e = tid; e < nt * nt; e += 256) {
        const int t = e / nt, u = e - t * nt;
        double s = acc[e];
#pragma unroll 8
        for (int r = 0; r < 32; ++r) s = fma(Kc[r * ldk + t], Ac[r * ntp + u], s);
        acc[e] = s;
      }
      if (tid < nt) {
        double s = macc[tid];
        for (int r = 0; r < 32; ++r) s = fma(Kc[r * ldk + tid], alc[r], s);
        macc[tid] = s;
      }
    }
    __syncthreads();
    for (int e = tid; e < nt * nt; e += 256) {
      const int t = e / nt, u = e - t * nt;
      double r2 = 0.0;
      for (int k = 0; k < d; ++k) {
        const double df = xts[k * ntp + t] - xts[k * ntp + u];
        r2 = fma(df, df, r2);
      }
      p.cov[(size_t)e * p.M + m] = ys * ys * (os * kappa_of<KIND>(r2) - acc[e]);
    }
    if (tid < nt) p.mean[(size_t)tid * p.M + m] = p.ybar[m] + ys * macc[tid];
  }
}

inline int launch_cond_caches(CondCachesParams p, int kernel, int num_sms, void* stream) {
  p.n_tp = cond_ntp(p.n_t);
  const size_t smem = cond_caches_smem_bytes(p.d, p.n_t, p.n_tp);
  if (smem > 227 * 1024) return SCAML_E_SMEM;
  const int grid = p.M < 2 * num_sms ? p.M : 2 * num_sms;
  return dispatch_kind(kernel, [&](auto K) {
    return launch(scaml_cond_caches_kernel<K.value>, grid, 256, smem, stream, p);
  });
}

inline int launch_cond_prepare(CondPrepParams p, int kernel, int num_sms, void* stream) {
  p.n_tp = cond_ntp(p.n_t);
  p.pw = cond_panel_width(p.n_pad, p.d, p.n_tp);
  if (p.pw == 0) return SCAML_E_SMEM;
  p.npanel = (p.n_tp + p.pw - 1) / p.pw;
  const size_t smem = cond_prep_smem_bytes(p.n_pad, p.d, p.pw);
  long long items = (long long)p.M * p.npanel;
  int grid = (int)(items < num_sms ? items : num_sms);
  return dispatch_kind(kernel, [&](auto K) {
    switch (p.pw) {
      case 8: return launch(scaml_cond_prepare_kernel<K.value, 1>, grid, kPredThreads, smem, stream, p);
      case 16: return launch(scaml_cond_prepare_kernel<K.value, 2>, grid, kPredThreads, smem, stream, p);
      case 32: return launch(scaml_cond_prepare_kernel<K.value, 4>, grid, kPredThreads, smem, stream, p);
      default: return launch(scaml_cond_prepare_kernel<K.value, 8>, grid, kPredThreads, smem, stream, p);
    }
  });
}

inline int launch_cond_combine(const CondCombineParams& p, int kernel, void* stream) {
  const size_t smem = sizeof(double) * kCombTasks * (p.d + 1);
  const long long blocks = (p.B * (long long)p.n_t + 255) / 256;
  const int rc = dispatch_kind(kernel, [&](auto K) {
    return launch(scaml_cond_combine_kernel<K.value>, stride_grid(blocks * p.ntsplit, 148 * 8), 256, smem, stream, p);
  });
  if (rc || p.ntsplit <= 1) return rc;
  return launch(scaml_cond_combine_finish_kernel, stride_grid(blocks, 148 * 8), 256, 0, stream, p);
}

}  // namespace scaml
