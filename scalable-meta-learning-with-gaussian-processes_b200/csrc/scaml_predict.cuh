// Weighted ScaML-GP prediction (K6-K9): for a tile of CT (64 or 32) candidates a CTA walks over the
// tasks of its split.  Per task it
// (1) builds k*(X_m, candidates) once in shared memory (padded k-major 32x32 tiles) together with the
//     mean partials k*^T alpha.  The squared distances come from the FP64 tensor cores as well:
//     r^2 = |a|^2 + |c|^2 - 2 a.c on inputs centred on the task's first point and length-scaled (the
//     quadratic expansion gpytorch itself evaluates, SURVEY A.4), i.e. the accumulator is initialised
//     with |a|^2 + |c|^2 and one DMMA per four input dimensions adds -2 a.c for an 8 x 8 block of
//     pairs: 1/64 + 1 FP64 instructions per pair instead of 3 d (load, subtract, fma per dimension),
//     which was what bound the assembly (issue slots, not the pipe).  Matern-1/2 keeps direct
//     differences (exp(-r) is not smooth in r^2 at coincident points).
// (2) streams the packed L_m^-1 tiles and forms V = L^-1 k* on the FP64 tensor cores (mma.sync
//     m8n8k4 -> DMMA).  The 8 warps work as TWO independent groups of 4 (named barriers, own 3-stage
//     cp.async ring each); group 0 owns the 32-row blocks 0, 3, 4, 7, ... of L^-1 and group 1 the blocks
//     1, 2, 5, 6, ... -- row block r has r + 1 tiles, so both groups stream the same number of tiles
//     (n_pad = 256: 18 each) where the former lock-step walk over (2I, 2I+1) pairs left the warps of the
//     even blocks idle one step in every super-row; the zero half of the diagonal tiles is skipped.
// (3) folds  w_m (ybar_m + ystd_m k*^T alpha_m)  and  w_m^2 ystd_m^2 (s_m - ||V||^2)  into
//     per-candidate accumulators that stay in registers for the whole task loop -> the reduction over
//     tasks happens inside the kernel in a fixed order (deterministic, no atomics).
// Reference: _compute_target_prior, scamlgp/model.py:108-135; posterior A.7 of SURVEY.md.
#pragma once
#ifdef SCAML_PRED_PROF
#include <cstdio>
#endif
#include "scaml_device.cuh"

namespace scaml {

constexpr int kPLd = 36;               // padded row stride of a staged tile (conflict-free DMMA fragment loads)
constexpr int kPTile = kBS * kPLd;     // 1152 doubles
constexpr int kPStages = 3;
constexpr int kPredThreads = 256;
constexpr int kPGroupThreads = 128;  // one product group = 4 warps

struct PredParams {
  const double* X;
  const int32_t* n_valid;
  const double* theta;  // [M][P] constrained
  const double* linv;   // packed C-layout tiles
  const double* alpha;  // [M][n_pad]
  const double* ybar;
  const double* ystd;
  const double* w;
  const double* Xc;  // [B][d]
  double* mean;
  double* var;
  double* part;  // [nsplit][2][B] when nsplit > 1
  int M, n_max, n_pad, d, B, nsplit, ntile, ct, alias;
  // CROSS variant (conditioning on target data, see scaml_cond.cuh)
  const double* condA;  // [M][n_pad][n_tp]  A_m = K_m^-1 K_m(X_m, X_t)
  double* cxp;          // [nsplit][B][n_tp] partials of sum_m c_m k*_m^T A_m
  int n_tp;
};

// shared memory (doubles): kst | rings | [auxA = xst] [auxB = xcs] | alp | xcr | red | vsq | invl, ctr (x2)
// xst / xcs hold d + 2 rows (the scaled coordinates, then 1 | |a|^2 resp. |c|^2 | 1: the operand rows that put the
// squared norms of r^2 = |a|^2 + |c|^2 - 2 a.c into the same tensor-core product) with strides n_pad + 4 / ct + 4
// (== 4 mod 16 doubles: the DMMA fragment loads of the distance product are bank-conflict free).  The per-task
// staging data is dead once k* is assembled, so it may share memory with the L^-1 rings (6 padded tiles, laid out
// [g0 s0 | g0 s1 | g1 s0 | g1 s1 | g0 s2 | g1 s2]):
//   alias 0  own memory
//   alias 1  auxA on the two third-stage slots, which the pipeline does not touch before the product loop: the
//            first two tiles of each group still stream in under the assembly
//   alias 2  auxA and auxB on the rings; streaming starts after the assembly
constexpr int kPAliasA = 2 * kPTile;
#ifdef SCAML_EMU
inline
#else
__host__ __device__ inline
#endif
size_t predict_auxA_doubles(int n_pad, int d) { return (size_t)(d + 2) * (n_pad + 4); }
#ifdef SCAML_EMU
inline
#else
__host__ __device__ inline
#endif
size_t predict_auxB_doubles(int d, int ct) { return (size_t)(d + 2) * (ct + 4); }
inline size_t predict_smem_bytes(int n_pad, int d, int ct, int alias) {
  const size_t kst = (size_t)(n_pad / kBS) * (ct / kBS) * kPTile;
  const size_t stage = (size_t)kPStages * 2 * kPTile;
  const size_t aux = (alias == 0 ? predict_auxA_doubles(n_pad, d) : 0) + (alias <= 1 ? predict_auxB_doubles(d, ct) : 0);
  return sizeof(double) * (kst + stage + aux + (size_t)n_pad + (size_t)d * ct + 4 * ct + 2 * ct + 4 * kMaxP + 8);
}
// candidate tile width / layout for (n_pad, d): widest tile that fits 227 KB, least aliasing first
inline bool predict_config(int n_pad, int d, int* ct, int* alias) {
  for (int c = 64; c >= 32; c -= 32)
    for (int a = 0; a <= 2; ++a) {
      if (a == 1 && predict_auxA_doubles(n_pad, d) > (size_t)kPAliasA) continue;
      if (a == 2 && predict_auxA_doubles(n_pad, d) + predict_auxB_doubles(d, c) > (size_t)kPStages * 2 * kPTile) continue;
      if (predict_smem_bytes(n_pad, d, c, a) <= 227 * 1024) {
        *ct = c, *alias = a;
        return true;
      }
    }
  return false;
}
inline int predict_nsplit(int M, int B, int num_sms, int ct) {
  const int ntile = (B + ct - 1) / ct;
  int ns = (2 * num_sms + ntile - 1) / ntile;
  if (ns < 1) ns = 1;
  if (ns > M) ns = M;
  return ns;
}
inline size_t predict_workspace_bytes(int M, int n_pad, int d, int B, int num_sms) {
  int ct = 64, alias = 0;
  if (!predict_config(n_pad, d, &ct, &alias)) return 0;
  const int ns = predict_nsplit(M, B, num_sms, ct);
  return ns > 1 ? sizeof(double) * 2 * (size_t)ns * (size_t)B : 0;
}

// one dense 32x32 tile (8 KB, contiguous) global -> padded shared rows: 2 x 16 B per thread (256 threads)
SCAML_DEVICE void ptile_async(double* sdst, const double* gsrc, int tid) {
#pragma unroll
  for (int u = 0; u < 2; ++u) {
    const int c2 = tid + u * kPredThreads;
    const int row = c2 >> 4, j = c2 & 15;
    cp_async16(sdst + row * kPLd + 2 * j, gsrc + row * kBS + 2 * j);
  }
}

// flat chunk q of a task: super-row I, 32-wide column block ck (0 .. 2I+1)
struct PChunk {
  int I, ck;
  SCAML_DEVICE void next() {
    if (++ck > 2 * I + 1) {
      ++I;
      ck = 0;
    }
  }
};
SCAML_DEVICE void pred_issue(const double* Lm, const PChunk& c, double* st, int tid) {
  if (c.ck <= 2 * c.I) ptile_async(st, Lm + (size_t)(tri(2 * c.I) + c.ck) * kTile, tid);
  ptile_async(st + kPTile, Lm + (size_t)(tri(2 * c.I + 1) + c.ck) * kTile, tid);
}

// ---- the prediction kernel's two product groups ---------------------------------------------------------- //
// barrier over the 4 warps of group gi (hardware barrier 1 + gi; barrier 0 is __syncthreads)
SCAML_DEVICE void group_sync(int gi) {
#ifdef SCAML_EMU
  cuemu::named_sync(1 + gi);
#else
  if (gi == 0) asm volatile("bar.sync 1, %0;\n" ::"n"(kPGroupThreads) : "memory");
  else asm volatile("bar.sync 2, %0;\n" ::"n"(kPGroupThreads) : "memory");
#endif
}
// ring slot s of group gi: [g0 s0 | g0 s1 | g1 s0 | g1 s1 | g0 s2 | g1 s2]
SCAML_DEVICE double* gslot(double* stage, int gi, int s) {
  return stage + (s < 2 ? 2 * gi + s : 4 + gi) * kPTile;
}
// one dense tile global -> padded shared rows by the 128 threads of a group: 4 x 16 B per thread
SCAML_DEVICE void gtile_async(double* sdst, const double* gsrc, int gtid) {
#pragma unroll
  for (int u = 0; u < 4; ++u) {
    const int c2 = gtid + u * kPGroupThreads;
    const int row = c2 >> 4, j = c2 & 15;
    cp_async16(sdst + row * kPLd + 2 * j, gsrc + row * kBS + 2 * j);
  }
}
// walk of a group over its row blocks: group 0: r = 0, 3, 4, 7, ..; group 1: r = 1, 2, 5, 6, ..; tiles ck = 0 .. r
struct GChunk {
  int r, ck;
  SCAML_DEVICE void next() {
    if (++ck > r) {
      r += (r & 1) ? 1 : 3;
      ck = 0;
    }
  }
};
SCAML_DEVICE int group_tiles(int gi, int nb) {
  int L = 0;
  for (int r = gi; r < nb; r += (r & 1) ? 1 : 3) L += r + 1;
  return L;
}

#ifdef SCAML_PRED_PROF  // diagnostics build: per-phase clock64 totals of CTA 0, printed by the kernel
#define PPROF(ph)                                  \
  do {                                             \
    if (threadIdx.x == PPROF_TID) {                \
      const long long now_ = clock64();            \
      pprof[ph] += now_ - pprof_last;              \
      pprof_last = now_;                           \
    }                                              \
  } while (0)
#ifndef PPROF_TID
#define PPROF_TID 0
#endif
#else
#define PPROF(ph) \
  do {            \
  } while (0)
#endif

template <int KIND, int CT, bool CROSS>
__global__ void __launch_bounds__(kPredThreads, 1) scaml_predict_kernel(const PredParams p) {
#ifdef SCAML_PRED_PROF
  long long pprof[8] = {0, 0, 0, 0, 0, 0, 0, 0};
  long long pprof_last = clock64();
#endif
  constexpr int NJ = CT / 32;   // 8-column DMMA tiles per warp in the product (warp tile: 32 rows x 8*NJ candidates)
  constexpr int CBT = CT / 32;  // kst tile columns
  constexpr int CS = CT + 4;    // row stride of the scaled candidates
  constexpr int QN = kPredThreads / CT;  // row phases of the thread <-> candidate passes (4 for CT = 64, 8 for CT = 32)
  // Matern-1/2 assembles k* from direct differences (thread <-> candidate), everything else through the tensor cores
  constexpr bool kDirect = (KIND == SCAML_KERNEL_MATERN12);
  // RBF: the tensor-core product delivers the ARGUMENT of the exponential, log(s) - r^2 / 2, directly -- operand scales
  // (a . c instead of -2 a . c, norms times -1/2) and log(outputscale) in the norm row of the task's points -- so the
  // exponential IS the scaled kernel value: no multiply by -1/2, none by the outputscale, and the rows beyond n_valid
  // get -1e4 there (exp -> 3e-308, whose square underflows to 0) instead of a select per pair
  constexpr bool kArg = (KIND == SCAML_KERNEL_RBF);
  constexpr double kCs = kArg ? 1.0 : -2.0, kNs = kArg ? -0.5 : 1.0;
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const int gi = warp >> 2, gtid = tid & (kPGroupThreads - 1);  // product group, thread index inside it
  const int col0 = (warp & 3) * 8 * NJ, cb = col0 >> 5, cin = col0 & 31;
  const int d = p.d, P = d + 2, n_pad = p.n_pad, dp = (d + 3) & ~3, XS = n_pad + 4;
  // the two norm rows ride in the padding of the contraction when there is room (d = 6: rows 6, 7 of 8); otherwise
  // the accumulators are initialised with |a|^2 + |c|^2 (one FP64 add per pair, no extra DMMA)
  const bool aug = (((d + 2) + 3) & ~3) == dp;
  const int dk = aug ? d + 2 : d;
  double* kst = sm;                                                // (n_pad/32) x CBT padded tiles [a][c]
  double* stage = kst + (size_t)(n_pad / kBS) * CBT * kPTile;      // 2 groups x kPStages padded tiles
  double* own = stage + kPStages * 2 * kPTile;                     // un-aliased staging data, then alp ..
  const size_t nA = predict_auxA_doubles(n_pad, d), nB = predict_auxB_doubles(d, CT);
  double* xst = (p.alias == 0) ? own : ((p.alias == 1) ? stage + 4 * kPTile : stage);  // [d+2][XS]
  double* xcs = (p.alias == 0) ? own + nA : ((p.alias == 1) ? own : xst + nA);        // [d+2][CS]
  double* alp = own + (p.alias == 0 ? nA : 0) + (p.alias <= 1 ? nB : 0);              // [n_pad]
  double* xcr = alp + n_pad;                                       // [d][CT] raw candidates
  double* red = xcr + d * CT;                                      // 4 x CT mean partials
  double* vsq = red + 4 * CT;                                      // 2 x CT
  double* invl2 = vsq + 2 * CT;                                    // 2 x (kMaxP reciprocal lengthscales | kMaxP centre)
  const double* nrm = xst + (size_t)(d + 1) * XS;                  // |a|^2 (row d + 1 of xst)
  const double* ncs = xcs + (size_t)d * CS;                        // |c|^2 (row d of xcs)
  int tcount = 0;
  const long long lstride = (long long)tri(n_pad / kBS) * kTile;
  const int items = p.ntile * p.nsplit;
  const int mper = (p.M + p.nsplit - 1) / p.nsplit;

  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int ct = it % p.ntile, spx = it / p.ntile;
    const int b0 = ct * CT;
    const int m_lo = spx * mper, m_hi = (m_lo + mper < p.M) ? m_lo + mper : p.M;
    __syncthreads();
    for (int i = tid; i < CT * d; i += kPredThreads) {
      const int c = i / d, k = i - c * d;
      xcr[k * CT + c] = (b0 + c < p.B) ? p.Xc[(size_t)(b0 + c) * d + k] : 0.0;
    }
    double macc = 0.0, vacc = 0.0;
    // CROSS: cx[i][jj] = 8x8 block (candidates 32 xt + 8 i + .., target columns 8 (jw + JS jj) + ..) of
    // sum_m c_m k*_m^T A_m, accumulated over ALL tasks of the split by the tensor cores.  CT = 64: the warp's
    // candidate tile column xt = warp & 1 and column blocks jw = warp >> 1, +4, ..; CT = 32: xt = 0, jw = warp, +8, ..
    constexpr int JS = (CT == 64) ? 4 : 8;
    const int xt = (CT == 64) ? (warp & 1) : 0, jw = (CT == 64) ? (warp >> 1) : warp;
    double cx[CROSS ? 4 : 1][CROSS ? 4 : 1][2];
#pragma unroll
    for (int i = 0; i < (CROSS ? 4 : 1); ++i)
#pragma unroll
      for (int jj = 0; jj < (CROSS ? 4 : 1); ++jj) cx[i][jj][0] = cx[i][jj][1] = 0.0;
    // Everything the NEXT task needs from global memory before its tiles -- its scalars, lengthscales, centre, point
    // `tid` (first kPreD dimensions) and alpha -- is fetched into registers while the tensor-core phase of the
    // current task runs, so that neither the task prologue nor the staging waits on L2
    constexpr int kPreD = 8;
    int pre_m = -1, nv_n = 0;
    double xpre[kPreD], apre = 0.0, wm_n = 0.0, os_n = 0.0, ys_n = 0.0, yb_n = 0.0, th_n = 1.0, ctr_n = 0.0;
#pragma unroll
    for (int k = 0; k < kPreD; ++k) xpre[k] = 0.0;
    for (int m = m_lo; m < m_hi; ++m) {
      const bool have = (pre_m == m);
      const double wm = have ? wm_n : p.w[m];
      if (wm == 0.0) continue;
      const int nv = have ? nv_n : (p.n_valid ? p.n_valid[m] : p.n_max);
      const int NS = (nv + kSB - 1) / kSB, npt = NS * kSB, nb = 2 * NS;
      const int L = group_tiles(gi, nb);  // tiles this group streams for this task
      const double* th = p.theta + (size_t)m * P;
      const double os = have ? os_n : th[d];
      const double ys = have ? ys_n : p.ystd[m], yb = have ? yb_n : p.ybar[m];
      const double* Lm = p.linv + (size_t)m * lstride;
      const double* Xm = p.X + (size_t)m * p.n_max * d;
      // x * (1/l) instead of x / l: an FP64 division is ~30 instructions per staged coordinate (<= 1 ulp apart)
      double* invl = invl2 + (tcount & 1) * 2 * kMaxP;
      double* ctr = invl + kMaxP;  // centre of the expansion: the task's first point (any point would do)
      ++tcount;
      if (tid < d) {
        invl[tid] = 1.0 / (have ? th_n : th[tid]);
        ctr[tid] = have ? ctr_n : Xm[tid];
      }
      const double nadd = kArg ? log(os) : 0.0;  // uniform; the norm row below carries it into every argument
      __syncthreads();  // previous task fully consumed (kst, stage, aux); invl, ctr visible
      PPROF(0);
      GChunk qi{gi, 0};
      int issued = 0;
      // start streaming L^-1 under the exp-heavy assembly below (always two commits: the wait<1> accounting of
      // the product loop needs them even when the group has a single tile)
      auto issue_first_two = [&]() {
#pragma unroll
        for (int u = 0; u < 2; ++u) {
          if (issued < L) {
            gtile_async(gslot(stage, gi, issued % kPStages), Lm + (size_t)(tri(qi.r) + qi.ck) * kTile, gtid);
            ++issued;
            qi.next();
          }
          cp_async_commit();
        }
      };
      if (p.alias <= 1) issue_first_two();
      {
        if (tid < npt) {  // one point per thread: no runtime integer division
          double nn = 0.0;
#pragma unroll
          for (int k = 0; k < kPreD; ++k)
            if (k < d) {
              const double x = have ? xpre[k] : ((tid < nv) ? Xm[(size_t)tid * d + k] : 0.0);
              const double v = (tid < nv) ? (x - ctr[k]) * invl[k] : 0.0;
              xst[k * XS + tid] = v;
              nn = fma(v, v, nn);
            }
          for (int k = kPreD; k < d; ++k) {
            const double v = (tid < nv) ? (Xm[(size_t)tid * d + k] - ctr[k]) * invl[k] : 0.0;
            xst[k * XS + tid] = v;
            nn = fma(v, v, nn);
          }
          xst[d * XS + tid] = 1.0;
          xst[(d + 1) * XS + tid] = (kArg && tid >= nv) ? -1e4 : fma(kNs, nn, nadd);
          alp[tid] = have ? apre : p.alpha[(size_t)m * n_pad + tid];
        }
        for (int a = tid + kPredThreads; a < npt; a += kPredThreads) {
          double nn = 0.0;
          for (int k = 0; k < d; ++k) {
            const double v = (a < nv) ? (Xm[(size_t)a * d + k] - ctr[k]) * invl[k] : 0.0;
            xst[k * XS + a] = v;
            nn = fma(v, v, nn);
          }
          xst[d * XS + a] = 1.0;
          xst[(d + 1) * XS + a] = (kArg && a >= nv) ? -1e4 : fma(kNs, nn, nadd);
          alp[a] = p.alpha[(size_t)m * n_pad + a];
        }
        if (tid < 4 * CT) {  // candidate c = tid / 4, dimensions k = tid % 4, + 4, ..; |c|^2 by a fixed-order quad sum
          const int c = tid >> 2;
          double nn = 0.0;
          for (int k = tid & 3; k < d; k += 4) {
            const double v = (xcr[k * CT + c] - ctr[k]) * invl[k];
            xcs[k * CS + c] = kCs * v;
            nn = fma(v, v, nn);
          }
          nn += __shfl_xor_sync(0xffffffffu, nn, 1);
          nn += __shfl_xor_sync(0xffffffffu, nn, 2);
          if ((tid & 3) == 0) {
            xcs[d * CS + c] = kNs * nn;
            xcs[(d + 1) * CS + c] = 1.0;
          }
        }
      }
      __syncthreads();
      PPROF(1);
      // ---- k*(X_m, candidates) and the mean partials k*^T alpha ------------------------- //
      // every thread leaves the assembly with one or two folded partials (mu_lo, mu_hi) for columns red_col (+1) and a
      // row of red[4][CT]: half of the threads store before the barrier, the other half add after it
      double mu_lo = 0.0, mu_hi = 0.0;
      int red_col = 0, red_row = 0, red_n = 1;
      bool red_store = false, red_add = false;
      if (kDirect) {
        // a thread owns one candidate and walks the task's points 8 at a time: 8 independent distance / exp
        // chains per thread keep the FP64 pipe busy (a single chain per thread is latency bound).
        constexpr int U = 8;
        static_assert(QN * U <= 64, "assembly pass must not run past the task's rows");
        const int c = tid % CT, q = tid / CT;
        double mu = 0.0;
        for (int a0 = q; a0 < npt; a0 += QN * U) {
          double r2[U];
#pragma unroll
          for (int u = 0; u < U; ++u) r2[u] = 0.0;
          for (int k = 0; k < d; ++k) {
            const double xc = -0.5 * xcs[k * CS + c];  // kDirect is a Matern kernel: scale -2
            const double* xr = xst + k * XS + a0;
#pragma unroll
            for (int u = 0; u < U; ++u) {
              const double df = xr[u * QN] - xc;
              r2[u] = fma(df, df, r2[u]);
            }
          }
          double kap[U];
          kappa_n<KIND, U, false>(r2, kap, kap);
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int a = a0 + u * QN;
            const double kv = ((a < nv) ? os : 0.0) * kap[u];
            kst[((a >> 5) * CBT + (c >> 5)) * kPTile + (a & 31) * kPLd + (c & 31)] = kv;
            mu = fma(kv, alp[a], mu);
          }
        }
        // fold the QN phases into red[4][CT] in a fixed order: phases 4..7 store before the barrier, 0..3 add after it
        mu_lo = mu, red_col = c;
        red_store = (QN == 4 || q >= 4), red_add = (QN > 4 && q < 4), red_n = 1;
        red_row = q & 3;
      } else {
        // warp <-> 32-row block of the task (rbk = warp, warp + 8, ..); per (row block, 32-candidate half, RI 8-row
        // groups) the lane holds the DMMA accumulator fragments of 8 RI pairs: rows 8 i2 + g, candidates 8 j + 2 t4 + e.
        // Operand rows beyond dk (the contraction is padded to a multiple of 4) are selected to zero.
        constexpr int RI = CROSS ? 1 : 2;  // CROSS keeps 32 more accumulators live: shorter exp batches
        double mu[CBT * 8];  // [h][j][e] -> 8 h + 2 j + e : sum over this lane's rows of k* alpha
#pragma unroll
        for (int v = 0; v < CBT * 8; ++v) mu[v] = 0.0;
        for (int rbk = warp; rbk < nb; rbk += 8) {
#pragma unroll
          for (int h = 0; h < CBT; ++h) {
            double nc[4][2];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
              const double2 v = *reinterpret_cast<const double2*>(ncs + 32 * h + 8 * j + 2 * t4);
              nc[j][0] = aug ? 0.0 : v.x, nc[j][1] = aug ? 0.0 : v.y;
            }
            const double* bq = xcs + t4 * CS + 32 * h + g;
#pragma unroll
            for (int ip = 0; ip < 4 / RI; ++ip) {
              const int arow = 32 * rbk + 8 * RI * ip + g;  // + 8 i2
              double r2[8 * RI];  // [i2][j][e] -> 8 i2 + 2 j + e
#pragma unroll
              for (int i2 = 0; i2 < RI; ++i2) {
                const double na = aug ? 0.0 : nrm[arow + 8 * i2];
#pragma unroll
                for (int j = 0; j < 4; ++j) r2[8 * i2 + 2 * j] = na + nc[j][0], r2[8 * i2 + 2 * j + 1] = na + nc[j][1];
              }
              const double* aq = xst + t4 * XS + arow;
              for (int ks = 0; ks < dp; ks += 4) {
                const bool kin = (ks + t4 < dk);
                double a[RI], b[4];
#pragma unroll
                for (int i2 = 0; i2 < RI; ++i2) a[i2] = kin ? aq[ks * XS + 8 * i2] : 0.0;
#pragma unroll
                for (int j = 0; j < 4; ++j) b[j] = kin ? bq[ks * CS + 8 * j] : 0.0;
#pragma unroll
                for (int i2 = 0; i2 < RI; ++i2)
#pragma unroll
                  for (int j = 0; j < 4; ++j) dmma884s(r2[8 * i2 + 2 * j], r2[8 * i2 + 2 * j + 1], a[i2], b[j]);
              }
              // cancellation may leave r^2 = -1e-16 where gpytorch clamps to 0: exp(+5e-17) rounds to 1 all the
              // same, and the Matern kernels clamp r^2 to >= 1e-30 themselves (an FP64 max is 7 instructions)
              if (kArg) exp_nonpos_n<8 * RI>(r2, r2);  // r2 holds log(s) - r^2 / 2 (<= log s; the exp takes small positive arguments)
              else kappa_n<KIND, 8 * RI, false>(r2, r2, r2);
              double* kt = kst + (size_t)(rbk * CBT + h) * kPTile + (8 * RI * ip + g) * kPLd + 2 * t4;
#pragma unroll
              for (int i2 = 0; i2 < RI; ++i2) {
                const double osa = (arow + 8 * i2 < nv) ? os : 0.0, al = alp[arow + 8 * i2];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                  const double k0 = kArg ? r2[8 * i2 + 2 * j] : osa * r2[8 * i2 + 2 * j];
                  const double k1 = kArg ? r2[8 * i2 + 2 * j + 1] : osa * r2[8 * i2 + 2 * j + 1];
                  *reinterpret_cast<double2*>(kt + 8 * i2 * kPLd + 8 * j) = make_double2(k0, k1);
                  mu[8 * h + 2 * j] = fma(k0, al, mu[8 * h + 2 * j]);
                  mu[8 * h + 2 * j + 1] = fma(k1, al, mu[8 * h + 2 * j + 1]);
                }
              }
            }
          }
        }
        // sum over the 8 row groups g (lane bits 2..4) by a halving butterfly: in every round a lane hands one half of
        // its values to the partner and keeps the sums of the other half -- 8 + 4 + 2 shuffles (CT = 64) instead of
        // 3 per value, a fixed pairwise order.  CT = 64 ends with columns 2 lane, 2 lane + 1 in the lane.
        {
          constexpr int NV = CBT * 8;
          const bool b4 = (lane & 16) != 0, b3 = (lane & 8) != 0, b2 = (lane & 4) != 0;
          double s1[NV / 2];
#pragma unroll
          for (int v = 0; v < NV / 2; ++v) {
            const double give = b4 ? mu[v] : mu[v + NV / 2], keep = b4 ? mu[v + NV / 2] : mu[v];
            s1[v] = keep + __shfl_xor_sync(0xffffffffu, give, 16);
          }
          double s2[NV / 4];
#pragma unroll
          for (int v = 0; v < NV / 4; ++v) {
            const double give = b3 ? s1[v] : s1[v + NV / 4], keep = b3 ? s1[v + NV / 4] : s1[v];
            s2[v] = keep + __shfl_xor_sync(0xffffffffu, give, 8);
          }
          double s3[NV / 8];
#pragma unroll
          for (int v = 0; v < NV / 8; ++v) {
            const double give = b2 ? s2[v] : s2[v + NV / 8], keep = b2 ? s2[v + NV / 8] : s2[v];
            s3[v] = keep + __shfl_xor_sync(0xffffffffu, give, 4);
          }
          // value index bits, most significant first, were chosen by lane bits 4, 3, 2
          if (CT == 64) {  // index = (h, j1, j0, e): h = b4, j = 2 b3 + b2, e = 0, 1 left -> columns 8 g + 2 t4 + e
            mu_lo = s3[0], mu_hi = s3[NV / 8 - 1], red_n = 2, red_col = 2 * lane;
          } else {         // index = (j1, j0, e): j = 2 b4 + b3, e = b2
            mu_lo = s3[0], red_n = 1, red_col = 8 * (2 * (int)b4 + (int)b3) + 2 * t4 + (int)b2;
          }
          red_store = (warp >= 4), red_add = (warp < 4), red_row = warp & 3;
        }
      }
      if (red_store) {
        red[red_row * CT + red_col] = mu_lo;
        if (red_n == 2) red[red_row * CT + red_col + 1] = mu_hi;
      }
      PPROF(2);
      __syncthreads();
      PPROF(3);
      if (p.alias == 2) issue_first_two();  // the staging data on the rings is dead (barrier above)
      if (red_add) {
        red[red_row * CT + red_col] += mu_lo;
        if (red_n == 2) red[red_row * CT + red_col + 1] += mu_hi;
      }
      if (CROSS) {
        // cx += (c_m k*)^T A_m : A-operand = k* (shared, this warp's 32-candidate tile column), B-operand = A_m.
        // A_m streams through the two third-stage ring slots -- idle until the product loop -- as [32 rows of one row
        // block] x [W = 8 JS target columns] tiles (row stride W + 4), double-buffered when two fit (W = 32), fetched
        // with cp.async by the whole CTA; in a tile every warp owns ONE 8-column block (jw) and the accumulator set
        // jj = column chunk.  (Round 1 read the B fragments straight from L2 with one item of register prefetch:
        // latency bound, 27 k cycles per task and candidate tile against 8 k of DMMA work.)
        constexpr int W = 8 * JS, LDW = W + 4, NBUF = (2 * kPTile) / (32 * LDW);
        static_assert(NBUF >= 1, "a CROSS tile must fit the two spare ring slots");
        double* xbuf = stage + 4 * kPTile;
        const int njt = p.n_tp >> 3;
        const int nchunk = (p.n_tp + W - 1) / W, nitems = nb * nchunk;
        const double cm = wm * wm * ys * ys;
        const double* Am = p.condA + (size_t)m * n_pad * p.n_tp;
        auto issue_item = [&](int item) {
          const int rbk = item / nchunk, c = item - rbk * nchunk;
          double* dst = xbuf + (NBUF == 2 ? (item & 1) : 0) * 32 * LDW;
          const double* src = Am + (size_t)(32 * rbk) * p.n_tp + W * c;
#pragma unroll
          for (int u = 0; u < (16 * W) / kPredThreads; ++u) {
            const int pc = tid + u * kPredThreads;
            const int row = pc / (W / 2), j2 = pc - row * (W / 2);
            if (W * c + 2 * j2 < p.n_tp) cp_async16(dst + row * LDW + 2 * j2, src + (size_t)row * p.n_tp + 2 * j2);
          }
          cp_async_commit();
        };
        const double* ks = kst + (size_t)xt * kPTile + t4 * kPLd + g;
        if (nitems > 0) issue_item(0);
        for (int item = 0; item < nitems; ++item) {
          cp_async_wait<0>();
          __syncthreads();  // tile `item` visible; every warp has finished the tile before it
          if (NBUF == 2 && item + 1 < nitems) issue_item(item + 1);
          const int rbk = item / nchunk, jj = item - rbk * nchunk;
          if (jw + JS * jj < njt) {
            const double* kr = ks + (size_t)rbk * CBT * kPTile;
            const double* br = xbuf + (NBUF == 2 ? (item & 1) : 0) * 32 * LDW + t4 * LDW + 8 * jw + g;
            // jj is warp-uniform but not a compile-time constant, and the accumulators must be indexed statically to
            // stay in registers: one copy of the loop per set behind a uniform branch.  (Selecting the set by
            // predicate inside ONE loop issued 16 DMMAs per step, 12 of them predicated off -- and a predicated-off
            // DMMA still holds the warp for its 16 issue cycles: the fused cross-covariance ran at a quarter of
            // the tensor-core rate.)
#define SCAML_CX_LOOP(Q)                                                  \
  _Pragma("unroll") for (int s = 0; s < 8; ++s) {                         \
    const double a[4] = {kr[0], kr[8], kr[16], kr[24]};                   \
    const double b = cm * br[0];                                          \
    kr += 4 * kPLd;                                                       \
    br += 4 * LDW;                                                        \
    _Pragma("unroll") for (int i = 0; i < 4; ++i) dmma884(cx[i][Q], a[i], b); \
  }
            if (jj == 0) {
              SCAML_CX_LOOP(0)
            } else if (jj == 1) {
              SCAML_CX_LOOP(1)
            } else if (jj == 2) {
              SCAML_CX_LOOP(2)
            } else {
              SCAML_CX_LOOP(3)
            }
#undef SCAML_CX_LOOP
          }
          if (NBUF == 1 && item + 1 < nitems) {
            __syncthreads();
            issue_item(item + 1);
          }
        }
        __syncthreads();  // the spare slots go back to the product groups
      }
      if (m + 1 < m_hi) {  // prefetch for the next task (lands during the product below)
        pre_m = m + 1;
        const double* th1 = p.theta + (size_t)(m + 1) * P;
        const double* X1 = p.X + (size_t)(m + 1) * p.n_max * d;
        wm_n = p.w[m + 1];
        nv_n = p.n_valid ? p.n_valid[m + 1] : p.n_max;
        os_n = th1[d];
        ys_n = p.ystd[m + 1];
        yb_n = p.ybar[m + 1];
        if (tid < d) {
          th_n = th1[tid];
          ctr_n = X1[tid];
        }
        // rows beyond the next task's n_valid are never used (staging masks them): no dependence on nv_n here
#pragma unroll
        for (int k = 0; k < kPreD; ++k) xpre[k] = (k < d && tid < p.n_max) ? X1[(size_t)tid * d + k] : 0.0;
        apre = (tid < n_pad) ? p.alpha[(size_t)(m + 1) * n_pad + tid] : 0.0;
      }
      // ---- V = L^-1 k*  on the FP64 tensor cores, column sums of squares ------------- //
      double acc[4][NJ][2];
      double vs[NJ][2];
#pragma unroll
      for (int j = 0; j < NJ; ++j) vs[j][0] = vs[j][1] = 0.0;
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < NJ; ++j) acc[i][j][0] = acc[i][j][1] = 0.0;
      GChunk qc{gi, 0};
      PPROF(4);
      for (int q = 0; q < L; ++q) {
        cp_async_wait<1>();
        group_sync(gi);  // tile q visible to the group; the group has finished reading tile q-1
        if (issued < L) {
          gtile_async(gslot(stage, gi, issued % kPStages), Lm + (size_t)(tri(qi.r) + qi.ck) * kTile, gtid);
          ++issued;
          qi.next();
        }
        cp_async_commit();  // always commit (possibly empty): keeps the wait<1> accounting uniform
        const bool dg = (qc.ck == qc.r);  // diagonal tile: L^-1(r, kk) = 0 for kk > r
        {
          const double* ar = gslot(stage, gi, q % kPStages) + t4 * kPLd + g;
          const double* br = kst + (qc.ck * CBT + cb) * kPTile + t4 * kPLd + cin + g;
#pragma unroll
          for (int s = 0; s < 8; ++s) {
            const double a[4] = {ar[0], ar[8], ar[16], ar[24]};
            double b[NJ];
#pragma unroll
            for (int j = 0; j < NJ; ++j) b[j] = br[8 * j];
            ar += 4 * kPLd;
            br += 4 * kPLd;
#pragma unroll
            for (int i = 0; i < 4; ++i)
              if (!dg || s < 2 * i + 2) {
#pragma unroll
                for (int j = 0; j < NJ; ++j) dmma884(acc[i][j], a[i], b[j]);
              }
          }
        }
        if (dg) {  // row block complete: ||V_r||^2 per candidate column
#pragma unroll
          for (int j = 0; j < NJ; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
#pragma unroll
              for (int i = 0; i < 4; ++i) {
                vs[j][e] = fma(acc[i][j][e], acc[i][j][e], vs[j][e]);
                acc[i][j][e] = 0.0;
              }
            }
        }
        qc.next();
      }
      cp_async_wait<0>();
      PPROF(5);
#pragma unroll
      for (int j = 0; j < NJ; ++j)
#pragma unroll
        for (int e = 0; e < 2; ++e) {
          double s = vs[j][e];
          s += __shfl_xor_sync(0xffffffffu, s, 4);
          s += __shfl_xor_sync(0xffffffffu, s, 8);
          s += __shfl_xor_sync(0xffffffffu, s, 16);
          if (g == 0) vsq[gi * CT + col0 + 8 * j + 2 * t4 + e] = s;
        }
      __syncthreads();
      if (tid < CT) {
        const double mu = ((red[tid] + red[CT + tid]) + red[2 * CT + tid]) + red[3 * CT + tid];
        const double ssq = vsq[tid] + vsq[CT + tid];
        macc = fma(wm, yb + ys * mu, macc);
        vacc = fma(wm * wm * ys * ys, os - ssq, vacc);
      }
      PPROF(6);
    }
    if (CROSS) {
      const int njt = p.n_tp >> 3;
      double* dst = p.cxp + (size_t)spx * p.B * p.n_tp;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int b = b0 + 32 * xt + 8 * i + g;
        if (b < p.B) {
#pragma unroll
          for (int jj = 0; jj < 4; ++jj)
            if (jw + JS * jj < njt)
              *reinterpret_cast<double2*>(dst + (size_t)b * p.n_tp + 8 * (jw + JS * jj) + 2 * t4) =
                  make_double2(cx[i][jj][0], cx[i][jj][1]);
        }
      }
    }
    if (tid < CT && b0 + tid < p.B) {
      if (p.nsplit == 1) {
        p.mean[b0 + tid] = macc;
        p.var[b0 + tid] = vacc;
      } else {
        p.part[((size_t)spx * 2 + 0) * p.B + b0 + tid] = macc;
        p.part[((size_t)spx * 2 + 1) * p.B + b0 + tid] = vacc;
      }
    }
  }
#ifdef SCAML_PRED_PROF
  if (blockIdx.x == 0 && threadIdx.x == PPROF_TID)
    printf("pprof tid %d: top %lld staging %lld assembly %lld asmbar %lld mean+prefetch %lld product %lld tail %lld\n",
           (int)threadIdx.x, pprof[0], pprof[1], pprof[2], pprof[3], pprof[4], pprof[5], pprof[6]);
#endif
}

__global__ void scaml_predict_reduce_kernel(const double* part, double* mean, double* var, int nsplit, int B) {
  for (int b = blockIdx.x * blockDim.x + threadIdx.x; b < B; b += gridDim.x * blockDim.x) {
    double m = 0.0, v = 0.0;
    for (int s = 0; s < nsplit; ++s) {
      m += part[((size_t)s * 2 + 0) * B + b];
      v += part[((size_t)s * 2 + 1) * B + b];
    }
    mean[b] = m;
    var[b] = v;
  }
}

// many splits (few candidates): one warp per candidate, lanes stride over the splits, fixed-order warp tree
__global__ void __launch_bounds__(128) scaml_predict_reduce_wide_kernel(const double* part, double* mean, double* var,
                                                                        int nsplit, int B) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, wpg = blockDim.x >> 5;
  for (int b = blockIdx.x * wpg + warp; b < B; b += gridDim.x * wpg) {
    double m = 0.0, v = 0.0;
    for (int s = lane; s < nsplit; s += 32) {
      m += part[((size_t)s * 2 + 0) * B + b];
      v += part[((size_t)s * 2 + 1) * B + b];
    }
    m = warp_sum(m);
    v = warp_sum(v);
    if (lane == 0) {
      mean[b] = m;
      var[b] = v;
    }
  }
}

// condA != null: also accumulate the cross-covariance partials into cxp (needs 64-candidate tiles: SCAML_E_SMEM
// otherwise); workspace layout: [nsplit][2][B] mean/var partials (nsplit > 1) -- cxp is a separate buffer
inline int launch_predict_weighted(const double* X, const int32_t* n_valid, const double* theta, const double* linv,
                                   const double* alpha, const double* ybar, const double* ystd, const double* w,
                                   const double* Xc, double* mean, double* var, double* workspace, int M, int n_max,
                                   int n_pad, int d, int B, int kernel, int num_sms, void* stream,
                                   const double* condA = nullptr, double* cxp = nullptr, int n_tp = 0) {
  PredParams p;
  p.condA = condA, p.cxp = cxp, p.n_tp = n_tp;
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.linv = linv, p.alpha = alpha, p.ybar = ybar, p.ystd = ystd;
  p.w = w, p.Xc = Xc, p.mean = mean, p.var = var, p.part = workspace;
  p.M = M, p.n_max = n_max, p.n_pad = n_pad, p.d = d, p.B = B;
  if (!predict_config(n_pad, d, &p.ct, &p.alias)) return SCAML_E_SMEM;
  if (condA != nullptr && (n_tp <= 0 || n_tp > 128 || (n_tp & 7))) return SCAML_E_UNSUPPORTED;
  p.ntile = (B + p.ct - 1) / p.ct;
  p.nsplit = predict_nsplit(M, B, num_sms, p.ct);
  const size_t smem = predict_smem_bytes(n_pad, d, p.ct, p.alias);
  long long items = (long long)p.ntile * p.nsplit;
  int grid = (int)(items < num_sms ? items : num_sms);
  const int rc = dispatch_kind(kernel, [&](auto K) {
    if (condA != nullptr)
      return p.ct == 64 ? launch(scaml_predict_kernel<K.value, 64, true>, grid, kPredThreads, smem, stream, p)
                        : launch(scaml_predict_kernel<K.value, 32, true>, grid, kPredThreads, smem, stream, p);
    return p.ct == 64 ? launch(scaml_predict_kernel<K.value, 64, false>, grid, kPredThreads, smem, stream, p)
                      : launch(scaml_predict_kernel<K.value, 32, false>, grid, kPredThreads, smem, stream, p);
  });
  if (rc != 0 || p.nsplit == 1) return rc;
  if (p.nsplit >= 32)  // by shape only
    return launch(scaml_predict_reduce_wide_kernel, stride_grid((B + 3) / 4, 1184), 128, 0, stream, workspace, mean,
                  var, p.nsplit, B);
  return launch(scaml_predict_reduce_kernel, stride_grid((B + 255) / 256, 1184), 256, 0, stream, workspace, mean, var,
                p.nsplit, B);
}

}  // namespace scaml
