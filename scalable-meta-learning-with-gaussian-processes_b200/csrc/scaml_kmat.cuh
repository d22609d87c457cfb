// Standalone batched kernel-matrix assembly (K1): K[m] = s * kappa(X_m / l) + noise * I,
// dense [M][n_max][n_max] fp64.  HBM-store bound (M * n^2 * 8 bytes); symmetry is used so
// every exp() is evaluated once: a CTA computes one 64x64 tile (ti >= tj) and stores it twice (as
// (ti,tj) rows and as the transposed (tj,ti) rows).
//   * squared distances on the FP64 tensor cores: r^2 = |a|^2 + |b|^2 - 2 a.b on inputs centred on
//     the task's first point and length-scaled (the quadratic expansion gpytorch evaluates, SURVEY
//     A.4): the accumulators start at |a|^2 + |b|^2 (one commutative add, so K stays bit-symmetric
//     inside the diagonal tiles as well) and a warp gets the -2 a.b of a 32 x 16 block from 8 DMMAs
//     per four input dimensions instead of 3 d FP64 instructions per pair.  Matern-1/2 (exp(-r), not
//     smooth in r^2 at r = 0) keeps direct differences.
//   * the tile goes through shared memory twice with conflict-free layouts -- row-major (stride 72:
//     the 16-byte fragment stores of a quarter warp fall into 8 different 16-byte slots) for the
//     (ti,tj) rows and column-major (stride 66: the 8-byte stores of a half warp fall into 16
//     different banks) for the transpose -- and leaves in whole rows: one warp instruction = 512 B
//     contiguous, every 32-byte sector written once.  (The round-1 layout, stride 65 with 4 x 4
//     register patches, ran 8-way conflicted stores: 85 % of the shared-memory pipe,
//     profiles/r2_kmat_kernel_ncu_summary.txt.)
// Reference call site: covar_module(X) + likelihood noise inside mll(model(X), y),
// scamlgp/utils.py:175-177; kernels scamlgp/model.py:44-70.
#pragma once
#include "scaml_device.cuh"

namespace scaml {

constexpr int kKXs = 68;   // row stride of the staged operands (== 4 mod 16: conflict-free DMMA fragment loads)
constexpr int kKTr = 72;   // row stride of the row-major staging tile
constexpr int kKTc = 66;   // row stride of the column-major (transposed) staging tile

struct KmatParams {
  const double* X;
  const int32_t* n_valid;
  const double* theta;  // [M][P] constrained
  double* K;
  int M, n_max, d, nt;  // nt = tiles per dimension
  long long items;      // M * nt*(nt+1)/2
};

// operand rows: d coordinates padded to a multiple of 4, + 1 row of squared norms
inline int kmat_rows(int d) { return ((d + 3) & ~3) + 1; }
inline size_t kmat_smem_bytes(int d) {
  return sizeof(double) * (2 * (size_t)kmat_rows(d) * kKXs + (size_t)kSB * kKTr + 2 * kMaxP);
}

template <int KIND>
__global__ void __launch_bounds__(256, 3) scaml_kmat_tile_kernel(const KmatParams p) {
  constexpr bool kDirect = (KIND == SCAML_KERNEL_MATERN12);
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const int rb = warp >> 2, cq = warp & 3;  // warp block: rows 32 rb .., columns 16 cq ..
  const int d = p.d, P = d + 2, dp = (d + 3) & ~3;
  double* xa = sm;                    // [dp + 1][kKXs] rows of tile ti: scaled coordinates (0 beyond d) | |a|^2
  double* xb = xa + (dp + 1) * kKXs;  // [dp + 1][kKXs] rows of tile tj: -2 x scaled coordinates | |b|^2
  double* T = xb + (dp + 1) * kKXs;   // 64 x kKTr row-major, then 64 x kKTc column-major
  double* invl = T + kSB * kKTr;   // [kMaxP] reciprocal lengthscales of the current task
  double* ctr = invl + kMaxP;      // [kMaxP] centre of the expansion (the task's first point)
  const int pairs = (p.nt * (p.nt + 1)) / 2;
  const bool vec_ok = (p.n_max % 2) == 0;
  for (long long it = blockIdx.x; it < p.items; it += gridDim.x) {
    const int m = (int)(it / pairs);
    const int pr = (int)(it - (long long)m * pairs);
    int ti = 0;
    while (tri(ti + 1) <= pr) ++ti;
    const int tj = pr - tri(ti);
    const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
    const double* th = p.theta + (size_t)m * P;
    const double* Xm = p.X + (size_t)m * p.n_max * d;
    // 128 points (64 rows of tile ti, 64 of tile tj) x d coordinates: thread -> (point tid / 2, coordinate parity),
    // no runtime integer division.  The raw coordinates are fetched into registers BEFORE the barrier (their latency
    // overlaps the previous tile's stores) and scaled by reciprocal lengthscales.
    const int pt = tid >> 1, kh = tid & 1;
    const int r = pt & 63;
    const int ga = (pt < kSB) ? ti * kSB + r : tj * kSB + r;
    double xq[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const int k = kh + 2 * u;
      xq[u] = (k < d && ga < p.n_max) ? __ldg(Xm + (size_t)ga * d + k) : 0.0;
    }
    if (tid < d) {
      invl[tid] = 1.0 / th[tid];
      ctr[tid] = __ldg(Xm + tid);
    }
    __syncthreads();  // invl, ctr visible (everyone has left the previous tile's epilogue: see the barriers below)
    {
      double* dst = (pt < kSB) ? xa : xb;
      const double sc = (pt < kSB) ? 1.0 : -2.0;
      double nn = 0.0;
#pragma unroll
      for (int u = 0; u < 4; ++u) {
        const int k = kh + 2 * u;
        if (k < d) {
          const double v = (ga < p.n_max) ? (xq[u] - ctr[k]) * invl[k] : 0.0;
          dst[k * kKXs + r] = sc * v;
          nn = fma(v, v, nn);
        }
      }
      for (int k = kh + 8; k < d; k += 2) {
        const double v = (ga < p.n_max) ? (__ldg(Xm + (size_t)ga * d + k) - ctr[k]) * invl[k] : 0.0;
        dst[k * kKXs + r] = sc * v;
        nn = fma(v, v, nn);
      }
      nn += __shfl_xor_sync(0xffffffffu, nn, 1);
      if (kh == 0) {
        dst[dp * kKXs + r] = nn;
        for (int k = d; k < dp; ++k) dst[k * kKXs + r] = 0.0;
      }
    }
    __syncthreads();
    const double os = th[d], noise = th[d + 1];
    double kv[16];  // [i][j][e] -> 4 i + 2 j + e : rows 32 rb + 8 i + g, columns 16 cq + 8 j + 2 t4 + e
    if (kDirect) {
#pragma unroll
      for (int u = 0; u < 16; ++u) kv[u] = 0.0;
      for (int k = 0; k < d; ++k) {
        double av[4], bv[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) av[i] = xa[k * kKXs + 32 * rb + 8 * i + g];
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const double2 b2 = *reinterpret_cast<const double2*>(xb + k * kKXs + 16 * cq + 8 * j + 2 * t4);
          bv[2 * j] = -0.5 * b2.x, bv[2 * j + 1] = -0.5 * b2.y;
        }
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const double df = av[i] - bv[c];
            kv[4 * i + c] = fma(df, df, kv[4 * i + c]);
          }
      }
    } else {
#pragma unroll
      for (int j = 0; j < 2; ++j) {
        const double2 nb = *reinterpret_cast<const double2*>(xb + dp * kKXs + 16 * cq + 8 * j + 2 * t4);
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const double na = xa[dp * kKXs + 32 * rb + 8 * i + g];
          kv[4 * i + 2 * j] = na + nb.x, kv[4 * i + 2 * j + 1] = na + nb.y;
        }
      }
      const double* aq = xa + t4 * kKXs + 32 * rb + g;
      const double* bq = xb + t4 * kKXs + 16 * cq + g;
      for (int ks = 0; ks < dp; ks += 4) {
        double a[4], b[2];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = aq[ks * kKXs + 8 * i];
#pragma unroll
        for (int j = 0; j < 2; ++j) b[j] = bq[ks * kKXs + 8 * j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j) dmma884s(kv[4 * i + 2 * j], kv[4 * i + 2 * j + 1], a[i], b[j]);
      }
    }
    kappa_n<KIND, 16, false>(kv, kv, kv);  // 16 independent exponentials, interleaved
    // interior tiles (off the diagonal, fully inside the valid range) need no per-element masks: CTA-uniform
    const bool interior = (ti != tj) && (ti * kSB + kSB <= nv);
    if (interior) {
#pragma unroll
      for (int u = 0; u < 16; ++u) kv[u] *= os;
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int a = ti * kSB + 32 * rb + 8 * i + g, b = tj * kSB + 16 * cq + 8 * j + 2 * t4 + e;
            double k = os * kv[4 * i + 2 * j + e];
            if (a == b) k = os + noise;  // kappa(0) = 1 exactly (the expansion leaves r^2 = +-1e-16 on the diagonal)
            if (a >= nv || b >= nv) k = (a == b) ? 1.0 : 0.0;
            kv[4 * i + 2 * j + e] = k;
          }
    }
    // (1) row-major staging, whole-row stores of tile (ti, tj)
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 2; ++j)
        *reinterpret_cast<double2*>(T + (32 * rb + 8 * i + g) * kKTr + 16 * cq + 8 * j + 2 * t4) =
            make_double2(kv[4 * i + 2 * j], kv[4 * i + 2 * j + 1]);
    __syncthreads();
    double* Km = p.K + (size_t)m * p.n_max * p.n_max;
    const int row0 = ti * kSB, col0 = tj * kSB;
    for (int rr = warp; rr < kSB; rr += 8) {
      const int gr = row0 + rr;
      if (gr >= p.n_max) break;
      double* q = Km + (size_t)gr * p.n_max + col0;
      const double2 v = *reinterpret_cast<const double2*>(T + rr * kKTr + 2 * lane);
      if (vec_ok && col0 + 2 * lane + 1 < p.n_max) {
        *reinterpret_cast<double2*>(q + 2 * lane) = v;
      } else {
        if (col0 + 2 * lane < p.n_max) q[2 * lane] = v.x;
        if (col0 + 2 * lane + 1 < p.n_max) q[2 * lane + 1] = v.y;
      }
    }
    // (2) off the diagonal: column-major staging of the same registers, whole-row stores of tile (tj, ti)
    if (ti != tj) {
      __syncthreads();  // row reads of T done
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e)
            T[(16 * cq + 8 * j + 2 * t4 + e) * kKTc + 32 * rb + 8 * i + g] = kv[4 * i + 2 * j + e];
      __syncthreads();
      for (int c = warp; c < kSB; c += 8) {
        const int gb = col0 + c;
        if (gb >= p.n_max) break;
        double* q = Km + (size_t)gb * p.n_max + row0;
        const double2 v = *reinterpret_cast<const double2*>(T + c * kKTc + 2 * lane);
        if (vec_ok && row0 + 2 * lane + 1 < p.n_max) {
          *reinterpret_cast<double2*>(q + 2 * lane) = v;
        } else {
          if (row0 + 2 * lane < p.n_max) q[2 * lane] = v.x;
          if (row0 + 2 * lane + 1 < p.n_max) q[2 * lane + 1] = v.y;
        }
      }
    }
    // no barrier here: the next iteration overwrites invl / ctr before its first barrier -- every thread has passed
    // this tile's later barriers, i.e. left its staging -- and xa / xb / T only after that barrier
  }
}

// ---- whole-task variant (the fast path: every shape whose scaled inputs fit kKTaskSmem) ------------------------- //
// A CTA stages the centred, scaled inputs of ONE task once (the tile kernel above re-stages 128 points for each of
// the nt (nt + 1) / 2 tiles: 5 x redundant at n = 256) and its 8 warps then walk the task's 32 x 16 blocks on their
// own -- no barrier and no shared-memory staging of the result: the DMMA accumulator fragment of a block leaves
// straight from registers, rows of the block as 16-byte stores (8 rows x 64 B per instruction) and, for the mirrored
// block, columns as 8-byte stores (4 rows x 64 B): whole 32-byte sectors in both directions.  Blocks strictly above
// the diagonal inside a diagonal tile are not computed at all (they are the mirror of a block below it).
#ifdef SCAML_EMU
constexpr size_t kKTaskSmem = 16 * 1024;  // CPU tests reach both kernels with small problems
#else
constexpr size_t kKTaskSmem = 100 * 1024;
#endif
inline size_t kmat_task_smem_bytes(int n_max, int d) {
  const int n_pad = ((n_max + kSB - 1) / kSB) * kSB;
  return sizeof(double) * ((size_t)kmat_rows(d) * (n_pad + 4) + 2 * kMaxP);
}

template <int KIND>
__global__ void __launch_bounds__(256, 3) scaml_kmat_task_kernel(const KmatParams p) {
  constexpr bool kDirect = (KIND == SCAML_KERNEL_MATERN12);
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const int d = p.d, P = d + 2, dp = (d + 3) & ~3;
  const int n_pad = p.nt * kSB, XS = n_pad + 4;
  double* xs = sm;                        // [dp + 1][XS]: scaled coordinates (0 beyond d) | squared norm
  double* invl = xs + (size_t)(dp + 1) * XS;
  double* ctr = invl + kMaxP;
  const double* nrm = xs + (size_t)dp * XS;
  const int pairs = (p.nt * (p.nt + 1)) / 2;
  const bool vec_ok = (p.n_max % 2) == 0;
  for (int m = blockIdx.x; m < p.M; m += gridDim.x) {
    const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
    const double* th = p.theta + (size_t)m * P;
    const double* Xm = p.X + (size_t)m * p.n_max * d;
    __syncthreads();  // every warp has finished the previous task's blocks
    if (tid < d) {
      invl[tid] = 1.0 / th[tid];
      ctr[tid] = __ldg(Xm + tid);
    }
    __syncthreads();
    for (int a = tid; a < n_pad; a += 256) {
      double nn = 0.0;
      for (int k = 0; k < d; ++k) {
        const double v = (a < p.n_max) ? (__ldg(Xm + (size_t)a * d + k) - ctr[k]) * invl[k] : 0.0;
        xs[k * XS + a] = v;
        nn = fma(v, v, nn);
      }
      for (int k = d; k < dp; ++k) xs[k * XS + a] = 0.0;
      xs[dp * XS + a] = nn;
    }
    __syncthreads();
    const double os = th[d], noise = th[d + 1];
    double* Km = p.K + (size_t)m * p.n_max * p.n_max;
    for (int u = warp; u < pairs * 8; u += 8) {
      const int pr = u >> 3, blk = u & 7;
      int ti = 0;
      while (tri(ti + 1) <= pr) ++ti;
      const int tj = pr - tri(ti);
      const int rb = blk >> 2, cq = blk & 3;
      const int r0 = ti * kSB + 32 * rb, c0 = tj * kSB + 16 * cq;  // first row / column of the block
      if (ti == tj && c0 >= r0 + 32) continue;                      // strictly above the diagonal: mirrored below
      if (r0 >= p.n_max || c0 >= p.n_max) continue;
      double kv[16];  // [i][j][e] -> 4 i + 2 j + e : rows r0 + 8 i + g, columns c0 + 8 j + 2 t4 + e
      if (kDirect) {
#pragma unroll
        for (int q = 0; q < 16; ++q) kv[q] = 0.0;
        for (int k = 0; k < d; ++k) {
          double av[4], bv[4];
#pragma unroll
          for (int i = 0; i < 4; ++i) av[i] = xs[k * XS + r0 + 8 * i + g];
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const double2 b2 = *reinterpret_cast<const double2*>(xs + k * XS + c0 + 8 * j + 2 * t4);
            bv[2 * j] = b2.x, bv[2 * j + 1] = b2.y;
          }
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              const double df = av[i] - bv[c];
              kv[4 * i + c] = fma(df, df, kv[4 * i + c]);
            }
        }
      } else {
#pragma unroll
        for (int j = 0; j < 2; ++j) {
          const double2 nb = *reinterpret_cast<const double2*>(nrm + c0 + 8 * j + 2 * t4);
#pragma unroll
          for (int i = 0; i < 4; ++i) {
            const double na = nrm[r0 + 8 * i + g];
            kv[4 * i + 2 * j] = na + nb.x, kv[4 * i + 2 * j + 1] = na + nb.y;  // commutative: K stays bit-symmetric
          }
        }
        const double* aq = xs + t4 * XS + r0 + g;
        const double* bq = xs + t4 * XS + c0 + g;
        for (int ks = 0; ks < dp; ks += 4) {
          double a[4], b[2];
#pragma unroll
          for (int i = 0; i < 4; ++i) a[i] = aq[ks * XS + 8 * i];
#pragma unroll
          for (int j = 0; j < 2; ++j) b[j] = -2.0 * bq[ks * XS + 8 * j];
#pragma unroll
          for (int i = 0; i < 4; ++i)
#pragma unroll
            for (int j = 0; j < 2; ++j) dmma884s(kv[4 * i + 2 * j], kv[4 * i + 2 * j + 1], a[i], b[j]);
        }
      }
#ifdef SCAML_KMAT_TABEXP
      kappa_n<KIND, 16, false>(kv, kv, kv);  // 16 independent exponentials, interleaved
#else
      // table-free exp: this kernel's scarce resource is the load / store pipe (78 % busy with the table variant, a
      // third of it table lookups), not the FP64 pipe
      kappa_n<KIND, 16, false, false>(kv, kv, kv);
#endif
      // blocks off the diagonal tiles and fully inside the valid range need no per-element masks: warp-uniform
      const bool interior = (ti != tj) && (r0 + 32 <= nv);
      if (interior) {
#pragma unroll
        for (int q = 0; q < 16; ++q) kv[q] *= os;
      } else {
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 2; ++j)
#pragma unroll
            for (int e = 0; e < 2; ++e) {
              const int a = r0 + 8 * i + g, b = c0 + 8 * j + 2 * t4 + e;
              double k = os * kv[4 * i + 2 * j + e];
              if (a == b) k = os + noise;  // kappa(0) = 1 exactly (the expansion leaves r^2 = +-1e-16 on the diagonal)
              if (a >= nv || b >= nv) k = (a == b) ? 1.0 : 0.0;
              kv[4 * i + 2 * j + e] = k;
            }
      }
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int a = r0 + 8 * i + g;
        if (a < p.n_max) {
          double* q = Km + (size_t)a * p.n_max + c0 + 2 * t4;
#pragma unroll
          for (int j = 0; j < 2; ++j) {
            const int b = c0 + 8 * j + 2 * t4;
            if (vec_ok && b + 1 < p.n_max) {
              *reinterpret_cast<double2*>(q + 8 * j) = make_double2(kv[4 * i + 2 * j], kv[4 * i + 2 * j + 1]);
            } else {
              if (b < p.n_max) q[8 * j] = kv[4 * i + 2 * j];
              if (b + 1 < p.n_max) q[8 * j + 1] = kv[4 * i + 2 * j + 1];
            }
          }
        }
      }
      // mirror: every block of an off-diagonal tile; inside a diagonal tile the blocks strictly below the diagonal
      if (ti != tj || c0 + 16 <= r0) {
#pragma unroll
        for (int j = 0; j < 2; ++j)
#pragma unroll
          for (int e = 0; e < 2; ++e) {
            const int b = c0 + 8 * j + 2 * t4 + e;
            if (b < p.n_max) {
              double* q = Km + (size_t)b * p.n_max + r0 + g;
#pragma unroll
              for (int i = 0; i < 4; ++i)
                if (r0 + 8 * i + g < p.n_max) q[8 * i] = kv[4 * i + 2 * j + e];
            }
          }
      }
    }
  }
}

// variant: 0 = by shape (whole-task kernel when the task's scaled inputs fit kKTaskSmem), 1 = tile kernel, 2 = task kernel
inline int launch_kmat(const double* X, const int32_t* n_valid, const double* theta, double* K, int M, int n_max,
                       int d, int kernel, void* stream, int variant = 0) {
  KmatParams p;
  p.X = X, p.n_valid = n_valid, p.theta = theta, p.K = K, p.M = M, p.n_max = n_max, p.d = d;
  p.nt = (n_max + kSB - 1) / kSB;
  p.items = (long long)M * ((p.nt * (p.nt + 1)) / 2);
  const size_t tsmem = kmat_task_smem_bytes(n_max, d);
  const bool task = (variant == 2) || (variant == 0 && tsmem <= kKTaskSmem);
  if (task && tsmem > 227 * 1024) return SCAML_E_SMEM;
  const size_t smem = task ? tsmem : kmat_smem_bytes(d);
  const int grid = stride_grid(task ? (long long)M : p.items, 148LL * 8 * 4);
  return dispatch_kind(kernel, [&](auto K) {
    return task ? launch(scaml_kmat_task_kernel<K.value>, grid, 256, smem, stream, p)
                : launch(scaml_kmat_tile_kernel<K.value>, grid, 256, smem, stream, p);
  });
}

}  // namespace scaml
