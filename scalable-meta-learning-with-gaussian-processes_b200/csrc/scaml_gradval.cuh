// Posterior VALUES from U = K_m^-1 K_m(X_m, Xc) (the gradient path has it anyway, scaml_grad.cuh): with u_m(x) in hand
// the weighted prior at a candidate needs no triangular product any more,
//   mean(x)     = sum_m w_m (ybar_m + ystd_m k*_m^T alpha_m)
//   var(x)      = sum_m c_m (s_m - k*_m^T u_m),                              c_m = w_m^2 ystd_m^2
//   cross(x, j) = sum_m c_m (K_m(x, x_tj) - k*_m^T A_m[:, j]),
// i.e. per task one [B x n] x [n x (n_t + 1)] product (A_m | alpha_m) on the FP64 tensor cores plus an elementwise
// k* . U sum -- O(n (n_t + d)) per (task, candidate) instead of the n^2 of the prediction kernel.  Same quantities as
// scaml_predict_conditioned (reference scamlgp/model.py:364-375, eval branch of ScaMLGP.forward, q = 1), used for the
// value half of one value-and-gradient evaluation of the acquisition optimiser.
//
// One CTA owns a contiguous split of the tasks x one tile of 64 candidates; per 32-row chunk of a task it builds the
// scaled k* chunk (c_m s_m kappa) in shared memory (thread <-> candidate, 8 rows each, U read coalesced for the
// variance term), stages A_m | alpha_m / (w_m ystd_m) next to it and contracts on DMMA (warp <-> 8 candidates, all
// column blocks); the accumulators persist over all tasks of the split (fixed order).  Partials go out in the layout
// scaml_cond_combine_kernel sums, a small kernel finishes mean / variance.
#pragma once
#include "scaml_cond.cuh"

namespace scaml {

struct GradValParams {
  const double* X;         // [M][n_max][d]
  const int32_t* n_valid;  // [M] or null
  const double* theta;     // [M][P] constrained
  const double* alpha;     // [M][n_pad]
  const double* ybar;      // [M]
  const double* ystd;      // [M]
  const double* w;         // [M]
  const double* Xc;        // [B][d]
  const double* U;         // [M][n_pad][B_p]
  const double* A;         // [M][n_pad][n_tp] (n_t > 0)
  double* cxp;             // [nsplit][B][n_tp] partial sum_m c_m k*_m^T A_m (n_t > 0)
  double* mvp;             // [nsplit][B][2]    partial sum_m w_m (ybar_m + ystd_m k*^T alpha) | sum_m c_m (s_m - k*^T u)
  double* mean;            // [B]
  double* var;             // [B]
  int M, n_max, n_pad, d, B, B_p, n_t, n_tp, nsplit, ntile;
};

constexpr int kGvThreads = 256;
constexpr int kGvCT = 64;                  // candidates per tile
constexpr int kGvLdk = kGvCT + 4;          // k* chunk row stride (= 4 mod 8: conflict-free DMMA A-fragments)
constexpr int kGvMaxCB = 17;               // column blocks: n_tp / 8 (<= 16) + the alpha block
inline int gv_lda(int n_tp) { return n_tp + 8 + 4; }
// shared memory (doubles): ks [32][68] | Ae [32][lda] | xs [32][d] | xcs [d][64] | il [kMaxP] | red [4][64]
inline size_t gradval_smem_bytes(int d, int n_tp) {
  return sizeof(double) * (32 * (size_t)kGvLdk + 32 * (size_t)gv_lda(n_tp) + 32 * (size_t)d + (size_t)d * kGvCT + kMaxP +
                           4 * kGvCT + 8);
}

template <int KIND, int NCB>
__global__ void __launch_bounds__(kGvThreads, (NCB <= 9 ? 2 : 1)) scaml_grad_values_kernel(const GradValParams p) {
  SCAML_DYN_SMEM(double, sm);
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31, g = lane >> 2, t4 = lane & 3;
  const int d = p.d, P = d + 2, n_pad = p.n_pad, nt = p.n_t, ntp = p.n_tp, lda = ntp + 12;
  const int ncb = ntp / 8 + 1;  // column blocks incl. the alpha block (column ntp)
  double* ks = sm;                          // [32][kGvLdk]
  double* Ae = ks + 32 * kGvLdk;            // [32][lda]
  double* xs = Ae + 32 * (size_t)lda;       // [32][d] raw inputs of the chunk
  double* xcs = xs + 32 * (size_t)d;        // [d][64] raw candidates of the tile
  double* il = xcs + (size_t)d * kGvCT;     // [kMaxP] 1 / l_k of the task
  double* red = il + kMaxP;                 // [4][64]
  const int cb_ = tid & 63, rg = tid >> 6;  // this thread: candidate cb_ of the tile, rows rg + 4 k of a chunk
  const int items = p.nsplit * p.ntile;
  for (int it = blockIdx.x; it < items; it += gridDim.x) {
    const int split = it / p.ntile, tile = it - split * p.ntile;
    const int b0 = tile * kGvCT;
    const int bme = b0 + cb_ < p.B ? b0 + cb_ : p.B - 1;  // dead candidates shadow the last one (never written)
    const int m_lo = (int)((long long)p.M * split / p.nsplit), m_hi = (int)((long long)p.M * (split + 1) / p.nsplit);
    __syncthreads();
    for (int i = tid; i < d * kGvCT; i += kGvThreads) {
      const int k = i / kGvCT, c = i - k * kGvCT;
      const int bb = b0 + c < p.B ? b0 + c : p.B - 1;
      xcs[i] = p.Xc[(size_t)bb * d + k];
    }
    double acc[NCB][2];
#pragma unroll
    for (int c = 0; c < NCB; ++c) acc[c][0] = acc[c][1] = 0.0;
    double vacc = 0.0, c0 = 0.0, c1 = 0.0;  // c0 / c1: the split's share of sum_m w_m ybar_m and sum_m c_m s_m
    for (int m = m_lo; m < m_hi; ++m) {
      const double wm = p.w[m];
      if (wm == 0.0) continue;  // pruned task (uniform over the CTA)
      const int nv = p.n_valid ? p.n_valid[m] : p.n_max;
      const double* th = p.theta + (size_t)m * P;
      const double sy = p.ystd[m], cmw = wm * sy, cos_ = cmw * cmw * th[d], ia = 1.0 / cmw;
      c0 = fma(wm, p.ybar[m], c0);
      c1 += cos_;
      const double* Xm = p.X + (size_t)m * p.n_max * d;
      const int nchunk = (nv + 31) >> 5;
      for (int ch = 0; ch < nchunk; ++ch) {
        __syncthreads();  // previous chunk's products are done with ks / Ae
        if (ch == 0 && tid < d) il[tid] = 1.0 / th[tid];
        for (int i = tid; i < 32 * d; i += kGvThreads) {
          const int r = 32 * ch + i / d;
          xs[i] = r < nv ? Xm[(size_t)32 * ch * d + i] : 0.0;
        }
        for (int i = tid; i < 32 * (ntp + 8); i += kGvThreads) {
          const int r = i / (ntp + 8), c = i - r * (ntp + 8), row = 32 * ch + r;
          double v = 0.0;
          if (row < nv) {
            if (c < ntp) v = p.A[((size_t)m * n_pad + row) * ntp + c];
            else if (c == ntp) v = p.alpha[(size_t)m * n_pad + row] * ia;
          }
          Ae[(size_t)r * lda + c] = v;
        }
        __syncthreads();
        {  // scaled k* chunk: ks[r][c] = c_m s_m kappa(x_c, X_m[row]); variance term with U (coalesced over candidates)
          double r2[8], kap[8], uq[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {  // U first: the loads fly under the distance / exp chains
            const int row = 32 * ch + rg + 4 * u;
            uq[u] = row < nv ? p.U[((size_t)m * n_pad + row) * p.B_p + bme] : 0.0;
            r2[u] = 0.0;
          }
          for (int k = 0; k < d; ++k) {
            const double xk = xcs[k * kGvCT + cb_], ik = il[k];
#pragma unroll
            for (int u = 0; u < 8; ++u) {
              const double df = (xk - xs[(rg + 4 * u) * d + k]) * ik;
              r2[u] = fma(df, df, r2[u]);
            }
          }
          kappa_n<KIND, 8, false>(r2, kap, kap);
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int r = rg + 4 * u, row = 32 * ch + r;
            const double kv = row < nv ? cos_ * kap[u] : 0.0;
            ks[r * kGvLdk + cb_] = kv;
            vacc = fma(kv, uq[u], vacc);
          }
        }
        __syncthreads();
        {  // out[cand][col] += sum_rows ks[row][cand] * Ae[row][col]; warp <-> candidates 8 warp .. 8 warp + 7
          const double* ar = ks + (size_t)t4 * kGvLdk + 8 * warp + g;
          const double* br = Ae + (size_t)t4 * lda + g;
#pragma unroll
          for (int s = 0; s < 8; ++s) {
            const double a = ar[(size_t)4 * s * kGvLdk];
#pragma unroll
            for (int c = 0; c < NCB; ++c)
              if (c < ncb) dmma884(acc[c], a, br[(size_t)4 * s * lda + 8 * c]);
          }
        }
      }
    }
    // ---- partials of this (split, tile) ------------------------------------------------------------------- //
    {
      const int cand = b0 + 8 * warp + g;  // d[e] = D[g][2 t4 + e]
#pragma unroll
      for (int c = 0; c < NCB; ++c) {
        if (c < ncb - 1) {
          if (cand < p.B)
            *reinterpret_cast<double2*>(p.cxp + ((size_t)split * p.B + cand) * ntp + 8 * c + 2 * t4) =
                make_double2(acc[c][0], acc[c][1]);
        } else if (c == ncb - 1) {
          if (cand < p.B && t4 == 0) p.mvp[((size_t)split * p.B + cand) * 2] = c0 + acc[c][0];
        }
      }
    }
    __syncthreads();
    red[rg * kGvCT + cb_] = vacc;
    __syncthreads();
    if (tid < kGvCT && b0 + tid < p.B)
      p.mvp[((size_t)split * p.B + b0 + tid) * 2 + 1] =
          c1 - ((red[tid] + red[kGvCT + tid]) + (red[2 * kGvCT + tid] + red[3 * kGvCT + tid]));
  }
}

// mean[b] = sum_s mvp[s][b][0];  var[b] = sum_s mvp[s][b][1]   (the splits carry their share of the constants; lanes
// stride over the splits, fixed-order warp tree)
__global__ void __launch_bounds__(64) scaml_grad_values_finish_kernel(const GradValParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int wpg = blockDim.x >> 5;
  for (long long b = (long long)blockIdx.x * wpg + warp; b < p.B; b += (long long)gridDim.x * wpg) {
    double a = 0.0, v = 0.0;
    for (int s = lane; s < p.nsplit; s += 32) {
      a += p.mvp[((size_t)s * p.B + b) * 2];
      v += p.mvp[((size_t)s * p.B + b) * 2 + 1];
    }
    a = warp_sum(a);
    v = warp_sum(v);
    if (lane == 0) {
      p.mean[b] = a;
      p.var[b] = v;
    }
  }
}

inline int gradval_nsplit(int M, int ntile, int num_sms) {
  int ns = (4 * num_sms + ntile - 1) / ntile;  // 2 CTAs / SM resident, 2 waves
  if (ns > M) ns = M;
  return ns < 1 ? 1 : ns;
}

inline int launch_grad_values(const GradValParams& p, int kernel, int num_sms, void* stream) {
  const size_t smem = gradval_smem_bytes(p.d, p.n_tp);
  if (smem > 227 * 1024) return SCAML_E_SMEM;
  const int grid = stride_grid(p.nsplit * p.ntile, 4 * num_sms);
  const int ncb = p.n_tp / 8 + 1;  // accumulator column blocks per warp: register variants 5 / 9 / 17
  const int rc = dispatch_kind(kernel, [&](auto K) {
    if (ncb <= 5) return launch(scaml_grad_values_kernel<K.value, 5>, grid, kGvThreads, smem, stream, p);
    if (ncb <= 9) return launch(scaml_grad_values_kernel<K.value, 9>, grid, kGvThreads, smem, stream, p);
    return launch(scaml_grad_values_kernel<K.value, kGvMaxCB>, grid, kGvThreads, smem, stream, p);
  });
  if (rc) return rc;
  const int fgrid = stride_grid(((long long)p.B + 1) / 2, 4LL * num_sms);  // one warp per candidate, two per CTA
  return launch(scaml_grad_values_finish_kernel, fgrid, 64, 0, stream, p);
}

}  // namespace scaml
