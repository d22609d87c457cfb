// Device-side batched projected L-BFGS update: E independent minimisations advance in lock-step, one WARP per
// row.  One call consumes the objective values / gradients at the trial points xt and produces the next trial
// points; the host only launches (objective kernel, this kernel) pairs and polls the number of active rows
// every few rounds -- no per-row host round trip (SURVEY 8f rank 2).  Replaces the per-task scipy L-BFGS-B loop
// behind botorch `fit_gpytorch_mll` (reference scamlgp/utils.py:175,190; defaults m = 10, gtol 1e-5,
// ftol 2.2e-9).  Semantics are those of scamlgp_b200/lbfgs.py (the torch statement of the same algorithm,
// kept as the checker in tests/test_lbfgs.py): Armijo backtracking with safeguarded quadratic interpolation,
// curvature pairs kept when s.y > 1e-10 |s||y|, active-set handling of simple lower bounds, steepest-descent
// restart when the two-loop direction is not a descent direction, NaN objective = rejected step.
// All reductions are fixed-order warp trees: deterministic and independent of the other rows in the batch.
// Two shapes of the same code (template WPR = warps per row): one warp per row for the source fits (tens of
// thousands of rows, D = d + 2) and one 8-warp CTA per row for the target fit (a handful of rows, D = M + d + 2 in the
// thousands -- one warp per row took 1.4 ms per update at M = 4096 and was 85 % of `ScaMLGPBO.report`).
#pragma once
#include "scaml_device.cuh"

namespace scaml {

enum { kLbActive = 1, kLbConverged = 2, kLbFailed = 4 };

struct LbfgsParams {
  double* x;      // [E][D] accepted iterates
  double* f;      // [E]
  double* g;      // [E][D]
  double* d;      // [E][D] search directions
  double* t;      // [E] step lengths
  double* S;      // [E][m][D]
  double* Y;      // [E][m][D]
  double* rho;    // [E][m]
  int32_t* count;     // [E] stored pairs
  int32_t* head;      // [E] next slot
  int32_t* iters;     // [E] accepted steps
  int32_t* ls_count;  // [E] consecutive rejections
  int32_t* flags;     // [E] kLb*
  double* xt;         // [E][D] in: evaluated trial points; out: next trial points
  const double* ft;   // [E]
  const double* gt;   // [E][D]
  const double* lower;  // [D] or null (-inf = free)
  int E, D, m, init, maxiter, max_ls;
  double gtol, ftol;
};

SCAML_DEVICE bool lb_finite(double v) { return v == v && fabs(v) <= 1.7976931348623157e308; }


// A row is worked on by WPR warps (WPR = 1: one warp, warp-level primitives only; WPR > 1: the whole CTA, which then
// holds exactly one row so that block barriers are row barriers and early exits are uniform).
template <int WPR>
struct LbRow {
  int li, lane, wir;  // thread index within the row group, lane, warp within the row
  double* red;        // shared scratch of the row group: WPR doubles
  SCAML_DEVICE void sync() const {
    if (WPR == 1) __syncwarp();
    else __syncthreads();
  }
  SCAML_DEVICE double sum(double v) const {  // fixed order: warp tree, then the warps of the row in order
    v = warp_sum(v);
    if (WPR == 1) return v;
    __syncthreads();
    if (lane == 0) red[wir] = v;
    __syncthreads();
    double s = 0.0;
    for (int w = 0; w < WPR; ++w) s += red[w];
    return s;
  }
  SCAML_DEVICE double max(double v) const {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if (WPR == 1) return v;
    __syncthreads();
    if (lane == 0) red[wir] = v;
    __syncthreads();
    double s = red[0];
    for (int w = 1; w < WPR; ++w) s = fmax(s, red[w]);
    return s;
  }
  SCAML_DEVICE bool any(int pred) const {
    pred = __any_sync(0xffffffffu, pred);
    if (WPR == 1) return pred != 0;
    return sum(pred ? 1.0 : 0.0) > 0.0;
  }
};
constexpr int kLbWideWarps = 8;   // warps per row of the wide variant
constexpr int kLbWideMinD = 512;  // rows at least this long take the wide variant

// d = -H gg (two-loop recursion over the row's circular history); the threads of the row stride over D.  al: m doubles of
// per-warp scratch.  gg = g with the fixed (bound-active) variables zeroed; d is zeroed there as well.
template <int WPR>
SCAML_DEVICE void lb_direction(const LbfgsParams& p, int e, const LbRow<WPR>& rw, double* al, int count, int head) {
  const int lane = rw.li;
  constexpr int kStride = 32 * WPR;
  const int D = p.D, m = p.m;
  const double* x = p.x + (size_t)e * D;
  const double* g = p.g + (size_t)e * D;
  double* d = p.d + (size_t)e * D;
  const double* S = p.S + (size_t)e * m * D;
  const double* Y = p.Y + (size_t)e * m * D;
  const double* rho = p.rho + (size_t)e * m;
  // q (held in d) = gg
  for (int i = lane; i < D; i += kStride) {
    const bool fixed = p.lower != nullptr && x[i] <= p.lower[i] && g[i] > 0.0;
    d[i] = fixed ? 0.0 : g[i];
  }
  rw.sync();
  for (int j = 0; j < m && j < count; ++j) {  // newest -> oldest
    const int idx = ((head - 1 - j) % m + m) % m;
    const double* s = S + (size_t)idx * D;
    const double* y = Y + (size_t)idx * D;
    double a = 0.0;
    for (int i = lane; i < D; i += kStride) a = fma(s[i], d[i], a);
    a = rw.sum(a) * rho[idx];
    if (lane == 0) al[j] = a;
    for (int i = lane; i < D; i += kStride) d[i] = fma(-a, y[i], d[i]);
    rw.sync();
  }
  double gamma = 1.0;
  if (count > 0) {
    const int idx0 = ((head - 1) % m + m) % m;
    const double* s = S + (size_t)idx0 * D;
    const double* y = Y + (size_t)idx0 * D;
    double sy = 0.0, yy = 0.0;
    for (int i = lane; i < D; i += kStride) {
      sy = fma(s[i], y[i], sy);
      yy = fma(y[i], y[i], yy);
    }
    sy = rw.sum(sy);
    yy = rw.sum(yy);
    if (yy > 0.0) gamma = sy / fmax(yy, 1e-300);
  }
  for (int i = lane; i < D; i += kStride) d[i] *= gamma;
  rw.sync();
  for (int j = (count < m ? count : m) - 1; j >= 0; --j) {  // oldest -> newest
    const int idx = ((head - 1 - j) % m + m) % m;
    const double* s = S + (size_t)idx * D;
    const double* y = Y + (size_t)idx * D;
    double b = 0.0;
    for (int i = lane; i < D; i += kStride) b = fma(y[i], d[i], b);
    b = rw.sum(b) * rho[idx];
    const double c = al[j] - b;
    for (int i = lane; i < D; i += kStride) d[i] = fma(c, s[i], d[i]);
    rw.sync();
  }
  // d = -r with fixed variables pinned; fall back to steepest descent if it is not a descent direction
  double slope = 0.0;
  for (int i = lane; i < D; i += kStride) {
    const bool fixed = p.lower != nullptr && x[i] <= p.lower[i] && g[i] > 0.0;
    const double v = fixed ? 0.0 : -d[i];
    d[i] = v;
    slope = fma(g[i], v, slope);
  }
  slope = rw.sum(slope);
  if (!(slope < 0.0)) {
    for (int i = lane; i < D; i += kStride) {
      const bool fixed = p.lower != nullptr && x[i] <= p.lower[i] && g[i] > 0.0;
      d[i] = fixed ? 0.0 : -g[i];
    }
  }
  rw.sync();
}

template <int WPR>
SCAML_DEVICE double lb_projected_grad_inf(const LbfgsParams& p, int e, const LbRow<WPR>& rw) {
  const int lane = rw.li;
  constexpr int kStride = 32 * WPR;
  const int D = p.D;
  const double* x = p.x + (size_t)e * D;
  const double* g = p.g + (size_t)e * D;
  double mx = 0.0;
  for (int i = lane; i < D; i += kStride) {
    double v = g[i];
    if (p.lower != nullptr) v = x[i] - fmax(x[i] - g[i], p.lower[i]);
    mx = fmax(mx, fabs(v));
  }
  return rw.max(mx);
}

constexpr int kLbWarps = 4;
constexpr int kLbMaxHistory = 32;

template <int WPR>
__global__ void __launch_bounds__(WPR == 1 ? kLbWarps * 32 : WPR * 32) scaml_lbfgs_step_kernel(const LbfgsParams p) {
  SCAML_DYN_SMEM(double, sm);  // per row group: kLbMaxHistory two-loop coefficients | WPR reduction slots
  constexpr int kStride = 32 * WPR;
  const int warp = threadIdx.x >> 5;
  const int grp = WPR == 1 ? warp : 0;               // row group within the CTA
  const int e = WPR == 1 ? blockIdx.x * kLbWarps + warp : blockIdx.x;
  if (e >= p.E) return;
  double* al = sm + grp * (kLbMaxHistory + WPR);
  LbRow<WPR> rw;
  rw.lane = threadIdx.x & 31, rw.wir = WPR == 1 ? 0 : warp, rw.li = WPR == 1 ? rw.lane : threadIdx.x;
  rw.red = al + kLbMaxHistory;
  const int lane = rw.li;  // "lane" below = index within the row group; loops stride by kStride
  const int D = p.D, m = p.m;
  double* x = p.x + (size_t)e * D;
  double* g = p.g + (size_t)e * D;
  double* d = p.d + (size_t)e * D;
  double* xt = p.xt + (size_t)e * D;
  const double* gt = p.gt + (size_t)e * D;
  int flags = p.init ? kLbActive : p.flags[e];
  if (!(flags & kLbActive)) return;
  // scalar state of the row: every lane reads it BEFORE lane 0 may rewrite it (no intra-warp read/write race);
  // updated copies live in registers (warp-uniform) and are stored once at the end
  const double f = p.init ? 0.0 : p.f[e];
  double tcur = p.init ? 0.0 : p.t[e];
  int count = p.init ? 0 : p.count[e], head = p.init ? 0 : p.head[e];
  int iters = p.init ? 0 : p.iters[e], lsc = p.init ? 0 : p.ls_count[e];
  double fnew = f;
  rw.sync();
  const double ft = p.ft[e];
  bool fin = lb_finite(ft);
  {
    int bad = 0;
    for (int i = lane; i < D; i += kStride) bad |= !lb_finite(gt[i]);
    fin = fin && !rw.any(bad);
  }
  bool fresh_dir = false;  // a new direction is needed (accepted step or initialisation)
  if (p.init) {
    for (int i = lane; i < D; i += kStride) {
      x[i] = xt[i];
      g[i] = fin ? gt[i] : 0.0;
    }
    rw.sync();
    fnew = ft;
    if (!fin) {
      flags = kLbFailed;
    } else if (lb_projected_grad_inf<WPR>(p, e, rw) <= p.gtol) {
      flags = kLbConverged;
    } else {
      fresh_dir = true;
    }
  } else {
    double dec = 0.0, ss = 0.0, sy = 0.0, yy = 0.0;
    for (int i = lane; i < D; i += kStride) {
      const double st = xt[i] - x[i];
      dec = fma(g[i], st, dec);
      if (fin) {
        const double y = gt[i] - g[i];
        ss = fma(st, st, ss);
        sy = fma(st, y, sy);
        yy = fma(y, y, yy);
      }
    }
    dec = rw.sum(dec);
    const bool ok = fin && (ft <= f + 1e-4 * dec);
    if (ok) {
      ss = rw.sum(ss), sy = rw.sum(sy), yy = rw.sum(yy);
      const bool upd = (sy > 1e-10 * sqrt(ss) * sqrt(yy)) && (sy > 0.0);
      if (upd) {
        double* s = p.S + ((size_t)e * m + head) * D;
        double* y = p.Y + ((size_t)e * m + head) * D;
        for (int i = lane; i < D; i += kStride) {
          s[i] = xt[i] - x[i];
          y[i] = gt[i] - g[i];
        }
        if (lane == 0) p.rho[(size_t)e * m + head] = 1.0 / sy;
        head = (head + 1) % m;
        count = count + 1 < m ? count + 1 : m;
      }
      const double rel = (f - ft) / fmax(fmax(fabs(f), fabs(ft)), 1.0);
      for (int i = lane; i < D; i += kStride) {
        x[i] = xt[i];
        g[i] = gt[i];
      }
      rw.sync();
      fnew = ft;
      iters += 1;
      lsc = 0;
      const bool conv = (lb_projected_grad_inf<WPR>(p, e, rw) <= p.gtol) || (rel <= p.ftol);
      if (conv) {
        flags = (flags & ~kLbActive) | kLbConverged;
      } else if (iters >= p.maxiter) {
        flags &= ~kLbActive;
      } else {
        fresh_dir = true;
      }
    } else {
      // rejected: shrink the step (quadratic interpolation, safeguarded)
      lsc += 1;
      const double denom = 2.0 * (ft - f - dec);
      const double tq = (fin && denom > 0.0) ? -dec / fmax(denom, 1e-300) : 0.5;
      tcur *= fmin(fmax(tq, 0.1), 0.5);
      if (lsc >= p.max_ls) {  // the line search has reached the resolution of the objective
        flags &= ~kLbActive;
        flags |= (iters > 0) ? kLbConverged : kLbFailed;
      }
    }
  }
  rw.sync();
  if (fresh_dir) {
    lb_direction<WPR>(p, e, rw, al, count, head);
    tcur = 1.0;
    if (count == 0) {  // no curvature yet: cautious first step min(1, 1/||d||)
      double dn = 0.0;
      for (int i = lane; i < D; i += kStride) dn = fma(d[i], d[i], dn);
      dn = sqrt(rw.sum(dn));
      tcur = fmin(1.0, 1.0 / fmax(dn, 1e-300));
    }
  }
  rw.sync();
  if (lane == 0) {
    p.f[e] = fnew;
    p.t[e] = tcur;
    p.count[e] = count, p.head[e] = head, p.iters[e] = iters, p.ls_count[e] = lsc;
    p.flags[e] = flags;
  }
  if (flags & kLbActive) {
    for (int i = lane; i < D; i += kStride) {
      double v = fma(tcur, d[i], x[i]);
      if (p.lower != nullptr) v = fmax(v, p.lower[i]);
      xt[i] = v;
    }
  }
}

inline int launch_lbfgs_step(const LbfgsParams& p, void* stream) {
  if (p.E <= 0 || p.D <= 0 || p.m <= 0 || p.m > kLbMaxHistory) return SCAML_E_ARG;
  const bool wide = p.D >= kLbWideMinD;  // by shape only: the reduction order of a row never depends on the batch
  const int grid = wide ? p.E : (p.E + kLbWarps - 1) / kLbWarps;
  const size_t smem = sizeof(double) * (wide ? (kLbMaxHistory + kLbWideWarps) : kLbWarps * (kLbMaxHistory + 1));
  if (wide) return launch(scaml_lbfgs_step_kernel<kLbWideWarps>, grid, kLbWideWarps * 32, smem, stream, p);
  return launch(scaml_lbfgs_step_kernel<1>, grid, kLbWarps * 32, smem, stream, p);
}

}  // namespace scaml
