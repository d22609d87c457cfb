// Device-side helpers shared by the ScaML-GP kernels, and the host-side launch and dispatch helpers (sm_100a; also
// compiles under the CPU logic emulation in emu/cuda_emu.h when SCAML_EMU is defined).
#pragma once

#ifdef SCAML_EMU
#include "emu/cuda_emu.h"
#define SCAML_DEVICE inline
#define SCAML_DYN_SMEM(type, name) type* name = reinterpret_cast<type*>(cuemu::ctx()->dyn_smem)
struct alignas(16) double2 {
  double x, y;
};
inline double2 make_double2(double x, double y) { return double2{x, y}; }
#else
#include <cuda_runtime.h>
#define SCAML_DEVICE __device__ __forceinline__
#define SCAML_DYN_SMEM(type, name) \
  extern __shared__ __align__(1024) unsigned char name##_raw_[]; \
  type* name = reinterpret_cast<type*>(name##_raw_)
#endif

#include <stdint.h>

#include <type_traits>

#include "../../include/scaml_b200.h"

namespace scaml {

constexpr int kBS = 32;           // tile edge
constexpr int kTile = kBS * kBS;  // doubles per tile (8 KB)
constexpr int kSB = 64;           // super-tile edge (2x2 tiles)
constexpr int kMaxP = 34;  // d <= 32
constexpr double kLog2Pi = 1.8378770664093454835606594728112;

// ----------------------------------------------------------------------------------- //
// async copies (LDGSTS, L2-only caching: the workspace is rewritten in place, L1 must
// never serve a stale line)
// ----------------------------------------------------------------------------------- //
SCAML_DEVICE void cp_async16(double* smem_dst, const double* gsrc) {
#ifdef SCAML_EMU
  std::memcpy(smem_dst, gsrc, 16);
#else
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gsrc) : "memory");
#endif
}
SCAML_DEVICE void cp_async_commit() {
#ifndef SCAML_EMU
  asm volatile("cp.async.commit_group;\n" ::: "memory");
#endif
}
template <int N>
SCAML_DEVICE void cp_async_wait() {
#ifndef SCAML_EMU
  asm volatile("cp.async.wait_group %0;\n" ::"n"(N) : "memory");
#endif
}

// streaming (evict-first) 16-byte global accesses for write-once / read-once scratch
SCAML_DEVICE void st_stream(double2* p, double2 v) {
#ifdef SCAML_EMU
  *p = v;
#else
  __stcs(p, v);
#endif
}
SCAML_DEVICE double2 ld_stream(const double2* p) {
#ifdef SCAML_EMU
  return *p;
#else
  return __ldcs(p);
#endif
}

// FP64 tensor-core MMA (DMMA): D(8x8) += A(8x4) * B(4x8).  Fragments (PTX ISA, mma.m8n8k4 .f64):
//   a    = A[lane>>2][lane&3]        b = B[lane&3][lane>>2]
//   d[e] = D[lane>>2][2*(lane&3)+e]
SCAML_DEVICE void dmma884(double (&d)[2], double a, double b) {
#ifdef SCAML_EMU
  cuemu::dmma884(d, a, b);
#else
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d[0]), "+d"(d[1])
               : "d"(a), "d"(b));
#endif
}

// the same with the two accumulator elements as separate scalars (accumulators kept in flat arrays)
SCAML_DEVICE void dmma884s(double& d0, double& d1, double a, double b) {
#ifdef SCAML_EMU
  double d[2] = {d0, d1};
  cuemu::dmma884(d, a, b);
  d0 = d[0], d1 = d[1];
#else
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};\n"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
#endif
}

SCAML_DEVICE double warp_sum(double v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

SCAML_DEVICE int tri(int i) { return (i * (i + 1)) >> 1; }

// ----------------------------------------------------------------------------------- //
// exp(x) for x <= 0, branch-free.  libdevice's exp() carries a slow-path branch, so the 8..16
// independent exponentials of an unrolled epilogue are emitted one after the other and each
// is a ~20-deep dependent DFMA chain (measured: "wait" stalls dominate the k* assembly).
// Without control flow the compiler interleaves them.  Table-driven: x = (64 n + j) ln2/64 + r,
// |r| <= ln2/128, exp(x) = 2^n * T[j] * (1 + r (1 + r/2 + r^2/6 + r^3/24 + r^4/120)) with
// T[j] = 2^(j/64) correctly rounded (64 doubles, read through the read-only data path: L1
// resident) -- 10 FP64 instructions and a dependent chain of 9 instead of 17 / 16 for the
// table-free degree-13 polynomial; truncation r^6/720 < 3.6e-17.  Max error < 1.5 ulp on
// [-708, 0] (tests/test_emu_kernels.py); arguments below -708 (incl. -inf) give exp(-708) =
// 3.3e-308 (a k* entry that small is 0 for every purpose), NaN propagates.
// ----------------------------------------------------------------------------------- //
#ifdef SCAML_EMU
#define SCAML_TABLE static const
#else
#define SCAML_TABLE __device__ const
#endif
SCAML_TABLE double kExp2Tab[64] = {
    0x1.0000000000000p+0, 0x1.02c9a3e778061p+0, 0x1.059b0d3158574p+0, 0x1.0874518759bc8p+0,
    0x1.0b5586cf9890fp+0, 0x1.0e3ec32d3d1a2p+0, 0x1.11301d0125b51p+0, 0x1.1429aaea92de0p+0,
    0x1.172b83c7d517bp+0, 0x1.1a35beb6fcb75p+0, 0x1.1d4873168b9aap+0, 0x1.2063b88628cd6p+0,
    0x1.2387a6e756238p+0, 0x1.26b4565e27cddp+0, 0x1.29e9df51fdee1p+0, 0x1.2d285a6e4030bp+0,
    0x1.306fe0a31b715p+0, 0x1.33c08b26416ffp+0, 0x1.371a7373aa9cbp+0, 0x1.3a7db34e59ff7p+0,
    0x1.3dea64c123422p+0, 0x1.4160a21f72e2ap+0, 0x1.44e086061892dp+0, 0x1.486a2b5c13cd0p+0,
    0x1.4bfdad5362a27p+0, 0x1.4f9b2769d2ca7p+0, 0x1.5342b569d4f82p+0, 0x1.56f4736b527dap+0,
    0x1.5ab07dd485429p+0, 0x1.5e76f15ad2148p+0, 0x1.6247eb03a5585p+0, 0x1.6623882552225p+0,
    0x1.6a09e667f3bcdp+0, 0x1.6dfb23c651a2fp+0, 0x1.71f75e8ec5f74p+0, 0x1.75feb564267c9p+0,
    0x1.7a11473eb0187p+0, 0x1.7e2f336cf4e62p+0, 0x1.82589994cce13p+0, 0x1.868d99b4492edp+0,
    0x1.8ace5422aa0dbp+0, 0x1.8f1ae99157736p+0, 0x1.93737b0cdc5e5p+0, 0x1.97d829fde4e50p+0,
    0x1.9c49182a3f090p+0, 0x1.a0c667b5de565p+0, 0x1.a5503b23e255dp+0, 0x1.a9e6b5579fdbfp+0,
    0x1.ae89f995ad3adp+0, 0x1.b33a2b84f15fbp+0, 0x1.b7f76f2fb5e47p+0, 0x1.bcc1e904bc1d2p+0,
    0x1.c199bdd85529cp+0, 0x1.c67f12e57d14bp+0, 0x1.cb720dcef9069p+0, 0x1.d072d4a07897cp+0,
    0x1.d5818dcfba487p+0, 0x1.da9e603db3285p+0, 0x1.dfc97337b9b5fp+0, 0x1.e502ee78b3ff6p+0,
    0x1.ea4afa2a490dap+0, 0x1.efa1bee615a27p+0, 0x1.f50765b6e4540p+0, 0x1.fa7c1819e90d8p+0,
};
#ifdef SCAML_EMU
SCAML_DEVICE int dbl_hi(double x) {
  int64_t b;
  std::memcpy(&b, &x, 8);
  return (int)(b >> 32);
}
SCAML_DEVICE int dbl_lo(double x) {
  int64_t b;
  std::memcpy(&b, &x, 8);
  return (int)(b & 0xffffffff);
}
SCAML_DEVICE double dbl_make(int hi, int lo) {
  const int64_t b = (int64_t)(((uint64_t)(uint32_t)hi << 32) | (uint32_t)lo);
  double x;
  std::memcpy(&x, &b, 8);
  return x;
}
SCAML_DEVICE double exp2_tab(int j) { return kExp2Tab[j]; }
#else
SCAML_DEVICE int dbl_hi(double x) { return __double2hiint(x); }
SCAML_DEVICE int dbl_lo(double x) { return __double2loint(x); }
SCAML_DEVICE double dbl_make(int hi, int lo) { return __hiloint2double(hi, lo); }
SCAML_DEVICE double exp2_tab(int j) { return __ldg(kExp2Tab + j); }
#endif

// U independent exponentials, written step-major so that the U dependent chains are interleaved in the
// instruction stream (in[u] <= 0; out may alias in).  Range handling is ONE clamp of the argument to >= -708
// (compare + two selects; NaN fails the compare and propagates through the FP64 chain, its low word is 0 on
// the GPU so that n = 0): below -708 the function returns exp(-708) = 3.3e-308 instead of a denormal or 0 --
// 18 instructions per value instead of 25 with per-value flush / NaN selects (the k* assemblies are bound by
// issue slots, not by the FP64 pipe).
// TAB = false: table-free variant, x = n ln2 + r, degree-13 polynomial (17 FP64 instructions, no load) for kernels
// whose load / store pipe is the scarce resource (kernel-matrix assembly).
template <int U, bool TAB = true>
SCAML_DEVICE void exp_nonpos_n(const double (&in)[U], double (&out)[U]) {
  const double kMagic = 6755399441055744.0;  // 1.5 * 2^52: adding it rounds to the nearest integer
  double r[U], p[U], tab[U];
  int n[U];
  if (TAB) {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const double x = (in[u] < -708.0) ? -708.0 : in[u];
      const double t = fma(x, 92.33248261689366, kMagic);  // 64 / ln 2
      const int k = dbl_lo(t);                             // round(64 x / ln 2) = 64 n + j, n >= -1022
      tab[u] = exp2_tab(k & 63);
      n[u] = k >> 6;
      const double kf = t - kMagic;
      // ln2/64 split: the high part has 35 significant bits, so kf * hi is exact for |kf| < 2^17
      r[u] = fma(kf, -0x1.1cf79abc9e3b4p-42, fma(kf, -0x1.62e42fef80000p-7, x));
      p[u] = fma(8.3333333333333332177e-03, r[u], 4.1666666666666664354e-02);  // 1/5!, 1/4!
#ifdef SCAML_EMU
      if (x != x) n[u] = 0;  // host NaNs keep their payload: low word not necessarily 0
#endif
    }
#pragma unroll
    for (int u = 0; u < U; ++u) p[u] = fma(p[u], r[u], 1.6666666666666665741e-01);
#pragma unroll
    for (int u = 0; u < U; ++u) p[u] = fma(p[u], r[u], 0.5);
#pragma unroll
    for (int u = 0; u < U; ++u) p[u] = fma(p[u], r[u], 1.0);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const double q = fma(tab[u], p[u] * r[u], tab[u]);  // T (1 + r poly): in [0.99, 2); NaN for NaN
      out[u] = dbl_make(dbl_hi(q) + n[u] * 1048576, dbl_lo(q));
    }
  } else {
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const double x = (in[u] < -708.0) ? -708.0 : in[u];
      const double t = fma(x, 1.4426950408889634074, kMagic);
      n[u] = dbl_lo(t);  // round(x / ln 2) >= -1022
      const double nf = t - kMagic;
      r[u] = fma(nf, -1.90821492927058770002e-10, fma(nf, -6.93147180369123816490e-01, x));
      p[u] = fma(1.6059043836821614599e-10, r[u], 2.0876756987868098979e-09);  // 1/13!, 1/12!
#ifdef SCAML_EMU
      if (x != x) n[u] = 0;
#endif
    }
    const double c[11] = {2.5052108385441718775e-08, 2.7557319223985890653e-07, 2.7557319223985892511e-06,
                          2.4801587301587301566e-05, 1.9841269841269841253e-04, 1.3888888888888889419e-03,
                          8.3333333333333332177e-03, 4.1666666666666664354e-02, 1.6666666666666665741e-01, 0.5, 1.0};
#pragma unroll
    for (int k = 0; k < 11; ++k)
#pragma unroll
      for (int u = 0; u < U; ++u) p[u] = fma(p[u], r[u], c[k]);
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const double q = fma(p[u], r[u], 1.0);  // in [0.7, 1.42]
      out[u] = dbl_make(dbl_hi(q) + n[u] * 1048576, dbl_lo(q));
    }
  }
}
SCAML_DEVICE double exp_nonpos(double x) {
  const double in[1] = {x};
  double out[1];
  exp_nonpos_n<1>(in, out);
  return out[0];
}

// ----------------------------------------------------------------------------------- //
// stationary kernels: kappa(r^2) and kd = -2 dkappa/dr^2 (SURVEY A.4/A.5)
// ----------------------------------------------------------------------------------- //
template <int KIND>
SCAML_DEVICE double kappa_of(double r2) {
  if (KIND == SCAML_KERNEL_RBF) return exp_nonpos(-0.5 * r2);
  const double r = sqrt(r2 < 1e-30 ? 1e-30 : r2);
  if (KIND == SCAML_KERNEL_MATERN12) return exp_nonpos(-r);
  if (KIND == SCAML_KERNEL_MATERN32) {
    const double s3 = 1.7320508075688772935;
    return (1.0 + s3 * r) * exp_nonpos(-s3 * r);
  }
  const double s5 = 2.2360679774997896964;
  return (1.0 + s5 * r + (5.0 / 3.0) * r * r) * exp_nonpos(-s5 * r);
}

template <int KIND>
SCAML_DEVICE void kappa_pair(double r2, double& k, double& kd) {
  if (KIND == SCAML_KERNEL_RBF) {
    k = exp_nonpos(-0.5 * r2);
    kd = k;
    return;
  }
  const double r = sqrt(r2 < 1e-30 ? 1e-30 : r2);
  if (KIND == SCAML_KERNEL_MATERN12) {
    k = exp_nonpos(-r);
    kd = (r2 > 0.0) ? k / r : 0.0;
    return;
  }
  if (KIND == SCAML_KERNEL_MATERN32) {
    const double s3 = 1.7320508075688772935;
    const double e = exp_nonpos(-s3 * r);
    k = (1.0 + s3 * r) * e;
    kd = 3.0 * e;
    return;
  }
  const double s5 = 2.2360679774997896964;
  const double e = exp_nonpos(-s5 * r);
  k = (1.0 + s5 * r + (5.0 / 3.0) * r * r) * e;
  kd = (5.0 / 3.0) * (1.0 + s5 * r) * e;
}

// U kernel values at once (independent chains interleaved): k[u] = kappa(r2[u]), kd[u] = -2 dkappa/dr^2
template <int KIND, int U, bool WITH_KD, bool TAB = true>
SCAML_DEVICE void kappa_n(const double (&r2)[U], double (&k)[U], double (&kd)[U]) {
  double arg[U], r[U], e[U];
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (KIND == SCAML_KERNEL_RBF) {
      arg[u] = -0.5 * r2[u];
    } else {
      r[u] = sqrt(r2[u] < 1e-30 ? 1e-30 : r2[u]);
      arg[u] = (KIND == SCAML_KERNEL_MATERN12)   ? -r[u]
               : (KIND == SCAML_KERNEL_MATERN32) ? -1.7320508075688772935 * r[u]
                                                 : -2.2360679774997896964 * r[u];
    }
  }
  exp_nonpos_n<U, TAB>(arg, e);
#pragma unroll
  for (int u = 0; u < U; ++u) {
    if (KIND == SCAML_KERNEL_RBF) {
      k[u] = e[u];
      if (WITH_KD) kd[u] = e[u];
    } else if (KIND == SCAML_KERNEL_MATERN12) {
      const double kk = e[u];
      if (WITH_KD) kd[u] = (r2[u] > 0.0) ? e[u] / r[u] : 0.0;
      k[u] = kk;
    } else if (KIND == SCAML_KERNEL_MATERN32) {
      const double kk = (1.0 + 1.7320508075688772935 * r[u]) * e[u];
      if (WITH_KD) kd[u] = 3.0 * e[u];
      k[u] = kk;
    } else {
      const double s5r = 2.2360679774997896964 * r[u];
      const double kk = (1.0 + s5r + (5.0 / 3.0) * r[u] * r[u]) * e[u];
      if (WITH_KD) kd[u] = (5.0 / 3.0) * (1.0 + s5r) * e[u];
      k[u] = kk;
    }
  }
}

// runtime-dispatched variant for the non-hot callers
SCAML_DEVICE double kappa_rt(int kind, double r2) {
  switch (kind) {
    case SCAML_KERNEL_RBF: return kappa_of<SCAML_KERNEL_RBF>(r2);
    case SCAML_KERNEL_MATERN12: return kappa_of<SCAML_KERNEL_MATERN12>(r2);
    case SCAML_KERNEL_MATERN32: return kappa_of<SCAML_KERNEL_MATERN32>(r2);
    default: return kappa_of<SCAML_KERNEL_MATERN52>(r2);
  }
}

// ----------------------------------------------------------------------------------- //
// priors (torch.distributions Gamma / LogNormal log densities) and the Interval transform
// ----------------------------------------------------------------------------------- //
SCAML_DEVICE double log_prior(int kind, double p1, double p2, double x) {
  if (kind == SCAML_PRIOR_GAMMA) return p1 * log(p2) + (p1 - 1.0) * log(x) - p2 * x - lgamma(p1);
  if (kind == SCAML_PRIOR_LOGNORMAL) {
    const double lx = log(x);
    const double t = lx - p1;
    return -lx - log(p2) - 0.5 * kLog2Pi - t * t / (2.0 * p2 * p2);
  }
  return 0.0;
}
SCAML_DEVICE double dlog_prior(int kind, double p1, double p2, double x) {
  if (kind == SCAML_PRIOR_GAMMA) return (p1 - 1.0) / x - p2;
  if (kind == SCAML_PRIOR_LOGNORMAL) return -1.0 / x - (log(x) - p1) / (p2 * p2 * x);
  return 0.0;
}
SCAML_DEVICE double sigmoid(double x) { return 1.0 / (1.0 + exp(-x)); }

// target points padded to whole 8-column DMMA blocks (shared by the conditioning and the gradient kernels)
inline int cond_ntp(int n_t) { return ((n_t + 7) / 8) * 8; }

// ----------------------------------------------------------------------------------- //
// host side: every kernel launch and every choice of a kernel-family template
// ----------------------------------------------------------------------------------- //
// kern<<<grid, block, smem, stream>>>(args...) on the GPU, CTA by CTA on the CPU emulation; 0 or the CUDA error.
// Dynamic shared memory above 48 KB needs the opt-in attribute.  It is per device and the sharded path drives several
// GPUs from one process, so it is set on every such launch rather than cached.
template <class... P, class... A>
inline int launch(void (*kern)(P...), dim3 grid, dim3 block, size_t smem, void* stream, const A&... args) {
#ifdef SCAML_EMU
  (void)stream;
  cuemu::launch(grid, block, smem, kern, args...);
  return 0;
#else
  if (smem > 48 * 1024) {
    const cudaError_t err = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (err != cudaSuccess) return (int)err;
  }
  kern<<<grid, block, smem, (cudaStream_t)stream>>>(args...);
  return (int)cudaGetLastError();
#endif
}

// CTAs of a kernel that strides over `work` items by gridDim.x: at most gpu_cap on the GPU.  The emulation runs CTAs
// one after another, so it runs two: enough to exercise the stride.
inline int stride_grid(long long work, long long gpu_cap = INT32_MAX) {
#ifdef SCAML_EMU
  gpu_cap = 2;
#endif
  return (int)(work < gpu_cap ? work : gpu_cap);
}

// f(std::integral_constant<int, SCAML_KERNEL_*>) for the kernel-family id `kernel`; SCAML_E_ARG outside 0..3
template <class F>
inline int dispatch_kind(int kernel, F&& f) {
  switch (kernel) {
    case SCAML_KERNEL_RBF: return f(std::integral_constant<int, SCAML_KERNEL_RBF>());
    case SCAML_KERNEL_MATERN12: return f(std::integral_constant<int, SCAML_KERNEL_MATERN12>());
    case SCAML_KERNEL_MATERN32: return f(std::integral_constant<int, SCAML_KERNEL_MATERN32>());
    case SCAML_KERNEL_MATERN52: return f(std::integral_constant<int, SCAML_KERNEL_MATERN52>());
    default: return SCAML_E_ARG;
  }
}

// f(std::integral_constant<int, DMAX>) for the kernels that keep per-dimension registers: DMAX = 8, 16 or 32 >= d
template <class F>
inline int dispatch_dmax(int d, F&& f) {
  if (d <= 8) return f(std::integral_constant<int, 8>());
  if (d <= 16) return f(std::integral_constant<int, 16>());
  return f(std::integral_constant<int, 32>());
}

}  // namespace scaml
