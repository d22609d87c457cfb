// CPU emulation of the handful of CUDA constructs the ScaML-GP kernels use.
//
// TEST INFRASTRUCTURE ONLY.  It lets the *same* kernel source be compiled with g++
// (-DSCAML_EMU) and executed one CTA at a time with one OS thread per CUDA thread, so
// the block-level algorithm (indexing, layouts, barriers' placement) can be checked
// against the oracle in the CPU-only CI container.  It is never loaded by the product
// package (scamlgp_b200 refuses to run without the sm_100a library and a GPU).
//
// Fidelity: __syncthreads / __syncwarp are real barriers, warp shuffles exchange through
// per-warp slots, cp.async is a synchronous memcpy.  Data races that the real hardware
// could expose between barriers are NOT detected (compute-sanitizer on the GPU box is
// used for that).
#pragma once
#include <cxxabi.h>
#include <dlfcn.h>
#include <pthread.h>
#include <sched.h>

#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <thread>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __restrict__
#define __launch_bounds__(...)
#define __shared__ static  // one CTA runs at a time; its OS threads share the static
#define __align__(n) alignas(n)

typedef void* cudaStream_t;
typedef int cudaError_t;
#define cudaSuccess 0

struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};

namespace cuemu {
struct BlockCtx {
  pthread_barrier_t bar;
  pthread_barrier_t wbar[64];
  pthread_barrier_t nbar[8];  // named barriers 1..8 (bar.sync id, 128): groups of four warps
  alignas(16) unsigned char slot[64][32][16];
  unsigned char* dyn_smem = nullptr;
  int nthreads = 0;
};
inline BlockCtx*& ctx() {
  static BlockCtx* c = nullptr;
  return c;
}
inline dim3& tIdx() {
  static thread_local dim3 t;
  return t;
}
inline dim3& bIdx() {
  static dim3 b;
  return b;
}
inline dim3& bDim() {
  static dim3 b;
  return b;
}
inline dim3& gDim() {
  static dim3 g;
  return g;
}
inline void block_sync() { pthread_barrier_wait(&ctx()->bar); }
inline void warp_sync() { pthread_barrier_wait(&ctx()->wbar[tIdx().x >> 5]); }
inline void named_sync(int id) { pthread_barrier_wait(&ctx()->nbar[id - 1]); }  // 128 participants
template <class T>
inline T shfl(T v, int src) {
  static_assert(sizeof(T) <= 16, "shfl payload");
  BlockCtx* c = ctx();
  const int w = tIdx().x >> 5, l = tIdx().x & 31;
  std::memcpy(c->slot[w][l], &v, sizeof(T));
  warp_sync();
  T r;
  std::memcpy(&r, c->slot[w][src & 31], sizeof(T));
  warp_sync();
  return r;
}

// mma.sync.m8n8k4.f64 with the PTX fragment layout (see scaml_device.cuh)
inline void dmma884(double (&d)[2], double a, double b) {
  BlockCtx* c = ctx();
  const int w = tIdx().x >> 5, l = tIdx().x & 31;
  double ab[2] = {a, b};
  std::memcpy(c->slot[w][l], ab, 16);
  warp_sync();
  const int g = l >> 2, t = l & 3;
  for (int k = 0; k < 4; ++k) {
    double ak[2], b0[2], b1[2];
    std::memcpy(ak, c->slot[w][g * 4 + k], 16);
    std::memcpy(b0, c->slot[w][(2 * t) * 4 + k], 16);
    std::memcpy(b1, c->slot[w][(2 * t + 1) * 4 + k], 16);
    d[0] = std::fma(ak[0], b0[1], d[0]);
    d[1] = std::fma(ak[0], b1[1], d[1]);
  }
  warp_sync();
}

// launch log: the demangled name of every kernel launched (e.g. "void scaml::scaml_grad_contract_kernel<0, 32>(...)"),
// so tests can check which template instantiation a shape dispatches to
inline std::vector<std::string>& launch_log() {
  static std::vector<std::string> v;
  return v;
}
template <class F>
void log_launch(F kernel) {
  Dl_info info;
  std::string name = "?";
  if (dladdr(reinterpret_cast<void*>(kernel), &info) != 0 && info.dli_sname != nullptr) {
    int status = 0;
    char* dem = abi::__cxa_demangle(info.dli_sname, nullptr, nullptr, &status);
    name = (status == 0 && dem != nullptr) ? dem : info.dli_sname;
    std::free(dem);
  }
  launch_log().push_back(name);
}

template <class F, class... A>
void launch(dim3 grid, dim3 block, size_t smem_bytes, F kernel, A... args) {
  log_launch(kernel);
  gDim() = grid;
  bDim() = block;
  const int nt = (int)block.x;
  const int nw = (nt + 31) / 32;
  for (unsigned long long b = 0; b < (unsigned long long)grid.x * grid.y * grid.z; ++b) {
    const dim3 cta((unsigned)(b % grid.x), (unsigned)(b / grid.x % grid.y), (unsigned)(b / grid.x / grid.y));
    BlockCtx c;
    c.nthreads = nt;
    pthread_barrier_init(&c.bar, nullptr, nt);
    for (int w = 0; w < nw; ++w) {
      int cnt = (w == nw - 1 && (nt & 31)) ? (nt & 31) : 32;
      pthread_barrier_init(&c.wbar[w], nullptr, cnt);
    }
    for (int i = 0; i < 8; ++i) pthread_barrier_init(&c.nbar[i], nullptr, nt < 128 ? nt : 128);
    void* mem = nullptr;
    if (posix_memalign(&mem, 1024, smem_bytes + 1024) != 0) abort();
    std::memset(mem, 0xCD, smem_bytes + 1024);  // poison: uninitialised smem reads show up as NaN-ish
    c.dyn_smem = (unsigned char*)mem;
    ctx() = &c;
    bIdx() = cta;
    std::vector<std::thread> th;
    th.reserve(nt);
    for (int t = 0; t < nt; ++t)
      th.emplace_back([=]() {
        tIdx() = dim3((unsigned)t, 0, 0);
        kernel(args...);
      });
    for (auto& t : th) t.join();
    // canary: a kernel that writes past the dynamic shared memory it asked for would corrupt a neighbour on the GPU
    for (size_t i = smem_bytes; i < smem_bytes + 1024; ++i)
      if (((unsigned char*)mem)[i] != 0xCD) {
        std::fprintf(stderr, "cuda_emu: CTA (%u, %u, %u) wrote past its %zu bytes of dynamic shared memory at %zu\n",
                     cta.x, cta.y, cta.z, smem_bytes, i);
        std::abort();
      }
    pthread_barrier_destroy(&c.bar);
    for (int w = 0; w < nw; ++w) pthread_barrier_destroy(&c.wbar[w]);
    for (int i = 0; i < 8; ++i) pthread_barrier_destroy(&c.nbar[i]);
    free(mem);
    ctx() = nullptr;
  }
}
}  // namespace cuemu

#define threadIdx (cuemu::tIdx())
#define blockIdx (cuemu::bIdx())
#define blockDim (cuemu::bDim())
#define gridDim (cuemu::gDim())

inline void __syncthreads() { cuemu::block_sync(); }
inline void __syncwarp(unsigned = 0xffffffffu) { cuemu::warp_sync(); }
template <class T>
inline T __shfl_sync(unsigned, T v, int src) {
  return cuemu::shfl(v, src);
}
template <class T>
inline T __shfl_xor_sync(unsigned, T v, int m) {
  return cuemu::shfl(v, (int)((threadIdx.x & 31) ^ m));
}
template <class T>
inline T __shfl_down_sync(unsigned, T v, int d) {
  int l = threadIdx.x & 31;
  return cuemu::shfl(v, l + d < 32 ? l + d : l);
}
inline int __any_sync(unsigned, int pred) {
  int v = pred ? 1 : 0;
  for (int o = 16; o > 0; o >>= 1) v |= cuemu::shfl(v, (int)((threadIdx.x & 31) ^ o));
  return v;
}
template <class T>
inline T __ldcg(const T* p) {
  return *p;
}
template <class T>
inline T __ldg(const T* p) {
  return *p;
}
inline void __threadfence_block() { __atomic_thread_fence(__ATOMIC_SEQ_CST); }
inline int atomicAdd(int* p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
inline double rsqrt(double x) { return 1.0 / std::sqrt(x); }
inline double fma_emu(double a, double b, double c) { return std::fma(a, b, c); }
using std::exp;
using std::fabs;
using std::fmax;
using std::isfinite;
using std::lgamma;
using std::log;
using std::sqrt;
