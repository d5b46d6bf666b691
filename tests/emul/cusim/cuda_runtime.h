// cusim/cuda_runtime.h -- TEST INFRASTRUCTURE, never part of the product.
//
// A stand-in for the CUDA runtime and the device language that lets the product's .cu sources be
// compiled by g++ and RUN ON THE HOST, so that the kernels' logic -- warp shuffles, ballots,
// shared-memory staging, block barriers, atomics -- can be exercised where there is no GPU
// (tests/test_sim.py; the build container has none).  It is a functional model, not a timing model:
//
//   * a kernel launch runs the blocks of the grid one after the other;
//   * the threads of a block are fibers (ucontext) scheduled round robin; a thread runs until it
//     reaches a barrier or a warp collective, where it waits for the others it names;
//   * __syncthreads / __syncwarp / __shfl*_sync / __ballot_sync / __any_sync / __reduce_*_sync are
//     rendezvous among the named lanes (lanes that have left the kernel count as arrived);
//   * atomics are the compiler's atomic builtins;
//   * __shared__ is `static thread_local` (one block per emulated device is alive at a time; the
//     ranks of a partitioned graph are threads), dynamic shared memory a buffer per block;
//   * streams and events are immediate; device memory is host memory;
//   * a cooperative launch keeps every block of its grid alive at once (grid-wide barriers).
//
// tests/emul/cusim_build.py rewrites `kernel<<<grid, block, smem, stream>>>(args)` into
// cusim::Launch(grid, block, smem, stream)(kernel)(args), `extern __shared__ T name[]` into a
// pointer to the block's buffer and cudaLaunchCooperativeKernel into its typed form; nothing else
// in the sources is touched.
#pragma once
#include <math.h>
#include <stddef.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <time.h>

#include <functional>
#include <type_traits>
#include <utility>

#define CUSIM 1

// ---------------------------------------------------------------- language
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __shared__ static thread_local      // ranks of a partitioned graph are threads (tests/test_sim.py)
#define __align__(n) alignas(n)
#define __constant__ static

struct uint2 { uint32_t x, y; };
struct alignas(8) uint2a { uint32_t x, y; };
struct alignas(16) uint4 { uint32_t x, y, z, w; };
struct uint3 { uint32_t x, y, z; };
struct int2 { int32_t x, y; };
struct float2 { float x, y; };
struct dim3 {
  uint32_t x, y, z;
  dim3(uint32_t x_ = 1, uint32_t y_ = 1, uint32_t z_ = 1) : x(x_), y(y_), z(z_) {}
};
static inline uint2 make_uint2(uint32_t x, uint32_t y) { return uint2{x, y}; }
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { return uint4{x, y, z, w}; }
static inline int2 make_int2(int32_t x, int32_t y) { return int2{x, y}; }
static inline float2 make_float2(float x, float y) { return float2{x, y}; }

typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorNotSupported = 801, cudaErrorMemoryAllocation = 2 };
typedef struct cusim_stream *cudaStream_t;
typedef struct cusim_event *cudaEvent_t;
enum cudaMemcpyKind { cudaMemcpyHostToHost, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };

namespace cusim {

struct ThreadCtx {              // what the running fiber sees
  uint3 tid;
};
struct BlockCtx {
  uint3 bid;
  dim3 bdim, gdim;
  void *dyn_smem;
};
extern thread_local ThreadCtx *T;
extern thread_local BlockCtx *B;

// rendezvous primitives (cusim.cpp)
void block_barrier();
// every lane named in mask deposits v; returns a pointer to the 32 deposited values and the mask of
// lanes that really arrived (lanes that left the kernel do not deposit)
const uint64_t *warp_collect(uint32_t mask, uint64_t v, uint32_t *arrived);
void warp_release();            // the caller has read the values

void run_grid(dim3 grid, dim3 block, size_t smem, const std::function<void()> &body);
void run_grid_coop(dim3 grid, dim3 block, size_t smem, const std::function<void()> &body);
void grid_barrier();
void set_order(uint64_t mode);

struct Launch {
  dim3 g, b;
  size_t smem;
  Launch(dim3 g_, dim3 b_, size_t smem_ = 0, cudaStream_t = nullptr) : g(g_), b(b_), smem(smem_) {}
  template <typename... P>
  struct Bound {
    const Launch &l;
    void (*k)(P...);
    template <typename... A>
    void operator()(A &&...a) const {
      void (*kk)(P...) = k;
      // arguments are copied once, as a launch does
      auto call = [kk, &a...]() { kk(static_cast<P>(a)...); };
      run_grid(l.g, l.b, l.smem, call);
    }
  };
  template <typename... P>
  Bound<P...> operator()(void (*k)(P...)) const { return Bound<P...>{*this, k}; }
};

// cooperative launch: cudaLaunchCooperativeKernel((const void *) k, grid, block, args, smem, stream)
// is rewritten into cusim::coop_launch(k, grid, block, args, smem, stream), which knows k's types
template <typename... P, size_t... I>
static inline void coop_call(void (*k)(P...), void **args, std::index_sequence<I...>) {
  k(*static_cast<typename std::remove_reference<P>::type *>(args[I])...);
}
template <typename... P>
static inline int coop_launch(void (*k)(P...), dim3 g, dim3 b, void **args, size_t smem, cudaStream_t) {
  auto call = [k, args]() { coop_call(k, args, std::index_sequence_for<P...>{}); };
  run_grid_coop(g, b, smem, call);
  return 0;
}

}  // namespace cusim

#define threadIdx (::cusim::T->tid)
#define blockIdx (::cusim::B->bid)
#define blockDim (::cusim::B->bdim)
#define gridDim (::cusim::B->gdim)

// ---------------------------------------------------------------- device functions
static inline void __syncthreads() { cusim::block_barrier(); }

static inline uint32_t cusim_lane() { return threadIdx.x & 31u; }

static inline void __syncwarp(uint32_t mask = 0xffffffffu) {
  uint32_t arrived;
  cusim::warp_collect(mask, 0, &arrived);
  cusim::warp_release();
}
static inline uint32_t __ballot_sync(uint32_t mask, int pred) {
  uint32_t arrived, r = 0;
  const uint64_t *v = cusim::warp_collect(mask, pred ? 1u : 0u, &arrived);
  for (uint32_t l = 0; l < 32; l++)
    if (((arrived >> l) & 1u) && v[l]) r |= 1u << l;
  cusim::warp_release();
  return r;
}
static inline int __any_sync(uint32_t mask, int pred) { return __ballot_sync(mask, pred) != 0u; }
static inline int __all_sync(uint32_t mask, int pred) {
  uint32_t arrived, r = 1;
  const uint64_t *v = cusim::warp_collect(mask, pred ? 1u : 0u, &arrived);
  for (uint32_t l = 0; l < 32; l++)
    if (((arrived >> l) & 1u) && !v[l]) r = 0;
  cusim::warp_release();
  return (int) r;
}
template <typename V>
static inline uint64_t cusim_bits(V v) {
  static_assert(sizeof(V) <= 8, "shuffle operand");
  uint64_t b = 0;
  memcpy(&b, &v, sizeof(V));
  return b;
}
template <typename V>
static inline V cusim_unbits(uint64_t b) {
  V v;
  memcpy(&v, &b, sizeof(V));
  return v;
}
template <typename V>
static inline V cusim_shfl_from(uint32_t mask, V var, uint32_t src, bool valid) {
  uint32_t arrived;
  const uint64_t *v = cusim::warp_collect(mask, cusim_bits(var), &arrived);
  V r = var;
  if (valid && ((arrived >> (src & 31u)) & 1u)) r = cusim_unbits<V>(v[src & 31u]);
  cusim::warp_release();
  return r;
}
template <typename V>
static inline V __shfl_sync(uint32_t mask, V var, int src, int width = 32) {
  (void) width;
  return cusim_shfl_from(mask, var, (uint32_t) src & 31u, true);
}
template <typename V>
static inline V __shfl_up_sync(uint32_t mask, V var, unsigned delta, int width = 32) {
  (void) width;
  const uint32_t l = cusim_lane();
  return cusim_shfl_from(mask, var, l - delta, l >= delta);
}
template <typename V>
static inline V __shfl_down_sync(uint32_t mask, V var, unsigned delta, int width = 32) {
  (void) width;
  const uint32_t l = cusim_lane();
  return cusim_shfl_from(mask, var, l + delta, l + delta < 32u);
}
template <typename V>
static inline V __shfl_xor_sync(uint32_t mask, V var, int lanemask, int width = 32) {
  (void) width;
  return cusim_shfl_from(mask, var, cusim_lane() ^ (uint32_t) lanemask, true);
}
template <typename V, typename F>
static inline V cusim_reduce(uint32_t mask, V var, F f) {
  uint32_t arrived;
  const uint64_t *v = cusim::warp_collect(mask, cusim_bits(var), &arrived);
  V r = var;
  for (uint32_t l = 0; l < 32; l++)
    if (((arrived & mask) >> l) & 1u) r = f(r, cusim_unbits<V>(v[l]));
  cusim::warp_release();
  return r;
}
static inline uint32_t __reduce_or_sync(uint32_t m, uint32_t v) { return cusim_reduce(m, v, [](uint32_t a, uint32_t b) { return a | b; }); }
static inline uint32_t __reduce_and_sync(uint32_t m, uint32_t v) { return cusim_reduce(m, v, [](uint32_t a, uint32_t b) { return a & b; }); }
static inline uint32_t __reduce_max_sync(uint32_t m, uint32_t v) { return cusim_reduce(m, v, [](uint32_t a, uint32_t b) { return a > b ? a : b; }); }
static inline uint32_t __reduce_min_sync(uint32_t m, uint32_t v) { return cusim_reduce(m, v, [](uint32_t a, uint32_t b) { return a < b ? a : b; }); }
static inline int __reduce_max_sync(uint32_t m, int v) { return cusim_reduce(m, v, [](int a, int b) { return a > b ? a : b; }); }
static inline int __reduce_min_sync(uint32_t m, int v) { return cusim_reduce(m, v, [](int a, int b) { return a < b ? a : b; }); }
static inline uint32_t __reduce_add_sync(uint32_t m, uint32_t v) {
  // own value is folded in by the loop as well: start from the neutral element
  uint32_t arrived;
  const uint64_t *p = cusim::warp_collect(m, v, &arrived);
  uint32_t r = 0;
  for (uint32_t l = 0; l < 32; l++)
    if (((arrived & m) >> l) & 1u) r += (uint32_t) p[l];
  cusim::warp_release();
  return r;
}

// atomics: GCC builtins -- the fibers of one emulated device share a host thread, but the ranks of
// a partitioned graph are threads that store into each other's buffers (peer memory)
template <typename A, typename V> static inline A atomicAdd(A *p, V v) { return __atomic_fetch_add(p, (A) v, __ATOMIC_SEQ_CST); }
template <typename A, typename V> static inline A atomicSub(A *p, V v) { return __atomic_fetch_sub(p, (A) v, __ATOMIC_SEQ_CST); }
template <typename A, typename V> static inline A atomicOr(A *p, V v) { return __atomic_fetch_or(p, (A) v, __ATOMIC_SEQ_CST); }
template <typename A, typename V> static inline A atomicAnd(A *p, V v) { return __atomic_fetch_and(p, (A) v, __ATOMIC_SEQ_CST); }
template <typename A, typename V> static inline A atomicExch(A *p, V v) { return __atomic_exchange_n(p, (A) v, __ATOMIC_SEQ_CST); }
template <typename A, typename V, typename W> static inline A atomicCAS(A *p, V cmp, W v) {
  A expected = (A) cmp;
  __atomic_compare_exchange_n(p, &expected, (A) v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST);
  return expected;
}
template <typename A, typename V> static inline A atomicMax(A *p, V v) {
  A o = __atomic_load_n(p, __ATOMIC_SEQ_CST);
  while ((A) v > o && !__atomic_compare_exchange_n(p, &o, (A) v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) {}
  return o;
}
template <typename A, typename V> static inline A atomicMin(A *p, V v) {
  A o = __atomic_load_n(p, __ATOMIC_SEQ_CST);
  while ((A) v < o && !__atomic_compare_exchange_n(p, &o, (A) v, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) {}
  return o;
}
static inline void __threadfence() {}
static inline void __threadfence_block() {}

template <typename V> static inline V __ldcs(const V *p) { return *p; }
template <typename V> static inline V __ldcg(const V *p) { return *p; }
template <typename V> static inline V __ldg(const V *p) { return *p; }
template <typename V> static inline void __stcs(V *p, V v) { *p = v; }
template <typename V> static inline void __stcg(V *p, V v) { *p = v; }

static inline int __popc(uint32_t x) { return __builtin_popcount(x); }
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __clz(int x) { return x == 0 ? 32 : __builtin_clz((uint32_t) x); }
static inline int __clzll(long long x) { return x == 0 ? 64 : __builtin_clzll((unsigned long long) x); }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline uint32_t __brev(uint32_t x) {
  uint32_t r = 0;
  for (int i = 0; i < 32; i++) r |= ((x >> i) & 1u) << (31 - i);
  return r;
}
// round-to-nearest float intrinsics: plain IEEE operations (the emulation is compiled with
// -ffp-contract=off, so nothing is fused)
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
static inline double __ddiv_rn(double a, double b) { return a / b; }
static inline double __dsqrt_rn(double a) { return sqrt(a); }
static inline float __fsqrt_rn(float a) { return sqrtf(a); }
static inline float __ll2float_rn(long long a) { return (float) a; }
static inline float __double2float_rn(double a) { return (float) a; }
static inline float __int2float_rn(int a) { return (float) a; }
static inline float __uint2float_rn(unsigned a) { return (float) a; }
static inline double __ll2double_rn(long long a) { return (double) a; }
static inline uint32_t __float_as_uint(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
static inline int __float_as_int(float f) { int u; memcpy(&u, &f, 4); return u; }
static inline float __uint_as_float(uint32_t u) { float f; memcpy(&f, &u, 4); return f; }
static inline float __int_as_float(int u) { float f; memcpy(&f, &u, 4); return f; }
static inline long long __double_as_longlong(double d) { long long u; memcpy(&u, &d, 8); return u; }
static inline double __longlong_as_double(long long u) { double d; memcpy(&d, &u, 8); return d; }
static inline unsigned long long __umul64hi(unsigned long long a, unsigned long long b) {
  return (unsigned long long) (((unsigned __int128) a * b) >> 64);
}
static inline uint32_t __umulhi(uint32_t a, uint32_t b) { return (uint32_t) (((uint64_t) a * b) >> 32); }

// CUDA's integer min / max overloads
#define CUSIM_MINMAX(TY) \
  static inline TY min(TY a, TY b) { return a < b ? a : b; } \
  static inline TY max(TY a, TY b) { return a > b ? a : b; }
CUSIM_MINMAX(int)
CUSIM_MINMAX(unsigned int)
CUSIM_MINMAX(long)
CUSIM_MINMAX(unsigned long)
CUSIM_MINMAX(long long)
CUSIM_MINMAX(unsigned long long)
static inline unsigned int min(unsigned int a, int b) { return a < (unsigned int) b ? a : (unsigned int) b; }
static inline unsigned int min(int a, unsigned int b) { return (unsigned int) a < b ? (unsigned int) a : b; }
static inline unsigned int max(unsigned int a, int b) { return a > (unsigned int) b ? a : (unsigned int) b; }
static inline unsigned int max(int a, unsigned int b) { return (unsigned int) a > b ? (unsigned int) a : b; }
static inline unsigned long min(unsigned long a, unsigned int b) { return a < b ? a : b; }
static inline unsigned long min(unsigned int a, unsigned long b) { return a < b ? a : b; }
static inline unsigned long max(unsigned long a, unsigned int b) { return a > b ? a : b; }
static inline unsigned long max(unsigned int a, unsigned long b) { return a > b ? a : b; }

// ---------------------------------------------------------------- runtime API
struct cudaDeviceProp {
  int multiProcessorCount;
  char name[64];
};
enum cudaDeviceAttr { cudaDevAttrCooperativeLaunch, cudaDevAttrMultiProcessorCount };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize, cudaFuncAttributePreferredSharedMemoryCarveout };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2, cudaIpcMemLazyEnablePeerAccess = 1 };
struct cudaIpcMemHandle_t { char reserved[64]; };

static inline cudaError_t cudaGetDeviceCount(int *n) { *n = 1; return cudaSuccess; }
static inline cudaError_t cudaSetDevice(int) { return cudaSuccess; }
static inline cudaError_t cudaGetDevice(int *d) { *d = 0; return cudaSuccess; }
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp *p, int) {
  memset(p, 0, sizeof(*p));
  p->multiProcessorCount = 2;                 // small grids: the persistent kernels size themselves by this
  strcpy(p->name, "cusim");
  return cudaSuccess;
}
static inline cudaError_t cudaDeviceGetAttribute(int *v, cudaDeviceAttr a, int) {
  *v = a == cudaDevAttrMultiProcessorCount ? 2 : 1;     // cooperative launch: every block alive at once
  return cudaSuccess;
}
static inline cudaError_t cudaGetLastError() { return cudaSuccess; }
static inline const char *cudaGetErrorString(cudaError_t) { return "cusim error"; }
static inline const char *cudaGetErrorName(cudaError_t) { return "cusimError"; }
// counted for the tests: allocations not yet freed (cusim_live_allocs), host synchronisations (cusim_stream_syncs)
namespace cusim { extern long long live_allocs; extern unsigned long long stream_syncs; }
static inline cudaError_t cudaMalloc(void **p, size_t n) {
  *p = calloc(n ? n : 1, 1);
  if (*p == nullptr) return cudaErrorMemoryAllocation;
  __atomic_add_fetch(&cusim::live_allocs, 1, __ATOMIC_RELAXED);
  return cudaSuccess;
}
template <typename P> static inline cudaError_t cudaMalloc(P **p, size_t n) { return cudaMalloc((void **) p, n); }
static inline cudaError_t cudaFree(void *p) {
  if (p != nullptr) __atomic_sub_fetch(&cusim::live_allocs, 1, __ATOMIC_RELAXED);
  free(p);
  return cudaSuccess;
}
static inline cudaError_t cudaMallocHost(void **p, size_t n) { return cudaMalloc(p, n); }
template <typename P> static inline cudaError_t cudaMallocHost(P **p, size_t n) { return cudaMalloc((void **) p, n); }
static inline cudaError_t cudaFreeHost(void *p) { return cudaFree(p); }
static inline cudaError_t cudaMemcpy(void *d, const void *s, size_t n, cudaMemcpyKind) { if (n) memmove(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemcpyAsync(void *d, const void *s, size_t n, cudaMemcpyKind, cudaStream_t = nullptr) { if (n) memmove(d, s, n); return cudaSuccess; }
static inline cudaError_t cudaMemset(void *d, int v, size_t n) { if (n) memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaMemsetAsync(void *d, int v, size_t n, cudaStream_t = nullptr) { if (n) memset(d, v, n); return cudaSuccess; }
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t *s, unsigned) { *s = (cudaStream_t) malloc(8); return cudaSuccess; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t s) { free(s); return cudaSuccess; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { __atomic_add_fetch(&cusim::stream_syncs, 1, __ATOMIC_RELAXED); return cudaSuccess; }
static inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned = 0) { return cudaSuccess; }
// events carry the host's clock: cudaEventElapsedTime is emulation time, useful only to see which
// kernel the emulation spends its rendezvous on
struct cusim_event { double t; };
static inline double cusim_now_ms() {
  struct timespec ts;
  clock_gettime(CLOCK_MONOTONIC, &ts);
  return ts.tv_sec * 1e3 + ts.tv_nsec * 1e-6;
}
static inline cudaError_t cudaEventCreate(cudaEvent_t *e) { *e = (cudaEvent_t) calloc(1, sizeof(cusim_event)); return cudaSuccess; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t *e, unsigned) { return cudaEventCreate(e); }
static inline cudaError_t cudaEventDestroy(cudaEvent_t e) { free(e); return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t e, cudaStream_t = nullptr) { e->t = cusim_now_ms(); return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventElapsedTime(float *ms, cudaEvent_t a, cudaEvent_t b) { *ms = (float) (b->t - a->t); return cudaSuccess; }
template <typename K> static inline cudaError_t cudaFuncSetAttribute(K, cudaFuncAttribute, int) { return cudaSuccess; }
template <typename K> static inline cudaError_t cudaOccupancyMaxActiveBlocksPerMultiprocessor(int *n, K, int, size_t) { *n = 1; return cudaSuccess; }
static inline cudaError_t cudaLaunchCooperativeKernel(const void *, dim3, dim3, void **, size_t, cudaStream_t) { return cudaErrorNotSupported; }
// peer memory: the ranks are threads of one process, a handle is the pointer itself
static inline cudaError_t cudaIpcGetMemHandle(cudaIpcMemHandle_t *h, void *p) { memset(h, 0, sizeof(*h)); memcpy(h->reserved, &p, sizeof(p)); return cudaSuccess; }
static inline cudaError_t cudaIpcOpenMemHandle(void **p, cudaIpcMemHandle_t h, unsigned) { memcpy(p, h.reserved, sizeof(*p)); return cudaSuccess; }
static inline cudaError_t cudaIpcCloseMemHandle(void *) { return cudaSuccess; }
