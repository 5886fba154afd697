// cuda_emu.h — DEVELOPMENT TOOL, NOT A PRODUCT PATH.
//
// A functional host emulation of the small CUDA subset the kernels in csrc/*.cuh use, so that kernel LOGIC can be
// debugged in the build container (which has nvcc but no GPU).  Each CTA is run as a set of cooperative fibers
// (one per CUDA thread, hand-rolled x86-64 context switch); __syncthreads / warp collectives are fiber barriers.
// Cooperative scheduling hides data races, so this checks algorithms, not the memory model: the real checks are the
// `-m gpu` parity tests and compute-sanitizer on a B200.  The package (mtscomp_b200/_native.py) never loads anything
// built from this header; only tools/emu_*.py and tests/test_emu_kernels.py do.
#pragma once
#ifndef MTSCOMP_EMU
#error "cuda_emu.h is only for -DMTSCOMP_EMU host builds"
#endif
#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <thread>
#include <vector>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __shared__ static thread_local
#define __constant__ static const
#define __launch_bounds__(...)
#define __align__(n) __attribute__((aligned(n)))

struct uint3 { unsigned x, y, z; };
struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct alignas(16) uint4 { unsigned x, y, z, w; };
struct alignas(8) uint2 { unsigned x, y; };
struct alignas(16) int4 { int x, y, z, w; };
struct alignas(4) ushort2 { unsigned short x, y; };
static inline uint4 make_uint4(unsigned x, unsigned y, unsigned z, unsigned w) { return uint4{x, y, z, w}; }
static inline uint2 make_uint2(unsigned x, unsigned y) { return uint2{x, y}; }

namespace emu {

extern "C" void emu_switch(void** save_sp, void* new_sp);

struct Warp {
  int count = 0;
  unsigned gen = 0;
  uint64_t x[32];
};

struct Block {
  std::vector<void*> sp;
  std::vector<char*> stacks;
  std::vector<char> done;
  std::vector<Warp> warps;
  void* sched_sp = nullptr;
  int cur = 0;
  unsigned nthreads = 0, alive = 0;
  int bar_count = 0;
  unsigned bar_gen = 0;
  long bar_acc = 0, bar_result = 0;
  long bar_and = 1, bar_and_result = 1;
  int nb_count[16] = {0};
  unsigned nb_gen[16] = {0};
  const std::function<void()>* body = nullptr;
};

extern thread_local Block* g_blk;
extern thread_local unsigned char* g_dyn_smem;

static inline void yield() {
  Block* b = g_blk;
  emu_switch(&b->sp[b->cur], b->sched_sp);
}

// Dynamic shared memory a launch may ask for: 48 KB unless the kernel's cudaFuncAttributeMaxDynamicSharedMemorySize
// says otherwise, and never more than the opt-in limit of an sm_100 block (sharedMemPerBlockOptin below).  A launch
// past its limit runs nothing and leaves cudaErrorInvalidValue for the next cudaGetLastError, as on the device.
static const size_t kDynSmemDefault = 48 * 1024, kDynSmemOptin = 232448;
extern thread_local int g_last_error;           // cudaGetLastError's slot (per host thread, as in the runtime)
int set_max_dyn_smem(const void* fn, int bytes);
template <class F> static inline const void* fn_addr(F f) { return reinterpret_cast<const void*>(f); }
void launch(const void* fn, dim3 grid, dim3 block, size_t smem, const std::function<void()>& body);

}  // namespace emu

extern thread_local uint3 threadIdx, blockIdx;
extern thread_local dim3 blockDim, gridDim;
static const int warpSize = 32;

// ---------------------------------------------------------------- barriers
static inline void __emu_release_block(emu::Block* b) {
  b->bar_count = 0;
  b->bar_result = b->bar_acc;
  b->bar_acc = 0;
  b->bar_and_result = b->bar_and;
  b->bar_and = 1;
  b->bar_gen++;
}
static inline void __syncthreads() {
  emu::Block* b = emu::g_blk;
  unsigned g = b->bar_gen;
  if (++b->bar_count == (int)b->alive) __emu_release_block(b);
  else while (b->bar_gen == g) emu::yield();
}
static inline int __syncthreads_or(int p) {
  emu::g_blk->bar_acc += (p != 0);
  __syncthreads();
  return emu::g_blk->bar_result != 0;
}
static inline int __syncthreads_count(int p) {
  emu::g_blk->bar_acc += (p != 0);
  __syncthreads();
  return (int)emu::g_blk->bar_result;
}
static inline int __syncthreads_and(int p) {
  emu::g_blk->bar_and &= (p != 0);
  __syncthreads();
  return emu::g_blk->bar_and_result != 0;
}
// named barrier: `count` threads of the CTA meet at barrier `id` (PTX bar.sync id, count)
static inline void __emu_named_barrier(int id, int count) {
  emu::Block* b = emu::g_blk;
  unsigned g = b->nb_gen[id];
  if (++b->nb_count[id] == count) { b->nb_count[id] = 0; b->nb_gen[id]++; }
  else while (b->nb_gen[id] == g) emu::yield();
}
static inline void __emu_named_barrier_arrive(int id, int count) {
  emu::Block* b = emu::g_blk;
  if (++b->nb_count[id] == count) { b->nb_count[id] = 0; b->nb_gen[id]++; }
}
static inline unsigned __emu_tid() { return threadIdx.x + blockDim.x * (threadIdx.y + blockDim.y * threadIdx.z); }
static inline emu::Warp& __emu_warp() { return emu::g_blk->warps[__emu_tid() >> 5]; }
static inline void __emu_wbar(unsigned mask) {
  emu::Warp& w = __emu_warp();
  unsigned g = w.gen;
  if (++w.count == __builtin_popcount(mask)) { w.count = 0; w.gen++; }
  else while (w.gen == g) emu::yield();
}
static inline void __syncwarp(unsigned mask = 0xffffffffu) { __emu_wbar(mask); }
static inline void __threadfence() {}
static inline void __threadfence_block() {}

// ---------------------------------------------------------------- warp collectives
template <class T> static inline uint64_t __emu_bits(T v) { uint64_t r = 0; memcpy(&r, &v, sizeof(T)); return r; }
template <class T> static inline T __emu_from(uint64_t r) { T v; memcpy(&v, &r, sizeof(T)); return v; }

template <class T> static inline T __shfl_sync(unsigned mask, T v, int src, int width = 32) {
  emu::Warp& w = __emu_warp();
  int lane = __emu_tid() & 31;
  w.x[lane] = __emu_bits(v);
  __emu_wbar(mask);
  int s = (lane & ~(width - 1)) | (src & (width - 1));
  T r = __emu_from<T>(w.x[s]);
  __emu_wbar(mask);
  return r;
}
template <class T> static inline T __shfl_up_sync(unsigned mask, T v, unsigned d, int width = 32) {
  emu::Warp& w = __emu_warp();
  int lane = __emu_tid() & 31;
  w.x[lane] = __emu_bits(v);
  __emu_wbar(mask);
  int s = lane - (int)d;
  if (s < (lane & ~(width - 1))) s = lane;
  T r = __emu_from<T>(w.x[s]);
  __emu_wbar(mask);
  return r;
}
template <class T> static inline T __shfl_down_sync(unsigned mask, T v, unsigned d, int width = 32) {
  emu::Warp& w = __emu_warp();
  int lane = __emu_tid() & 31;
  w.x[lane] = __emu_bits(v);
  __emu_wbar(mask);
  int s = lane + (int)d;
  if (s >= (lane & ~(width - 1)) + width) s = lane;
  T r = __emu_from<T>(w.x[s]);
  __emu_wbar(mask);
  return r;
}
template <class T> static inline T __shfl_xor_sync(unsigned mask, T v, int m, int width = 32) {
  emu::Warp& w = __emu_warp();
  int lane = __emu_tid() & 31;
  w.x[lane] = __emu_bits(v);
  __emu_wbar(mask);
  T r = __emu_from<T>(w.x[lane ^ m]);
  __emu_wbar(mask);
  return r;
}
static inline unsigned __ballot_sync(unsigned mask, int p) {
  emu::Warp& w = __emu_warp();
  int lane = __emu_tid() & 31;
  w.x[lane] = (p != 0);
  __emu_wbar(mask);
  unsigned r = 0;
  for (int l = 0; l < 32; l++) if (((mask >> l) & 1) && w.x[l]) r |= 1u << l;
  __emu_wbar(mask);
  return r;
}
static inline int __any_sync(unsigned mask, int p) { return __ballot_sync(mask, p) != 0; }
static inline int __all_sync(unsigned mask, int p) { return __ballot_sync(mask, p) == mask; }
template <class T> static inline unsigned __match_any_sync(unsigned mask, T v) {
  emu::Warp& w = __emu_warp();
  int lane = __emu_tid() & 31;
  w.x[lane] = __emu_bits(v);
  __emu_wbar(mask);
  unsigned r = 0;
  for (int l = 0; l < 32; l++) if (((mask >> l) & 1) && w.x[l] == w.x[lane]) r |= 1u << l;
  __emu_wbar(mask);
  return r;
}
static inline unsigned __activemask() { return 0xffffffffu; }

// ---------------------------------------------------------------- atomics (CTAs may run on several OS threads)
template <class T> static inline T atomicAdd(T* p, T v) { return __atomic_fetch_add(p, v, __ATOMIC_RELAXED); }
template <class T> static inline T atomicSub(T* p, T v) { return __atomic_fetch_sub(p, v, __ATOMIC_RELAXED); }
template <class T> static inline T atomicOr(T* p, T v) { return __atomic_fetch_or(p, v, __ATOMIC_RELAXED); }
template <class T> static inline T atomicAnd(T* p, T v) { return __atomic_fetch_and(p, v, __ATOMIC_RELAXED); }
template <class T> static inline T atomicExch(T* p, T v) { return __atomic_exchange_n(p, v, __ATOMIC_RELAXED); }
template <class T> static inline T atomicMax(T* p, T v) {
  T o = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (o < v && !__atomic_compare_exchange_n(p, &o, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return o;
}
template <class T> static inline T atomicMin(T* p, T v) {
  T o = __atomic_load_n(p, __ATOMIC_RELAXED);
  while (o > v && !__atomic_compare_exchange_n(p, &o, v, true, __ATOMIC_RELAXED, __ATOMIC_RELAXED)) {}
  return o;
}
template <class T> static inline T atomicCAS(T* p, T cmp, T v) {
  __atomic_compare_exchange_n(p, &cmp, v, false, __ATOMIC_RELAXED, __ATOMIC_RELAXED);
  return cmp;
}

// ---------------------------------------------------------------- integer intrinsics
static inline int __popc(unsigned x) { return __builtin_popcount(x); }
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __clz(int x) { return x ? __builtin_clz((unsigned)x) : 32; }
static inline int __clzll(long long x) { return x ? __builtin_clzll((unsigned long long)x) : 64; }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline unsigned __brev(unsigned x) {
  x = ((x >> 1) & 0x55555555u) | ((x & 0x55555555u) << 1);
  x = ((x >> 2) & 0x33333333u) | ((x & 0x33333333u) << 2);
  x = ((x >> 4) & 0x0f0f0f0fu) | ((x & 0x0f0f0f0fu) << 4);
  return __builtin_bswap32(x);
}
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned s) {
  return (unsigned)(((((uint64_t)hi) << 32) | lo) >> (s & 31));
}
static inline unsigned __funnelshift_l(unsigned lo, unsigned hi, unsigned s) {
  return (unsigned)((((((uint64_t)hi) << 32) | lo) << (s & 31)) >> 32);
}
static inline unsigned __byte_perm(unsigned x, unsigned y, unsigned s) {
  uint64_t v = (((uint64_t)y) << 32) | x;
  unsigned r = 0;
  for (int i = 0; i < 4; i++) {
    unsigned sel = (s >> (4 * i)) & 0xf;
    unsigned b = (unsigned)(v >> (8 * (sel & 7))) & 0xff;
    if (sel & 8) b = (b & 0x80) ? 0xff : 0;
    r |= b << (8 * i);
  }
  return r;
}
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((uint64_t)a * b) >> 32); }
template <class T> static inline T __ldg(const T* p) { return *p; }

// ---------------------------------------------------------------- IEEE operations rounded one at a time (no contraction)
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsub_rn(float a, float b) { return a - b; }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline double __dadd_rn(double a, double b) { return a + b; }
static inline double __dsub_rn(double a, double b) { return a - b; }
static inline double __dmul_rn(double a, double b) { return a * b; }
using std::max;
using std::min;
static inline unsigned min(unsigned a, int b) { return a < (unsigned)b ? a : (unsigned)b; }
static inline unsigned min(int a, unsigned b) { return (unsigned)a < b ? (unsigned)a : b; }
static inline unsigned max(unsigned a, int b) { return a > (unsigned)b ? a : (unsigned)b; }
static inline unsigned max(int a, unsigned b) { return (unsigned)a > b ? (unsigned)a : b; }

// ---------------------------------------------------------------- runtime API subset
typedef int cudaError_t;
typedef void* cudaStream_t;
struct __emu_event { std::chrono::steady_clock::time_point t; };
typedef __emu_event* cudaEvent_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2, cudaErrorInvalidValue = 11 };
enum cudaMemcpyKind { cudaMemcpyHostToHost, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2, cudaHostAllocDefault = 0 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8, cudaFuncAttributePreferredSharedMemoryCarveout = 9 };
enum { cudaSharedmemCarveoutMaxShared = 100 };
static inline const char* cudaGetErrorString(cudaError_t e) {
  return e == cudaSuccess ? "no error" : e == cudaErrorInvalidValue ? "invalid argument"
       : e == cudaErrorMemoryAllocation ? "out of memory" : "emu error";
}
static inline cudaError_t cudaGetLastError() { cudaError_t e = emu::g_last_error; emu::g_last_error = 0; return e; }
static inline cudaError_t cudaPeekAtLastError() { return emu::g_last_error; }
static inline cudaError_t cudaSetDevice(int) { return 0; }
static inline cudaError_t cudaGetDevice(int* d) { *d = 0; return 0; }
static inline cudaError_t cudaGetDeviceCount(int* n) { *n = 1; return 0; }
static inline cudaError_t cudaMalloc(void** p, size_t n) { *p = aligned_alloc(256, (n + 255) / 256 * 256 + 256); return *p ? 0 : 2; }
static inline cudaError_t cudaFree(void* p) { free(p); return 0; }
static inline cudaError_t cudaMallocHost(void** p, size_t n) { return cudaMalloc(p, n); }
static inline cudaError_t cudaHostAlloc(void** p, size_t n, unsigned) { return cudaMalloc(p, n); }
static inline cudaError_t cudaFreeHost(void* p) { free(p); return 0; }
static inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind, cudaStream_t = 0) { memmove(d, s, n); return 0; }
static inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { memmove(d, s, n); return 0; }
static inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = 0) { memset(d, v, n); return 0; }
static inline cudaError_t cudaMemset(void* d, int v, size_t n) { memset(d, v, n); return 0; }
static inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = (void*)1; return 0; }
static inline cudaError_t cudaStreamCreate(cudaStream_t* s) { *s = (void*)1; return 0; }
static inline cudaError_t cudaStreamDestroy(cudaStream_t) { return 0; }
static inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return 0; }
static inline cudaError_t cudaDeviceSynchronize() { return 0; }
static inline cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = new __emu_event; return 0; }
static inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = new __emu_event; return 0; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t e) { delete e; return 0; }
static inline cudaError_t cudaEventRecord(cudaEvent_t e, cudaStream_t = 0) { e->t = std::chrono::steady_clock::now(); return 0; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return 0; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned = 0) { return 0; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t a, cudaEvent_t b) {
  *ms = std::chrono::duration<float, std::milli>(b->t - a->t).count();
  return 0;
}
template <class F> static inline cudaError_t cudaFuncSetAttribute(F f, cudaFuncAttribute a, int v) {
  return a == cudaFuncAttributeMaxDynamicSharedMemorySize ? emu::set_max_dyn_smem(emu::fn_addr(f), v) : 0;
}
struct cudaDeviceProp { int multiProcessorCount; int major, minor; size_t sharedMemPerBlockOptin; char name[64]; size_t totalGlobalMem; };
static inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) {
  p->multiProcessorCount = 8; p->major = 10; p->minor = 0; p->sharedMemPerBlockOptin = 232448;
  p->totalGlobalMem = (size_t)8 << 30;
  snprintf(p->name, sizeof p->name, "host-emulation"); return 0;
}
static inline cudaError_t cudaMemGetInfo(size_t* f, size_t* t) { *f = (size_t)8 << 30; *t = (size_t)8 << 30; return 0; }
struct cudaPointerAttributes { int type; };
enum { cudaMemoryTypeUnregistered = 0, cudaMemoryTypeHost = 1, cudaMemoryTypeDevice = 2 };
static inline cudaError_t cudaPointerGetAttributes(cudaPointerAttributes* a, const void*) { a->type = 2; return 0; }

#define MTS_LAUNCH(kernel, grid, block, smem, stream, ...) \
  emu::launch(emu::fn_addr(kernel), (grid), (block), (smem), [&]() { kernel(__VA_ARGS__); })
#define MTS_DYN_SMEM(name) unsigned char* name = emu::g_dyn_smem
