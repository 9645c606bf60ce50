// HOST EMULATION of the sliver of CUDA that graph staging uses — test infrastructure only (tests/test_emu_staging_cpu.py).
// The staging kernels (graph_build.cu) are simple data-parallel loops without intra-block communication, so they can
// run on the CPU unchanged: every "thread" of a launch is executed to completion, one after the other.  "Device"
// memory is host memory.  Nothing here is part of the product; libcugraph_c.so is never built with it.
#pragma once
#ifndef B200_HOST_EMU
#error "emu/cuda_runtime.h is only for -DB200_HOST_EMU builds"
#endif
#include <algorithm>
#include <chrono>
#include <climits>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __launch_bounds__(...)
#define __shared__ static

struct uint3 { unsigned x{0}, y{0}, z{0}; };
struct dim3 {
  unsigned x{1}, y{1}, z{1};
  dim3(unsigned a = 1, unsigned b = 1, unsigned c = 1) : x(a), y(b), z(c) {}
};
struct uint2 { unsigned x, y; };
struct int2 { int x, y; };
inline int2 make_int2(int a, int b) { return {a, b}; }
struct uint4 { unsigned x, y, z, w; };
struct int4 { int x, y, z, w; };
struct double2 { double x, y; };
struct float4 { float x, y, z, w; };
struct float2 { float x, y; };
inline float2 make_float2(float a, float b) { return {a, b}; }
inline double2 make_double2(double a, double b) { return {a, b}; }
inline float4 make_float4(float a, float b, float c, float d) { return {a, b, c, d}; }
inline uint2 make_uint2(unsigned a, unsigned b) { return {a, b}; }
inline uint4 make_uint4(unsigned a, unsigned b, unsigned c, unsigned d) { return {a, b, c, d}; }
inline int4 make_int4(int a, int b, int c, int d) { return {a, b, c, d}; }

inline thread_local uint3 threadIdx, blockIdx;
inline thread_local dim3 blockDim, gridDim;

// ------------------------------------------------------------------------------------------------------------
// SIMT execution model.  A launch runs its CTAs one after the other; the threads of a CTA are FIBERS (ucontext) on the
// calling OS thread, resumed round-robin.  A fiber runs until it finishes or blocks in __syncthreads() / a warp
// collective (__shfl*_sync, __ballot_sync, ...), which complete when every live lane named by the mask has arrived.
// Sequential, deterministic, no data races; kernels whose CTAs wait for each other would deadlock (none here do —
// a CTA that finds no work left by its predecessors simply exits).
// ------------------------------------------------------------------------------------------------------------
#include <functional>
#include <ucontext.h>
#include <vector>

namespace emu {

constexpr int kMaxThreads  = 1024;
constexpr size_t kStackLen = 256 * 1024;
enum { IDLE = 0, RUN = 1, WAIT_WARP = 2, WAIT_CTA = 3, DONE = 4 };

struct warp_state_t {
  unsigned live{0}, arrived{0}, need{0}, out_mask{0};
  unsigned long long in[32], out[32];
};
struct cta_state_t {
  ucontext_t sched;
  ucontext_t ctx[kMaxThreads];
  char* stack[kMaxThreads] = {};
  int state[kMaxThreads]   = {};
  bool started[kMaxThreads] = {};
  int n{0}, cur{-1}, live{0}, cta_arrived{0};
  bool in_fiber{false};
  std::function<void()> body;
  warp_state_t warp[kMaxThreads / 32];
};
inline cta_state_t& cta()
{
  static cta_state_t* c = new cta_state_t();
  return *c;
}
inline bool in_fiber() { return cta().in_fiber; }

inline void yield_to_scheduler()
{
  cta_state_t& C = cta();
  swapcontext(&C.ctx[C.cur], &C.sched);
}
inline void fiber_main()
{
  cta_state_t& C = cta();
  for (;;) {  // pooled: a finished fiber is resumed with the next CTA's body
    C.body();
    C.state[C.cur] = DONE;
    yield_to_scheduler();
  }
}
inline void release_warp_if_complete(cta_state_t& C, int w)
{
  warp_state_t& W = C.warp[w];
  if (W.arrived == 0) return;
  if ((W.arrived & W.live) != (W.need & W.live)) return;
  for (int l = 0; l < 32; ++l) W.out[l] = W.in[l];
  W.out_mask = W.arrived;
  for (int l = 0; l < 32; ++l)
    if ((W.arrived >> l) & 1u) C.state[w * 32 + l] = RUN;
  W.arrived = 0;
}
inline void release_cta_if_complete(cta_state_t& C)
{
  if (C.cta_arrived == 0 || C.cta_arrived != C.live) return;
  for (int t = 0; t < C.n; ++t)
    if (C.state[t] == WAIT_CTA) C.state[t] = RUN;
  C.cta_arrived = 0;
}
inline void run_cta(int n)
{
  cta_state_t& C = cta();
  C.n = n; C.live = n; C.cta_arrived = 0;
  for (int w = 0; w < (n + 31) / 32; ++w) {
    const int lanes = std::min(32, n - w * 32);
    C.warp[w].live    = lanes == 32 ? 0xffffffffu : ((1u << lanes) - 1u);
    C.warp[w].arrived = 0;
  }
  for (int t = 0; t < n; ++t) C.state[t] = RUN;
  C.in_fiber = true;
  int done   = 0;
  while (done < n) {
    bool progressed = false;
    for (int t = 0; t < n; ++t) {
      if (C.state[t] != RUN) continue;
      progressed = true;
      C.cur      = t;
      threadIdx.x = (unsigned)t;
      if (!C.started[t]) {
        if (!C.stack[t]) C.stack[t] = (char*)std::malloc(kStackLen);
        getcontext(&C.ctx[t]);
        C.ctx[t].uc_stack.ss_sp   = C.stack[t];
        C.ctx[t].uc_stack.ss_size = kStackLen;
        C.ctx[t].uc_link          = nullptr;
        makecontext(&C.ctx[t], (void (*)())fiber_main, 0);
        C.started[t] = true;
      }
      swapcontext(&C.sched, &C.ctx[t]);
      const int w = t >> 5;
      if (C.state[t] == DONE) {
        ++done;
        --C.live;
        C.warp[w].live &= ~(1u << (t & 31));
        release_warp_if_complete(C, w);
        release_cta_if_complete(C);
      } else if (C.state[t] == WAIT_WARP) {
        release_warp_if_complete(C, w);
      } else if (C.state[t] == WAIT_CTA) {
        release_cta_if_complete(C);
      }
    }
    if (!progressed) {
      std::fprintf(stderr, "emu: deadlock in block %u (a collective or barrier some live threads never reach)\n", blockIdx.x);
      std::abort();
    }
  }
  C.in_fiber = false;
  C.cur      = -1;
}

// all live lanes named by `mask` exchange one 64-bit value
inline unsigned warp_collect(unsigned mask, unsigned long long v, unsigned long long (&out)[32])
{
  cta_state_t& C = cta();
  const int t = C.cur, w = t >> 5, l = t & 31;
  if (!C.in_fiber || mask == (1u << l)) {  // outside a launch, or a one-lane "collective"
    for (int i = 0; i < 32; ++i) out[i] = v;
    return 1u << (l & 31);
  }
  warp_state_t& W = C.warp[w];
  W.in[l] = v;
  W.need  = mask;
  W.arrived |= 1u << l;
  C.state[t] = WAIT_WARP;
  yield_to_scheduler();
  for (int i = 0; i < 32; ++i) out[i] = W.out[i];
  return W.out_mask;
}

}  // namespace emu

template <typename F>
inline void emu_launch(long long grid, long long block, F&& body)
{
  if (block > emu::kMaxThreads) { std::fprintf(stderr, "emu: block of %lld threads\n", block); std::abort(); }
  gridDim        = dim3((unsigned)grid);
  blockDim       = dim3((unsigned)block);
  emu::cta().body = [&] { body(); };
  for (long long b = 0; b < grid; ++b) {
    blockIdx.x = (unsigned)b;
    emu::run_cta((int)block);
  }
}

// ---- runtime API
typedef int cudaError_t;
enum { cudaSuccess = 0, cudaErrorMemoryAllocation = 2 };
typedef struct emu_stream_t* cudaStream_t;
typedef struct emu_event_t* cudaEvent_t;
typedef void* cudaMemPool_t;
enum cudaMemcpyKind { cudaMemcpyHostToHost, cudaMemcpyHostToDevice, cudaMemcpyDeviceToHost, cudaMemcpyDeviceToDevice, cudaMemcpyDefault };
enum { cudaStreamNonBlocking = 1, cudaEventDisableTiming = 2 };
enum cudaMemPoolAttr { cudaMemPoolAttrReleaseThreshold = 4 };
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };
struct cudaDeviceProp {
  int multiProcessorCount{4};
  int l2CacheSize{1 << 20};
};

inline const char* cudaGetErrorString(cudaError_t) { return "emulated CUDA error"; }
inline const char* cudaGetErrorName(cudaError_t) { return "cudaErrorEmu"; }
inline cudaError_t cudaGetLastError() { return cudaSuccess; }
inline cudaError_t cudaGetDevice(int* d) { *d = 0; return cudaSuccess; }
inline cudaError_t cudaGetDeviceProperties(cudaDeviceProp* p, int) { *p = cudaDeviceProp{}; return cudaSuccess; }
inline cudaError_t cudaDeviceGetDefaultMemPool(cudaMemPool_t* p, int) { *p = nullptr; return cudaSuccess; }
inline cudaError_t cudaMemPoolSetAttribute(cudaMemPool_t, cudaMemPoolAttr, void*) { return cudaSuccess; }
inline cudaError_t cudaMalloc(void** p, size_t n) { *p = std::malloc(n ? n : 1); return *p ? cudaSuccess : cudaErrorMemoryAllocation; }
template <typename T> inline cudaError_t cudaMalloc(T** p, size_t n) { return cudaMalloc((void**)p, n); }
inline cudaError_t cudaMallocAsync(void** p, size_t n, cudaStream_t) { return cudaMalloc(p, n); }
template <typename T> inline cudaError_t cudaMallocAsync(T** p, size_t n, cudaStream_t s) { return cudaMallocAsync((void**)p, n, s); }
inline cudaError_t cudaMallocHost(void** p, size_t n) { return cudaMalloc(p, n); }
template <typename T> inline cudaError_t cudaMallocHost(T** p, size_t n) { return cudaMalloc((void**)p, n); }
inline cudaError_t cudaFree(void* p) { std::free(p); return cudaSuccess; }
inline cudaError_t cudaFreeAsync(void* p, cudaStream_t) { std::free(p); return cudaSuccess; }
inline cudaError_t cudaFreeHost(void* p) { std::free(p); return cudaSuccess; }
inline cudaError_t cudaMemcpy(void* d, const void* s, size_t n, cudaMemcpyKind) { if (n) std::memmove(d, s, n); return cudaSuccess; }
inline cudaError_t cudaMemcpyAsync(void* d, const void* s, size_t n, cudaMemcpyKind k, cudaStream_t = nullptr) { return cudaMemcpy(d, s, n, k); }
inline cudaError_t cudaMemset(void* d, int v, size_t n) { if (n) std::memset(d, v, n); return cudaSuccess; }
inline cudaError_t cudaMemsetAsync(void* d, int v, size_t n, cudaStream_t = nullptr) { return cudaMemset(d, v, n); }
inline cudaError_t cudaStreamCreateWithFlags(cudaStream_t* s, unsigned) { *s = (cudaStream_t)std::malloc(8); return cudaSuccess; }
inline cudaError_t cudaStreamCreate(cudaStream_t* s) { return cudaStreamCreateWithFlags(s, 0); }
inline cudaError_t cudaStreamDestroy(cudaStream_t s) { std::free(s); return cudaSuccess; }
inline cudaError_t cudaStreamSynchronize(cudaStream_t) { return cudaSuccess; }
inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned = 0) { return cudaSuccess; }
inline cudaError_t cudaEventCreateWithFlags(cudaEvent_t* e, unsigned) { *e = (cudaEvent_t)std::malloc(8); return cudaSuccess; }
inline cudaError_t cudaEventCreate(cudaEvent_t* e) { return cudaEventCreateWithFlags(e, 0); }
inline cudaError_t cudaEventDestroy(cudaEvent_t e) { std::free(e); return cudaSuccess; }
// an event holds the host time of its record (8 bytes): work is synchronous here, so that IS when the "stream" got there
inline cudaError_t cudaEventRecord(cudaEvent_t e, cudaStream_t = nullptr)
{
  const double t = std::chrono::duration<double, std::milli>(std::chrono::steady_clock::now().time_since_epoch()).count();
  std::memcpy(e, &t, sizeof(t));
  return cudaSuccess;
}
inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
inline cudaError_t cudaDeviceSynchronize() { return cudaSuccess; }
inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t a, cudaEvent_t b)
{
  double ta, tb;
  std::memcpy(&ta, a, sizeof(ta));
  std::memcpy(&tb, b, sizeof(tb));
  *ms = (float)(tb - ta);
  return cudaSuccess;
}
template <typename F> inline cudaError_t cudaFuncSetAttribute(F, cudaFuncAttribute, int) { return cudaSuccess; }

// ---- device intrinsics (sequential semantics)
template <typename T> inline T atomicAdd(T* p, T v) { T o = *p; *p = o + v; return o; }
template <typename T> inline T atomicMin(T* p, T v) { T o = *p; if (v < o) *p = v; return o; }
template <typename T> inline T atomicMax(T* p, T v) { T o = *p; if (v > o) *p = v; return o; }
template <typename T> inline T atomicOr(T* p, T v) { T o = *p; *p = o | v; return o; }
inline unsigned __float_as_uint(float f) { unsigned u; std::memcpy(&u, &f, 4); return u; }
inline float __uint_as_float(unsigned u) { float f; std::memcpy(&f, &u, 4); return f; }
inline long long __double_as_longlong(double d) { long long u; std::memcpy(&u, &d, 8); return u; }
template <typename T> inline T __ldg(const T* p) { return *p; }
template <typename T> inline unsigned long long emu_bits(T v) { unsigned long long b = 0; static_assert(sizeof(T) <= 8, "shuffle width"); std::memcpy(&b, &v, sizeof(T)); return b; }
template <typename T> inline T emu_from_bits(unsigned long long b) { T v; std::memcpy(&v, &b, sizeof(T)); return v; }
inline int emu_lane() { return (int)(threadIdx.x & 31); }
template <typename T> inline T emu_shfl_from(unsigned mask, T v, int src)
{
  unsigned long long out[32];
  const unsigned pm = emu::warp_collect(mask, emu_bits(v), out);
  if (src < 0 || src > 31 || !((pm >> src) & 1u)) src = emu_lane();  // out of range / not participating: own value
  return emu_from_bits<T>(out[src]);
}
template <typename T> inline T __shfl_sync(unsigned m, T v, int src, int width = 32)
{
  return emu_shfl_from(m, v, (src & (width - 1)) + (emu_lane() & ~(width - 1)));
}
template <typename T> inline T __shfl_xor_sync(unsigned m, T v, int o, int = 32) { return emu_shfl_from(m, v, emu_lane() ^ o); }
template <typename T> inline T __shfl_down_sync(unsigned m, T v, int o, int = 32) { return emu_shfl_from(m, v, emu_lane() + o); }
template <typename T> inline T __shfl_up_sync(unsigned m, T v, int o, int = 32) { return emu_shfl_from(m, v, emu_lane() - o); }
inline unsigned __ballot_sync(unsigned m, int p)
{
  unsigned long long out[32];
  const unsigned pm = emu::warp_collect(m, p ? 1ull : 0ull, out);
  unsigned r = 0;
  for (int i = 0; i < 32; ++i)
    if (((pm >> i) & 1u) && out[i]) r |= 1u << i;
  return r;
}
inline int __all_sync(unsigned m, int p)
{
  unsigned long long out[32];
  const unsigned pm = emu::warp_collect(m, p ? 1ull : 0ull, out);
  for (int i = 0; i < 32; ++i)
    if (((pm >> i) & 1u) && !out[i]) return 0;
  return 1;
}
inline int __any_sync(unsigned m, int p) { return __ballot_sync(m, p) != 0; }
template <typename T> inline unsigned __match_any_sync(unsigned m, T v)
{
  unsigned long long out[32];
  const unsigned pm = emu::warp_collect(m, emu_bits(v), out);
  const unsigned long long mine = emu_bits(v);
  unsigned r = 0;
  for (int i = 0; i < 32; ++i)
    if (((pm >> i) & 1u) && out[i] == mine) r |= 1u << i;
  return r;
}
inline unsigned __reduce_or_sync(unsigned m, unsigned v)
{
  unsigned long long out[32];
  const unsigned pm = emu::warp_collect(m, (unsigned long long)v, out);
  unsigned r = 0;
  for (int i = 0; i < 32; ++i)
    if ((pm >> i) & 1u) r |= (unsigned)out[i];
  return r;
}
template <typename T> inline T __reduce_add_sync(unsigned m, T v)
{
  unsigned long long out[32];
  const unsigned pm = emu::warp_collect(m, emu_bits(v), out);
  T r = 0;
  for (int i = 0; i < 32; ++i)
    if ((pm >> i) & 1u) r += emu_from_bits<T>(out[i]);
  return r;
}
inline unsigned __activemask() { return 1u << emu_lane(); }  // worst-case divergence: every lane on its own
inline void __syncwarp(unsigned m = 0xffffffffu) { unsigned long long out[32]; emu::warp_collect(m, 0ull, out); }
inline void __threadfence() {}  // CTAs run one after the other: every write is visible
inline void __syncthreads()
{
  emu::cta_state_t& C = emu::cta();
  if (!C.in_fiber) return;
  C.state[C.cur] = emu::WAIT_CTA;
  ++C.cta_arrived;
  emu::yield_to_scheduler();
}
inline int __popc(unsigned v) { return __builtin_popcount(v); }
inline int __popcll(unsigned long long v) { return __builtin_popcountll(v); }
inline int __ffsll(long long v) { return __builtin_ffsll(v); }
inline int __ffs(int v) { return __builtin_ffs(v); }
inline int __clz(int v) { return v ? __builtin_clz((unsigned)v) : 32; }
inline float __int_as_float(int i) { float f; std::memcpy(&f, &i, 4); return f; }
inline int __float_as_int(float f) { int i; std::memcpy(&i, &f, 4); return i; }
inline double __longlong_as_double(long long i) { double f; std::memcpy(&f, &i, 8); return f; }
template <typename T> inline T atomicExch(T* p, T v) { T o = *p; *p = v; return o; }
template <typename T> inline T atomicCAS(T* p, T c, T v) { T o = *p; if (o == c) *p = v; return o; }
