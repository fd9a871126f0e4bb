// cuda_emu.h -- a tiny single-process SIMT emulator used ONLY by the CPU-side tests.
//
// TEST INFRASTRUCTURE, NOT A FALLBACK.  The product (mdn_sfm_b200) never loads anything built with this
// header.  Its purpose: there is no GPU in the build container, so `tests/emu/build_emu.py` compiles the
// UNMODIFIED kernel source mdn_sfm_b200/csrc/mdn_loss.cu with g++ against this shim and the not-gpu tests
// execute the very same tile / halo / reduction logic on host buffers to catch indexing and adjoint bugs
// before a gpurun round trip.  Every CUDA thread of a block is a ucontext fiber; __syncthreads() and warp
// shuffles are block-wide rendezvous points of a round-robin scheduler, so block-uniform kernels run
// deterministically.  Approximate intrinsics (__expf, __fdividef, ...) map to the exact libm functions.
#pragma once
#include <ucontext.h>

#include <algorithm>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <vector>

#define MDN_EMU 1
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __launch_bounds__(...)
#define __grid_constant__
#define __shared__ static
#define __align__(x) __attribute__((aligned(x)))

struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct float2 { float x, y; };
struct float4 { float x, y, z, w; };
static inline float4 make_float4(float a, float b, float c, float d) { return float4{a, b, c, d}; }
static inline float2 make_float2(float a, float b) { return float2{a, b}; }
struct int2 { int x, y; };
static inline int2 make_int2(int a, int b) { return int2{a, b}; }

typedef void* cudaStream_t;
typedef int cudaError_t;
enum { cudaSuccess = 0 };
static inline cudaError_t cudaGetLastError() { return cudaSuccess; }
static inline const char* cudaGetErrorString(cudaError_t) { return "emu"; }
static inline cudaError_t cudaMemsetAsync(void* p, int v, size_t n, cudaStream_t) { memset(p, v, n); return cudaSuccess; }
typedef void* cudaEvent_t;
static inline cudaError_t cudaEventCreate(cudaEvent_t* e) { *e = nullptr; return cudaSuccess; }
static inline cudaError_t cudaEventRecord(cudaEvent_t, cudaStream_t) { return cudaSuccess; }
static inline cudaError_t cudaEventSynchronize(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaEventElapsedTime(float* ms, cudaEvent_t, cudaEvent_t) { *ms = 0.f; return cudaSuccess; }
static inline cudaError_t cudaEventDestroy(cudaEvent_t) { return cudaSuccess; }
static inline cudaError_t cudaStreamWaitEvent(cudaStream_t, cudaEvent_t, unsigned) { return cudaSuccess; }
enum cudaFuncAttribute { cudaFuncAttributeMaxDynamicSharedMemorySize = 8 };
template <class T> static inline cudaError_t cudaFuncSetAttribute(T, cudaFuncAttribute, int) { return cudaSuccess; }

namespace mdn_emu {

struct Fiber {
  ucontext_t ctx;
  std::vector<char> stack;
  bool done = false;
};

struct State {
  dim3 tid, bid, bdim, gdim;
  ucontext_t sched;
  std::vector<Fiber> fibers;
  int cur = 0;
  std::vector<char> smem;
  std::vector<uint32_t> xchg;
  const std::function<void()>* body = nullptr;
};
inline State& st() { static State s; return s; }

inline void yield_to_scheduler() {
  State& s = st();
  swapcontext(&s.fibers[s.cur].ctx, &s.sched);
}
inline void fiber_entry() {
  State& s = st();
  (*s.body)();
  s.fibers[s.cur].done = true;
  swapcontext(&s.fibers[s.cur].ctx, &s.sched);
}

inline void launch(dim3 grid, dim3 block, size_t smem_bytes, const std::function<void()>& body) {
  State& s = st();
  const int nthr = (int)(block.x * block.y * block.z);
  s.bdim = block; s.gdim = grid; s.body = &body;
  s.smem.assign(smem_bytes + 64, 0);
  s.xchg.assign(nthr, 0);
  if ((int)s.fibers.size() < nthr) s.fibers.resize(nthr);
  for (unsigned bz = 0; bz < grid.z; ++bz)
  for (unsigned by = 0; by < grid.y; ++by)
  for (unsigned bx = 0; bx < grid.x; ++bx) {
    std::fill(s.smem.begin(), s.smem.end(), (char)0xCD);  // poison: catches reads of never-written shared memory
    for (int t = 0; t < nthr; ++t) {
      Fiber& f = s.fibers[t];
      if (f.stack.empty()) f.stack.resize(256 * 1024);
      f.done = false;
      getcontext(&f.ctx);
      f.ctx.uc_stack.ss_sp = f.stack.data();
      f.ctx.uc_stack.ss_size = f.stack.size();
      f.ctx.uc_link = &s.sched;
      makecontext(&f.ctx, (void (*)())fiber_entry, 0);
    }
    int alive = nthr;
    while (alive > 0) {
      int finished = 0, yielded = 0;
      for (int t = 0; t < nthr; ++t) {
        Fiber& f = s.fibers[t];
        if (f.done) continue;
        s.cur = t;
        s.tid = dim3(t % block.x, (t / block.x) % block.y, t / (block.x * block.y));
        s.bid = dim3(bx, by, bz);
        swapcontext(&s.sched, &f.ctx);
        if (f.done) ++finished; else ++yielded;
      }
      if (finished && yielded) {
        fprintf(stderr, "mdn_emu: divergent barrier (some threads exited while others wait)\n");
        abort();
      }
      alive -= finished;
    }
  }
}

inline uint32_t exchange(uint32_t v, int src_tid) {
  State& s = st();
  s.xchg[s.cur] = v;
  yield_to_scheduler();
  uint32_t r = s.xchg[src_tid];
  yield_to_scheduler();
  return r;
}
}  // namespace mdn_emu

#define threadIdx (mdn_emu::st().tid)
#define blockIdx (mdn_emu::st().bid)
#define blockDim (mdn_emu::st().bdim)
#define gridDim (mdn_emu::st().gdim)
#define MDN_DYN_SMEM(name) float* name = reinterpret_cast<float*>((reinterpret_cast<uintptr_t>(mdn_emu::st().smem.data()) + 63) & ~uintptr_t(63))
#define MDN_LAUNCH(kernel, grid, block, smem, stream, ...) \
  mdn_emu::launch(grid, block, smem, [=]() { kernel(__VA_ARGS__); })

static inline void __syncthreads() { mdn_emu::yield_to_scheduler(); }
static inline void __threadfence() {}
static inline float __shfl_xor_sync(unsigned, float v, int lanemask) {
  uint32_t u; memcpy(&u, &v, 4);
  u = mdn_emu::exchange(u, mdn_emu::st().cur ^ lanemask);
  float r; memcpy(&r, &u, 4); return r;
}
static inline unsigned __shfl_xor_sync(unsigned, unsigned v, int lanemask) {
  return mdn_emu::exchange(v, mdn_emu::st().cur ^ lanemask);
}
static inline int __shfl_xor_sync(unsigned, int v, int lanemask) {
  return (int)mdn_emu::exchange((uint32_t)v, mdn_emu::st().cur ^ lanemask);
}

// lane - delta / lane + delta of the caller's warp; lanes without such a neighbour keep their own value (like the hardware)
static inline float __shfl_up_sync(unsigned, float v, unsigned delta) {
  uint32_t u; memcpy(&u, &v, 4);
  const int cur = mdn_emu::st().cur, lane = cur & 31;
  u = mdn_emu::exchange(u, lane >= (int)delta ? cur - (int)delta : cur);
  float r; memcpy(&r, &u, 4); return r;
}
static inline float __shfl_down_sync(unsigned, float v, unsigned delta) {
  uint32_t u; memcpy(&u, &v, 4);
  const int cur = mdn_emu::st().cur, lane = cur & 31;
  u = mdn_emu::exchange(u, lane + (int)delta <= 31 ? cur + (int)delta : cur);
  float r; memcpy(&r, &u, 4); return r;
}
static inline void __syncwarp(unsigned = 0xffffffffu) { mdn_emu::yield_to_scheduler(); }
static inline float __shfl_sync(unsigned, float v, int src_lane) {
  uint32_t u; memcpy(&u, &v, 4);
  u = mdn_emu::exchange(u, (mdn_emu::st().cur & ~31) | src_lane);
  float r; memcpy(&r, &u, 4); return r;
}
// vote over the 32 lanes of the caller's warp (all lanes of the warp must call it), built on the shuffle rendezvous
static inline int __all_sync(unsigned, int pred) {
  unsigned v = pred ? 1u : 0u;
  for (int m = 16; m >= 1; m >>= 1) v &= mdn_emu::exchange(v, mdn_emu::st().cur ^ m);
  return (int)v;
}
// one bit per lane of the caller's warp (all 32 lanes call it): OR-butterfly over the shuffle rendezvous
static inline unsigned __ballot_sync(unsigned, int pred) {
  unsigned v = pred ? (1u << (mdn_emu::st().cur & 31)) : 0u;
  for (int m = 16; m >= 1; m >>= 1) v |= mdn_emu::exchange(v, mdn_emu::st().cur ^ m);
  return v;
}
static inline unsigned __funnelshift_r(unsigned lo, unsigned hi, unsigned shift) {
  return (unsigned)(((((unsigned long long)hi) << 32) | lo) >> (shift & 31));
}

template <class T> static inline T __ldg(const T* p) { return *p; }
template <class T> static inline T __ldcg(const T* p) { return *p; }
static inline float __fmul_rn(float a, float b) { volatile float r = a * b; return r; }
static inline float __fadd_rn(float a, float b) { volatile float r = a + b; return r; }
static inline float __fsub_rn(float a, float b) { volatile float r = a - b; return r; }
static inline float __fdiv_rn(float a, float b) { volatile float r = a / b; return r; }
static inline float __fmaf_rn(float a, float b, float c) { return fmaf(a, b, c); }
static inline float __fsqrt_rn(float a) { return sqrtf(a); }
static inline float __frcp_rn(float a) { return 1.0f / a; }
static inline float __fdividef(float a, float b) { return a / b; }
static inline float __saturatef(float a) { return !(a > 0.f) ? 0.f : (a > 1.f ? 1.f : a); }   // NaN -> 0 like the hardware
#define __expf(a) expf(a)
#define __logf(a) logf(a)
using std::max;
using std::min;
static inline float rsqrtf(float a) { return 1.0f / sqrtf(a); }
static inline int __float2int_rd(float a) {
  if (!(a == a)) return 0;
  float f = floorf(a);
  if (f >= 2147483520.f) return 2147483647;
  if (f <= -2147483648.f) return -2147483647 - 1;
  return (int)f;
}
static inline unsigned __float_as_uint(float a) { unsigned u; memcpy(&u, &a, 4); return u; }
static inline float __uint_as_float(unsigned u) { float a; memcpy(&a, &u, 4); return a; }
static inline unsigned long long atomicMax(unsigned long long* p, unsigned long long v) {
  unsigned long long o = *p; if (v > o) *p = v; return o;
}
static inline unsigned atomicAdd(unsigned* p, unsigned v) { unsigned o = *p; *p = o + v; return o; }
static inline unsigned atomicInc(unsigned* p, unsigned lim) { unsigned o = *p; *p = (o >= lim) ? 0 : o + 1; return o; }
