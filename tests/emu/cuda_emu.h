// cuda_emu.h — minimal SIMT emulator so the *unmodified* kernel source
// (roboticsplayroompybullet_b200/csrc/prb_kernels.cuh) can be compiled with g++ and
// executed on the CPU by the `-m "not gpu"` tests.
//
// TEST HARNESS ONLY.  The product library (libprb_b200.so) is built by nvcc for
// sm_100a and never includes this file; there is no CPU fallback in the product.
//
// Model: one CUDA thread = one fiber (own stack); the fibers of a block are scheduled
// round-robin and only switch at warp-synchronous points (__syncwarp, shuffles,
// ballots, __syncthreads), which is exactly the set of places where a real warp's lanes
// exchange data.  Switching uses _setjmp/_longjmp after a one-time makecontext start.
#pragma once
#include <math.h>
#include <setjmp.h>
#include <stdint.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <ucontext.h>

#include <algorithm>
#include <functional>
#include <vector>

#define PRB_EMU 1
#define __global__
#define __device__
#define __host__
#define __forceinline__ inline
#define __noinline__
#define __restrict__
#define __launch_bounds__(...)
#define __maxnreg__(n)
#define __grid_constant__
#define __shared__ static
#define __constant__ static

struct emu_dim3 { unsigned x = 1, y = 1, z = 1; };
struct float2 { float x, y; };
struct float3 { float x, y, z; };
struct float4 { float x, y, z, w; };
static inline float2 make_float2(float x, float y) { float2 r = {x, y}; return r; }
static inline float3 make_float3(float x, float y, float z) { float3 r = {x, y, z}; return r; }
static inline float4 make_float4(float x, float y, float z, float w) { float4 r = {x, y, z, w}; return r; }

namespace emu {
struct Fiber {
  ucontext_t uc;
  jmp_buf jb;
  char* stack = nullptr;
  emu_dim3 tid;
  bool done = false, started = false;
};
struct Warp {
  unsigned gen = 0, arrived = 0;
  uint32_t buf[32];
  unsigned ballot = 0;
  unsigned ggen[32] = {0}, garr[32] = {0};   // sub-warp groups (partial masks), keyed by the mask's lowest lane
};
static std::vector<Fiber> fibers;
static std::vector<Warp> warps;
static int cur = 0, nthreads = 0;
static emu_dim3 g_blockIdx, g_blockDim, g_gridDim;
static jmp_buf sched_jb;
static std::function<void()> body;
static unsigned block_gen = 0, block_arrived = 0;

static inline void switch_to_scheduler() {
  if (_setjmp(fibers[cur].jb) == 0) _longjmp(sched_jb, 1);
}
static void fiber_entry() {
  body();
  fibers[cur].done = true;
  _longjmp(sched_jb, 1);
}
static inline void yield() { switch_to_scheduler(); }
static inline void warp_barrier() {
  Warp& w = warps[cur / 32];
  unsigned width = std::min(32, nthreads - (cur / 32) * 32);
  unsigned g = w.gen;
  if (++w.arrived == width) { w.arrived = 0; w.gen++; }
  else while (w.gen == g) yield();
}
static inline void block_barrier() {
  unsigned g = block_gen;
  if (++block_arrived == (unsigned)nthreads) { block_arrived = 0; block_gen++; }
  else while (block_gen == g) yield();
}
// barrier among the lanes of a partial mask (e.g. a quad): exited lanes of other groups do not take part
static inline void group_barrier(unsigned mask) {
  Warp& w = warps[cur / 32];
  const int key = __builtin_ctz(mask);
  const unsigned width = __builtin_popcount(mask);
  unsigned g = w.ggen[key];
  if (++w.garr[key] == width) { w.garr[key] = 0; w.ggen[key]++; }
  else while (w.ggen[key] == g) yield();
}
static const size_t STACK = 256 * 1024;

template <class F>
void launch_y(emu_dim3 grid, emu_dim3 block, unsigned by, F f) {
  g_gridDim = grid; g_blockDim = block;
  nthreads = block.x;
  for (unsigned b = 0; b < grid.x; b++) {
    g_blockIdx.x = b; g_blockIdx.y = by;
    fibers.assign(nthreads, Fiber());
    warps.assign((nthreads + 31) / 32, Warp());
    block_gen = block_arrived = 0;
    body = f;
    for (int t = 0; t < nthreads; t++) {
      fibers[t].tid.x = t;
      fibers[t].stack = (char*)malloc(STACK);
      getcontext(&fibers[t].uc);
      fibers[t].uc.uc_stack.ss_sp = fibers[t].stack;
      fibers[t].uc.uc_stack.ss_size = STACK;
      fibers[t].uc.uc_link = nullptr;
      makecontext(&fibers[t].uc, fiber_entry, 0);
    }
    int remaining = nthreads;
    volatile int next = 0;
    while (remaining > 0) {
      int t = next; next = (next + 1) % nthreads;
      if (fibers[t].done) continue;
      cur = t;
      if (_setjmp(sched_jb) == 0) {
        if (!fibers[t].started) { fibers[t].started = true; setcontext(&fibers[t].uc); }
        else _longjmp(fibers[t].jb, 1);
      }
      if (fibers[cur].done && fibers[cur].stack) { remaining--; }
    }
    for (int t = 0; t < nthreads; t++) free(fibers[t].stack);
  }
}
template <class F>
void launch(emu_dim3 grid, emu_dim3 block, F f) { launch_y(grid, block, 0, f); }
}  // namespace emu

#define threadIdx (emu::fibers[emu::cur].tid)
#define blockIdx (emu::g_blockIdx)
#define blockDim (emu::g_blockDim)
#define gridDim (emu::g_gridDim)

using std::min;
using std::max;

static inline void __syncwarp(unsigned mask = 0xffffffffu) { if (mask == 0xffffffffu) emu::warp_barrier(); else emu::group_barrier(mask); }
static inline void __syncthreads() { emu::block_barrier(); }
template <class T>
static inline T emu_shfl_group(unsigned mask, T v, int src) {
  static_assert(sizeof(T) == 4, "32-bit shuffles only");
  emu::Warp& w = emu::warps[emu::cur / 32];
  int lane = emu::cur % 32;
  memcpy(&w.buf[lane], &v, 4);
  emu::group_barrier(mask);
  T r; memcpy(&r, &w.buf[src & 31], 4);
  emu::group_barrier(mask);
  return r;
}
template <class T>
static inline T emu_shfl(T v, int src) {
  static_assert(sizeof(T) == 4, "32-bit shuffles only");
  emu::Warp& w = emu::warps[emu::cur / 32];
  int lane = emu::cur % 32;
  memcpy(&w.buf[lane], &v, 4);
  emu::warp_barrier();
  T r; memcpy(&r, &w.buf[src & 31], 4);
  emu::warp_barrier();
  return r;
}
template <class T> static inline T __shfl_sync(unsigned mask, T v, int src) { return mask == 0xffffffffu ? emu_shfl(v, src) : emu_shfl_group(mask, v, src); }
template <class T> static inline T __shfl_xor_sync(unsigned mask, T v, int m) {
  return mask == 0xffffffffu ? emu_shfl(v, (emu::cur % 32) ^ m) : emu_shfl_group(mask, v, (emu::cur % 32) ^ m);
}
template <class T> static inline T __shfl_down_sync(unsigned, T v, int d) { int l = emu::cur % 32; return emu_shfl(v, l + d < 32 ? l + d : l); }
template <class T> static inline T __shfl_up_sync(unsigned, T v, int d) { int l = emu::cur % 32; return emu_shfl(v, l - d >= 0 ? l - d : l); }
static inline unsigned __ballot_sync(unsigned, int pred) {
  emu::Warp& w = emu::warps[emu::cur / 32];
  int lane = emu::cur % 32;
  w.buf[lane] = pred ? 1u : 0u;
  emu::warp_barrier();
  unsigned r = 0;
  unsigned width = std::min(32, emu::nthreads - (emu::cur / 32) * 32);
  for (unsigned i = 0; i < width; i++) r |= (w.buf[i] & 1u) << i;
  emu::warp_barrier();
  return r;
}
static inline int __any_sync(unsigned m, int p) { return __ballot_sync(m, p) != 0; }
static inline int __all_sync(unsigned m, int p) { return __ballot_sync(m, !p) == 0; }
static inline int __popc(unsigned x) { return __builtin_popcount(x); }
static inline int __popcll(unsigned long long x) { return __builtin_popcountll(x); }
static inline int __ffs(int x) { return __builtin_ffs(x); }
static inline int __ffsll(long long x) { return __builtin_ffsll(x); }
static inline int __clz(int x) { return x == 0 ? 32 : __builtin_clz((unsigned)x); }
template <class T> static inline T atomicAdd(T* p, T v) { T o = *p; *p = o + v; return o; }
template <class T> static inline T __ldg(const T* p) { return *p; }
static inline float rsqrtf(float x) { return 1.0f / sqrtf(x); }
static inline float __frcp_rn(float x) { return 1.0f / x; }
static inline float __fdividef(float a, float b) { return a / b; }
static inline float __fmul_rn(float a, float b) { return a * b; }
static inline float __fadd_rn(float a, float b) { return a + b; }
static inline float __fsqrt_rn(float a) { return sqrtf(a); }
static inline float __fdiv_rn(float a, float b) { return a / b; }
static inline void sincosf_emu(float x, float* s, float* c) { *s = sinf(x); *c = cosf(x); }
#ifndef sincosf
#define sincosf(x, s, c) sincosf_emu(x, s, c)
#endif
static inline float fminf_(float a, float b) { return a < b ? a : b; }
static inline unsigned __umulhi(unsigned a, unsigned b) { return (unsigned)(((uint64_t)a * b) >> 32); }
static inline float __uint2float_rn(unsigned x) { return (float)x; }
static inline float __int_as_float(int x) { float f; memcpy(&f, &x, 4); return f; }
static inline int __float_as_int(float x) { int i; memcpy(&i, &x, 4); return i; }
