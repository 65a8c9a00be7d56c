// Host-side emulation of the small CUDA subset the srst kernels use -- TEST INFRASTRUCTURE ONLY.
//
// The build container has nvcc but no GPU, so kernel index logic cannot be exercised there.
// This header lets the *unmodified* kernel sources (srgan_st_b200/csrc/*.cuh) compile with g++
// (-DSRST_EMULATE) and run one OS thread per CUDA thread, blocks executed one after another, with
// __syncthreads() mapped to a std::barrier and warp shuffles to a per-warp exchange buffer.
// It is slow and is used only by tests/test_emu_*.py on tiny shapes; the product library
// (libsrst.so, built by nvcc for sm_100a) never contains or calls any of this.
#pragma once
#include <atomic>
#include <barrier>
#include <cmath>
#include <cstdint>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <mutex>
#include <thread>
#include <vector>

struct dim3 {
  unsigned x, y, z;
  dim3(unsigned x_ = 1, unsigned y_ = 1, unsigned z_ = 1) : x(x_), y(y_), z(z_) {}
};
struct alignas(8) float2 { float x, y; };
struct alignas(16) float4 { float x, y, z, w; };
struct alignas(16) int4 { int x, y, z, w; };
static inline float2 make_float2(float x, float y) { return float2{x, y}; }
static inline float4 make_float4(float x, float y, float z, float w) { return float4{x, y, z, w}; }

typedef int cudaError_t;
typedef void* cudaStream_t;
enum { cudaSuccess = 0, cudaErrorInvalidValue = 1 };
static inline cudaError_t cudaGetLastError() { return 0; }
static inline cudaError_t cudaPeekAtLastError() { return 0; }

#define __global__
#define __device__
#define __host__
#define __forceinline__ inline __attribute__((always_inline))
#define __restrict__ __restrict
#define __launch_bounds__(...)
#define __grid_constant__
// Static __shared__ arrays become function-local statics of the kernels.  tests/emu/shared.ld (with -fdata-sections)
// gathers every local static of a function named *_kernel into one range, so that launch() can poison them before
// every block, like dynamic shared memory: a kernel that reads a static array it did not write in the same block sees
// the poison instead of the previous block's (finite, plausible) values.  (g++ ignores a section attribute on a local
// static of a function template, hence the linker script.)
#define __shared__ static
#define __align__(n) __attribute__((aligned(n)))

// Bounds of that range (set by shared.ld; both null when the library was linked without it).
extern "C" unsigned char __start_srst_emu_shared[] __attribute__((weak, visibility("hidden")));
extern "C" unsigned char __stop_srst_emu_shared[] __attribute__((weak, visibility("hidden")));

namespace emu {
// Byte that fills dynamic and static shared memory before every block.  0xCD (the float -4.3e8) by default; 0xFF
// makes every float a NaN and every int -1, so that a read of never-written shared memory cannot hide behind a
// zero weight.  Set through srst_emu_set_poison().
inline int g_smem_poison = 0xCD;
struct BlockCtx {
  std::unique_ptr<std::barrier<>> bar;
  std::vector<std::unique_ptr<std::barrier<>>> warp_bar;
  std::vector<uint64_t> warp_xchg;  // 32 slots per warp
  unsigned char* dyn_smem = nullptr;
  unsigned nthreads = 0;
  std::mutex named_mu;
  std::map<int, std::unique_ptr<std::barrier<>>> named;  // bar.sync/bar.arrive id -> barrier(count)
  std::barrier<>* named_bar(int id, int count) {
    std::lock_guard<std::mutex> lk(named_mu);
    auto& b = named[id];
    if (!b) b = std::make_unique<std::barrier<>>(count);
    return b.get();
  }
};
inline BlockCtx* g_block = nullptr;
inline dim3 g_blockDim, g_gridDim;
inline thread_local dim3 t_threadIdx, t_blockIdx;
inline thread_local unsigned t_linear_tid = 0;

template <class F>
void launch(dim3 grid, dim3 block, size_t smem_bytes, F&& body) {
  g_blockDim = block;
  g_gridDim = grid;
  const unsigned nt = block.x * block.y * block.z;
  const unsigned nwarps = (nt + 31) / 32;
  std::vector<unsigned char> smem(smem_bytes + 64);
  unsigned char* smem_aligned =
      reinterpret_cast<unsigned char*>((reinterpret_cast<uintptr_t>(smem.data()) + 63) & ~uintptr_t(63));
  for (unsigned bz = 0; bz < grid.z; ++bz)
    for (unsigned by = 0; by < grid.y; ++by)
      for (unsigned bx = 0; bx < grid.x; ++bx) {
        BlockCtx ctx;
        ctx.nthreads = nt;
        ctx.bar = std::make_unique<std::barrier<>>(nt);
        for (unsigned w = 0; w < nwarps; ++w) {
          unsigned lanes = std::min(32u, nt - 32 * w);
          ctx.warp_bar.emplace_back(std::make_unique<std::barrier<>>(lanes));
        }
        ctx.warp_xchg.assign(32 * nwarps, 0);
        std::memset(smem_aligned, g_smem_poison, smem_bytes);  // poison: uninitialised reads become visible
        if (__start_srst_emu_shared && __stop_srst_emu_shared > __start_srst_emu_shared)
          std::memset(__start_srst_emu_shared, g_smem_poison, __stop_srst_emu_shared - __start_srst_emu_shared);
        ctx.dyn_smem = smem_aligned;
        g_block = &ctx;
        std::vector<std::thread> ths;
        ths.reserve(nt);
        for (unsigned t = 0; t < nt; ++t) {
          ths.emplace_back([&, t]() {
            t_linear_tid = t;
            t_threadIdx = dim3(t % block.x, (t / block.x) % block.y, t / (block.x * block.y));
            t_blockIdx = dim3(bx, by, bz);
            body();
          });
        }
        for (auto& th : ths) th.join();
        g_block = nullptr;
      }
}

template <class T>
inline T warp_exchange(T v, int src_lane) {
  static_assert(sizeof(T) <= 8, "");
  BlockCtx* c = g_block;
  unsigned w = t_linear_tid / 32, lane = t_linear_tid % 32;
  uint64_t bits = 0;
  std::memcpy(&bits, &v, sizeof(T));
  c->warp_xchg[32 * w + lane] = bits;
  c->warp_bar[w]->arrive_and_wait();
  unsigned lanes = std::min(32u, c->nthreads - 32 * w);
  T out = v;
  if (src_lane >= 0 && (unsigned)src_lane < lanes) {
    uint64_t b2 = c->warp_xchg[32 * w + src_lane];
    std::memcpy(&out, &b2, sizeof(T));
  }
  c->warp_bar[w]->arrive_and_wait();
  return out;
}
inline unsigned warp_ballot(bool pred) {
  BlockCtx* c = g_block;
  unsigned w = t_linear_tid / 32, lane = t_linear_tid % 32;
  c->warp_xchg[32 * w + lane] = pred ? 1u : 0u;
  c->warp_bar[w]->arrive_and_wait();
  unsigned lanes = std::min(32u, c->nthreads - 32 * w), mask = 0;
  for (unsigned l = 0; l < lanes; ++l) mask |= (unsigned)(c->warp_xchg[32 * w + l] & 1u) << l;
  c->warp_bar[w]->arrive_and_wait();
  return mask;
}
}  // namespace emu

// Test hook exported by the emulation library only (the header is compiled into exactly one translation unit):
// the shared-memory poison byte of later launches; returns the previous one.
extern "C" __attribute__((visibility("default"))) int srst_emu_set_poison(int byte) {
  const int old = emu::g_smem_poison;
  emu::g_smem_poison = byte & 0xFF;
  return old;
}

#define threadIdx (emu::t_threadIdx)
#define blockIdx (emu::t_blockIdx)
#define blockDim (emu::g_blockDim)
#define gridDim (emu::g_gridDim)

static inline void __syncthreads() { emu::g_block->bar->arrive_and_wait(); }
static inline void __syncwarp(unsigned = 0xffffffffu) {
  emu::g_block->warp_bar[emu::t_linear_tid / 32]->arrive_and_wait();
}
// named barriers (PTX bar.sync / bar.arrive with an id and a participating-thread count)
static inline void emu_bar_sync(int id, int count) { emu::g_block->named_bar(id, count)->arrive_and_wait(); }
static inline void emu_bar_arrive(int id, int count) { (void)emu::g_block->named_bar(id, count)->arrive(); }
static inline void __threadfence_block() { std::atomic_thread_fence(std::memory_order_seq_cst); }
static inline void __threadfence() { std::atomic_thread_fence(std::memory_order_seq_cst); }

template <class T> static inline T __shfl_xor_sync(unsigned, T v, int m) {
  return emu::warp_exchange(v, int(emu::t_linear_tid % 32) ^ m);
}
template <class T> static inline T __shfl_down_sync(unsigned, T v, int d) {
  int src = int(emu::t_linear_tid % 32) + d;
  return emu::warp_exchange(v, src < 32 ? src : -1);
}
template <class T> static inline T __shfl_sync(unsigned, T v, int src) { return emu::warp_exchange(v, src & 31); }
template <class T> static inline T __shfl_up_sync(unsigned, T v, int d) {
  int src = int(emu::t_linear_tid % 32) - d;
  return emu::warp_exchange(v, src >= 0 ? src : -1);
}
static inline unsigned __ballot_sync(unsigned, int pred) { return emu::warp_ballot(pred != 0); }
static inline int __popcll(unsigned long long v) { return __builtin_popcountll(v); }
static inline int __popc(unsigned v) { return __builtin_popcount(v); }
static inline int __ffsll(long long v) { return __builtin_ffsll(v); }

static inline unsigned atomicAdd(unsigned* p, unsigned v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
static inline int atomicAdd(int* p, int v) { return __atomic_fetch_add(p, v, __ATOMIC_SEQ_CST); }
static inline float atomicAdd(float* p, float v) {
  uint32_t* ip = reinterpret_cast<uint32_t*>(p);
  uint32_t old = __atomic_load_n(ip, __ATOMIC_SEQ_CST);
  for (;;) {
    float f;
    std::memcpy(&f, &old, 4);
    float nf = f + v;
    uint32_t nb;
    std::memcpy(&nb, &nf, 4);
    if (__atomic_compare_exchange_n(ip, &old, nb, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST)) return f;
  }
}

template <class T> static inline T __ldg(const T* p) { return *p; }
template <class T> static inline T __ldcg(const T* p) { return *reinterpret_cast<const volatile T*>(p); }
static inline float __ldcg(const float* p) { return *reinterpret_cast<const volatile float*>(p); }

using std::max;
using std::min;
static inline float __int_as_float(int i) { float f; std::memcpy(&f, &i, 4); return f; }
static inline int __float_as_int(float f) { int i; std::memcpy(&i, &f, 4); return i; }
static inline float rsqrtf(float x) { return 1.0f / std::sqrt(x); }
static inline float __frsqrt_rn(float x) { return 1.0f / std::sqrt(x); }
static inline float __frcp_rn(float x) { return 1.0f / x; }
static inline float __fdividef(float a, float b) { return a / b; }
#define __logf(x) std::log((float)(x))
static inline float __fmul_rn(float a, float b) { volatile float r = a * b; return r; }
static inline float __fadd_rn(float a, float b) { volatile float r = a + b; return r; }
static inline float __fsub_rn(float a, float b) { volatile float r = a - b; return r; }
static inline float __fdiv_rn(float a, float b) { volatile float r = a / b; return r; }
static inline float __fsqrt_rn(float a) { volatile float r = std::sqrt(a); return r; }
static inline float __fmaf_rn(float a, float b, float c) { return std::fma(a, b, c); }
static inline float2 __ffma2_rn(float2 a, float2 b, float2 c) {
  return float2{std::fma(a.x, b.x, c.x), std::fma(a.y, b.y, c.y)};
}
static inline float2 __fmul2_rn(float2 a, float2 b) { return float2{a.x * b.x, a.y * b.y}; }
static inline float2 __fadd2_rn(float2 a, float2 b) { return float2{a.x + b.x, a.y + b.y}; }
