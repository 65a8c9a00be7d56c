// Common device-side helpers for the srst kernels (sm_100a).
//
// Compiles two ways:
//   nvcc  -gencode arch=compute_100a,code=sm_100a   -> the product (libsrst.so)
//   g++   -DSRST_EMULATE                            -> tests/emu host emulation (test infra only;
//                                                      one OS thread per CUDA thread, used to
//                                                      check index logic without a GPU)
#pragma once

#ifdef SRST_EMULATE
#include "cuda_emu.h"
#define SRST_DYN_SMEM(T, name) T* name = reinterpret_cast<T*>(emu::g_block->dyn_smem)
#define SRST_LAUNCH(kernel, grid, block, smem, stream, ...) \
  emu::launch((grid), (block), (smem), [&]() { kernel(__VA_ARGS__); })
#define SRST_SET_SMEM(kernel, bytes) (0)
#define SRST_LAUNCH_PDL(kernel, grid, block, smem, stream, P) SRST_LAUNCH(kernel, grid, block, smem, stream, P)
#else
#include <cuda_runtime.h>
#include <cstdlib>
#define SRST_DYN_SMEM(T, name) extern __shared__ __align__(128) unsigned char name##_raw_[]; \
  T* name = reinterpret_cast<T*>(name##_raw_)
#define SRST_LAUNCH(kernel, grid, block, smem, stream, ...) \
  kernel<<<(grid), (block), (smem), (cudaStream_t)(stream)>>>(__VA_ARGS__)
#define SRST_SET_SMEM(kernel, bytes) \
  cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(bytes))
// Launch with programmatic stream serialization (PDL): the grid may be scheduled while the previous
// kernel of the stream is still draining; the kernel itself calls pdl_wait() before it touches
// global memory, so only launch latency and CTA set-up overlap.  SRST_PDL=0 turns it off.
#define SRST_LAUNCH_PDL(kernel, grid, block, smem, stream, P)                                   \
  do {                                                                                           \
    cudaLaunchConfig_t cfg_ = {};                                                                \
    cfg_.gridDim = (grid); cfg_.blockDim = (block); cfg_.dynamicSmemBytes = (smem);              \
    cfg_.stream = (cudaStream_t)(stream);                                                        \
    cudaLaunchAttribute at_[1];                                                                  \
    at_[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;                              \
    at_[0].val.programmaticStreamSerializationAllowed = 1;                                       \
    cfg_.attrs = at_; cfg_.numAttrs = srst::pdl_enabled() ? 1 : 0;                               \
    cudaLaunchKernelEx(&cfg_, kernel, P);                                                        \
  } while (0)
#endif

#define SRST_DEV __device__ __forceinline__

namespace srst {

#ifndef SRST_EMULATE
inline bool pdl_enabled() {
  static const bool on = [] { const char* e = std::getenv("SRST_PDL"); return !(e && e[0] == '0'); }();
  return on;
}
#endif
// Programmatic dependent launch hooks (no-ops for kernels launched without the PDL attribute):
// pdl_wait() blocks until the previous kernel of the stream has completed and its writes are
// visible; pdl_trigger() lets the next PDL-launched kernel of the stream start its own launch.
#ifdef SRST_EMULATE
SRST_DEV void pdl_wait() {}
SRST_DEV void pdl_trigger() {}
#else
SRST_DEV void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
SRST_DEV void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

constexpr int round_up4(int x) { return (x + 3) / 4 * 4; }
constexpr int round_dn4(int x) { return x / 4 * 4; }
// Shared-memory row pitch (floats): >= w, multiple of 4 (16-byte rows for LDS.128) and == 4 mod 8,
// so that 8 lanes reading float4s from 8 consecutive rows hit 8 distinct 16-byte bank groups.
constexpr int smem_pitch(int w) {
  int p = round_up4(w);
  while (p % 8 != 4) p += 4;
  return p;
}
constexpr int cmax(int a, int b) { return a > b ? a : b; }
constexpr int cmin(int a, int b) { return a < b ? a : b; }

SRST_DEV float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }
SRST_DEV void st4(float* p, float4 v) { *reinterpret_cast<float4*>(p) = v; }
SRST_DEV float4 ldg4(const float* p) { return __ldg(reinterpret_cast<const float4*>(p)); }
#ifdef SRST_EMULATE
SRST_DEV float4 ldcg4(const float* p) { return *reinterpret_cast<const float4*>(p); }
#else
SRST_DEV float4 ldcg4(const float* p) { return __ldcg(reinterpret_cast<const float4*>(p)); }  // L2 (data written by this kernel)
#endif

// torchvision rgb_to_grayscale weights (reference loss.py:400-401).
constexpr float kGrayR = 0.2989f, kGrayG = 0.587f, kGrayB = 0.114f;
// One fixed contraction, so that every load path of every kernel rounds a pixel the same way (the compiler is
// otherwise free to fuse either product into an FMA, and two code sites then differ in the last bit).
SRST_DEV float gray_of(float r, float g, float b) { return __fmaf_rn(kGrayB, b, __fmaf_rn(kGrayR, r, __fmul_rn(kGrayG, g))); }

// Raw SFU approximations (MUFU.RSQ / MUFU.LG2 / MUFU.RCP, <= 2 ulp) without the denormal/special
// fix-up code that rsqrtf()/__logf()/__fdividef() add; callers guarantee normal-range inputs.
#ifdef SRST_EMULATE
SRST_DEV float fast_rsqrt(float x) { return 1.0f / std::sqrt(x); }
SRST_DEV float fast_lg2(float x) { return std::log2(x); }
SRST_DEV float fast_rcp(float x) { return 1.0f / x; }
#else
SRST_DEV float fast_rsqrt(float x) { float y; asm("rsqrt.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
SRST_DEV float fast_lg2(float x) { float y; asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
SRST_DEV float fast_rcp(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
#endif

// NaN-propagating minimum of three (one FMNMX3.NAN on sm_100a): any NaN operand gives NaN.
#ifdef SRST_EMULATE
SRST_DEV float min3_nan(float a, float b, float c) {
  if (a != a || b != b || c != c) return std::nanf("");
  return std::fmin(a, std::fmin(b, c));
}
#else
SRST_DEV float min3_nan(float a, float b, float c) {
  float d;
  asm("min.NaN.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
  return d;
}
#endif

// 16-byte asynchronous global->shared copy (LDGSTS); `valid == false` zero-fills the destination
// without reading `gsrc` (src-size 0), which implements the reference's zero padding for free.
#ifdef SRST_EMULATE
SRST_DEV void cp_async16(float* sdst, const float* gsrc, bool valid) {
  if (valid) std::memcpy(sdst, gsrc, 16); else std::memset(sdst, 0, 16);
}
SRST_DEV void cp_async4(float* sdst, const float* gsrc) { *sdst = *gsrc; }
SRST_DEV void cp_async_commit() {}
SRST_DEV void cp_async_wait_all() {}
#else
SRST_DEV void cp_async16(float* sdst, const float* gsrc, bool valid) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(sdst);
  const int sz = valid ? 16 : 0;
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(s), "l"(gsrc), "r"(sz) : "memory");
}
SRST_DEV void cp_async4(float* sdst, const float* gsrc) {
  const unsigned s = (unsigned)__cvta_generic_to_shared(sdst);
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(s), "l"(gsrc) : "memory");
}
SRST_DEV void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
SRST_DEV void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }
#endif

// TMA (cp.async.bulk.tensor) staging of a 3-D box [bp planes][bh rows][bw cols] of an fp32 tensor
// viewed as [P planes][H][W] into shared memory.  One thread issues ONE instruction for the whole
// box; coordinates may start outside the tensor (negative or past the end) and the hardware fills
// those elements with zeros -- the reference's zero padding.  The first box column must be a multiple of
// 4 floats (16 bytes) all the same: a box starting at x = -10 raises "illegal instruction" on B200 (measured,
// round 2); the emulation aborts on it.  Completion is signalled on an mbarrier that every consumer thread polls.
#ifdef SRST_EMULATE
struct SrstTmap { const float* base; int W, H, P; };
// The emulated mbarrier keeps (completed phases) in its low and (bytes still expected) in its high 32 bits, so that
// tma_wait really waits for the issuing thread (OS threads run ahead of each other just like warps do).
SRST_DEV void tma_barrier_init(unsigned long long* mbar) { __atomic_store_n(mbar, 0ull, __ATOMIC_SEQ_CST); }
SRST_DEV void tma_expect(unsigned long long* mbar, unsigned bytes) {
  __atomic_fetch_add(mbar, (unsigned long long)bytes << 32, __ATOMIC_SEQ_CST);
}
SRST_DEV void tma_load_3d(unsigned long long* mbar, float* dst, const SrstTmap* m, int x, int y, int z, int bw,
                          int bh, int bp) {
  if ((x & 3) != 0 || (bw & 3) != 0) { std::fprintf(stderr, "emulated TMA: box column %d / width %d not a multiple of 4\n", x, bw); std::abort(); }
  for (int p = 0; p < bp; ++p)
    for (int r = 0; r < bh; ++r)
      for (int c = 0; c < bw; ++c) {
        const int gx = x + c, gy = y + r, gp = z + p;
        const bool ok = gx >= 0 && gx < m->W && gy >= 0 && gy < m->H && gp >= 0 && gp < m->P;
        dst[(p * bh + r) * bw + c] = ok ? m->base[((size_t)gp * m->H + gy) * m->W + gx] : 0.f;
      }
  const unsigned long long bytes = (unsigned long long)bp * bh * bw * sizeof(float);
  const unsigned long long after = __atomic_sub_fetch(mbar, bytes << 32, __ATOMIC_SEQ_CST);
  if ((after >> 32) == 0) __atomic_fetch_add(mbar, 1ull, __ATOMIC_SEQ_CST);  // the phase is complete
}
SRST_DEV void tma_wait(unsigned long long* mbar, unsigned parity = 0) {
  while (((unsigned)__atomic_load_n(mbar, __ATOMIC_SEQ_CST) & 1u) == parity) std::this_thread::yield();
}
SRST_DEV void fence_async_smem() {}
#else
}  // namespace srst
#include <cuda.h>
namespace srst {
typedef CUtensorMap SrstTmap;
// One mbarrier can collect several box copies: init (one arriving thread), announce the total byte
// count once, then issue the copies.  (bw, bh, bp) repeat the box dimensions encoded in the tensor
// map; only the emulation reads them.
SRST_DEV void tma_barrier_init(unsigned long long* mbar) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(bar) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
SRST_DEV void tma_expect(unsigned long long* mbar, unsigned bytes) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(mbar);
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
SRST_DEV void tma_load_3d(unsigned long long* mbar, float* dst, const SrstTmap* m, int x, int y, int z, int bw,
                          int bh, int bp) {
  (void)bw; (void)bh; (void)bp;
  const unsigned bar = (unsigned)__cvta_generic_to_shared(mbar);
  const unsigned sdst = (unsigned)__cvta_generic_to_shared(dst);
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];"
      ::"r"(sdst), "l"(reinterpret_cast<unsigned long long>(m)), "r"(x), "r"(y), "r"(z), "r"(bar)
      : "memory");
}
// Waits for the phase of `mbar` with the given parity (0 for the first use of a barrier, then alternating).
SRST_DEV void tma_wait(unsigned long long* mbar, unsigned parity = 0) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(mbar);
  unsigned done = 0;
  while (!done) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
  }
}
// Orders this thread's earlier generic-proxy accesses to shared memory before later async-proxy (TMA) writes.
SRST_DEV void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
#endif

// Counting mbarriers for multi-stage shared-memory pipelines (the patch-search kernel's candidate chunks): `count`
// arrivals complete a phase; mbar_wait(parity) returns once the phase with that parity (0 for the first, then
// alternating) has completed.  cp_async_mbar_arrive makes the calling thread's arrival wait for all of its earlier
// cp.async copies.  The wait is bounded: a protocol error traps instead of hanging the GPU.
#ifdef SRST_EMULATE
// emulated state: pending arrivals (bits 0..19) | expected count (20..39) | completed phases (40..)
SRST_DEV void mbar_init(unsigned long long* b, unsigned count) {
  __atomic_store_n(b, (unsigned long long)count | ((unsigned long long)count << 20), __ATOMIC_SEQ_CST);
}
SRST_DEV void mbar_arrive(unsigned long long* b) {
  unsigned long long v = __atomic_load_n(b, __ATOMIC_SEQ_CST), nv;
  do {
    const unsigned long long pending = (v & 0xFFFFFull) - 1, expected = (v >> 20) & 0xFFFFFull, phase = v >> 40;
    nv = pending ? ((v & ~0xFFFFFull) | pending) : (expected | (expected << 20) | ((phase + 1) << 40));
  } while (!__atomic_compare_exchange_n(b, &v, nv, false, __ATOMIC_SEQ_CST, __ATOMIC_SEQ_CST));
}
SRST_DEV void cp_async_mbar_arrive(unsigned long long* b) { mbar_arrive(b); }  // emulated copies are synchronous
SRST_DEV void mbar_wait(unsigned long long* b, unsigned parity) {
  while (((__atomic_load_n(b, __ATOMIC_SEQ_CST) >> 40) & 1ull) == parity) std::this_thread::yield();
}
#else
SRST_DEV void mbar_init(unsigned long long* b, unsigned count) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(b);
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
SRST_DEV void mbar_arrive(unsigned long long* b) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(b);
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
SRST_DEV void cp_async_mbar_arrive(unsigned long long* b) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(b);
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}
SRST_DEV void mbar_wait(unsigned long long* b, unsigned parity) {
  const unsigned bar = (unsigned)__cvta_generic_to_shared(b);
  unsigned done = 0;
  for (int spin = 0; !done; ++spin) {
    asm volatile(
        "{\n\t.reg .pred p;\n\tmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\tselp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(done)
        : "r"(bar), "r"(parity)
        : "memory");
    if (spin > (1 << 24)) __trap();
  }
}
#endif

// Named barriers for producer/consumer warp roles: `n` = number of participating threads.
#ifdef SRST_EMULATE
SRST_DEV void bar_sync(int id, int n) { emu_bar_sync(id, n); }
SRST_DEV void bar_arrive(int id, int n) { emu_bar_arrive(id, n); }
#else
SRST_DEV void bar_sync(int id, int n) { asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(n) : "memory"); }
SRST_DEV void bar_arrive(int id, int n) { asm volatile("bar.arrive %0, %1;" ::"r"(id), "r"(n) : "memory"); }
#endif

// Optional phase time stamps (tools/phase_timing.py; compiled in only with -DSRST_TIMING, never in the product
// library): thread 0 of every CTA records %globaltimer at the phase boundaries of its first tile.
#if defined(SRST_TIMING) && !defined(SRST_EMULATE)
__device__ long long* g_srst_timing = nullptr;
SRST_DEV void srst_stamp(int slot) {
  if (g_srst_timing && threadIdx.x == 0) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_srst_timing[(size_t)blockIdx.x * 32 + slot] = t;
  }
}
#define SRST_STAMP(slot) srst_stamp(slot)
#else
#define SRST_STAMP(slot) ((void)0)
#endif

SRST_DEV float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// Per-image form of the deterministic loss reduction (reduction='none'), run by every thread of the CTA that drew
// the last ticket.  The grid is laid out image-major, so partials[b * per .. (b + 1) * per) are image b's CTAs: one
// warp per image sums them in double in a fixed order (lane-strided, then a fixed shuffle tree), zeroes them again and
// writes out[b] = sum * scale.
SRST_DEV void reduce_partials_per_image(float* partials, int B, unsigned int per, double scale, float* out) {
  const int lane = threadIdx.x & 31;
  for (int b = threadIdx.x >> 5; b < B; b += blockDim.x >> 5) {
    float* p = partials + (size_t)b * per;
    double acc = 0.0;
    for (unsigned int i = lane; i < per; i += 32) {
      acc += (double)__ldcg(p + i);
      p[i] = 0.f;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) out[b] = (float)(acc * scale);
  }
}

}  // namespace srst
