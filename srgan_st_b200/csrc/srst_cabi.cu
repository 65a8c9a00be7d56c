// C ABI of libsrst.so (declared in include/srst.h).  Host-side launch logic only: validates
// arguments, picks a compiled tile configuration and enqueues the sm_100a kernels on the caller's
// stream.  No allocation, no synchronisation, no global state, no CPU fallback.
//
// The same file compiles with g++ -DSRST_EMULATE into tests/emu/_build/libsrst_emu.so, a
// test-only host emulation used to check kernel index logic in the GPU-less build container.
#include "../../include/srst.h"

#include <cstdlib>
#include <cstring>

#include <type_traits>

#include "st_kernels.cuh"
#include "st_march.cuh"
#include "bb_generic.cuh"
#include "st_generic.cuh"
#include "bb_kernels.cuh"

namespace srst {

static inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// Tuning knobs are read from the environment ONCE (first use); srst_st_force_cfg() overrides the
// tile choice at run time (tests cover every compiled shape through it).
static int env_int_once(const char* name, int dflt) {
  const char* s = std::getenv(name);
  return (s && *s) ? std::atoi(s) : dflt;
}
static int g_force_fwd = -2, g_force_bwd = -2;  // -2: not initialised, -1: library's own choice
static int g_force_chunk = -2;                  // row blocks per chunk of the marching forward (0 / -1: own choice)
static int forced_fwd() {
  if (g_force_fwd == -2) g_force_fwd = env_int_once("SRST_ST_FWD_CFG", -1);
  return g_force_fwd;
}
static int forced_chunk() {
  if (g_force_chunk == -2) g_force_chunk = env_int_once("SRST_ST_CHUNK_BLOCKS", -1);
  return g_force_chunk;
}
static int forced_bwd() {
  if (g_force_bwd == -2) g_force_bwd = env_int_once("SRST_ST_BWD_CFG", -1);
  return g_force_bwd;
}

// ---- compiled structure-tensor tile configurations (reference default radii: r_sigma 2, r_rho 8) ----
// Only shapes the dispatcher can pick are compiled (the sweeps that selected them: profiles/r02_tile_sweep.log; the
// round-1 shapes that lost them are gone).  Forward cfg ids: 0-2 tiled (unaligned tensors / fall-back), 3-4 marching.
//                       TH  TW  RS CSB RG RK MINB CHU
using Fwd0 = StFwdCfg<32, 64, 16, 4, 2, 8, 3, 0, true>;  // large images, 256 threads, unrolled: three CTAs per SM; plane-split vertical items
using Fwd1 = StFwdCfg<24, 96, 8, 4, 2, 8, 2, 0>;   // full-width strip of a 96-wide crop (no horizontal halo), 288 threads, unrolled
using Fwd2 = StFwdCfg<24, 96, 8, 4, 2, 8, 3, 0>;   // Fwd1 with three CTAs per SM (72 registers): multi-wave batches of 96-wide crops
// cfg 3, 4: the row-marching kernel (st_march.cuh), 96- and 112-column strips -- the default whenever TMA can
// fetch the images; the tiled shapes above remain for unaligned tensors and as the fall-back.  Cfg 3 runs the crop
// layout (March96X: no x halo) on images no wider than 96 columns.
using March96 = StMarchCfg<96, 2, 8>;
using March96X = StMarchCfg<96, 2, 8, 8, true>;
using March112 = StMarchCfg<112, 2, 8>;
constexpr int kNumFwdCfg = 5, kFwdMarch96 = 3, kFwdMarch112 = 4;
//                       TH  TW  RS   NT RG RK MINB CSD PIPE XFULL
using Bwd0 = StBwdCfg<28, 56, 16, 256, 2, 8, 2, 8, true>;  // large images: persistent CTAs, the next tile's boxes prefetched
// cfg 1: full-width strips of crops (W <= 96, no x halo); the strip height is picked from the batch (crop_bwd)
using Bwd1 = StBwdCfg<12, 96, 8, 224, 2, 8, 2, 8, true, true>;     // persistent 12-row strips
using Bwd1W = StBwdCfg<24, 96, 14, 192, 2, 8, 2, 8, false, true>;  // 24-row strips, one tile per CTA
constexpr int kNumBwdCfg = 2;

constexpr int kMinFwdTH = 16, kMinFwdTW = 48;  // finest forward work split (workspace sizing): 16-row chunks, 48-wide tiles

static int sm_count() {
#ifdef SRST_EMULATE
  return 2;
#else
  static int cached[64] = {};
  int dev = 0;
  if (cudaGetDevice(&dev) != cudaSuccess || dev < 0 || dev >= 64) return 148;
  if (cached[dev] == 0) {
    int n = 0;
    if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    cached[dev] = n;
  }
  return cached[dev];
#endif
}

// Opt in to > 48 KB of dynamic shared memory once per (kernel, device).
// `Tag` makes the once-flag unique per kernel instantiation (all kernels of one direction share a
// function-pointer type).
template <class Tag, class K>
static int ensure_smem(K kernel, size_t bytes) {
#ifdef SRST_EMULATE
  (void)kernel; (void)bytes;
  return 0;
#else
  static bool done[64] = {};
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return (int)e;
  if (dev >= 0 && dev < 64 && done[dev]) return 0;
  e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
  if (e != cudaSuccess) return (int)e;
  if (dev >= 0 && dev < 64) done[dev] = true;
  return 0;
#endif
}

// Copies the (2*rs+1)- and (2*rk+1)-tap filters into the compiled radii (RG >= rs, RK >= rk),
// centred and zero-padded: a filter with extra zero taps at both ends is the same filter.
template <int RG, int RK>
static void fill_taps(StTaps<RG, RK>& t, const float* g, const float* dg, int rs, const float* k, int rk) {
  for (int i = 0; i <= 2 * RG; ++i) {
    const int j = i - (RG - rs);
    t.g[i] = (j >= 0 && j <= 2 * rs) ? g[j] : 0.f;
    t.dg[i] = (j >= 0 && j <= 2 * rs) ? dg[j] : 0.f;
  }
  for (int i = 0; i <= 2 * RK; ++i) {
    const int j = i - (RK - rk);
    t.k[i] = (j >= 0 && j <= 2 * rk) ? k[j] : 0.f;
  }
  // tap pairs (t[u], t[u-1]) for the row-pair (FFMA2) vertical passes
  for (int u = 0; u <= 2 * RG + 1; ++u) {
    t.gp[u] = make_float2(u <= 2 * RG ? t.g[u] : 0.f, u >= 1 ? t.g[u - 1] : 0.f);
    t.dgp[u] = make_float2(u <= 2 * RG ? t.dg[u] : 0.f, u >= 1 ? t.dg[u - 1] : 0.f);
  }
  for (int u = 0; u <= 2 * RK + 1; ++u) t.kp[u] = make_float2(u <= 2 * RK ? t.k[u] : 0.f, u >= 1 ? t.k[u - 1] : 0.f);
}

// The filled tap block depends on the caller's tap values only: keep the last one per radius class
// and thread (a training loop calls with the same sigma / rho every step).
template <int RG, int RK>
static const StTaps<RG, RK>& cached_taps(const float* g, const float* dg, int rs, const float* k, int rk) {
  struct Entry { bool valid = false; int rs = 0, rk = 0; float g[2 * RG + 1], dg[2 * RG + 1], k[2 * RK + 1]; StTaps<RG, RK> taps; };
  static thread_local Entry e;
  const bool hit = e.valid && e.rs == rs && e.rk == rk && std::memcmp(e.g, g, sizeof(float) * (2 * rs + 1)) == 0 &&
                   std::memcmp(e.dg, dg, sizeof(float) * (2 * rs + 1)) == 0 &&
                   std::memcmp(e.k, k, sizeof(float) * (2 * rk + 1)) == 0;
  if (!hit) {
    e.rs = rs; e.rk = rk;
    std::memcpy(e.g, g, sizeof(float) * (2 * rs + 1));
    std::memcpy(e.dg, dg, sizeof(float) * (2 * rs + 1));
    std::memcpy(e.k, k, sizeof(float) * (2 * rk + 1));
    fill_taps(e.taps, g, dg, rs, k, rk);
    e.valid = true;
  }
  return e.taps;
}

// Tensor map of an fp32 tensor viewed as [planes][rows][cols] with a [box_p][box_h][box_w] box (no
// swizzle, zero OOB fill).  Returns false when TMA cannot be used (unaligned tensor, row pitch not a
// multiple of 16 bytes, driver entry point missing): the kernel then stages with plain loads.
// Encoding costs a driver call, so the last few maps are kept per thread, keyed by everything that
// goes into them (a training loop re-uses the same saved-tensor addresses step after step).
static bool make_plane_map(SrstTmap* map, const float* base, long long planes, int rows, int cols, int box_w, int box_h,
                           int box_p) {
#ifdef SRST_EMULATE
  (void)box_w; (void)box_h; (void)box_p;
  map->base = base; map->W = cols; map->H = rows; map->P = (int)planes;
  return true;
#else
  typedef CUresult (*EncodeFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                               const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                               CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
  static EncodeFn encode = nullptr;
  static bool looked_up = false;
  if (!looked_up) {
    void* fn = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      encode = reinterpret_cast<EncodeFn>(fn);
    looked_up = true;
  }
  if (!encode || !aligned16(base) || (cols % 4) != 0 || box_w > 256 || box_h > 256 || (box_w % 4) != 0) return false;
  struct Key { const float* base; long long planes; int rows, cols, bw, bh, bp; };
  struct Entry { Key key; CUtensorMap map; bool valid; };
  constexpr int kSlots = 16;
  static thread_local Entry cache[kSlots] = {};
  static thread_local int next = 0;
  const Key key{base, planes, rows, cols, box_w, box_h, box_p};
  for (int i = 0; i < kSlots; ++i) {
    const Entry& c = cache[i];
    if (c.valid && c.key.base == key.base && c.key.planes == key.planes && c.key.rows == key.rows &&
        c.key.cols == key.cols && c.key.bw == key.bw && c.key.bh == key.bh && c.key.bp == key.bp) {
      *map = c.map;
      return true;
    }
  }
  const cuuint64_t dims[3] = {(cuuint64_t)cols, (cuuint64_t)rows, (cuuint64_t)planes};
  const cuuint64_t strides[2] = {(cuuint64_t)cols * 4, (cuuint64_t)cols * rows * 4};
  const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_p};
  const cuuint32_t estr[3] = {1, 1, 1};
  if (encode(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, const_cast<float*>(base), dims, strides, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return false;
  Entry& slot = cache[next];
  next = (next + 1) % kSlots;
  slot.key = key; slot.map = *map; slot.valid = true;
  return true;
#endif
}

// once-flag tag per forward / backward instantiation (PI: the per-image reduction, reduction='none'; MAP: the
// distance map)
template <class C, bool PX, bool HR, bool PI = false, bool MAP = false> struct FwdTag {};
template <class C, bool PX, bool PI = false> struct BwdTag {};

template <class C, bool PX = false, bool PI = false, bool MAP = false>
static int launch_st_forward(StFwdParamsT<C::RG, C::RK, MAP>& P, void* stream) {
  P.tiles_x = (P.W + C::TW - 1) / C::TW;
  P.tiles_y = (P.H + C::TH - 1) / C::TH;
  const long long ntiles = (long long)P.B * P.tiles_x * P.tiles_y;
  if (ntiles <= 0 || ntiles > 0x7fffffffLL) return SRST_E_SHAPE;
  int e;
  if (P.ds_hr) {
    if ((e = ensure_smem<FwdTag<C, PX, true, PI, MAP>>(st_forward_kernel<C, PX, true, PI, MAP>, C::SMEM_BYTES)) != 0) return e;
    SRST_LAUNCH_PDL((st_forward_kernel<C, PX, true, PI, MAP>), dim3((unsigned)ntiles), dim3(C::NT), C::SMEM_BYTES, stream, P);
  } else {
    if ((e = ensure_smem<FwdTag<C, PX, false, PI, MAP>>(st_forward_kernel<C, PX, false, PI, MAP>, C::SMEM_BYTES)) != 0) return e;
    SRST_LAUNCH_PDL((st_forward_kernel<C, PX, false, PI, MAP>), dim3((unsigned)ntiles), dim3(C::NT), C::SMEM_BYTES, stream, P);
  }
  return (int)cudaGetLastError();
}

// Row-marching forward.  Returns kMarchUnusable when the images cannot be fetched by TMA (the caller then uses a
// tiled shape).  Chunking: whole strips when B * strips already fills the machine, otherwise each strip is cut
// into as many row chunks as there are idle SMs (a chunk costs one extra 16-row block of gradient + horizontal work).
constexpr int kMarchUnusable = -1000;
template <class C, bool PX, bool HR, bool PI = false, bool MAP = false> struct MarchTag {};
template <class C, bool PX = false, bool PI = false, bool MAP = false>
static int launch_st_march(const StFwdParamsT<C::RG, C::RK, MAP>& F, void* stream) {
  static thread_local StMarchParamsT<C::RG, C::RK, MAP> MP_tls;
  auto& MP = MP_tls;  // a plain reference: the emulation's kernel threads must see THIS thread's instance
  if (!F.vec4) return kMarchUnusable;
  if (C::XFULL && F.W > C::TW) return SRST_E_SHAPE;  // the crop layout has one strip, at x = 0
  if (!make_plane_map(&MP.sr_map, F.sr, (long long)F.B * 3, F.H, F.W, C::BW, C::RS, 3) ||
      !make_plane_map(&MP.hr_map, F.hr, (long long)F.B * 3, F.H, F.W, C::BW, C::RS, 3))
    return kMarchUnusable;
  MP.F = F;
  if constexpr (MAP) MP.map_out = F.map_out;
  const int nblk = (F.H + C::RS - 1) / C::RS;
  MP.nstrips = (F.W + C::TW - 1) / C::TW;
  const long long base = (long long)F.B * MP.nstrips;
  long long nch = 1;
  const int slots = sm_count() * C::MINB;
  if (base < slots) nch = slots / base;
  if (nch > nblk) nch = nblk;
  int cb = (int)((nblk + nch - 1) / nch);
  if (forced_chunk() > 0) cb = forced_chunk() < nblk ? forced_chunk() : nblk;
  MP.chunk_blocks = cb;
  MP.nchunks = (nblk + cb - 1) / cb;
  const long long grid = base * MP.nchunks;
  if (grid <= 0 || grid > 0x7fffffffLL) return SRST_E_SHAPE;
  int e;
  if (F.ds_hr) {
    if ((e = ensure_smem<MarchTag<C, PX, true, PI, MAP>>(st_forward_march_kernel<C, PX, true, PI, MAP>, C::SMEM_BYTES)) != 0)
      return e;
    SRST_LAUNCH_PDL((st_forward_march_kernel<C, PX, true, PI, MAP>), dim3((unsigned)grid), dim3(C::NT), C::SMEM_BYTES, stream, MP);
  } else {
    if ((e = ensure_smem<MarchTag<C, PX, false, PI, MAP>>(st_forward_march_kernel<C, PX, false, PI, MAP>, C::SMEM_BYTES)) != 0)
      return e;
    SRST_LAUNCH_PDL((st_forward_march_kernel<C, PX, false, PI, MAP>), dim3((unsigned)grid), dim3(C::NT), C::SMEM_BYTES, stream, MP);
  }
  return (int)cudaGetLastError();
}

template <class C, bool PX = false, bool PI = false>
static int launch_st_backward(StBwdParams<C::RG, C::RK>& P, void* stream) {
  if (C::XFULL && P.W > C::TW) return SRST_E_SHAPE;  // the tile layout assumes one tile in x
  static const bool tma_env = env_int_once("SRST_ST_BWD_TMA", 1) != 0;
  const int Hp = (P.H + 1) / 2;
  P.use_tma = (tma_env && P.vec4 && aligned16(P.ixy) &&
               make_plane_map(&P.ds_map, P.ds, (long long)P.B * 3, P.H, P.W, C::SW, C::SH, 3) &&
               make_plane_map(&P.ixy_map, P.ixy, (long long)P.B * 2, Hp, 2 * P.W, C::PI, C::EH / 2, 2)) ? 1 : 0;
  P.tiles_x = (P.W + C::TW - 1) / C::TW;
  P.tiles_y = (P.H + C::TH - 1) / C::TH;
  const long long nblk = (long long)P.B * P.tiles_x * P.tiles_y;
  if (nblk <= 0 || nblk > 0x7fffffffLL) return SRST_E_SHAPE;
  int e = ensure_smem<BwdTag<C, PX, PI>>(st_backward_kernel<C, PX, PI>, C::SMEM_BYTES);
  if (e) return e;
  long long grid = nblk;
  if (C::PIPE && P.use_tma) {  // persistent: one wave of resident CTAs, each looping over tiles
    const long long slots = (long long)sm_count() * C::MINB;
    if (grid > slots) grid = slots;
  }
  SRST_LAUNCH_PDL((st_backward_kernel<C, PX, PI>), dim3((unsigned)grid), dim3(C::NT), C::SMEM_BYTES, stream, P);
  return (int)cudaGetLastError();
}

static int pick_fwd_cfg(int B, int H, int W) {
  const int forced = forced_fwd();
  if (forced >= 0 && forced < kNumFwdCfg) return forced;
  // measured on B200 (profiles/r02_tile_sweep.log): full-width 24x96 strips win on 96-wide crops -- two CTAs per SM
  // while the batch is a single wave, the 72-register variant (three CTAs per SM) once there are several waves of
  // strips; the 32x64 tile with three CTAs per SM wins on large images (all unrolled kernels)
  if (W <= 96) return ((long long)B * ((H + 23) / 24) >= 6LL * sm_count()) ? 2 : 1;
  return 0;
}
// Strip width of the marching kernel: the one that pads the image width least (cost = strips * (TW + 2 RK) columns
// of gradient work); 96 columns or 112 (15 warps: four per scheduler, 128 registers).
static int pick_march_cfg(int W) {
  const int forced = forced_fwd();
  if (forced == kFwdMarch96 || forced == kFwdMarch112) return forced;
  if (forced >= 0) return -1;  // a tiled shape was asked for
  static const bool off = env_int_once("SRST_ST_MARCH", 1) == 0;
  if (off) return -1;
  const long long c96 = (long long)((W + 95) / 96) * (96 + 16), c112 = (long long)((W + 111) / 112) * (112 + 16);
  return c96 <= c112 ? kFwdMarch96 : kFwdMarch112;
}
static int pick_bwd_cfg(int B, int H, int W) {
  const int forced = forced_bwd();
  if (forced >= 0 && forced < kNumBwdCfg) return forced;
  // measured on B200 (profiles/r02_tile_sweep.log, r07_bwd_crop_sweep.log): full-width strips on 96-wide crops, the 28x56
  // tile on large images
  (void)B; (void)H;
  return W <= 96 ? 1 : 0;
}

}  // namespace srst

using namespace srst;

extern "C" {

int srst_version(void) { return SRST_VERSION; }

const char* srst_error_string(int code) {
  switch (code) {
    case 0: return "ok";
    case SRST_E_INVALID: return "srst: invalid argument (null pointer, non-positive size or bad enum)";
    case SRST_E_UNSUPPORTED: return "srst: filter radius / patch geometry not compiled into libsrst";
    case SRST_E_WORKSPACE: return "srst: workspace missing, misaligned or too small";
    case SRST_E_SHAPE: return "srst: image shape not usable by this entry point";
    default: break;
  }
#ifndef SRST_EMULATE
  if (code > 0) return cudaGetErrorString((cudaError_t)code);
#endif
  return "srst: unknown error";
}

// Compiled radius classes: r_sigma is padded up to 2 or 4, r_rho up to 4, 8 or 12 (zero taps).
// (2, 8) -- the reference default sigma=0.5, rho=2.0 -- has the tuned tile shapes; the other
// classes use one generic shape each.
static bool st_compiled(int r_sigma, int r_rho) { return r_sigma >= 1 && r_sigma <= 4 && r_rho >= 1 && r_rho <= 12; }
int srst_st_supported(int r_sigma, int r_rho) {
  if (st_compiled(r_sigma, r_rho)) return 1;
  return (r_sigma >= 1 && r_sigma <= kGenMaxR && r_rho >= 1 && r_rho <= kGenMaxR) ? 2 : 0;  // 2: generic-radius path
}

#if defined(SRST_TIMING) && !defined(SRST_EMULATE)
// tools-only build: where the kernels write their phase time stamps (32 slots per CTA); NULL turns them off
int srst_debug_set_timing(long long* device_buffer) {
  return (int)cudaMemcpyToSymbol(g_srst_timing, &device_buffer, sizeof(device_buffer));
}
#endif

int srst_st_num_cfgs(int backward) { return backward ? kNumBwdCfg : kNumFwdCfg; }

int srst_st_force_chunk_blocks(int blocks) {
  g_force_chunk = blocks > 0 ? blocks : -1;
  return 0;
}

int srst_st_force_cfg(int fwd_cfg, int bwd_cfg) {
  if (fwd_cfg < -1 || fwd_cfg >= kNumFwdCfg || bwd_cfg < -1 || bwd_cfg >= kNumBwdCfg) return SRST_E_INVALID;
  g_force_fwd = fwd_cfg;
  g_force_bwd = bwd_cfg;
  return 0;
}

static size_t st_partials_bytes(int B, int H, int W) {
  // one float per CTA of the finest compiled tiling + the ticket counter, rounded to 256 bytes
  const size_t tiles = (size_t)B * ((H + kMinFwdTH - 1) / kMinFwdTH) * ((W + kMinFwdTW - 1) / kMinFwdTW);
  return ((tiles + 4) * sizeof(float) + 255) / 256 * 256;
}

size_t srst_st_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return 2 * st_partials_bytes(B, H, W);  // ST partials + ticket | partials of the fused Pixel term
}

static size_t gen_plane_bytes(int B, int H, int W) { return ((size_t)B * H * W * sizeof(float) + 255) / 256 * 256; }
constexpr int kGenFwdPlanes = 11, kGenBwdPlanes = 5;

size_t srst_st_workspace_bytes_r(int B, int H, int W, int r_sigma, int r_rho) {
  const size_t base = srst_st_workspace_bytes(B, H, W);
  const int sup = srst_st_supported(r_sigma, r_rho);
  if (base == 0 || sup == 0) return 0;
  if (sup == 1) return base;
  return base + kGenMaxPartials * sizeof(float) + kGenFwdPlanes * gen_plane_bytes(B, H, W);
}

size_t srst_st_backward_workspace_bytes(int B, int H, int W, int r_sigma, int r_rho) {
  if (B <= 0 || H <= 0 || W <= 0 || srst_st_supported(r_sigma, r_rho) != 2) return 0;
  return kGenBwdPlanes * gen_plane_bytes(B, H, W);
}

size_t srst_st_ixy_floats(int B, int H, int W) {
  if (B <= 0 || H <= 0 || W <= 0) return 0;
  return (size_t)B * 2 * ((H + 1) / 2) * (size_t)W * 2;
}

}  // extern "C"

namespace srst {

struct StCall {
  // forward: sr, hr -> ds_sr, ds_hr, ixy_sr, ixy_hr, loss_out ; backward: ixy, ds, grad_out -> d_img
  const float *sr = nullptr, *hr = nullptr, *ixy = nullptr, *ds = nullptr, *grad_out = nullptr;
  float *ds_sr = nullptr, *ds_hr = nullptr, *ixy_sr = nullptr, *ixy_hr = nullptr, *loss_out = nullptr, *d_img = nullptr;
  int px = 0;                                            // forward: also reduce the fused Pixel (MSE) term into loss_out[1]
  int per_image = 0;                                     // reduction='none': loss_out / grad_out / grad_px are [B], and
                                                         // the MSE terms go to loss_out[B .. 2B)
  const float *px_img = nullptr, *px_other = nullptr, *grad_px = nullptr;  // backward: image pair + upstream gradient of the MSE term
  float* map_out = nullptr;                              // forward: also store the per-pixel distances [B,H,W]
  int unit_scale = 0;                                    // backward: ds already carries the upstream gradient of each
                                                         // pixel and grad_out is a device 1.0f (no 1/(B H W))
  int B = 0, H = 0, W = 0, normalize = 1, vec4 = 0;
  float eps = 0.f;
  void* workspace = nullptr;
  const float *g = nullptr, *dg = nullptr, *k = nullptr;
  int rs = 0, rk = 0;
  void* stream = nullptr;
};

// one tile shape with the batch or the per-image reduction (c.per_image), or the distance map (c.map_out, never
// together with PX); PX: the fused Pixel term
template <class C, bool PX, int RG, int RK>
static int tiled_fwd(StFwdMapParams<RG, RK>& P, const StCall& c) {
  if (c.map_out) return launch_st_forward<C, false, false, true>(P, c.stream);
  return c.per_image ? launch_st_forward<C, PX, true>(P, c.stream) : launch_st_forward<C, PX>(P, c.stream);
}
template <class C, bool PX>
static int march_fwd(const StFwdMapParams<C::RG, C::RK>& P, const StCall& c) {
  if (c.map_out) return launch_st_march<C, false, false, true>(P, c.stream);
  return c.per_image ? launch_st_march<C, PX, true>(P, c.stream) : launch_st_march<C, PX>(P, c.stream);
}
template <class C, bool PX, int RG, int RK>
static int tiled_bwd(StBwdParams<RG, RK>& P, const StCall& c) {
  return c.per_image ? launch_st_backward<C, PX, true>(P, c.stream) : launch_st_backward<C, PX>(P, c.stream);
}

template <int RG, int RK>
static int st_forward_rr(const StCall& c) {
  static thread_local StFwdMapParams<RG, RK> P;  // ~0.5 KB of taps: filled in place, passed by reference to the launcher
  P.map_out = c.map_out;
  P.sr = c.sr; P.hr = c.hr; P.ds_sr = c.ds_sr; P.ds_hr = c.ds_hr; P.ixy_sr = c.ixy_sr; P.ixy_hr = c.ixy_hr;
  P.ticket = reinterpret_cast<unsigned int*>(c.workspace);
  P.partials = reinterpret_cast<float*>(c.workspace) + 4;
  P.px_partials = c.px ? reinterpret_cast<float*>(reinterpret_cast<char*>(c.workspace) + st_partials_bytes(c.B, c.H, c.W))
                       : nullptr;
  P.loss_out = c.loss_out;
  P.B = c.B; P.H = c.H; P.W = c.W; P.tiles_x = P.tiles_y = 0;
  P.normalize = c.normalize; P.vec4 = c.vec4; P.eps = c.eps;
  P.inv_count = (float)(1.0 / ((double)(c.per_image ? 1 : c.B) * c.H * c.W));
  P.taps = cached_taps<RG, RK>(c.g, c.dg, c.rs, c.k, c.rk);
  if constexpr (RG == 2 && RK == 8) {
    const int mcfg = pick_march_cfg(c.W);
    if (mcfg >= 0) {
      int e;
      if (mcfg == kFwdMarch96 && c.W <= March96X::TW)
        e = c.px ? march_fwd<March96X, true>(P, c) : march_fwd<March96X, false>(P, c);
      else if (mcfg == kFwdMarch96) e = c.px ? march_fwd<March96, true>(P, c) : march_fwd<March96, false>(P, c);
      else e = c.px ? march_fwd<March112, true>(P, c) : march_fwd<March112, false>(P, c);
      if (e != kMarchUnusable) return e;
    }
    int cfg = pick_fwd_cfg(c.B, c.H, c.W);
    if (cfg >= kFwdMarch96) cfg = (c.W <= 96) ? 1 : 0;  // a marching shape was forced but TMA cannot fetch these tensors
    if (c.px) {  // the fused Pixel term is compiled into the two default tile shapes only
      if (cfg != 0 && c.W <= 96) return tiled_fwd<Fwd1, true>(P, c);
      return tiled_fwd<Fwd0, true>(P, c);
    }
    switch (cfg) {
      case 1: return tiled_fwd<Fwd1, false>(P, c);
      case 2: return tiled_fwd<Fwd2, false>(P, c);
      default: return tiled_fwd<Fwd0, false>(P, c);
    }
  } else {
    using G = StFwdCfg<32, 64, 16, 4, RG, RK, (RK <= 8 ? 2 : 1), 0>;
    return c.px ? tiled_fwd<G, true>(P, c) : tiled_fwd<G, false>(P, c);
  }
}

// Crop-width backward (cfg 1, W <= 96).  12-row strips while they fit one round of the resident CTAs (16 x 96 rows:
// 128 strips on 296 slots); beyond that the 24-row strips, whose taller tiles stage and filter fewer halo rows per
// output row: one round instead of two at 64 x 96 rows, and less work per row at 1024 (measured on B200:
// profiles/r07_bwd_crop_sweep.log).
template <bool PX>
static int crop_bwd(StBwdParams<2, 8>& P, const StCall& c) {
  const long long slots = (long long)sm_count() * Bwd1::MINB;
  if ((long long)c.B * ((c.H + Bwd1::TH - 1) / Bwd1::TH) <= slots) return tiled_bwd<Bwd1, PX>(P, c);
  return tiled_bwd<Bwd1W, PX>(P, c);
}

template <int RG, int RK>
static int st_backward_rr(const StCall& c) {
  static thread_local StBwdParams<RG, RK> P;
  P.use_tma = 0;
  P.ds = c.ds; P.ixy = c.ixy; P.grad_out = c.grad_out; P.d_img = c.d_img;
  P.img = c.px_img; P.px_other = c.px_other; P.grad_px = c.grad_px;
  P.B = c.B; P.H = c.H; P.W = c.W; P.tiles_x = P.tiles_y = 0;
  P.vec4 = c.vec4;
  P.inv_count = c.unit_scale ? 1.0f : (float)(1.0 / ((double)(c.per_image ? 1 : c.B) * c.H * c.W));
  P.taps = cached_taps<RG, RK>(c.g, c.dg, c.rs, c.k, c.rk);
  if constexpr (RG == 2 && RK == 8) {
    if (c.px_other) {  // the fused Pixel term is compiled into the two default tile shapes
      if (c.W <= Bwd1::TW) return crop_bwd<true>(P, c);
      return tiled_bwd<Bwd0, true>(P, c);
    }
    if (c.W <= Bwd1::TW && pick_bwd_cfg(c.B, c.H, c.W) == 1) return crop_bwd<false>(P, c);
    return tiled_bwd<Bwd0, false>(P, c);  // cfg 1 forced on an image wider than its strips runs cfg 0
  } else {
    using G = StBwdCfg<24, 64, (24 + 2 * RG) / 2, 256, RG, RK, (RK <= 8 ? 2 : 1), 4>;
    return c.px_other ? tiled_bwd<G, true>(P, c) : tiled_bwd<G, false>(P, c);
  }
}

// ---- generic-radius path (st_generic.cuh): any radius up to kGenMaxR, scratch planes in the workspace ----
static void gen_fill_taps(StGenTaps& t, const StCall& c) {
  t.rs = c.rs; t.rk = c.rk;
  std::memcpy(t.g, c.g, sizeof(float) * (2 * c.rs + 1));
  std::memcpy(t.dg, c.dg, sizeof(float) * (2 * c.rs + 1));
  std::memcpy(t.k, c.k, sizeof(float) * (2 * c.rk + 1));
}

static int st_forward_generic(const StCall& c, size_t workspace_bytes) {
  if (workspace_bytes < srst_st_workspace_bytes_r(c.B, c.H, c.W, c.rs, c.rk)) return SRST_E_WORKSPACE;
  const size_t npix = (size_t)c.B * c.H * c.W, pb = gen_plane_bytes(c.B, c.H, c.W);
  if (npix > 0x7fffffffULL * (size_t)kGenNT) return SRST_E_SHAPE;
  char* w = reinterpret_cast<char*>(c.workspace);
  float* partials = reinterpret_cast<float*>(w + srst_st_workspace_bytes(c.B, c.H, c.W));
  char* planes = reinterpret_cast<char*>(partials + kGenMaxPartials);
  auto plane = [&](int i) { return reinterpret_cast<float*>(planes + (size_t)i * pb); };
  float* S[2] = {plane(0), plane(3)};  // smoothed tensors of SR / HR (3 planes each); T1, T2 of an image live in its S first
  float* V = plane(6);                 // vertical pass of the products (3 planes), shared by the two images
  float* IXY = plane(9);               // Ix, Iy (2 planes) when the caller does not save them
  static thread_local StGenParams P_tls;
  StGenParams& P = P_tls;
  P.B = c.B; P.H = c.H; P.W = c.W; P.scale = 0.f;
  gen_fill_taps(P.taps, c);
  const unsigned nblk = (unsigned)((npix + kGenNT - 1) / kGenNT);
  for (int img = 0; img < 2; ++img) {
    float* ixy = img ? c.ixy_hr : c.ixy_sr;
    if (!ixy) ixy = IXY;
    float* T1 = S[img];
    float* T2 = S[img] + pb / sizeof(float);
    P.in0 = img ? c.hr : c.sr; P.in1 = P.in2 = nullptr; P.out0 = T1; P.out1 = T2;
    SRST_LAUNCH(gen_gray_v_kernel, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
    P.in0 = T1; P.in1 = T2; P.out0 = ixy; P.out1 = nullptr;
    SRST_LAUNCH(gen_grad_h_kernel, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
    P.in0 = ixy; P.in1 = nullptr; P.out0 = V;
    SRST_LAUNCH(gen_prod_v_kernel, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
    P.in0 = V; P.out0 = S[img];
    SRST_LAUNCH(gen_smooth_h_kernel, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
  }
  StGenChainParams Q;
  Q.s1 = S[0]; Q.s2 = S[1]; Q.ds_sr = c.ds_sr; Q.ds_hr = c.ds_hr; Q.partials = partials;
  Q.ticket = reinterpret_cast<unsigned int*>(c.workspace); Q.loss_out = c.loss_out;
  Q.B = c.B; Q.H = c.H; Q.W = c.W; Q.normalize = c.normalize; Q.eps = c.eps;
  if (c.per_image) {
    // CTAs that each stay inside one image, image-major; their partials go where the compiled classes keep theirs
    // (B * ceil(H/16) * ceil(W/48) slots after the ticket), so any B fits
    const size_t plane_blocks = ((size_t)c.H * c.W + kGenNT - 1) / kGenNT;
    const size_t slots = (size_t)((c.H + kMinFwdTH - 1) / kMinFwdTH) * ((c.W + kMinFwdTW - 1) / kMinFwdTW);
    size_t per = (size_t)kGenMaxPartials / (size_t)c.B;
    per = per < 1 ? 1 : per;
    per = per < plane_blocks ? per : plane_blocks;
    per = per < slots ? per : slots;
    if ((size_t)c.B * per > 0x7fffffffULL) return SRST_E_SHAPE;
    Q.partials = reinterpret_cast<float*>(c.workspace) + 4;
    Q.inv_count = (float)(1.0 / ((double)c.H * c.W));
    SRST_LAUNCH(gen_chain_kernel<true>, dim3((unsigned)(c.B * per)), dim3(kGenNT), 0, c.stream, Q);
    return (int)cudaGetLastError();
  }
  Q.inv_count = (float)(1.0 / ((double)c.B * c.H * c.W));
  const unsigned ngrid = nblk < (unsigned)kGenMaxPartials ? nblk : (unsigned)kGenMaxPartials;
  if (c.map_out) {
    StGenChainMapParams M;
    static_cast<StGenChainParams&>(M) = Q;
    M.map_out = c.map_out;
    SRST_LAUNCH((gen_chain_kernel<false, true>), dim3(ngrid), dim3(kGenNT), 0, c.stream, M);
    return (int)cudaGetLastError();
  }
  SRST_LAUNCH(gen_chain_kernel<false>, dim3(ngrid), dim3(kGenNT), 0, c.stream, Q);
  return (int)cudaGetLastError();
}

static int st_backward_generic(const StCall& c, void* workspace, size_t workspace_bytes) {
  if (!workspace || !aligned16(workspace) ||
      workspace_bytes < srst_st_backward_workspace_bytes(c.B, c.H, c.W, c.rs, c.rk))
    return SRST_E_WORKSPACE;
  const size_t npix = (size_t)c.B * c.H * c.W, pb = gen_plane_bytes(c.B, c.H, c.W);
  if (npix > 0x7fffffffULL * (size_t)kGenNT) return SRST_E_SHAPE;
  char* w = reinterpret_cast<char*>(workspace);
  float* V = reinterpret_cast<float*>(w);            // Ch(k) ds: 3 planes; U1, U2 re-use its first two
  float* DI = reinterpret_cast<float*>(w + 3 * pb);  // dIx, dIy
  // the kernels index [B][n][H][W] densely: the plane stride inside a scratch region is H*W floats, not pb
  static thread_local StGenParams P_tls;
  StGenParams& P = P_tls;
  P.B = c.B; P.H = c.H; P.W = c.W;
  P.scale = c.unit_scale ? 1.0f : (float)(1.0 / ((double)(c.per_image ? 1 : c.B) * c.H * c.W));
  gen_fill_taps(P.taps, c);
  const unsigned nblk = (unsigned)((npix + kGenNT - 1) / kGenNT);
  P.in0 = c.ds; P.in1 = P.in2 = nullptr; P.out0 = V; P.out1 = nullptr;
  SRST_LAUNCH(gen_smooth_v_kernel, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
  P.in0 = V; P.in1 = c.ixy; P.out0 = DI;
  SRST_LAUNCH(gen_bwd_prod_kernel, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
  P.in0 = DI; P.in1 = nullptr; P.out0 = V;
  SRST_LAUNCH(gen_bwd_gh_kernel, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
  P.in0 = V; P.in1 = c.grad_out; P.out0 = c.d_img;
  if (c.per_image) SRST_LAUNCH(gen_bwd_gv_kernel<true>, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
  else SRST_LAUNCH(gen_bwd_gv_kernel<false>, dim3(nblk), dim3(kGenNT), 0, c.stream, P);
  return (int)cudaGetLastError();
}

static int st_dispatch(const StCall& c, bool forward) {
  const int rg = c.rs <= 2 ? 2 : 4;
  const int rk = c.rk <= 4 ? 4 : (c.rk <= 8 ? 8 : 12);
#define SRST_RR(RG_, RK_) \
  if (rg == RG_ && rk == RK_) return forward ? st_forward_rr<RG_, RK_>(c) : st_backward_rr<RG_, RK_>(c);
  SRST_RR(2, 8) SRST_RR(2, 4) SRST_RR(2, 12) SRST_RR(4, 4) SRST_RR(4, 8) SRST_RR(4, 12)
#undef SRST_RR
  return SRST_E_UNSUPPORTED;
}

}  // namespace srst

// srst_st_forward and srst_st_forward_per_image: the same checks and dispatch; per_image selects the [B] reduction
// (srst_st_forward_map: map_out set, per_image 0)
static int st_forward_entry(const float* sr, const float* hr, int B, int H, int W, const float* g, const float* dg,
                            int r_sigma, const float* k, int r_rho, int normalize, float eps, float* loss_out,
                            float* ds_sr, float* ds_hr, float* ixy_sr, float* ixy_hr, void* workspace,
                            size_t workspace_bytes, void* stream, int per_image, float* map_out = nullptr) {
  if (!sr || !hr || !g || !dg || !k || !loss_out || B <= 0 || H <= 0 || W <= 0) return SRST_E_INVALID;
  if (!srst_st_supported(r_sigma, r_rho)) return SRST_E_UNSUPPORTED;
  if (!workspace || !aligned16(workspace) || workspace_bytes < srst_st_workspace_bytes(B, H, W))
    return SRST_E_WORKSPACE;
  StCall c;
  c.sr = sr; c.hr = hr; c.ds_sr = ds_sr; c.ds_hr = ds_hr; c.ixy_sr = ixy_sr; c.ixy_hr = ixy_hr; c.loss_out = loss_out;
  c.B = B; c.H = H; c.W = W; c.normalize = normalize ? 1 : 0; c.eps = eps;
  c.vec4 = (W % 4 == 0 && aligned16(sr) && aligned16(hr) && (!ds_sr || aligned16(ds_sr)) &&
            (!ds_hr || aligned16(ds_hr)) && (!ixy_sr || aligned16(ixy_sr)) && (!ixy_hr || aligned16(ixy_hr))) ? 1 : 0;
  c.workspace = workspace; c.g = g; c.dg = dg; c.k = k; c.rs = r_sigma; c.rk = r_rho; c.stream = stream;
  c.per_image = per_image;
  c.map_out = map_out;
  if (!st_compiled(r_sigma, r_rho)) return st_forward_generic(c, workspace_bytes);
  return st_dispatch(c, true);
}

// (srst_st_backward_map: ds = the weighted scratch planes, grad_out = the unit slot, unit_scale 1)
static int st_backward_entry(const float* ixy, const float* ds, const float* grad_out, int B, int H, int W,
                             const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float* d_img,
                             void* workspace, size_t workspace_bytes, void* stream, int per_image, int unit_scale = 0) {
  if (!ixy || !ds || !grad_out || !g || !dg || !k || !d_img || B <= 0 || H <= 0 || W <= 0) return SRST_E_INVALID;
  if (!srst_st_supported(r_sigma, r_rho)) return SRST_E_UNSUPPORTED;
  StCall c;
  c.ixy = ixy; c.ds = ds; c.grad_out = grad_out; c.d_img = d_img;
  c.B = B; c.H = H; c.W = W;
  c.vec4 = (W % 4 == 0 && aligned16(d_img) && aligned16(ds)) ? 1 : 0;
  c.g = g; c.dg = dg; c.k = k; c.rs = r_sigma; c.rk = r_rho; c.stream = stream;
  c.per_image = per_image;
  c.unit_scale = unit_scale;
  if (!st_compiled(r_sigma, r_rho)) return st_backward_generic(c, workspace, workspace_bytes);
  return st_dispatch(c, false);
}

extern "C" {

int srst_st_forward(const float* sr, const float* hr, int B, int H, int W, const float* g, const float* dg,
                    int r_sigma, const float* k, int r_rho, int normalize, float eps, float* loss_out,
                    float* ds_sr, float* ds_hr, float* ixy_sr, float* ixy_hr, void* workspace,
                    size_t workspace_bytes, void* stream) {
  return st_forward_entry(sr, hr, B, H, W, g, dg, r_sigma, k, r_rho, normalize, eps, loss_out, ds_sr, ds_hr, ixy_sr,
                          ixy_hr, workspace, workspace_bytes, stream, 0);
}

int srst_st_forward_per_image(const float* sr, const float* hr, int B, int H, int W, const float* g, const float* dg,
                              int r_sigma, const float* k, int r_rho, int normalize, float eps, float* loss_out,
                              float* ds_sr, float* ds_hr, float* ixy_sr, float* ixy_hr, void* workspace,
                              size_t workspace_bytes, void* stream) {
  return st_forward_entry(sr, hr, B, H, W, g, dg, r_sigma, k, r_rho, normalize, eps, loss_out, ds_sr, ds_hr, ixy_sr,
                          ixy_hr, workspace, workspace_bytes, stream, 1);
}

int srst_st_backward_ws(const float* ixy, const float* ds, const float* grad_out, int B, int H, int W,
                        const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float* d_img,
                        void* workspace, size_t workspace_bytes, void* stream) {
  return st_backward_entry(ixy, ds, grad_out, B, H, W, g, dg, r_sigma, k, r_rho, d_img, workspace, workspace_bytes,
                           stream, 0);
}

int srst_st_backward_per_image(const float* ixy, const float* ds, const float* grad_out, int B, int H, int W,
                               const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float* d_img,
                               void* workspace, size_t workspace_bytes, void* stream) {
  return st_backward_entry(ixy, ds, grad_out, B, H, W, g, dg, r_sigma, k, r_rho, d_img, workspace, workspace_bytes,
                           stream, 1);
}

int srst_st_backward(const float* ixy, const float* ds, const float* grad_out, int B, int H, int W,
                     const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float* d_img,
                     void* stream) {
  return srst_st_backward_ws(ixy, ds, grad_out, B, H, W, g, dg, r_sigma, k, r_rho, d_img, nullptr, 0, stream);
}

int srst_st_forward_map(const float* sr, const float* hr, int B, int H, int W, const float* g, const float* dg,
                        int r_sigma, const float* k, int r_rho, int normalize, float eps, float* loss_out,
                        float* map_out, float* ds_sr, float* ds_hr, float* ixy_sr, float* ixy_hr, void* workspace,
                        size_t workspace_bytes, void* stream) {
  if (!map_out) return SRST_E_INVALID;
  return st_forward_entry(sr, hr, B, H, W, g, dg, r_sigma, k, r_rho, normalize, eps, loss_out, ds_sr, ds_hr, ixy_sr,
                          ixy_hr, workspace, workspace_bytes, stream, 0, map_out);
}

// workspace of srst_st_backward_map: the weighted ds planes [B,3,H,W], the unit slot, then the generic-radius scratch
static size_t st_map_ds_bytes(int B, int H, int W) { return ((size_t)B * 3 * H * W * sizeof(float) + 255) / 256 * 256; }
constexpr size_t kMapUnitBytes = 256;

size_t srst_st_backward_map_workspace_bytes(int B, int H, int W, int r_sigma, int r_rho) {
  if (B <= 0 || H <= 0 || W <= 0 || !srst_st_supported(r_sigma, r_rho)) return 0;
  return st_map_ds_bytes(B, H, W) + kMapUnitBytes + srst_st_backward_workspace_bytes(B, H, W, r_sigma, r_rho);
}

int srst_st_backward_map(const float* ixy, const float* ds, const float* grad_map, int B, int H, int W,
                         const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float* d_img,
                         void* workspace, size_t workspace_bytes, void* stream) {
  if (!ixy || !ds || !grad_map || !g || !dg || !k || !d_img || B <= 0 || H <= 0 || W <= 0) return SRST_E_INVALID;
  if (!srst_st_supported(r_sigma, r_rho)) return SRST_E_UNSUPPORTED;
  if (!workspace || !aligned16(workspace) ||
      workspace_bytes < srst_st_backward_map_workspace_bytes(B, H, W, r_sigma, r_rho))
    return SRST_E_WORKSPACE;
  const size_t plane = (size_t)H * W, ds_bytes = st_map_ds_bytes(B, H, W);
  float* wds = reinterpret_cast<float*>(workspace);
  float* unit = reinterpret_cast<float*>(reinterpret_cast<char*>(workspace) + ds_bytes);
  const bool vec4 = W % 4 == 0 && aligned16(ds) && aligned16(grad_map);
  const size_t items = (size_t)B * plane / (vec4 ? 4 : 1);
  const size_t want = (items + kMapNT - 1) / kMapNT, cap = (size_t)sm_count() * 16;
  const dim3 grid((unsigned)(want < cap ? want : cap));
  if (vec4) SRST_LAUNCH(st_map_scale_kernel<true>, grid, dim3(kMapNT), 0, stream, ds, grad_map, wds, unit, B, plane);
  else SRST_LAUNCH(st_map_scale_kernel<false>, grid, dim3(kMapNT), 0, stream, ds, grad_map, wds, unit, B, plane);
  if (const int e = (int)cudaGetLastError()) return e;
  return st_backward_entry(ixy, wds, unit, B, H, W, g, dg, r_sigma, k, r_rho, d_img, unit + kMapUnitBytes / sizeof(float),
                           workspace_bytes - ds_bytes - kMapUnitBytes, stream, 0, 1);
}

}  // extern "C"

// srst_stpx_forward and srst_stpx_forward_per_image: the same checks and dispatch; per_image selects the [2][B] output
static int stpx_forward_entry(const float* sr, const float* hr, int B, int H, int W, const float* g, const float* dg,
                              int r_sigma, const float* k, int r_rho, int normalize, float eps, float* loss2_out,
                              float* ds_sr, float* ixy_sr, void* workspace, size_t workspace_bytes, void* stream,
                              int per_image) {
  if (!sr || !hr || !g || !dg || !k || !loss2_out || B <= 0 || H <= 0 || W <= 0) return SRST_E_INVALID;
  if (!st_compiled(r_sigma, r_rho)) return SRST_E_UNSUPPORTED;  // the generic-radius path has no fused / feature variant
  if (!workspace || !aligned16(workspace) || workspace_bytes < srst_st_workspace_bytes(B, H, W))
    return SRST_E_WORKSPACE;
  StCall c;
  c.sr = sr; c.hr = hr; c.ds_sr = ds_sr; c.ixy_sr = ixy_sr; c.loss_out = loss2_out; c.px = 1;
  c.B = B; c.H = H; c.W = W; c.normalize = normalize ? 1 : 0; c.eps = eps;
  c.vec4 = (W % 4 == 0 && aligned16(sr) && aligned16(hr) && (!ds_sr || aligned16(ds_sr)) &&
            (!ixy_sr || aligned16(ixy_sr))) ? 1 : 0;
  c.workspace = workspace; c.g = g; c.dg = dg; c.k = k; c.rs = r_sigma; c.rk = r_rho; c.stream = stream;
  c.per_image = per_image;
  return st_dispatch(c, true);
}

static int stpx_backward_entry(const float* sr, const float* hr, const float* ixy, const float* ds, const float* grad_st,
                               const float* grad_px, int B, int H, int W, const float* g, const float* dg, int r_sigma,
                               const float* k, int r_rho, float* d_sr, void* stream, int per_image) {
  if (!sr || !hr || !ixy || !ds || !grad_st || !grad_px || !g || !dg || !k || !d_sr || B <= 0 || H <= 0 || W <= 0)
    return SRST_E_INVALID;
  if (!st_compiled(r_sigma, r_rho)) return SRST_E_UNSUPPORTED;  // the generic-radius path has no fused / feature variant
  StCall c;
  c.ixy = ixy; c.ds = ds; c.grad_out = grad_st; c.d_img = d_sr; c.px_img = sr; c.px_other = hr; c.grad_px = grad_px;
  c.B = B; c.H = H; c.W = W;
  c.vec4 = (W % 4 == 0 && aligned16(sr) && aligned16(hr) && aligned16(d_sr) && aligned16(ds)) ? 1 : 0;
  c.g = g; c.dg = dg; c.k = k; c.rs = r_sigma; c.rk = r_rho; c.stream = stream;
  c.per_image = per_image;
  return st_dispatch(c, false);
}

extern "C" {

int srst_stpx_forward(const float* sr, const float* hr, int B, int H, int W, const float* g, const float* dg,
                      int r_sigma, const float* k, int r_rho, int normalize, float eps, float* loss2_out, float* ds_sr,
                      float* ixy_sr, void* workspace, size_t workspace_bytes, void* stream) {
  return stpx_forward_entry(sr, hr, B, H, W, g, dg, r_sigma, k, r_rho, normalize, eps, loss2_out, ds_sr, ixy_sr,
                            workspace, workspace_bytes, stream, 0);
}

int srst_stpx_forward_per_image(const float* sr, const float* hr, int B, int H, int W, const float* g, const float* dg,
                                int r_sigma, const float* k, int r_rho, int normalize, float eps, float* loss2_out,
                                float* ds_sr, float* ixy_sr, void* workspace, size_t workspace_bytes, void* stream) {
  return stpx_forward_entry(sr, hr, B, H, W, g, dg, r_sigma, k, r_rho, normalize, eps, loss2_out, ds_sr, ixy_sr,
                            workspace, workspace_bytes, stream, 1);
}

int srst_stpx_backward(const float* sr, const float* hr, const float* ixy, const float* ds, const float* grad_st,
                       const float* grad_px, int B, int H, int W, const float* g, const float* dg, int r_sigma,
                       const float* k, int r_rho, float* d_sr, void* stream) {
  return stpx_backward_entry(sr, hr, ixy, ds, grad_st, grad_px, B, H, W, g, dg, r_sigma, k, r_rho, d_sr, stream, 0);
}

int srst_stpx_backward_per_image(const float* sr, const float* hr, const float* ixy, const float* ds,
                                 const float* grad_st, const float* grad_px, int B, int H, int W, const float* g,
                                 const float* dg, int r_sigma, const float* k, int r_rho, float* d_sr, void* stream) {
  return stpx_backward_entry(sr, hr, ixy, ds, grad_st, grad_px, B, H, W, g, dg, r_sigma, k, r_rho, d_sr, stream, 1);
}

}  // extern "C"

namespace srst {
template <int RG, int RK>
static int st_features_rr(const float* img, int B, int H, int W, const float* g, const float* dg, int rs, const float* k, int rk,
                          float* J, float* eig, float* orient, float* coher, int vec4, void* stream) {
  using C = StFwdCfg<32, 64, 16, 4, RG, RK, (RK <= 8 ? 2 : 1), 0>;
  static thread_local StFeatParams<RG, RK> P;
  P.img = img; P.J = J; P.eig = eig; P.orient = orient; P.coher = coher;
  P.B = B; P.H = H; P.W = W; P.vec4 = vec4;
  P.tiles_x = (W + C::TW - 1) / C::TW;
  P.tiles_y = (H + C::TH - 1) / C::TH;
  const long long ntiles = (long long)B * P.tiles_x * P.tiles_y;
  if (ntiles <= 0 || ntiles > 0x7fffffffLL) return SRST_E_SHAPE;
  P.taps = cached_taps<RG, RK>(g, dg, rs, k, rk);
  struct FeatTag {};
  int e = ensure_smem<FeatTag>(st_features_kernel<C>, C::SMEM_BYTES);
  if (e) return e;
  const StFeatParams<RG, RK>& Pr = P;  // (the emulation runs kernel bodies on other OS threads: never name a thread_local there)
  SRST_LAUNCH(st_features_kernel<C>, dim3((unsigned)ntiles), dim3(C::NT), C::SMEM_BYTES, stream, Pr);
  return (int)cudaGetLastError();
}
}  // namespace srst

extern "C" int srst_st_features(const float* img, int B, int H, int W, const float* g, const float* dg, int r_sigma,
                                const float* k, int r_rho, float* J_out, float* eig_out, float* orient_out,
                                float* coher_out, void* stream) {
  if (!img || !g || !dg || !k || B <= 0 || H <= 0 || W <= 0) return SRST_E_INVALID;
  if (!J_out && !eig_out && !orient_out && !coher_out) return SRST_E_INVALID;
  if (!st_compiled(r_sigma, r_rho)) return SRST_E_UNSUPPORTED;  // the generic-radius path has no fused / feature variant
  const int vec4 = (W % 4 == 0 && aligned16(img)) ? 1 : 0;
  const int rg = r_sigma <= 2 ? 2 : 4;
  const int rk = r_rho <= 4 ? 4 : (r_rho <= 8 ? 8 : 12);
#define SRST_FT(RG_, RK_) \
  if (rg == RG_ && rk == RK_) \
    return st_features_rr<RG_, RK_>(img, B, H, W, g, dg, r_sigma, k, r_rho, J_out, eig_out, orient_out, coher_out, vec4, stream);
  SRST_FT(2, 8) SRST_FT(2, 4) SRST_FT(2, 12) SRST_FT(4, 4) SRST_FT(4, 8) SRST_FT(4, 12)
#undef SRST_FT
  return SRST_E_UNSUPPORTED;
}

// ---- Best-Buddy entry points ---------------------------------------------------------------
extern "C" {

size_t srst_bb_workspace_bytes(int B, int H, int W) {
  if (B <= 0 || H < 12 || W < 12) return 0;
  return bb_carve(nullptr, bb_geom(B, H, W)).total_bytes;
}

// grid of the grid-stride zero-fill: never more CTAs than the buffer has 256-element slices
static unsigned fill_grid(size_t n, unsigned cap) {
  const size_t want = (n + 255) / 256;
  return (unsigned)(want < 1 ? 1 : (want < cap ? want : cap));
}

static int bb_launch_pyramid(const float* gt, const BbGeom& g, float* o2, float* o4, void* stream) {
  const size_t n = (size_t)g.B * 3 * ((size_t)g.H2 * g.W2 + (size_t)g.H4 * g.W4);
  const unsigned nblk = (unsigned)((n + 255) / 256);
  SRST_LAUNCH(bb_pyramid_kernel, dim3(nblk), dim3(256), 0, stream, gt, o2, o4, g.B * 3, g.H, g.W, g.H2, g.W2,
              g.H4, g.W4);
  return (int)cudaGetLastError();
}

int srst_bb_pyramid(const float* gt, int B, int H, int W, float* out2, float* out4, void* stream) {
  if (!gt || !out2 || !out4 || B <= 0) return SRST_E_INVALID;
  if (H < 12 || W < 12) return SRST_E_SHAPE;
  return bb_launch_pyramid(gt, bb_geom(B, H, W), out2, out4, stream);
}

}  // extern "C"

// Splits the search norm off `criterion` (dist_norm, utils.py:166-172; the backward entry points ignore it): what is
// left must be L1 or L2.
static int bb_criterion(int& criterion, bool& dist_l1) {
  dist_l1 = (criterion & SRST_BB_DIST_L1) != 0;
  criterion &= ~SRST_BB_DIST_L1;
  return (criterion == SRST_BB_L1 || criterion == SRST_BB_L2) ? 0 : SRST_E_INVALID;
}

// Arguments of the default-geometry patch entry points, after their NULL / B <= 0 check: criterion, shape, then the
// gt2 / gt4 pairing.
static int bb_check(int& criterion, bool& dist_l1, int B, int H, int W, const float* gt2, const float* gt4) {
  if (const int e = bb_criterion(criterion, dist_l1)) return e;
  if (H < 12 || W < 12 || B > 65535) return SRST_E_SHAPE;
  return (gt2 == nullptr) != (gt4 == nullptr) ? SRST_E_INVALID : 0;
}

// The caller's coarse levels of gt, or the library's own built into pyr2 / pyr4 (workspace).
static int bb_levels(const float* gt, const BbGeom& g, const float*& gt2, const float*& gt4, float* pyr2, float* pyr4,
                     void* stream) {
  if (gt2) return 0;
  gt2 = pyr2;
  gt4 = pyr4;
  return bb_launch_pyramid(gt, g, pyr2, pyr4, stream);
}

static int zero_fill(float* p, size_t n, void* stream) {
#ifdef SRST_EMULATE
  std::memset(p, 0, sizeof(float) * n);
  return 0;
#else
  return (int)cudaMemsetAsync(p, 0, sizeof(float) * n, (cudaStream_t)stream);
#endif
}

// PI: reduction='none' (srst_patch_forward_per_image): loss_out is [B].  MAP (srst_patch_forward_map): loss_out[0] as
// the scalar entry points, and map_out [B][N] the per-query means
template <int MODE, bool PI = false, bool MAP = false>
static int bb_forward_impl(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W,
                           float alpha, float beta, int criterion, int64_t* idx_out, float* loss_out, void* workspace,
                           size_t workspace_bytes, void* stream, const PstTaps& tp = PstTaps{}, float* map_out = nullptr) {
  static_assert(!(PI && MAP), "one output form");
  constexpr int D = BbDesc<MODE>::D;
  if (!sr || !gt || !idx_out || !loss_out || (MAP && !map_out) || B <= 0) return SRST_E_INVALID;
  bool dist_l1;
  int e = bb_check(criterion, dist_l1, B, H, W, gt2, gt4);
  if (e) return e;
  const BbGeom g = bb_geom(B, H, W);
  if (!workspace || !aligned16(workspace)) return SRST_E_WORKSPACE;
  const BbWorkspace w = bb_carve(workspace, g, D);
  if (workspace_bytes < w.total_bytes) return SRST_E_WORKSPACE;
  if ((e = bb_levels(gt, g, gt2, gt4, w.pyr2, w.pyr4, stream)) != 0) return e;
  const int npack = g.Npad > g.Mpad ? g.Npad : g.Mpad;
  SRST_LAUNCH(bb_pack_kernel<MODE>, dim3((npack + 255) / 256, B), dim3(256), 0, stream, sr, gt, gt2, gt4, w.mats,
              w.per_image, g, tp);
  if ((e = (int)cudaGetLastError()) != 0) return e;
  if (dist_l1)
    SRST_LAUNCH(bb_search_l1_kernel<D>, dim3(g.Npad / BB_QT, B), dim3(BB_NT), 0, stream, w.mats, w.per_image, g, alpha, beta,
                idx_out);
  else {
    struct SearchTag {};
    constexpr size_t dyn = bb_search_dyn_smem<D>();
    if ((e = ensure_smem<SearchTag>(bb_search_kernel<D, MODE == 2>, dyn)) != 0) return e;
    SRST_LAUNCH((bb_search_kernel<D, MODE == 2>), dim3(g.Npad / BB_QT, B), dim3(BB_NT), dyn, stream, w.mats, w.per_image, g,
                alpha, beta, idx_out);
  }
  if ((e = (int)cudaGetLastError()) != 0) return e;
  if constexpr (PI) {
    // ceil(N / BB_NT) CTAs per image, so that none spans two images.  That can be more CTAs than w.partials has slots
    // for; their partials go over the library's own x1/2 pyramid level instead (the loss kernel reads only the
    // descriptor matrices, and every backward entry point rebuilds that level).  It holds 3 (H/2)(W/2) >= N / 256 + 1
    // floats per image.
    const unsigned per = (unsigned)((g.N + BB_NT - 1) / BB_NT);
    SRST_LAUNCH((bb_loss_kernel<D, true>), dim3(per * (unsigned)B), dim3(BB_NT), 0, stream, w.mats, w.per_image, g, idx_out,
                criterion, w.pyr2, w.ticket, loss_out);
    return (int)cudaGetLastError();
  }
  const unsigned nl = (unsigned)(((size_t)B * g.N + BB_NT - 1) / BB_NT);
  if constexpr (MAP)
    SRST_LAUNCH((bb_loss_kernel<D, false, true>), dim3(nl), dim3(BB_NT), 0, stream, w.mats, w.per_image, g, idx_out,
                criterion, w.partials, w.ticket, loss_out, map_out);
  else
    SRST_LAUNCH(bb_loss_kernel<D>, dim3(nl), dim3(BB_NT), 0, stream, w.mats, w.per_image, g, idx_out, criterion,
                w.partials, w.ticket, loss_out);
  return (int)cudaGetLastError();
}

extern "C" {

int srst_bb_forward(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W,
                    float alpha, float beta, int criterion, int64_t* idx_out, float* loss_out, void* workspace,
                    size_t workspace_bytes, void* stream) {
  return bb_forward_impl<0>(sr, gt, gt2, gt4, B, H, W, alpha, beta, criterion, idx_out, loss_out, workspace,
                            workspace_bytes, stream);
}

int srst_gram_forward(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W,
                      float alpha, float beta, int criterion, int64_t* idx_out, float* loss_out, void* workspace,
                      size_t workspace_bytes, void* stream) {
  return bb_forward_impl<1>(sr, gt, gt2, gt4, B, H, W, alpha, beta, criterion, idx_out, loss_out, workspace,
                            workspace_bytes, stream);
}

}  // extern "C"

// Central five taps (offsets -2..2) of a (2r+1)-tap filter: all a 3x3 patch image can see.
static void central5(const float* t, int r, float (&o)[5]) {
  for (int i = 0; i < 5; ++i) {
    const int j = r + i - 2;
    o[i] = (j >= 0 && j <= 2 * r) ? t[j] : 0.f;
  }
}
static int pst_taps(const float* g, const float* dg, int r_sigma, const float* k, int r_rho, PstTaps& tp) {
  if (!g || !dg || !k || r_sigma < 1 || r_rho < 1 || r_sigma > 4096 || r_rho > 4096) return SRST_E_INVALID;
  central5(g, r_sigma, tp.g);
  central5(dg, r_sigma, tp.dg);
  central5(k, r_rho, tp.k);
  return 0;
}

// PI: reduction='none' (srst_patch_backward_per_image): grad_out is [B]; MAP (srst_patch_backward_map): [B][N]
template <int MODE, bool PI = false, bool MAP = false>
static int patch_backward_impl(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                               const float* grad_out, int B, int H, int W, int criterion, float* d_sr, void* workspace,
                               size_t workspace_bytes, void* stream, const PstTaps& tp = PstTaps{}) {
  if (!sr || !gt || !idx || !grad_out || !d_sr || B <= 0) return SRST_E_INVALID;
  bool dist_l1;
  int e = bb_check(criterion, dist_l1, B, H, W, gt2, gt4);
  if (e) return e;
  const BbGeom g = bb_geom(B, H, W);
  if (!gt2) {  // the workspace only has to hold the library's own pyramid levels
    if (!workspace || !aligned16(workspace)) return SRST_E_WORKSPACE;
    const BbWorkspace w = bb_carve(workspace, g);
    if (workspace_bytes < w.total_bytes) return SRST_E_WORKSPACE;
    if ((e = bb_levels(gt, g, gt2, gt4, w.pyr2, w.pyr4, stream)) != 0) return e;
  }
  if constexpr (MODE == 0) {  // one thread per pixel of d_sr
    const size_t total = (size_t)B * 3 * H * W;
    SRST_LAUNCH((bb_backward_kernel<PI, MAP>), dim3((unsigned)((total + 255) / 256)), dim3(256), 0, stream, sr, gt, gt2, gt4,
                idx, grad_out, g, criterion, d_sr);
  } else {  // one thread per patch: pixels outside every patch keep a zero gradient
    if ((H % 3 != 0 || W % 3 != 0) && (e = zero_fill(d_sr, (size_t)B * 3 * H * W, stream)) != 0) return e;
    const size_t total = (size_t)B * g.N;
    if constexpr (MODE == 1)
      SRST_LAUNCH((gram_backward_kernel<false, PI, MAP>), dim3((unsigned)((total + 255) / 256)), dim3(256), 0, stream, sr, gt,
                  gt2, gt4, idx, grad_out, g, criterion, d_sr, nullptr, nullptr);
    else
      SRST_LAUNCH((pst_backward_kernel<false, PI, MAP>), dim3((unsigned)((total + 127) / 128)), dim3(128), 0, stream, sr, gt,
                  gt2, gt4, idx, grad_out, g, tp, criterion, d_sr, nullptr, nullptr);
  }
  return (int)cudaGetLastError();
}

extern "C" {

int srst_pst_forward(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W,
                     const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float alpha, float beta,
                     int criterion, int64_t* idx_out, float* loss_out, void* workspace, size_t workspace_bytes,
                     void* stream) {
  PstTaps tp;
  const int e = pst_taps(g, dg, r_sigma, k, r_rho, tp);
  if (e) return e;
  return bb_forward_impl<2>(sr, gt, gt2, gt4, B, H, W, alpha, beta, criterion, idx_out, loss_out, workspace,
                            workspace_bytes, stream, tp);
}

int srst_bb_backward(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                     const float* grad_out, int B, int H, int W, int criterion, float* d_sr, void* workspace,
                     size_t workspace_bytes, void* stream) {
  return patch_backward_impl<0>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, criterion, d_sr, workspace, workspace_bytes,
                                stream);
}

int srst_gram_backward(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                       const float* grad_out, int B, int H, int W, int criterion, float* d_sr, void* workspace,
                       size_t workspace_bytes, void* stream) {
  return patch_backward_impl<1>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, criterion, d_sr, workspace, workspace_bytes,
                                stream);
}

int srst_pst_backward(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                      const float* grad_out, int B, int H, int W, const float* g, const float* dg, int r_sigma,
                      const float* k, int r_rho, int criterion, float* d_sr, void* workspace, size_t workspace_bytes,
                      void* stream) {
  PstTaps tp;
  const int e = pst_taps(g, dg, r_sigma, k, r_rho, tp);
  if (e) return e;
  return patch_backward_impl<2>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, criterion, d_sr, workspace, workspace_bytes,
                                stream, tp);
}

}  // extern "C"

// srst_patch_backward_gt, and the d_gt half of srst_patch_backward_per_image (PI: grad_out is [B]) and of
// srst_patch_backward_map (MAP: grad_out is [B][N])
template <bool PI, bool MAP = false>
static int patch_backward_gt_impl(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                                  const int64_t* idx, const float* grad_out, int B, int H, int W, const float* g,
                                  const float* dg, int r_sigma, const float* k, int r_rho, int criterion, float* d_gt,
                                  void* workspace, size_t workspace_bytes, void* stream) {
  if (!sr || !gt || !idx || !grad_out || !d_gt || B <= 0 || mode < 0 || mode > 2) return SRST_E_INVALID;
  bool dist_l1;
  int e = bb_check(criterion, dist_l1, B, H, W, gt2, gt4);
  if (e) return e;
  PstTaps tp = {};
  if (mode == 2 && (e = pst_taps(g, dg, r_sigma, k, r_rho, tp)) != 0) return e;
  const BbGeom gm = bb_geom(B, H, W);
  if (!workspace || !aligned16(workspace)) return SRST_E_WORKSPACE;
  const BbWorkspace w = bb_carve(workspace, gm);
  if (workspace_bytes < w.total_bytes) return SRST_E_WORKSPACE;
  if ((e = bb_levels(gt, gm, gt2, gt4, w.pyr2, w.pyr4, stream)) != 0) return e;
  // gradient images of the two coarse levels: in the descriptor-matrix region of the workspace (dead after the forward)
  const size_t n0 = (size_t)B * 3 * H * W, n2 = (size_t)B * 3 * gm.H2 * gm.W2, n4 = (size_t)B * 3 * gm.H4 * gm.W4;
  float* d2 = w.mats;
  float* d4 = d2 + (n2 + 3) / 4 * 4;
  if ((n2 + 3) / 4 * 4 + n4 > w.per_image * (size_t)B) return SRST_E_WORKSPACE;
  SRST_LAUNCH(bb_fill_zero_kernel, dim3(fill_grid(n0, 592)), dim3(256), 0, stream, d_gt, n0);
  SRST_LAUNCH(bb_fill_zero_kernel, dim3(fill_grid((n2 + 3) / 4 * 4 + n4, 148)), dim3(256), 0, stream, d2, (n2 + 3) / 4 * 4 + n4);
  const size_t total = (size_t)B * gm.N;
  if (mode == 0)
    SRST_LAUNCH((bb_backward_gt_kernel<PI, MAP>), dim3((unsigned)((total + 255) / 256)), dim3(256), 0, stream, sr, gt, gt2,
                gt4, idx, grad_out, gm, criterion, d_gt, d2, d4);
  else if (mode == 1)
    SRST_LAUNCH((gram_backward_kernel<true, PI, MAP>), dim3((unsigned)((total + 255) / 256)), dim3(256), 0, stream, sr, gt,
                gt2, gt4, idx, grad_out, gm, criterion, d_gt, d2, d4);
  else
    SRST_LAUNCH((pst_backward_kernel<true, PI, MAP>), dim3((unsigned)((total + 127) / 128)), dim3(128), 0, stream, sr, gt,
                gt2, gt4, idx, grad_out, gm, tp, criterion, d_gt, d2, d4);
  SRST_LAUNCH(bb_pyramid_adjoint_kernel, dim3((unsigned)((n2 + n4 + 255) / 256)), dim3(256), 0, stream, d2, d4, d_gt, B * 3,
              H, W, gm.H2, gm.W2, gm.H4, gm.W4);
  return (int)cudaGetLastError();
}

extern "C" {

int srst_patch_backward_gt(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                           const int64_t* idx, const float* grad_out, int B, int H, int W, const float* g, const float* dg,
                           int r_sigma, const float* k, int r_rho, int criterion, float* d_gt, void* workspace,
                           size_t workspace_bytes, void* stream) {
  return patch_backward_gt_impl<false>(mode, sr, gt, gt2, gt4, idx, grad_out, B, H, W, g, dg, r_sigma, k, r_rho, criterion,
                                       d_gt, workspace, workspace_bytes, stream);
}

}  // extern "C"

// srst_patch_forward_per_image (PI) and srst_patch_forward_map (MAP): `mode` picks the descriptor
template <bool PI, bool MAP>
static int patch_forward_mode(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H,
                              int W, const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float alpha,
                              float beta, int criterion, int64_t* idx_out, float* loss_out, float* map_out, void* workspace,
                              size_t workspace_bytes, void* stream) {
  switch (mode) {
    case 0:
      return bb_forward_impl<0, PI, MAP>(sr, gt, gt2, gt4, B, H, W, alpha, beta, criterion, idx_out, loss_out, workspace,
                                         workspace_bytes, stream, PstTaps{}, map_out);
    case 1:
      return bb_forward_impl<1, PI, MAP>(sr, gt, gt2, gt4, B, H, W, alpha, beta, criterion, idx_out, loss_out, workspace,
                                         workspace_bytes, stream, PstTaps{}, map_out);
    case 2: {
      PstTaps tp;
      const int e = pst_taps(g, dg, r_sigma, k, r_rho, tp);
      if (e) return e;
      return bb_forward_impl<2, PI, MAP>(sr, gt, gt2, gt4, B, H, W, alpha, beta, criterion, idx_out, loss_out, workspace,
                                         workspace_bytes, stream, tp, map_out);
    }
    default: return SRST_E_INVALID;
  }
}

// srst_patch_backward_per_image (PI) and srst_patch_backward_map (MAP): d_sr and / or d_gt in one call
template <bool PI, bool MAP>
static int patch_backward_mode(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                               const int64_t* idx, const float* grad_out, int B, int H, int W, const float* g,
                               const float* dg, int r_sigma, const float* k, int r_rho, int criterion, float* d_sr,
                               float* d_gt, void* workspace, size_t workspace_bytes, void* stream) {
  if ((!d_sr && !d_gt) || mode < 0 || mode > 2) return SRST_E_INVALID;
  int e = 0;
  if (d_sr) {
    PstTaps tp;
    if (mode == 2 && (e = pst_taps(g, dg, r_sigma, k, r_rho, tp)) != 0) return e;
    if (mode == 0) e = patch_backward_impl<0, PI, MAP>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, criterion, d_sr, workspace,
                                                       workspace_bytes, stream);
    else if (mode == 1) e = patch_backward_impl<1, PI, MAP>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, criterion, d_sr,
                                                            workspace, workspace_bytes, stream);
    else e = patch_backward_impl<2, PI, MAP>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, criterion, d_sr, workspace,
                                             workspace_bytes, stream, tp);
    if (e) return e;
  }
  if (d_gt)
    e = patch_backward_gt_impl<PI, MAP>(mode, sr, gt, gt2, gt4, idx, grad_out, B, H, W, g, dg, r_sigma, k, r_rho, criterion,
                                        d_gt, workspace, workspace_bytes, stream);
  return e;
}

extern "C" {

int srst_patch_forward_per_image(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4, int B,
                                 int H, int W, const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                                 float alpha, float beta, int criterion, int64_t* idx_out, float* loss_out,
                                 void* workspace, size_t workspace_bytes, void* stream) {
  return patch_forward_mode<true, false>(mode, sr, gt, gt2, gt4, B, H, W, g, dg, r_sigma, k, r_rho, alpha, beta, criterion,
                                         idx_out, loss_out, nullptr, workspace, workspace_bytes, stream);
}

int srst_patch_backward_per_image(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                                  const int64_t* idx, const float* grad_out, int B, int H, int W, const float* g,
                                  const float* dg, int r_sigma, const float* k, int r_rho, int criterion, float* d_sr,
                                  float* d_gt, void* workspace, size_t workspace_bytes, void* stream) {
  return patch_backward_mode<true, false>(mode, sr, gt, gt2, gt4, idx, grad_out, B, H, W, g, dg, r_sigma, k, r_rho,
                                          criterion, d_sr, d_gt, workspace, workspace_bytes, stream);
}

int srst_patch_forward_map(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H,
                           int W, const float* g, const float* dg, int r_sigma, const float* k, int r_rho, float alpha,
                           float beta, int criterion, int64_t* idx_out, float* loss_out, float* map_out, void* workspace,
                           size_t workspace_bytes, void* stream) {
  return patch_forward_mode<false, true>(mode, sr, gt, gt2, gt4, B, H, W, g, dg, r_sigma, k, r_rho, alpha, beta, criterion,
                                         idx_out, loss_out, map_out, workspace, workspace_bytes, stream);
}

int srst_patch_backward_map(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                            const int64_t* idx, const float* grad_map, int B, int H, int W, const float* g, const float* dg,
                            int r_sigma, const float* k, int r_rho, int criterion, float* d_sr, float* d_gt,
                            void* workspace, size_t workspace_bytes, void* stream) {
  return patch_backward_mode<false, true>(mode, sr, gt, gt2, gt4, idx, grad_map, B, H, W, g, dg, r_sigma, k, r_rho,
                                          criterion, d_sr, d_gt, workspace, workspace_bytes, stream);
}

}  // extern "C"

// ---- Best-Buddy loss, arbitrary patch geometry (bb_generic.cuh) -----------------------------------------------
static int bbg_prepare(const float* gt, const float*& gt2, const float*& gt4, int B, int H, int W, const BbgGeom& g,
                       void* workspace, size_t workspace_bytes, BbgWorkspace& w, void* stream) {
  if (!workspace || !aligned16(workspace)) return SRST_E_WORKSPACE;
  w = bbg_carve(workspace, g);
  if (workspace_bytes < w.total_bytes) return SRST_E_WORKSPACE;
  if ((gt2 == nullptr) != (gt4 == nullptr)) return SRST_E_INVALID;
  return bb_levels(gt, bb_geom(B, H, W), gt2, gt4, w.pyr2, w.pyr4, stream);
}

extern "C" {

int srst_bbg_supported(int ksize, int pad, int stride) {
  return (ksize >= 1 && ksize <= BBG_MAXK && pad >= 0 && pad <= 64 && stride >= 1 && stride <= 4096) ? 1 : 0;
}

size_t srst_bbg_workspace_bytes(int B, int H, int W, int ksize, int pad, int stride) {
  if (!bbg_geom_ok(B, H, W, ksize, pad, stride)) return 0;
  return bbg_carve(nullptr, bbg_geom(B, H, W, ksize, pad, stride)).total_bytes;
}

long long srst_bbg_num_patches(int H, int W, int ksize, int pad, int stride) {
  if (!bbg_geom_ok(1, H, W, ksize, pad, stride)) return 0;
  return bbg_geom(1, H, W, ksize, pad, stride).N;
}

}  // extern "C"

// srst_bbg_forward / srst_bbg_forward_per_image (PI: loss_out is [B]) / srst_bbg_forward_map (MAP: map_out [B][N])
template <bool PI, bool MAP = false>
static int bbg_forward_impl(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W,
                            int ksize, int pad, int stride, float alpha, float beta, int criterion, int64_t* idx_out,
                            float* loss_out, void* workspace, size_t workspace_bytes, void* stream,
                            float* map_out = nullptr) {
  static_assert(!(PI && MAP), "one output form");
  if (!sr || !gt || !idx_out || !loss_out || (MAP && !map_out) || B <= 0) return SRST_E_INVALID;
  bool dist_l1;
  int e = bb_criterion(criterion, dist_l1);
  if (e) return e;
  if (!srst_bbg_supported(ksize, pad, stride)) return SRST_E_UNSUPPORTED;
  if (!bbg_geom_ok(B, H, W, ksize, pad, stride)) return SRST_E_SHAPE;
  const BbgGeom g = bbg_geom(B, H, W, ksize, pad, stride);
  BbgWorkspace w;
  if ((e = bbg_prepare(gt, gt2, gt4, B, H, W, g, workspace, workspace_bytes, w, stream)) != 0) return e;
  struct BbgSearchTag {};
  const size_t dyn = bbg_search_smem(3 * BBG_MAXK * BBG_MAXK);  // one opt-in covers every ksize
  if ((e = ensure_smem<BbgSearchTag>(bbg_search_kernel, dyn)) != 0) return e;
  SRST_LAUNCH(bbg_pack_kernel, dim3((unsigned)((w.Mpad + 255) / 256), (unsigned)B), dim3(256), 0, stream, gt, gt2, gt4, g,
              w.ymat, w.y_per_image, w.Mpad);
  if ((e = (int)cudaGetLastError()) != 0) return e;
  SRST_LAUNCH(bbg_search_kernel, dim3((unsigned)((g.N + BBG_QT - 1) / BBG_QT), (unsigned)B), dim3(BBG_NT),
              bbg_search_smem(g.D), stream, sr, gt, w.ymat, w.y_per_image, w.Mpad, g, alpha, beta, dist_l1 ? 1 : 0, idx_out);
  if ((e = (int)cudaGetLastError()) != 0) return e;
  if constexpr (PI) {
    // ceil(N / BBG_NT) CTAs per image, so that none spans two images; their partials go over the candidate matrices,
    // which only the search reads ((D + 1) Mpad >= N floats per image)
    const unsigned per = (unsigned)((g.N + BBG_NT - 1) / BBG_NT);
    SRST_LAUNCH(bbg_loss_kernel<true>, dim3(per * (unsigned)B), dim3(BBG_NT), 0, stream, sr, gt, gt2, gt4, g, idx_out,
                criterion, w.ymat, w.ticket, loss_out);
    return (int)cudaGetLastError();
  }
  const unsigned nl = (unsigned)(((size_t)B * g.N + BBG_NT - 1) / BBG_NT);
  if constexpr (MAP)
    SRST_LAUNCH((bbg_loss_kernel<false, true>), dim3(nl), dim3(BBG_NT), 0, stream, sr, gt, gt2, gt4, g, idx_out, criterion,
                w.partials, w.ticket, loss_out, map_out);
  else
    SRST_LAUNCH(bbg_loss_kernel<false>, dim3(nl), dim3(BBG_NT), 0, stream, sr, gt, gt2, gt4, g, idx_out, criterion,
                w.partials, w.ticket, loss_out);
  return (int)cudaGetLastError();
}

// srst_bbg_backward / srst_bbg_backward_per_image (PI: grad_out is [B]) / srst_bbg_backward_map (MAP: [B][N])
template <bool PI, bool MAP = false>
static int bbg_backward_impl(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                             const float* grad_out, int B, int H, int W, int ksize, int pad, int stride, int criterion,
                             float* d_sr, float* d_gt, void* workspace, size_t workspace_bytes, void* stream) {
  if (!sr || !gt || !idx || !grad_out || (!d_sr && !d_gt) || B <= 0) return SRST_E_INVALID;
  bool dist_l1;
  int e = bb_criterion(criterion, dist_l1);
  if (e) return e;
  if (!srst_bbg_supported(ksize, pad, stride)) return SRST_E_UNSUPPORTED;
  if (!bbg_geom_ok(B, H, W, ksize, pad, stride)) return SRST_E_SHAPE;
  const BbgGeom g = bbg_geom(B, H, W, ksize, pad, stride);
  BbgWorkspace w;
  if ((e = bbg_prepare(gt, gt2, gt4, B, H, W, g, workspace, workspace_bytes, w, stream)) != 0) return e;
  const size_t n0 = (size_t)B * 3 * H * W;
  if (d_sr) {
    SRST_LAUNCH((bbg_backward_kernel<PI, MAP>), dim3((unsigned)((n0 + 255) / 256)), dim3(256), 0, stream, sr, gt, gt2, gt4,
                idx, grad_out, g, criterion, d_sr);
    if ((e = (int)cudaGetLastError()) != 0) return e;
  }
  if (d_gt) {
    const size_t n2 = (size_t)B * 3 * g.L[1].H * g.L[1].W, n4 = (size_t)B * 3 * g.L[2].H * g.L[2].W;
    SRST_LAUNCH(bb_fill_zero_kernel, dim3(fill_grid(n0, 592)), dim3(256), 0, stream, d_gt, n0);
    SRST_LAUNCH(bb_fill_zero_kernel, dim3(fill_grid((n2 + 3) / 4 * 4 + n4, 148)), dim3(256), 0, stream, w.d2, (n2 + 3) / 4 * 4 + n4);
    const size_t total = (size_t)B * g.N * 3;
    SRST_LAUNCH((bbg_backward_gt_kernel<PI, MAP>), dim3((unsigned)((total + 255) / 256)), dim3(256), 0, stream, sr, gt, gt2,
                gt4, idx, grad_out, g, criterion, d_gt, w.d2, w.d4);
    SRST_LAUNCH(bb_pyramid_adjoint_kernel, dim3((unsigned)((n2 + n4 + 255) / 256)), dim3(256), 0, stream, w.d2, w.d4, d_gt,
                B * 3, H, W, g.L[1].H, g.L[1].W, g.L[2].H, g.L[2].W);
    if ((e = (int)cudaGetLastError()) != 0) return e;
  }
  return 0;
}

extern "C" {

int srst_bbg_forward(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W, int ksize,
                     int pad, int stride, float alpha, float beta, int criterion, int64_t* idx_out, float* loss_out,
                     void* workspace, size_t workspace_bytes, void* stream) {
  return bbg_forward_impl<false>(sr, gt, gt2, gt4, B, H, W, ksize, pad, stride, alpha, beta, criterion, idx_out, loss_out,
                                 workspace, workspace_bytes, stream);
}

int srst_bbg_forward_per_image(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W,
                               int ksize, int pad, int stride, float alpha, float beta, int criterion, int64_t* idx_out,
                               float* loss_out, void* workspace, size_t workspace_bytes, void* stream) {
  return bbg_forward_impl<true>(sr, gt, gt2, gt4, B, H, W, ksize, pad, stride, alpha, beta, criterion, idx_out, loss_out,
                                workspace, workspace_bytes, stream);
}

int srst_bbg_backward(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                      const float* grad_out, int B, int H, int W, int ksize, int pad, int stride, int criterion,
                      float* d_sr, float* d_gt, void* workspace, size_t workspace_bytes, void* stream) {
  return bbg_backward_impl<false>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, ksize, pad, stride, criterion, d_sr, d_gt,
                                  workspace, workspace_bytes, stream);
}

int srst_bbg_backward_per_image(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                                const float* grad_out, int B, int H, int W, int ksize, int pad, int stride, int criterion,
                                float* d_sr, float* d_gt, void* workspace, size_t workspace_bytes, void* stream) {
  return bbg_backward_impl<true>(sr, gt, gt2, gt4, idx, grad_out, B, H, W, ksize, pad, stride, criterion, d_sr, d_gt,
                                 workspace, workspace_bytes, stream);
}

int srst_bbg_forward_map(const float* sr, const float* gt, const float* gt2, const float* gt4, int B, int H, int W,
                         int ksize, int pad, int stride, float alpha, float beta, int criterion, int64_t* idx_out,
                         float* loss_out, float* map_out, void* workspace, size_t workspace_bytes, void* stream) {
  return bbg_forward_impl<false, true>(sr, gt, gt2, gt4, B, H, W, ksize, pad, stride, alpha, beta, criterion, idx_out,
                                       loss_out, workspace, workspace_bytes, stream, map_out);
}

int srst_bbg_backward_map(const float* sr, const float* gt, const float* gt2, const float* gt4, const int64_t* idx,
                          const float* grad_map, int B, int H, int W, int ksize, int pad, int stride, int criterion,
                          float* d_sr, float* d_gt, void* workspace, size_t workspace_bytes, void* stream) {
  return bbg_backward_impl<false, true>(sr, gt, gt2, gt4, idx, grad_map, B, H, W, ksize, pad, stride, criterion, d_sr, d_gt,
                                        workspace, workspace_bytes, stream);
}

}  // extern "C"
