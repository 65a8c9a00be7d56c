// Row-marching structure-tensor forward for sm_100a: the default forward of the reference radius class
// (sigma = 0.5, rho = 2.0; loss.py:384) whenever the images can be fetched by TMA (W % 4 == 0, 16-byte aligned).
//
// One CTA owns a column strip (TW columns) of one image pair and marches down a chunk of its rows in blocks
// of 16.  Nothing is recomputed vertically: a ring of horizontally smoothed product rows lives in shared
// memory, so every row goes through the gradient and the horizontal rho-pass exactly once per chunk (the
// tiled kernel in st_kernels.cuh recomputes a 16-row halo per 24..32-row tile).  The CTA is split in two
// thread groups that work on different blocks at the same time:
//
//   producers (NP threads)  raw RGB rows (TMA box, one block ahead) -> gray -> Ix, Iy (saved for the backward)
//                           -> products + HORIZONTAL rho-pass (the 24-column Ix, Iy window is read once for
//                           all three products) -> ring rows
//   consumers (NC threads)  VERTICAL rho-pass over the ring for both images -> per-pixel chain (utils.py:236-279
//                           and its adjoint) -> loss partial + ds stores; a thread owns one column and eight rows,
//                           so S1 and S2 of a pixel meet in registers without any exchange
//
// Step k of the march has two halves separated by CTA barriers:
//   Y_k : producers: gradients of block k            | consumers: vertical pass of output block k-2
//   X_k : producers: horizontal pass of block k,     | consumers: chain + stores of output block k-2
//         then gray conversion of block k+1 and the
//         TMA request for block k+2
// The ring holds two blocks (32 rows); block k overwrites block k-2, which the consumers finished reading
// in Y_k.  H block k covers rows y0 - RK + 16k .., output block j rows y0 + 16j .. and needs H blocks j, j+1.
//
// Per pixel pair of the image the kernel executes ~400 FP32 lane-operations (tiled kernel: ~570) and moves
// ~250 bytes through shared memory (tiled: ~450); see DESIGN.md section 3.
#pragma once
#include "st_kernels.cuh"

namespace srst {

// tools/march_bench.cu only: run-time ablation mask (skip a phase) to measure what each phase costs
#ifdef SRST_MARCH_ABL
__device__ int g_march_abl = 0;
#define MARCH_ON(bit) (((g_march_abl >> (bit)) & 1) == 0)
#endif
#ifdef SRST_MARCH_STAMPS
__device__ long long* g_march_stamp = nullptr;  // [grid][128] %globaltimer stamps of producer thread 0 (slots 0..63) and consumer thread 0 (64..127)
SRST_DEV void march_stamp(bool who, int slot) {
  if (g_march_stamp && who && slot < 64) {
    long long t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    g_march_stamp[(size_t)blockIdx.x * 128 + slot + (threadIdx.x ? 64 : 0)] = t;
  }
}
#define MSTAMP(who, slot) march_stamp(who, slot)
#else
#define MSTAMP(who, slot) ((void)0)
#endif
#ifndef SRST_MARCH_ABL
#define MARCH_ON(bit) true
#endif

template <int RG, int RK>
struct StMarchParams {
  SrstTmap sr_map;  // sr viewed as [B*3][H][W]; box [3][16][BW]
  SrstTmap hr_map;
  StFwdParams<RG, RK> F;
  int nstrips, nchunks, chunk_blocks;  // grid = B * nchunks * nstrips; a chunk = chunk_blocks * 16 rows
};
// MAP: the distance map [B,H,W] (see StFwdMapParams)
template <int RG, int RK>
struct StMarchMapParams : StMarchParams<RG, RK> {
  float* map_out;
};
template <int RG, int RK, bool MAP>
using StMarchParamsT = std::conditional_t<MAP, StMarchMapParams<RG, RK>, StMarchParams<RG, RK>>;

// XFULL: crop layout, for images no wider than the strip (W <= TW, so x0 == 0).  Every x-halo column is outside
// the image, so its gray values and gradients are zeros: the raw box and the gray conversion cover the TW image
// columns only, the gradient items the NSEGH image segments only, and the zero columns that the edge windows read
// (gray: GXH per side, Ix / Iy: RK per side) are written once per CTA.  The gradient and horizontal items are
// mapped so that a warp holds 4 consecutive row pairs (xitem): a warp whose rows are all outside the image skips
// the arithmetic of both passes.
template <int TW_, int RG_, int RK_, int CR_ = 8, bool XFULL_ = false>
struct StMarchCfg {
  static constexpr bool XFULL = XFULL_;
  static constexpr int TW = TW_, RG = RG_, RK = RK_;
  static constexpr int CR = CR_, CQ = CR_ / 2;       // rows / row pairs of a block that one consumer thread owns (8 or 4 rows)
  static constexpr int RS = 16, NQ = 8;             // rows / row pairs per block
  // x halo of the gray rows; a multiple of 4: TMA wants the first box column 16-byte aligned, and the crop
  // layout's gray rows start 16-byte aligned too (its halo is the RG zero columns of the edge windows)
  static constexpr int GXH = XFULL ? round_up4(RG) : round_up4(RK + RG);
  static constexpr int GOFF = GXH - RK - RG;        // gray columns left of the window of gradient segment 0 (x0 - RK ..)
  static constexpr int GW = TW + 2 * GXH;           // width of the gray rows
  static constexpr int BX = XFULL ? 0 : -GXH;       // first raw box column relative to x0
  static constexpr int BW = XFULL ? TW : GW;        // width of the raw box
  static constexpr int GP = NQ + RG;                // gray row pairs held: RG carried from the previous block + 8 new
  static constexpr int PG = smem_pitch(2 * GW);
  static constexpr int DW = TW + 2 * RK, PD = smem_pitch(2 * DW);  // Ix, Iy rows (x halo RK)
  static constexpr int NSEGB = DW / 8, NSEGH = TW / 8;             // 8-column items of the gradient / horizontal pass
  static constexpr int PH = smem_pitch(2 * TW);
  static constexpr int BWIN = 8 + 2 * RG;           // gray window of a gradient item
  static constexpr int HWIN = 8 + 2 * RK;           // Ix, Iy window of a horizontal item
  static constexpr int NIN = RK + CQ;               // ring row pairs a consumer reads for its CQ output row pairs
  static constexpr int NP = 2 * NQ * NSEGB;         // producers: one gradient item each (2 images x 8 row pairs x segments)
  static constexpr int NH = 2 * NQ * NSEGH;         // horizontal items (the first NH producers; XFULL: gradient items too)
  static constexpr int NC = (RS / CR) * TW;         // consumers: column x row part of the block
  static constexpr int NT = NP + NC;
  static constexpr int RAW_IMG = 3 * RS * BW;       // one TMA box
  static constexpr int GRAY_IMG = GP * PG, D_PLANE = NQ * PD, H_PLANE = 2 * NQ * PH;
  static constexpr int GRAY_OFF = (2 * RAW_IMG + 31) / 32 * 32;
  static constexpr int D_OFF = GRAY_OFF + 4 * GRAY_IMG;   // two gray buffers (block parity) x two images
  static constexpr int H_OFF = D_OFF + 4 * D_PLANE;
  static constexpr int SMEM_FLOATS = H_OFF + 6 * H_PLANE;
  static constexpr size_t SMEM_BYTES = sizeof(float) * SMEM_FLOATS;
  static constexpr int MINB = SMEM_BYTES <= 112 * 1024 ? 2 : 1;  // CTAs per SM
  static_assert(CR == 8 || CR == 4, "march: consumer rows");
  static_assert(RG % 2 == 0 && RK == 8, "march: radii (two ring blocks cover 16 + 2 RK rows; 8-column items aligned to the strip)");
  static_assert(TW % 16 == 0 && NP % 32 == 0 && NC % 32 == 0 && NT <= 1024, "march: strip width");
  static_assert(BW % 4 == 0 && BW <= 256 && (RAW_IMG * 4) % 128 == 0 && GOFF % 2 == 0, "march: TMA box");
  static_assert(NH <= NP && NP - NH == 32 && TW / 2 <= 64, "march: horizontal items; one copy warp, two float4 per lane and row pair");

  // Crop layout item map: item i < NH -> row pair q, image, image segment seg (columns 8 seg ..).  A warp holds row
  // pairs 4h .. 4h+3 (h = warp / XWH) of 8 consecutive (image, segment) pairs; a quarter-warp holds those 4 row
  // pairs of 2 adjacent segments of one image.
  static constexpr int XWH = NH / 64;  // warps per half block
  __host__ __device__ static constexpr void xitem(int i, int& q, int& img, int& seg) {
    const int w = i >> 5, l = i & 31;
    q = 4 * (w / XWH) + (l & 3);
    const int c = 8 * (w % XWH) + 2 * (l >> 3) + ((l >> 2) & 1);
    img = c / NSEGH;
    seg = c % NSEGH;
  }
  // 16-byte bank group of every LDS.128 / STS.128 address of the crop items (the window steps move all lanes of a
  // quarter-warp alike): gray window (gradient), Ix / Iy row (gradient store, horizontal window), ring row (store).
  // A quarter-warp is one shared-memory wavefront when its 8 lanes hit 8 distinct groups.
  __host__ __device__ static constexpr bool xitem_conflict_free() {
    for (int g = 0; g < NH / 8; ++g)
      for (int a = 0; a < 2 * 4; ++a) {  // address kind x ring / gray parity
        unsigned seen = 0;
        for (int l = 0; l < 8; ++l) {
          int q = 0, img = 0, seg = 0;
          xitem(8 * g + l, q, img, seg);
          const int par = a & 1;
          int off = 0;
          switch (a >> 1) {
            case 0: off = (par * 2 + img) * GRAY_IMG + q * PG + 2 * (8 * (seg + RK / 8) + GOFF); break;
            case 1: off = img * 2 * D_PLANE + q * PD + 2 * (8 * (seg + RK / 8)); break;
            case 2: off = img * 2 * D_PLANE + q * PD + 2 * (8 * seg); break;
            default: off = img * 3 * H_PLANE + (8 * par + q) * PH + 2 * (8 * seg); break;
          }
          if (off % 4 != 0) return false;
          seen |= 1u << ((off / 4) % 8);
        }
        if (seen != 0xffu) return false;
      }
    return true;
  }
  static_assert(!XFULL || (NQ == 8 && NSEGH % 4 == 0 && GXH >= RG), "march crop layout: 4 row pairs x 8 items per warp");
};

// The per-pixel chain on RAW tensors: same mathematics as st_pixel2 with the normalisation folded in.  With
// s1 = 1/sqrt(det S1 + eps), s2 likewise and s = s1 s2, the normalised matrix adj(S1^)S2^ is s times the raw one
// (trace T = s T', discriminant s^2 disc'), so the six normalising multiplies and their adjoints disappear:
//   dT' = s dT, ddisc' = s^2 ddisc, and with Q = s ds = T dT + 2 disc ddisc:  d(det S1) = -Q s1^2 / 2.
// Operand negations are kept out of the packed instructions (one -c, one -h up front).
template <bool WANT_SR, bool WANT_HR>
SRST_DEV float2 st_pixel2_raw(float2 a, float2 b, float2 c, float2 e, float2 f, float2 h, bool normalize, float eps,
                              StPixelGrad2& G) {
  constexpr float kLn2 = 0.6931471805599453f;
  const float2 eps2 = bcast2(eps), m1 = bcast2(-1.0f), half = bcast2(0.5f);
  const float2 nc = mul2(c, m1), nh = mul2(h, m1);
  float2 s1 = bcast2(1.0f), s2 = bcast2(1.0f);
  if (normalize) {
    s1 = rsqrt_nr2(add2(ffma2(a, b, mul2(c, nc)), eps2));
    s2 = rsqrt_nr2(add2(ffma2(e, f, mul2(h, nh)), eps2));
  }
  const float2 s = mul2(s1, s2);
  const float2 nch = mul2(nc, h);
  const float2 Ar = ffma2(b, e, nch), Br = ffma2(a, f, nch);
  const float2 Cr = ffma2(b, h, mul2(nc, f)), Dr = ffma2(a, h, mul2(nc, e));
  const float2 Tr = add2(Ar, Br);
  const float2 ambr = ffma2(Br, m1, Ar);
  const float2 discr = ffma2(mul2(Cr, Dr), bcast2(4.0f), mul2(ambr, ambr));
  const float2 ss = mul2(s, s);
  const float2 disc_raw = mul2(ss, discr);
  const float2 T = mul2(s, Tr);
  const float2 disc = make_float2((disc_raw.x < eps) ? eps : disc_raw.x, (disc_raw.y < eps) ? eps : disc_raw.y);
  const float2 ir = rsq2(disc);
  const float2 r = mul2(disc, ir);
  const float2 hT = mul2(half, T);
  const float2 l1r = ffma2(bcast2(-0.5f), r, hT), l2r = ffma2(half, r, hT);
  const float2 l1 = make_float2((l1r.x < 1.0f) ? 1.0f : l1r.x, (l1r.y < 1.0f) ? 1.0f : l1r.y);
  const float2 l2 = make_float2((l2r.x < 1.0f) ? 1.0f : l2r.x, (l2r.y < 1.0f) ? 1.0f : l2r.y);
  const float2 L1 = mul2(bcast2(kLn2), lg22(l1)), L2 = mul2(bcast2(kLn2), lg22(l2));
  const float2 arg = ffma2(L1, L1, ffma2(L2, L2, eps2));
  const float2 inv_d = rsq2(arg);
  const float2 d = mul2(arg, inv_d);
  if (WANT_SR || WANT_HR) {
    const float2 q1 = mul2(mul2(L1, inv_d), rcp2(l1)), q2 = mul2(mul2(L2, inv_d), rcp2(l2));
    // clamp sub-gradients (pass where raw >= 1); x*0 keeps NaN like torch
    const float2 dl1 = make_float2((l1r.x >= 1.0f) ? q1.x : l1r.x * 0.0f, (l1r.y >= 1.0f) ? q1.y : l1r.y * 0.0f);
    const float2 dl2 = make_float2((l2r.x >= 1.0f) ? q2.x : l2r.x * 0.0f, (l2r.y >= 1.0f) ? q2.y : l2r.y * 0.0f);
    const float2 dsum = add2(dl1, dl2);            // 2 dT
    const float2 wq = mul2(ffma2(dl1, m1, dl2), ir);  // 4 ddisc
    const float2 w = make_float2((disc_raw.x >= eps) ? wq.x : disc_raw.x * 0.0f,
                                 (disc_raw.y >= eps) ? wq.y : disc_raw.y * 0.0f);
    const float2 dTr = mul2(mul2(s, half), dsum);
    const float2 dd2 = mul2(mul2(ss, half), w);    // 2 ddisc'
    const float2 dambr = mul2(ambr, dd2);
    const float2 dd4 = add2(dd2, dd2);
    const float2 dCr = mul2(Dr, dd4), dDr = mul2(Cr, dd4);
    const float2 dAr = add2(dTr, dambr), dBr = ffma2(dambr, m1, dTr);
    const float2 dAB = add2(dTr, dTr);             // dA' + dB'
    float2 Qn = make_float2(0.f, 0.f);             // -Q/2 = -(T dsum + disc w) / 4
    if (normalize) Qn = mul2(ffma2(T, dsum, mul2(disc_raw, w)), bcast2(-0.25f));
    if (WANT_SR) {
      float2 da = ffma2(dBr, f, mul2(dDr, h));
      float2 db = ffma2(dAr, e, mul2(dCr, h));
      float2 dc = mul2(ffma2(dAB, h, ffma2(dCr, f, mul2(dDr, e))), m1);
      if (normalize) {
        const float2 dp = mul2(Qn, mul2(s1, s1));  // d / d(det S1)
        da = ffma2(dp, b, da);
        db = ffma2(dp, a, db);
        dc = ffma2(add2(dp, dp), nc, dc);
      }
      G.da = da; G.db = db; G.dc = dc;
    }
    if (WANT_HR) {
      float2 de = ffma2(dAr, b, mul2(dDr, nc));
      float2 df = ffma2(dBr, a, mul2(dCr, nc));
      float2 dh = ffma2(dAB, nc, ffma2(dCr, b, mul2(dDr, a)));
      if (normalize) {
        const float2 dp = mul2(Qn, mul2(s2, s2));
        de = ffma2(dp, f, de);
        df = ffma2(dp, e, df);
        dh = ffma2(add2(dp, dp), nh, dh);
      }
      G.de = de; G.df = df; G.dh = dh;
    }
  }
  return d;
}

// PER_IMG: reduction='none' -- loss_out[b] is the mean over image b's pixels (P.inv_count = 1 / (H W)) instead of
// loss_out[0] over the batch; with PX, loss_out[B + b] is image b's mean squared difference over its 3 H W values.
// MAP: also stores every pixel's distance into MP.map_out [B,H,W] (the loss and the other outputs are unchanged).
template <class C, bool PX = false, bool WANT_HR = false, bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(C::NT, C::MINB)
st_forward_march_kernel(const __grid_constant__ StMarchParamsT<C::RG, C::RK, MAP> MP) {
  static_assert(!(MAP && (PX || PER_IMG)), "the distance map comes with the batch loss only");
  static_assert(!C::XFULL || C::xitem_conflict_free(), "march crop layout: a quarter-warp's 16-byte accesses share a bank group");
  SRST_DYN_SMEM(float, smem);
  __shared__ float s_red[32];
  __shared__ unsigned int s_last;
  [[maybe_unused]] __shared__ float s_red_px[PX ? 32 : 1];
  __shared__ __align__(8) unsigned long long s_mbar;
  const auto& P = MP.F;
  const auto& tp = P.taps;
  constexpr int RG = C::RG, RK = C::RK, NQ = C::NQ;

  float* sRaw = smem;                 // [2 images][3][16][GW]   TMA destination
  float* sGray = smem + C::GRAY_OFF;  // [block parity][2 images][GP row pairs][PG]   row-pair interleaved
  float* sD = smem + C::D_OFF;        // [2][Ix|Iy][8][PD]
  float* sH = smem + C::H_OFF;        // [2][3][16 ring row pairs][PH]

  const int tid = threadIdx.x;
  const bool producer = tid < C::NP;
  int t = blockIdx.x;
  const int strip = t % MP.nstrips;
  t /= MP.nstrips;
  const int chunk = t % MP.nchunks;
  const int b = t / MP.nchunks;
  const int H = P.H, W = P.W;
  const int x0 = strip * C::TW;
  const int y0 = chunk * MP.chunk_blocks * C::RS;
  const int y1 = min(H, y0 + MP.chunk_blocks * C::RS);
  const int NB = (y1 - y0 + C::RS - 1) / C::RS;  // output blocks; H blocks 0..NB
  const size_t plane = (size_t)H * W;
  const size_t img_off = (size_t)b * 3 * plane;
  const bool norm = P.normalize != 0;

  MSTAMP(tid == 0, 0);
  if (tid == 0) tma_barrier_init(&s_mbar);
  pdl_wait();     // previous kernel of the stream is complete (it may have produced sr or used the workspace)
  pdl_trigger();
  __syncthreads();  // the barrier is initialised before anyone polls it

  // first image row of H block k
  auto hb = [&](int k) { return y0 - RK + C::RS * k; };
  // raw rows of block k = the 16 NEW gray rows its gradients need: hb(k) + RG ..  (blocks 1.. only: block 0 is
  // loaded directly while the first box is in flight)
  auto issue_raw = [&](int k) {
    tma_expect(&s_mbar, (unsigned)(2 * C::RAW_IMG * sizeof(float)));
    tma_load_3d(&s_mbar, sRaw, &MP.sr_map, x0 + C::BX, hb(k) + RG, b * 3, C::BW, C::RS, 3);
    tma_load_3d(&s_mbar, sRaw + C::RAW_IMG, &MP.hr_map, x0 + C::BX, hb(k) + RG, b * 3, C::BW, C::RS, 3);
  };
  [[maybe_unused]] float pxsum = 0.f;
  // raw box of block k -> gray row pairs RG .. RG+7 of gray buffer k&1; item = image x row pair x 4 columns
  auto convert = [&](int k) {
    constexpr int C4 = C::BW / 4;
    float* gbuf = sGray + (k & 1) * 2 * C::GRAY_IMG;
    for (int it = tid; it < 2 * NQ * C4; it += C::NP) {
      const int c4 = it % C4, rr = it / C4;
      const int q = rr % NQ, img = rr / NQ;
      const float* r0 = sRaw + img * C::RAW_IMG + (2 * q) * C::BW + 4 * c4;
      const float4 R0 = ld4(r0), G0 = ld4(r0 + C::RS * C::BW), B0 = ld4(r0 + 2 * C::RS * C::BW);
      const float4 R1 = ld4(r0 + C::BW), G1 = ld4(r0 + C::BW + C::RS * C::BW), B1 = ld4(r0 + C::BW + 2 * C::RS * C::BW);
      float* o = gbuf + img * C::GRAY_IMG + (RG + q) * C::PG + 8 * c4 + 2 * (C::GXH + C::BX);
      st4(o, make_float4(gray_of(R0.x, G0.x, B0.x), gray_of(R1.x, G1.x, B1.x), gray_of(R0.y, G0.y, B0.y),
                         gray_of(R1.y, G1.y, B1.y)));
      st4(o + 4, make_float4(gray_of(R0.z, G0.z, B0.z), gray_of(R1.z, G1.z, B1.z), gray_of(R0.w, G0.w, B0.w),
                             gray_of(R1.w, G1.w, B1.w)));
    }
    if constexpr (PX) {
      // fused Pixel term: squared RGB difference over the rows of this raw block that belong to the chunk
      constexpr int C2 = C::TW / 2;
      const int ry0 = hb(k) + RG;
      for (int it = tid; it < C::RS * C2; it += C::NP) {
        const int c2 = it % C2, r = it / C2;
        const int gy = ry0 + r, gx = x0 + 2 * c2;
        if (gy < y0 || gy >= y1 || gx >= W) continue;
        const float* ps = sRaw + r * C::BW - C::BX + 2 * c2;
        float acc = 0.f;
#pragma unroll
        for (int ch = 0; ch < 3; ++ch) {
          const float2 u = ld2(ps + ch * C::RS * C::BW), v = ld2(ps + C::RAW_IMG + ch * C::RS * C::BW);
          const float d0 = u.x - v.x, d1 = u.y - v.y;
          acc = fmaf(d0, d0, acc);
          acc = fmaf(d1, d1, acc);
        }
        pxsum += acc;
      }
    }
  };

  if (tid == 0) {
    issue_raw(1);  // H blocks 0..NB, NB >= 1: block 1 always exists
  }
  {
    // Block 0 (its RG carried row pairs and its 8 new ones: image rows hb(0) - RG .. hb(0) + RG + 15) comes straight
    // from global memory while the box of block 1 is in flight; item = row pair x 4 columns of BOTH images, spread
    // over ALL threads of the CTA (the consumers have nothing else to do yet).
    constexpr int C4 = C::BW / 4;
    for (int it = tid; it < C::GP * C4; it += C::NT) {
      const int c4 = it % C4, pr = it / C4;
      const int gx = x0 + C::BX + 4 * c4;
      const bool xin = gx >= 0 && gx < W;  // x0 + BX and W are multiples of 4: a float4 is all-in or all-out
      float4 v[2][2][3];                   // [image][row of the pair][channel]
      bool ok[2];
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const int gy = hb(0) - RG + 2 * pr + hf;
        ok[hf] = xin && gy >= 0 && gy < H;
        if (ok[hf]) {
          const size_t o = img_off + (size_t)gy * W + gx;
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) { v[0][hf][ch] = ldg4(P.sr + o + ch * plane); v[1][hf][ch] = ldg4(P.hr + o + ch * plane); }
        } else {
#pragma unroll
          for (int ch = 0; ch < 3; ++ch) { v[0][hf][ch] = make_float4(0.f, 0.f, 0.f, 0.f); v[1][hf][ch] = make_float4(0.f, 0.f, 0.f, 0.f); }
        }
      }
#pragma unroll
      for (int img = 0; img < 2; ++img) {
        const float4 *a0 = v[img][0], *a1 = v[img][1];
        float* o = sGray + img * C::GRAY_IMG + pr * C::PG + 8 * c4 + 2 * (C::GXH + C::BX);
        st4(o, make_float4(gray_of(a0[0].x, a0[1].x, a0[2].x), gray_of(a1[0].x, a1[1].x, a1[2].x),
                           gray_of(a0[0].y, a0[1].y, a0[2].y), gray_of(a1[0].y, a1[1].y, a1[2].y)));
        st4(o + 4, make_float4(gray_of(a0[0].z, a0[1].z, a0[2].z), gray_of(a1[0].z, a1[1].z, a1[2].z),
                               gray_of(a0[0].w, a0[1].w, a0[2].w), gray_of(a1[0].w, a1[1].w, a1[2].w)));
        if (pr >= NQ) {  // the last RG row pairs of block 0 are the first RG of block 1 (the other gray buffer)
          float* o1 = o + 2 * C::GRAY_IMG - NQ * C::PG;
          st4(o1, ld4(o));
          st4(o1 + 4, ld4(o + 4));
        }
      }
      if constexpr (PX) {
        if (gx >= x0 && gx < x0 + C::TW) {
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            const int gy = hb(0) - RG + 2 * pr + hf;
            if (!ok[hf] || gy < y0 || gy >= y1) continue;
            float acc = 0.f;
#pragma unroll
            for (int ch = 0; ch < 3; ++ch) {
              const float4 u = v[0][hf][ch], w = v[1][hf][ch];
              const float d0 = u.x - w.x, d1 = u.y - w.y, d2 = u.z - w.z, d3 = u.w - w.w;
              acc = fmaf(d0, d0, acc); acc = fmaf(d1, d1, acc); acc = fmaf(d2, d2, acc); acc = fmaf(d3, d3, acc);
            }
            pxsum += acc;
          }
        }
      }
    }
    if constexpr (C::XFULL) {
      // the zero columns of the edge windows, which nothing else writes: gray columns -GXH .. -1 and TW .. TW+GXH-1
      // of every gray row pair (both buffers, both images), Ix / Iy columns -RK .. -1 and TW .. TW+RK-1
      constexpr int GZ = C::GXH / 2, DZ = RK / 2;  // float4 per row pair and side
      constexpr int NG = 4 * C::GP * 2 * GZ, ND = 4 * NQ * 2 * DZ;
      for (int it = tid; it < NG + ND; it += C::NT) {
        float* o;
        if (it < NG) {
          const int r = it / (2 * GZ), u = it % (2 * GZ);
          o = sGray + r * C::PG + (u < GZ ? 4 * u : 2 * (C::GXH + C::TW) + 4 * (u - GZ));
        } else {
          const int r = (it - NG) / (2 * DZ), u = (it - NG) % (2 * DZ);
          o = sD + r * C::PD + (u < DZ ? 4 * u : 2 * (RK + C::TW) + 4 * (u - DZ));
        }
        st4(o, make_float4(0.f, 0.f, 0.f, 0.f));
      }
    }
  }
  __syncthreads();

  // consumer state: the smoothed tensors of this thread's column, 4 row pairs, both images
  const int ct = tid - C::NP;
  const int chalf = producer ? 0 : ct / C::TW, ccol = producer ? 0 : ct % C::TW;
  float2 S1[3][C::CQ], S2[3][C::CQ];
  float lsum = 0.f;
  const int Hp = (H + 1) >> 1;

  // Named barriers (0 is __syncthreads): kBarP among the producers; kBarH "ring block complete" (producers arrive,
  // consumers wait); kBarV "ring slot free" (consumers arrive, producers wait).  The two groups are coupled by these
  // hand-shakes only, so the latency-bound chain of the consumers overlaps whatever the producers are doing.
  constexpr int kBarP = 1, kBarH = 2, kBarV = 3;
  MSTAMP(tid == 0, 1);        // prologue done
  MSTAMP(tid == C::NP, 1);
  if (producer) {
#pragma unroll 1
    for (int k = 0; k <= NB; ++k) {
      {
        // gradients of block k: Ix, Iy on 8 row pairs x DW columns of both images; zero outside the image (the
        // reference zero-pads the PRODUCTS, utils.py:225-230); strip-interior items save them for the backward.
        // Crop layout: the image columns only (segments 1 .. NSEGH of the DW columns), on the first NH producers.
        if (!C::XFULL || tid < C::NH) {
        int q, seg, img;
        if constexpr (C::XFULL) {
          C::xitem(tid, q, img, seg);
          seg += RK / 8;
        } else {
          q = tid & 7;
          const int rest = tid >> 3;
          seg = rest % C::NSEGB;
          img = rest / C::NSEGB;
        }
        const int gy = hb(k) + 2 * q, gx0 = x0 - RK + 8 * seg;
        float2 Ix[8], Iy[8];
        if (gy + 1 >= 0 && gy < H && gx0 + 7 >= 0 && gx0 < W && MARCH_ON(3)) {
          const float* p = sGray + ((k & 1) * 2 + img) * C::GRAY_IMG + q * C::PG + 2 * (8 * seg + C::GOFF);
          grad_rowpair<RG, 8, C::BWIN, RG, C::PG, true>(p, p, tp, Ix, Iy);
          if (!(gy >= 0 && gy + 1 < H && gx0 >= 0 && gx0 + 8 <= W)) {  // straddles the image border: mask
            const bool r0 = gy >= 0, r1 = gy + 1 < H;
#pragma unroll
            for (int j = 0; j < 8; ++j) {
              const bool ok = (gx0 + j >= 0) && (gx0 + j < W);
              Ix[j].x = (ok && r0) ? Ix[j].x : 0.f;
              Ix[j].y = (ok && r1) ? Ix[j].y : 0.f;
              Iy[j].x = (ok && r0) ? Iy[j].x : 0.f;
              Iy[j].y = (ok && r1) ? Iy[j].y : 0.f;
            }
          }
        } else {
#pragma unroll
          for (int j = 0; j < 8; ++j) { Ix[j] = make_float2(0.f, 0.f); Iy[j] = make_float2(0.f, 0.f); }
        }
        float* o0 = sD + (img * 2) * C::D_PLANE + q * C::PD + 2 * (8 * seg);
        float* o1 = o0 + C::D_PLANE;
#pragma unroll
        for (int j = 0; j < 8; j += 2) {
          st4(o0 + 2 * j, make_float4(Ix[j].x, Ix[j].y, Ix[j + 1].x, Ix[j + 1].y));
          st4(o1 + 2 * j, make_float4(Iy[j].x, Iy[j].y, Iy[j + 1].x, Iy[j + 1].y));
        }
        }
        MSTAMP(tid == 0, 2 + 6 * k);  // gradients done
        // gray rows of block k+1 into the other gray buffer (its box was requested one half-step ago)
        if (k + 1 <= NB) {
          if (MARCH_ON(7)) tma_wait(&s_mbar, (unsigned)(k & 1));  // box of block k+1 is the k-th use of the barrier
          MSTAMP(tid == 0, 3 + 6 * k);  // box arrived
          if (MARCH_ON(4)) convert(k + 1);
          MSTAMP(tid == 0, 4 + 6 * k);  // converted
        }
      }
      bar_sync(kBarP, C::NP);  // Ix, Iy of block k and the gray rows of block k+1 are complete; the raw box is free
      MSTAMP(tid == 0, 5 + 6 * k);
      if (k >= 1) bar_sync(kBarV, C::NT);  // k == 1: the consumers have seen block 0; k >= 2: they are done with block k-2
      MSTAMP(tid == 0, 6 + 6 * k);
      {
        if (tid >= C::NH) {
          // The producers beyond the horizontal items (one warp: the x halo of the gradient items) do the copies.
          // Every producer is done with the raw box (block k+1 was converted in Y_k): request block k+2.
          const int lane = tid - C::NH;
          constexpr int NL = C::NP - C::NH;
          if (lane == 0 && k + 2 <= NB) {
            fence_async_smem();
            issue_raw(k + 2);
          }
          // the last RG gray row pairs of block k+1 are the first RG of block k+2 (gray buffer k&1 again)
          if (k + 2 <= NB) {
            const float* src = sGray + ((k + 1) & 1) * 2 * C::GRAY_IMG + NQ * C::PG + 4 * lane;
            float* dst = sGray + (k & 1) * 2 * C::GRAY_IMG + 4 * lane;
            constexpr int N4 = RG * (C::PG / 4), NIT = (N4 + NL - 1) / NL;  // RG consecutive row pairs = one contiguous run
            float4 v[2][NIT];
#pragma unroll
            for (int img = 0; img < 2; ++img)
#pragma unroll
              for (int i = 0; i < NIT; ++i)
                if (lane + i * NL < N4) v[img][i] = ld4(src + img * C::GRAY_IMG + 4 * NL * i);
#pragma unroll
            for (int img = 0; img < 2; ++img)
#pragma unroll
              for (int i = 0; i < NIT; ++i)
                if (lane + i * NL < N4) st4(dst + img * C::GRAY_IMG + 4 * NL * i, v[img][i]);
          }
          // save Ix, Iy of block k for the backward: the strip-interior columns of the D rows that belong to this
          // chunk, copied out with fully coalesced 16-byte stores (a row pair of a plane is 2*TW contiguous floats);
          // four row pairs are loaded before they are stored so that the copy is not one long LDS -> STG chain
          if (MARCH_ON(6)) {
            constexpr int E4 = C::TW / 2;  // float4 per row pair
            const int n4 = min(E4, (W - x0) / 2);
            const bool c0 = lane < n4, c1 = lane + NL < n4;
            const size_t rstride = 2 * (size_t)W, pstride = (size_t)Hp * rstride;
            const int gp0 = hb(k) >> 1;  // first row pair of the block (hb(k) is even; negative above the image)
#pragma unroll
            for (int img = 0; img < (WANT_HR ? 2 : 1); ++img) {
              float* ixy = img ? P.ixy_hr : P.ixy_sr;
              if (!ixy) continue;
              float* g0 = ixy + (size_t)b * 2 * pstride + 2 * (size_t)x0 + 4 * lane;
#pragma unroll
              for (int pl = 0; pl < 2; ++pl) {
#pragma unroll
                for (int qb = 0; qb < NQ; qb += 4) {
                  float4 va[4], vb[4];
#pragma unroll
                  for (int u = 0; u < 4; ++u) {
                    const float* so = sD + (img * 2 + pl) * C::D_PLANE + (qb + u) * C::PD + 2 * RK + 4 * lane;
                    va[u] = ld4(so);
                    if (E4 > NL) vb[u] = c1 ? ld4(so + 4 * NL) : make_float4(0.f, 0.f, 0.f, 0.f);
                  }
#pragma unroll
                  for (int u = 0; u < 4; ++u) {
                    const int gy = hb(k) + 2 * (qb + u);
                    if (gy >= y0 && gy < y1) {
                      float* go = g0 + pl * pstride + (size_t)(gp0 + qb + u) * rstride;
                      if (c0) st4(go, va[u]);
                      if (E4 > NL && c1) st4(go + 4 * NL, vb[u]);
                    }
                  }
                }
              }
            }
          }
        }
        // products + horizontal rho-pass of block k -> ring row pairs 8*(k&1) ..; item = image x row pair x 8 columns.
        // Scatter form: window column j contributes k[j - o] to output column o, so Ix, Iy are read once.
        if (tid < C::NH && MARCH_ON(2)) {
          int q, seg, img;
          if constexpr (C::XFULL) {
            C::xitem(tid, q, img, seg);
          } else {
            q = tid & 7;
            const int rest = tid >> 3;
            seg = rest % C::NSEGH;
            img = rest / C::NSEGH;
          }
          const float* pix = sD + (img * 2) * C::D_PLANE + q * C::PD + 2 * (8 * seg);
          const float* piy = pix + C::D_PLANE;
          float2 acc[3][8];
#pragma unroll
          for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int o = 0; o < 8; ++o) acc[c][o] = make_float2(0.f, 0.f);
          const int gyh = hb(k) + 2 * q;
          if (gyh + 1 >= 0 && gyh < H) {  // a row pair outside the image holds Ix = Iy = 0: its smoothed products are zeros
#pragma unroll
          for (int m = 0; m < C::HWIN / 2; ++m) {
            const float4 xv = ld4(pix + 4 * m), yv = ld4(piy + 4 * m);
#pragma unroll
            for (int hcol = 0; hcol < 2; ++hcol) {
              const int j = 2 * m + hcol;
              const float2 ix = hcol ? make_float2(xv.z, xv.w) : make_float2(xv.x, xv.y);
              const float2 iy = hcol ? make_float2(yv.z, yv.w) : make_float2(yv.x, yv.y);
              const float2 pxx = mul2(ix, ix), pyy = mul2(iy, iy), pxy = mul2(ix, iy);
#pragma unroll
              for (int o = 0; o < 8; ++o) {
                const int tap = j - o;
                if (tap >= 0 && tap <= 2 * RK) {
                  acc[0][o] = ffma2(pxx, bcast2(tp.k[tap]), acc[0][o]);
                  acc[1][o] = ffma2(pyy, bcast2(tp.k[tap]), acc[1][o]);
                  acc[2][o] = ffma2(pxy, bcast2(tp.k[tap]), acc[2][o]);
                }
              }
            }
          }
          }
          float* o = sH + (img * 3) * C::H_PLANE + (8 * (k & 1) + q) * C::PH + 2 * (8 * seg);
#pragma unroll
          for (int c = 0; c < 3; ++c)
#pragma unroll
            for (int jj = 0; jj < 8; jj += 2)
              st4(o + c * C::H_PLANE + 2 * jj, make_float4(acc[c][jj].x, acc[c][jj].y, acc[c][jj + 1].x, acc[c][jj + 1].y));
        }
      }
      MSTAMP(tid == 0, 7 + 6 * k);  // horizontal pass done
      __threadfence_block();
      bar_arrive(kBarH, C::NT);  // ring block k is complete
      bar_sync(kBarP, C::NP);    // every producer is done with Ix, Iy of block k; the carried gray rows are in place
    }
  } else {
    bar_sync(kBarH, C::NT);    // ring block 0
    bar_arrive(kBarV, C::NT);
#pragma unroll 1
    for (int jb = 0; jb < NB; ++jb) {
      const int k = jb + 2;
      bar_sync(kBarH, C::NT);  // ring block jb+1
      MSTAMP(tid == C::NP, 2 + 3 * jb);  // block available
      if (MARCH_ON(1)) {
      // vertical rho-pass of output block j = k-2 from ring blocks j, j+1: this thread's column, output row
      // pairs 4*chalf .. +3, input ring row pairs 4*chalf .. 4*chalf + NIN - 1 (relative to block j)
      const int j = k - 2;
      const int rp0 = 8 * (j & 1) + C::CQ * chalf;
#pragma unroll
      for (int img = 0; img < 2; ++img) {
        float2 acc[3][C::CQ];
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int o = 0; o < C::CQ; ++o) acc[c][o] = make_float2(0.f, 0.f);
        const float* base = sH + (img * 3) * C::H_PLANE + 2 * ccol;
#pragma unroll
        for (int i = 0; i < C::NIN; ++i) {
          const float* p = base + ((rp0 + i) & 15) * C::PH;
          const float2 v0 = ld2(p), v1 = ld2(p + C::H_PLANE), v2 = ld2(p + 2 * C::H_PLANE);
#pragma unroll
          for (int o = 0; o < C::CQ; ++o) {
            const int u0 = 2 * (i - o);  // tap-pair index of the even input row for output pair o
            if (u0 >= 0 && u0 <= 2 * RK + 1) {
              acc[0][o] = ffma2(bcast2(v0.x), tp.kp[u0], acc[0][o]);
              acc[1][o] = ffma2(bcast2(v1.x), tp.kp[u0], acc[1][o]);
              acc[2][o] = ffma2(bcast2(v2.x), tp.kp[u0], acc[2][o]);
            }
            if (u0 + 1 >= 0 && u0 + 1 <= 2 * RK + 1) {
              acc[0][o] = ffma2(bcast2(v0.y), tp.kp[u0 + 1], acc[0][o]);
              acc[1][o] = ffma2(bcast2(v1.y), tp.kp[u0 + 1], acc[1][o]);
              acc[2][o] = ffma2(bcast2(v2.y), tp.kp[u0 + 1], acc[2][o]);
            }
          }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c)
#pragma unroll
          for (int o = 0; o < C::CQ; ++o) {
            if (img == 0) S1[c][o] = acc[c][o];
            else S2[c][o] = acc[c][o];
          }
      }
      }
      MSTAMP(tid == C::NP, 3 + 3 * jb);  // vertical pass done
      if (jb + 2 <= NB) bar_arrive(kBarV, C::NT);  // ring slot jb&1 may be overwritten (block jb+2)
      if (MARCH_ON(0)) {
      // per-pixel chain + stores of output block j: rows y0 + 16j + 8*chalf + 2o (+1), column x0 + ccol
      const int j = k - 2;
      const int gx = x0 + ccol;
      const int ry = y0 + C::RS * j + C::CR * chalf;
      if (gx < W) {
        float* ps = P.ds_sr ? P.ds_sr + img_off + (size_t)ry * W + gx : nullptr;
        [[maybe_unused]] float* ph = WANT_HR ? P.ds_hr + img_off + (size_t)ry * W + gx : nullptr;
        [[maybe_unused]] float* pm = nullptr;
        if constexpr (MAP) pm = MP.map_out + (size_t)b * plane + (size_t)ry * W + gx;
        // all four pixel pairs are evaluated unconditionally (rows past the chunk hold finite filler) so that the
        // compiler can interleave their SFU / FMA dependency chains; only the loss and the stores are masked
#pragma unroll
        for (int o = 0; o < C::CQ; ++o) {
          const int gy = ry + 2 * o;
          StPixelGrad2 G;
          G.da = G.db = G.dc = G.de = G.df = G.dh = make_float2(0.f, 0.f);
          const float2 d = st_pixel2_raw<true, WANT_HR>(S1[0][o], S1[1][o], S1[2][o], S2[0][o], S2[1][o], S2[2][o], norm,
                                                        P.eps, G);
          const bool one = gy < y1, two = gy + 1 < y1;
          lsum += one ? d.x : 0.f;
          lsum += two ? d.y : 0.f;
          if (ps && MARCH_ON(5)) {
            if (one) { ps[0] = G.da.x; ps[plane] = G.db.x; ps[2 * plane] = G.dc.x; }
            if (two) { ps[W] = G.da.y; ps[plane + W] = G.db.y; ps[2 * plane + W] = G.dc.y; }
            ps += 2 * W;
          }
          if constexpr (WANT_HR) {
            if (one) { ph[0] = G.de.x; ph[plane] = G.df.x; ph[2 * plane] = G.dh.x; }
            if (two) { ph[W] = G.de.y; ph[plane + W] = G.df.y; ph[2 * plane + W] = G.dh.y; }
            ph += 2 * W;
          }
          if constexpr (MAP) {
            if (one) pm[0] = d.x;
            if (two) pm[W] = d.y;
            pm += 2 * W;
          }
        }
      }
      }
    }
  }

  MSTAMP(tid == C::NP, 4 + 3 * (NB - 1));  // last chain done
  // Deterministic loss reduction: block partial -> workspace; the last block to finish sums all
  // partials in a fixed order (double) and re-zeroes the workspace for the next call.
  lsum = warp_sum(lsum);
  if constexpr (PX) pxsum = warp_sum(pxsum);
  if ((tid & 31) == 0) {
    s_red[tid >> 5] = lsum;
    if constexpr (PX) s_red_px[tid >> 5] = pxsum;
  }
  __syncthreads();
  if (tid == 0) {
    float bs = 0.f;
    for (int w = 0; w < C::NT / 32; ++w) bs += s_red[w];
    P.partials[blockIdx.x] = bs;
    if constexpr (PX) {
      float bp = 0.f;
      for (int w = 0; w < C::NT / 32; ++w) bp += s_red_px[w];
      P.px_partials[blockIdx.x] = bp;
    }
    __threadfence();
    const unsigned int tk = atomicAdd(P.ticket, 1u);
    s_last = (tk == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if constexpr (PER_IMG) {
    if (s_last) {  // image-major grid: image b owns nchunks * nstrips consecutive CTAs
      __threadfence();
      reduce_partials_per_image(P.partials, P.B, gridDim.x / P.B, (double)P.inv_count, P.loss_out);
      if constexpr (PX)
        reduce_partials_per_image(P.px_partials, P.B, gridDim.x / P.B, (double)P.inv_count / 3.0, P.loss_out + P.B);
      if (tid == 0) *P.ticket = 0u;
    }
  } else if (s_last) {
    __threadfence();
    if (tid < 32) {
      double acc = 0.0;
      [[maybe_unused]] double accp = 0.0;
      for (unsigned int i = tid; i < gridDim.x; i += 32) {
        acc += (double)__ldcg(P.partials + i);
        P.partials[i] = 0.f;
        if constexpr (PX) {
          accp += (double)__ldcg(P.px_partials + i);
          P.px_partials[i] = 0.f;
        }
      }
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) {
        acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if constexpr (PX) accp += __shfl_xor_sync(0xffffffffu, accp, o);
      }
      if (tid == 0) {
        P.loss_out[0] = (float)(acc * (double)P.inv_count);
        if constexpr (PX) P.loss_out[1] = (float)(accp * (double)P.inv_count / 3.0);
        *P.ticket = 0u;
      }
    }
  }
}

}  // namespace srst
