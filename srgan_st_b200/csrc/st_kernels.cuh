// Fused structure-tensor loss kernels for sm_100a (forward and backward).
//
// What the reference does with ~100 ATen launches per direction (loss.py:399-413,
// utils.py:212-279) is done here by ONE kernel per direction:
//
//   st_forward_kernel : RGB tile (+halo) of SR and HR -> grayscale -> Gaussian-derivative
//                       gradients Ix, Iy -> products -> separable rho-smoothing -> per-pixel
//                       det-normalise, adj(S1)*S2, eigenvalues, log-distance  -> block partial of
//                       the loss, the per-pixel d(distance)/d(Jxx,Jyy,Jxy) ("ds" planes) AND the
//                       gradient planes Ix, Iy ("ixy", row-pair interleaved) the backward re-uses.
//   st_backward_kernel: ds planes + saved Ix, Iy (two TMA box copies) -> adjoint rho-smoothing ->
//                       product rule -> adjoint derivative filters -> grayscale weights -> d_img.
//
// Both are FP32 CUDA-core stencils (no tensor cores by design: see DESIGN.md).  The measured
// bound on B200 is the FP32 pipe (128 lane-FMA/clk/SM, tools/ubench_fma.cu), not HBM, so the
// design minimises issue slots per FMA:
//   * every shared-memory plane is stored ROW-PAIR INTERLEAVED: element (row r, col c) lives at
//     (r/2)*pitch + 2*c + (r&1), so a float2 holds one column of two adjacent rows;
//   * every filter pass works on such row pairs with packed fma.rn.f32x2 (SASS FFMA2): horizontal
//     passes multiply a register pair by one tap broadcast from the constant bank, vertical passes
//     multiply one value (broadcast) by the tap PAIR (k[t], k[t-1]) that maps it onto the two
//     output rows.  Both operand forms are native (FFMA2 Rd, Ra.F32, URb.F32x2, Rc), so a 17-tap
//     pass costs 17 issue slots per pixel pair and no register moves;
//   * horizontal passes are register-blocked (4 or 8 columns x 2 rows per thread, LDS.128 on a pitch
//     == 4 mod 8, lanes grouped so that every quarter-warp hits eight distinct 16-byte bank groups:
//     ItemMap), vertical passes own one column and RS rows (conflict-free LDS.64/STS.64);
//   * taps live in kernel parameters and every tap index is a compile-time constant;
//   * the forward runs the SR and the HR image through ONE copy of the filter code (a rolled loop)
//     and parks each image's smoothed tensor in a thread-private shared-memory slot, so the
//     per-pixel chain starts with an empty register file (no spills) and is itself a rolled loop.
#pragma once
#include <type_traits>

#include "srst_device.cuh"

namespace srst {

template <int RG, int RK>
struct StTaps {
  float g[2 * RG + 1];    // Gaussian(sigma), utils.py:194-205
  float dg[2 * RG + 1];   // its derivative taps, utils.py:206
  float k[2 * RK + 1];    // Gaussian(rho)
  // tap pairs (t[u], t[u-1]) with zeros outside the support: input row u of a row pair's window
  // contributes t[u] to the even output row and t[u-1] to the odd one.
  float2 gp[2 * RG + 2];
  float2 dgp[2 * RG + 2];
  float2 kp[2 * RK + 2];
};

// Saved gradient planes ("ixy"): [B][2][ceil(H/2)][W][2] fp32 -- plane 0 = Ix, plane 1 = Iy, each stored
// row-pair interleaved exactly like the shared-memory planes (rows 2p and 2p+1 of column c are the
// two floats at ((b*2+plane)*Hp + p)*2W + 2c), so that the backward fetches its tile with one TMA box.
SRST_DEV size_t ixy_offset(int b, int plane, int Hp, int W, int rowpair, int col) {
  return (((size_t)b * 2 + plane) * Hp + rowpair) * (size_t)(2 * W) + 2 * (size_t)col;
}

template <int RG, int RK>
struct StFwdParams {
  const float* sr;
  const float* hr;
  float* ds_sr;   // [B,3,H,W] or null
  float* ds_hr;   // [B,3,H,W] or null
  float* ixy_sr;  // saved gradient planes of SR (see ixy_offset) or null
  float* ixy_hr;
  float* partials;
  float* px_partials;  // null, or per-CTA partials of sum (sr-hr)^2: the fused "Pixel" MSE term (warmup.py:88-96)
  unsigned int* ticket;
  float* loss_out;     // [0] = ST loss; [1] = MSE when px_partials is set
  int B, H, W, tiles_x, tiles_y;
  int normalize;
  int vec4;  // 1: W % 4 == 0 and all base pointers 16-byte aligned
  float eps;
  float inv_count;
  StTaps<RG, RK> taps;
};

// MAP forward (srst_st_forward_map): the distance of every pixel also goes to map_out [B,H,W].  A derived type, so
// that the parameter layout of the other instantiations stays as it is.
template <int RG, int RK>
struct StFwdMapParams : StFwdParams<RG, RK> {
  float* map_out;
};
template <int RG, int RK, bool MAP>
using StFwdParamsT = std::conditional_t<MAP, StFwdMapParams<RG, RK>, StFwdParams<RG, RK>>;

template <int RG, int RK>
struct StBwdParams {
  SrstTmap ds_map;   // tensor map of ds viewed as [B*3][H][W]            (valid when use_tma)
  SrstTmap ixy_map;  // tensor map of ixy viewed as [B*2][ceil(H/2)][2W]  (valid when use_tma)
  const float* ds;
  const float* ixy;
  const float* grad_out;
  const float* img;       // fused Pixel term only: the image d_img belongs to ...
  const float* px_other;  // ... and the other image of the pair: adds grad_px * 2 (img - other) / (3 B H W) to d_img
  const float* grad_px;   // upstream gradient of the MSE term (device scalar)
  float* d_img;
  int B, H, W, tiles_x, tiles_y;
  int vec4;
  int use_tma;
  float inv_count;
  StTaps<RG, RK> taps;
};


SRST_DEV float2 ffma2(float2 a, float2 b, float2 c) { return __ffma2_rn(a, b, c); }
SRST_DEV float2 bcast2(float v) { return make_float2(v, v); }
SRST_DEV float2 ld2(const float* p) { return *reinterpret_cast<const float2*>(p); }
SRST_DEV void st2(float* p, float2 v) { *reinterpret_cast<float2*>(p) = v; }


// ------------------------------------------------------------------------------------------------
// Per-pixel chain: utils.py:236-279 forward and its adjoint.
//   S1 = (a,b,c) raw SR tensor (Jxx,Jyy,Jxy); S2 = (e,f,h) raw HR tensor.
// The discriminant is evaluated as (A-B)^2 + 4CD, algebraically equal to the reference's
// (A+B)^2 - 4(AB-CD) (utils.py:261) but without its catastrophic cancellation near A=B=1.
// NaN/clamp behaviour follows torch: clamp(min) keeps NaN; clamp gradient passes where x >= min.
// Transcendentals use the SFU (MUFU.RSQ/LG2/RCP): rsqrt of the two determinants gets one Newton
// step (they scale everything downstream); the rest stay at SFU accuracy (<= 2 ulp), far inside
// the 1e-5 / 1e-4 parity budget, at ~1/10 of the issue slots of sqrtf/logf/division.
// ------------------------------------------------------------------------------------------------
struct StPixelGrad {
  float da, db, dc;  // d dist / d (a,b,c)
  float de, df, dh;  // d dist / d (e,f,h)
};

SRST_DEV float rsqrt_nr(float x) {
  const float y = fast_rsqrt(x);
  return y * fmaf(-0.5f * x, y * y, 1.5f);  // one Newton step; NaN for x < 0 like 1/sqrt(x)
}

// Packed form of st_pixel: the same chain on TWO pixels at once (.x = even row, .y = odd row of a
// row pair), every add/mul/fma issued as FADD2/FMUL2/FFMA2; SFU ops and selects stay per lane.
struct StPixelGrad2 {
  float2 da, db, dc, de, df, dh;
};
SRST_DEV float2 mul2(float2 a, float2 b) { return __fmul2_rn(a, b); }
SRST_DEV float2 add2(float2 a, float2 b) { return __fadd2_rn(a, b); }
SRST_DEV float2 neg2(float2 a) { return make_float2(-a.x, -a.y); }
SRST_DEV float2 sub2(float2 a, float2 b) { return __fadd2_rn(a, neg2(b)); }
SRST_DEV float2 rsq2(float2 a) { return make_float2(fast_rsqrt(a.x), fast_rsqrt(a.y)); }
SRST_DEV float2 rcp2(float2 a) { return make_float2(fast_rcp(a.x), fast_rcp(a.y)); }
SRST_DEV float2 lg22(float2 a) { return make_float2(fast_lg2(a.x), fast_lg2(a.y)); }
SRST_DEV float2 rsqrt_nr2(float2 x) {
  const float2 y = rsq2(x);
  return mul2(y, ffma2(mul2(bcast2(-0.5f), x), mul2(y, y), bcast2(1.5f)));
}

template <bool WANT_SR, bool WANT_HR>
SRST_DEV float2 st_pixel2(float2 a, float2 b, float2 c, float2 e, float2 f, float2 h, bool normalize, float eps,
                          StPixelGrad2& G) {
  constexpr float kLn2 = 0.6931471805599453f;
  const float2 eps2 = bcast2(eps);
  float2 iq1 = bcast2(1.0f), iq2 = bcast2(1.0f);
  if (normalize) {
    iq1 = rsqrt_nr2(add2(ffma2(a, b, neg2(mul2(c, c))), eps2));
    iq2 = rsqrt_nr2(add2(ffma2(e, f, neg2(mul2(h, h))), eps2));
  }
  const float2 ah = mul2(a, iq1), bh = mul2(b, iq1), ch = mul2(c, iq1);
  const float2 eh = mul2(e, iq2), fh = mul2(f, iq2), hh = mul2(h, iq2);
  const float2 nchh = neg2(mul2(ch, hh));
  const float2 A = ffma2(bh, eh, nchh);
  const float2 Bm = ffma2(ah, fh, nchh);
  const float2 Cc = ffma2(bh, hh, neg2(mul2(ch, fh)));
  const float2 Dd = ffma2(ah, hh, neg2(mul2(ch, eh)));
  const float2 T = add2(A, Bm);
  const float2 amb = sub2(A, Bm);
  const float2 disc_raw = ffma2(amb, amb, mul2(bcast2(4.0f), mul2(Cc, Dd)));
  const float2 disc = make_float2((disc_raw.x < eps) ? eps : disc_raw.x, (disc_raw.y < eps) ? eps : disc_raw.y);
  const float2 ir = rsq2(disc);
  const float2 r = mul2(disc, ir);
  const float2 hT = mul2(bcast2(0.5f), T);
  const float2 l1r = ffma2(bcast2(-0.5f), r, hT), l2r = ffma2(bcast2(0.5f), r, hT);
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
    const float2 dr = mul2(bcast2(0.5f), sub2(dl2, dl1));
    const float2 dq = mul2(mul2(bcast2(0.5f), dr), ir);
    const float2 ddisc = make_float2((disc_raw.x >= eps) ? dq.x : disc_raw.x * 0.0f,
                                     (disc_raw.y >= eps) ? dq.y : disc_raw.y * 0.0f);
    const float2 dT = ffma2(mul2(bcast2(2.0f), T), ddisc, mul2(bcast2(0.5f), add2(dl1, dl2)));
    const float2 dd4 = mul2(bcast2(4.0f), ddisc);
    const float2 dA = ffma2(neg2(dd4), Bm, dT);
    const float2 dB = ffma2(neg2(dd4), A, dT);
    const float2 dC = mul2(dd4, Dd);
    const float2 dD = mul2(dd4, Cc);
    if (WANT_SR) {
      const float2 dah = ffma2(dB, fh, mul2(dD, hh));
      const float2 dbh = ffma2(dA, eh, mul2(dC, hh));
      const float2 dch = neg2(ffma2(add2(dA, dB), hh, ffma2(dC, fh, mul2(dD, eh))));
      if (normalize) {
        const float2 s = ffma2(a, dah, ffma2(b, dbh, mul2(c, dch)));
        const float2 ddet = mul2(mul2(mul2(bcast2(-0.5f), s), mul2(iq1, iq1)), iq1);
        G.da = ffma2(dah, iq1, mul2(ddet, b));
        G.db = ffma2(dbh, iq1, mul2(ddet, a));
        G.dc = ffma2(dch, iq1, mul2(mul2(bcast2(-2.0f), ddet), c));
      } else {
        G.da = dah; G.db = dbh; G.dc = dch;
      }
    }
    if (WANT_HR) {
      const float2 deh = ffma2(dA, bh, neg2(mul2(dD, ch)));
      const float2 dfh = ffma2(dB, ah, neg2(mul2(dC, ch)));
      const float2 dhh = ffma2(neg2(add2(dA, dB)), ch, ffma2(dC, bh, mul2(dD, ah)));
      if (normalize) {
        const float2 s = ffma2(e, deh, ffma2(f, dfh, mul2(h, dhh)));
        const float2 ddet = mul2(mul2(mul2(bcast2(-0.5f), s), mul2(iq2, iq2)), iq2);
        G.de = ffma2(deh, iq2, mul2(ddet, f));
        G.df = ffma2(dfh, iq2, mul2(ddet, e));
        G.dh = ffma2(dhh, iq2, mul2(mul2(bcast2(-2.0f), ddet), h));
      } else {
        G.de = deh; G.df = dfh; G.dh = dhh;
      }
    }
  }
  return d;
}

// ------------------------------------------------------------------------------------------------
// Shared building blocks (row-pair interleaved planes: float2 at rp*PITCH + 2*col)
// ------------------------------------------------------------------------------------------------

// Load the RGB pixels of rows [gy0, gy0+ROWS) x cols [gx0, gx0+COLS) of image `base` ([3,H,W]),
// convert to grayscale, store row-pair interleaved into sG; zero outside the image (the reference
// zero-pads: padding='same', utils.py:219-222).  ROWS even; gx0 and COLS multiples of 4.
// DEPTH items (6 x LDG.128 each) are in flight per thread before the first conversion.
// PX: the fused Pixel term -- when `px_other` (the other image of the pair) is given, the squared RGB
// difference over the tile interior rows [iy0, iy1) x cols [ix0, ix1) is accumulated into *px_acc.
template <int ROWS, int COLS, int PITCH, int NT, int DEPTH, bool PX = false>
SRST_DEV void load_gray_tile(float* sG, const float* __restrict__ base, int H, int W, int gy0, int gx0,
                             bool vec4, int tid, int iy0 = 0, int iy1 = 0, int ix0 = 0, int ix1 = 0,
                             const float* __restrict__ px_other = nullptr, float* px_acc = nullptr) {
  constexpr int C4 = COLS / 4;
  constexpr int NITEM = (ROWS / 2) * C4;
  const size_t plane = (size_t)H * W;
  if (vec4) {
#pragma unroll 1
    for (int it0 = tid; it0 < NITEM; it0 += DEPTH * NT) {
      float4 R[DEPTH][2], Gc[DEPTH][2], Bc[DEPTH][2];
      bool ok[DEPTH][2];
#pragma unroll
      for (int u = 0; u < DEPTH; ++u) {
        const int it = it0 + u * NT;
        const int q = it / C4, c4 = it - q * C4;
        const int gx = gx0 + 4 * c4;
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          const int gy = gy0 + 2 * q + hf;
          ok[u][hf] = (it < NITEM) && gy >= 0 && gy < H && gx >= 0 && gx < W;  // W % 4 == 0: all-in or all-out
          if (ok[u][hf]) {
            const float* p = base + (size_t)gy * W + gx;
            R[u][hf] = ldg4(p); Gc[u][hf] = ldg4(p + plane); Bc[u][hf] = ldg4(p + 2 * plane);
          }
        }
      }
#pragma unroll
      for (int u = 0; u < DEPTH; ++u) {
        const int it = it0 + u * NT;
        if (it >= NITEM) break;
        const int q = it / C4, c4 = it - q * C4;
        float v[2][4];
#pragma unroll
        for (int hf = 0; hf < 2; ++hf) {
          if (ok[u][hf]) {
            v[hf][0] = gray_of(R[u][hf].x, Gc[u][hf].x, Bc[u][hf].x);
            v[hf][1] = gray_of(R[u][hf].y, Gc[u][hf].y, Bc[u][hf].y);
            v[hf][2] = gray_of(R[u][hf].z, Gc[u][hf].z, Bc[u][hf].z);
            v[hf][3] = gray_of(R[u][hf].w, Gc[u][hf].w, Bc[u][hf].w);
          } else {
            v[hf][0] = v[hf][1] = v[hf][2] = v[hf][3] = 0.f;
          }
        }
        float* o = sG + q * PITCH + 8 * c4;
        st4(o, make_float4(v[0][0], v[1][0], v[0][1], v[1][1]));
        st4(o + 4, make_float4(v[0][2], v[1][2], v[0][3], v[1][3]));
        if (PX && px_other) {  // fused Pixel term: squared RGB difference to the other image, tile interior only
          const int gx = gx0 + 4 * c4;
#pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            const int gy = gy0 + 2 * q + hf;
            if (ok[u][hf] && gy >= iy0 && gy < iy1 && gx >= ix0 && gx < ix1) {
              const float* po = px_other + (size_t)gy * W + gx;
              const float4 a = ldg4(po), b = ldg4(po + plane), c = ldg4(po + 2 * plane);
              float sacc = 0.f;
              float d;
              d = R[u][hf].x - a.x; sacc = fmaf(d, d, sacc); d = R[u][hf].y - a.y; sacc = fmaf(d, d, sacc);
              d = R[u][hf].z - a.z; sacc = fmaf(d, d, sacc); d = R[u][hf].w - a.w; sacc = fmaf(d, d, sacc);
              d = Gc[u][hf].x - b.x; sacc = fmaf(d, d, sacc); d = Gc[u][hf].y - b.y; sacc = fmaf(d, d, sacc);
              d = Gc[u][hf].z - b.z; sacc = fmaf(d, d, sacc); d = Gc[u][hf].w - b.w; sacc = fmaf(d, d, sacc);
              d = Bc[u][hf].x - c.x; sacc = fmaf(d, d, sacc); d = Bc[u][hf].y - c.y; sacc = fmaf(d, d, sacc);
              d = Bc[u][hf].z - c.z; sacc = fmaf(d, d, sacc); d = Bc[u][hf].w - c.w; sacc = fmaf(d, d, sacc);
              *px_acc += sacc;
            }
          }
        }
      }
    }
  } else {
    for (int it = tid; it < NITEM; it += NT) {
      const int q = it / C4, c4 = it - q * C4;
      const int gx = gx0 + 4 * c4;
      float v[2][4];
#pragma unroll
      for (int hf = 0; hf < 2; ++hf) {
        const int gy = gy0 + 2 * q + hf;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const int x = gx + j;
          v[hf][j] = 0.f;
          if (gy >= 0 && gy < H && x >= 0 && x < W) {
            const float* p = base + (size_t)gy * W + x;
            v[hf][j] = gray_of(__ldg(p), __ldg(p + plane), __ldg(p + 2 * plane));
            if (PX && px_other && gy >= iy0 && gy < iy1 && x >= ix0 && x < ix1) {
              const float* po = px_other + (size_t)gy * W + x;
              const float d0 = __ldg(p) - __ldg(po), d1 = __ldg(p + plane) - __ldg(po + plane);
              const float d2 = __ldg(p + 2 * plane) - __ldg(po + 2 * plane);
              *px_acc += fmaf(d0, d0, fmaf(d1, d1, d2 * d2));
            }
          }
        }
      }
      float* o = sG + q * PITCH + 8 * c4;
      st4(o, make_float4(v[0][0], v[1][0], v[0][1], v[1][1]));
      st4(o + 4, make_float4(v[0][2], v[1][2], v[0][3], v[1][3]));
    }
  }
}

// Gaussian-derivative filter pair on a row pair, CS output columns:
//   ox = (A * dg|) * g-     oy = (B * g|) * dg-       (utils.py:219-222; A == B == gray forward)
// pa / pb point at (first input row pair, window start column) of planes A / B; the window is WIN
// columns wide and the CS outputs are centred at window columns CEN..CEN+CS-1.  RG+1 input row pairs
// feed the two output rows through the tap pairs dgp / gp.
template <int RG, int CS, int WIN, int CEN, bool SAME, class Taps>
SRST_DEV void grad_rowpair_rows(const float* const (&pa)[RG + 1], const float* const (&pb)[RG + 1], const Taps& tp,
                                float2 (&ox)[CS], float2 (&oy)[CS]) {
  static_assert(RG % 2 == 0 && WIN % 2 == 0, "row-pair gradient needs an even radius");
  float2 tA[WIN], tB[WIN];
#pragma unroll
  for (int j = 0; j < WIN; ++j) { tA[j] = make_float2(0.f, 0.f); tB[j] = make_float2(0.f, 0.f); }
#pragma unroll
  for (int q = 0; q <= RG; ++q) {
    float2 va[WIN], vb[WIN];
#pragma unroll
    for (int m = 0; m < WIN / 2; ++m) {
      const float4 t = ld4(pa[q] + 4 * m);
      va[2 * m] = make_float2(t.x, t.y);
      va[2 * m + 1] = make_float2(t.z, t.w);
      if (!SAME) {
        const float4 u = ld4(pb[q] + 4 * m);
        vb[2 * m] = make_float2(u.x, u.y);
        vb[2 * m + 1] = make_float2(u.z, u.w);
      }
    }
#pragma unroll
    for (int j = CEN - RG; j < CEN + CS + RG; ++j) {
      const float2 a = va[j], b = SAME ? va[j] : vb[j];
      // input rows 2q (.x) and 2q+1 (.y) of the window
      tA[j] = ffma2(bcast2(a.x), tp.dgp[2 * q], tA[j]);
      tA[j] = ffma2(bcast2(a.y), tp.dgp[2 * q + 1], tA[j]);
      tB[j] = ffma2(bcast2(b.x), tp.gp[2 * q], tB[j]);
      tB[j] = ffma2(bcast2(b.y), tp.gp[2 * q + 1], tB[j]);
    }
  }
#pragma unroll
  for (int j = 0; j < CS; ++j) {
    float2 sx = make_float2(0.f, 0.f), sy = make_float2(0.f, 0.f);
#pragma unroll
    for (int t = 0; t <= 2 * RG; ++t) {
      sx = ffma2(tA[CEN + j + t - RG], bcast2(tp.g[t]), sx);
      if (t != RG) sy = ffma2(tB[CEN + j + t - RG], bcast2(tp.dg[t]), sy);  // dg[RG] == 0
    }
    ox[j] = sx;
    oy[j] = sy;
  }
}

// Same, for planes whose RG+1 input row pairs are PITCH floats apart.
template <int RG, int CS, int WIN, int CEN, int PITCH, bool SAME, class Taps>
SRST_DEV void grad_rowpair(const float* pa, const float* pb, const Taps& tp, float2 (&ox)[CS], float2 (&oy)[CS]) {
  const float* ra[RG + 1];
  const float* rb[RG + 1];
#pragma unroll
  for (int q = 0; q <= RG; ++q) { ra[q] = pa + q * PITCH; rb[q] = pb + q * PITCH; }
  grad_rowpair_rows<RG, CS, WIN, CEN, SAME>(ra, rb, tp, ox, oy);
}

// Horizontal rho-pass on a row pair, 4 output columns: out[j] = sum_t k[t] * v[CEN + j + t - RK].
template <int RK, int CS, int WIN, int CEN, class Taps>
SRST_DEV void smooth_h_rowpair_n(const float* row, const Taps& tp, float2 (&out)[CS]) {
  float2 v[WIN];
#pragma unroll
  for (int m = 0; m < WIN / 2; ++m) {
    const float4 t = ld4(row + 4 * m);
    v[2 * m] = make_float2(t.x, t.y);
    v[2 * m + 1] = make_float2(t.z, t.w);
  }
#pragma unroll
  for (int j = 0; j < CS; ++j) {
    float2 s = make_float2(0.f, 0.f);
#pragma unroll
    for (int t = 0; t <= 2 * RK; ++t) s = ffma2(v[CEN + j + t - RK], bcast2(tp.k[t]), s);
    out[j] = s;
  }
}
// Chain + stores for one thread's 2 x 4 pixels; returns the sum of the valid distances.
// MAP: the distances also go to `map` (image b's [H,W] plane of the map), under the masks of the ds stores.
template <bool WANT_HR, bool MAP = false>
SRST_DEV float st_chain_store(const float2 (&S1)[3][4], const float2 (&S2)[3][4], bool norm, float eps,
                              float* __restrict__ ds_sr, float* __restrict__ ds_hr, size_t img_off, int H, int W,
                              int gy0, int gx0, bool vec4, float* __restrict__ map = nullptr) {
  float lsum = 0.f;
  float2 gs[3][4], gh[3][4];
  [[maybe_unused]] float2 dm[4];
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    StPixelGrad2 G;
    G.da = G.db = G.dc = G.de = G.df = G.dh = make_float2(0.f, 0.f);
    const float2 d = st_pixel2<true, WANT_HR>(S1[0][j], S1[1][j], S1[2][j], S2[0][j], S2[1][j], S2[2][j], norm, eps, G);
    const bool okx = gx0 + j < W;
    lsum += (okx && gy0 < H) ? d.x : 0.f;
    lsum += (okx && gy0 + 1 < H) ? d.y : 0.f;
    gs[0][j] = G.da; gs[1][j] = G.db; gs[2][j] = G.dc;
    if (WANT_HR) { gh[0][j] = G.de; gh[1][j] = G.df; gh[2][j] = G.dh; }
    if constexpr (MAP) dm[j] = d;
  }
  if (gx0 >= W) return lsum;
  const size_t plane = (size_t)H * W;
#pragma unroll
  for (int hf = 0; hf < 2; ++hf) {
    if (gy0 + hf >= H) continue;
    const size_t o = img_off + (size_t)(gy0 + hf) * W + gx0;
    if constexpr (MAP) {
      float* m = map + (size_t)(gy0 + hf) * W + gx0;
      const float m0 = hf ? dm[0].y : dm[0].x, m1 = hf ? dm[1].y : dm[1].x;
      const float m2 = hf ? dm[2].y : dm[2].x, m3 = hf ? dm[3].y : dm[3].x;
      if (vec4 && (reinterpret_cast<uintptr_t>(map) & 15u) == 0) {
        st4(m, make_float4(m0, m1, m2, m3));
      } else {
        const float mm[4] = {m0, m1, m2, m3};
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (gx0 + j < W) m[j] = mm[j];
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float v0 = hf ? gs[c][0].y : gs[c][0].x, v1 = hf ? gs[c][1].y : gs[c][1].x;
      const float v2 = hf ? gs[c][2].y : gs[c][2].x, v3 = hf ? gs[c][3].y : gs[c][3].x;
      float w0 = 0.f, w1 = 0.f, w2 = 0.f, w3 = 0.f;
      if (WANT_HR) {
        w0 = hf ? gh[c][0].y : gh[c][0].x; w1 = hf ? gh[c][1].y : gh[c][1].x;
        w2 = hf ? gh[c][2].y : gh[c][2].x; w3 = hf ? gh[c][3].y : gh[c][3].x;
      }
      if (vec4) {
        if (ds_sr) st4(ds_sr + o + c * plane, make_float4(v0, v1, v2, v3));
        if (WANT_HR) st4(ds_hr + o + c * plane, make_float4(w0, w1, w2, w3));
      } else {
        const float vv[4] = {v0, v1, v2, v3}, ww[4] = {w0, w1, w2, w3};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          if (gx0 + j < W) {
            if (ds_sr) ds_sr[o + c * plane + j] = vv[j];
            if (WANT_HR) ds_hr[o + c * plane + j] = ww[j];
          }
        }
      }
    }
  }
  return lsum;
}

// ------------------------------------------------------------------------------------------------
// Lane -> item mapping of the register-blocked (row pair x CS columns) phases.  An item reads
// LDS.128 windows at q*PITCH + 2*CS*seg + const with PITCH == 4 mod 8, i.e. 16-byte bank group
// (q*odd + (CS/2)*seg) mod 8.  A quarter-warp (the unit one LDS.128 wavefront serves) is conflict
// free when its eight lanes are 8 consecutive q of one seg, or 2 q x 4 seg (CS == 4), or 4 q x 2 seg
// (CS == 8).  The group shape is picked from the row-pair count so that no lane pattern straddles a
// segment boundary the way a plain it -> (it / NQ, it % NQ) split does when NQ % 8 != 0 (round 1:
// 16 % of the backward's shared-memory wavefronts were such conflicts).
// ------------------------------------------------------------------------------------------------
template <int NQ_, int NSEG_, int CS_>
struct ItemMap {
  static constexpr int NQ = NQ_, NSEG = NSEG_, CS = CS_;
  static constexpr int GQ = (NQ % 8 == 0) ? 8 : (CS == 4 ? 2 : 4);
  static constexpr int GS = 8 / GQ;
  static constexpr int NQG = (NQ + GQ - 1) / GQ, NSG = (NSEG + GS - 1) / GS;
  static constexpr int SLOTS = NQG * NSG * 8;
  static_assert(CS == 4 || CS == 8, "ItemMap: 4- or 8-column items");
  SRST_DEV static bool decode(int it, int& q, int& seg) {
    const int g = it >> 3, l = it & 7;
    const int gs = g / NQG, gq = g - gs * NQG;
    q = gq * GQ + (l % GQ);
    seg = gs * GS + (l / GQ);
    return q < NQ && seg < NSEG;
  }
};

// ------------------------------------------------------------------------------------------------
// Forward
// ------------------------------------------------------------------------------------------------
template <int TH_, int TW_, int RS_, int CSB_, int RG_, int RK_, int MINB_, int CHU_ = 1, bool CSPLIT_ = false, int LDEPTH_ = 2>
struct StFwdCfg {
  // CSPLIT: the vertical pass hands out (plane, row segment, column) items instead of (row segment, column): used
  // when columns x segments alone leave a large part of the CTA idle (32x64 tile: 160 items for 256 threads).
  static constexpr bool CSPLIT = CSPLIT_;
  static constexpr int TH = TH_, TW = TW_, RS = RS_, CSB = CSB_, RG = RG_, RK = RK_, MINB = MINB_;
  // CHU > 0: ROLLED kernel -- SR and HR run through one copy of the filter code, both smoothed tensors are
  //          parked in thread-private shared-memory slots and the per-pixel chain is a loop over the thread's four
  //          pixel pairs, CHU of them in flight (half the code, no spills, 24 * NT floats of shared memory more).
  // CHU == 0: UNROLLED kernel -- two inlined copies of the filter phases, the SR tensor waits in registers while
  //          the HR image is processed, chain on all eight pixels at once (more registers, less shared memory:
  //          what lets the large-image tile keep three CTAs per SM).
  static constexpr int CHU = CHU_;
  static constexpr bool ROLLED = CHU_ > 0;
  static constexpr int LDEPTH = LDEPTH_;  // gray-tile items (6 x LDG.128 each) in flight per thread
  static constexpr int HXD = round_up4(RK);  // x halo of the gradient (D) and V regions
  static constexpr int OFF = round_up4(RG);
  static constexpr int HXG = HXD + OFF;      // x halo of the gray (G) region
  static constexpr int GH = TH + 2 * (RG + RK), GW = TW + 2 * HXG, PG = smem_pitch(2 * GW);
  static constexpr int DH = TH + 2 * RK, DW = TW + 2 * HXD, PD = smem_pitch(2 * DW);
  static constexpr int PV = PD;
  static constexpr int NSEG = TH / RS;
  static constexpr int BW_LO = (OFF - RG) / 2 * 2, BW_HI = (OFF + CSB + RG + 1) / 2 * 2, BWIN = BW_HI - BW_LO;
  static constexpr int DW_LO = (HXD - RK) / 2 * 2, DW_HI = (HXD + 4 + RK + 1) / 2 * 2, DWIN = DW_HI - DW_LO;
  using MapB = ItemMap<DH / 2, DW / CSB, CSB>;  // gradient items
  using MapD = ItemMap<TH / 2, TW / 4, 4>;      // horizontal-pass items == the thread's 2 x 4 output pixels
  static constexpr int NT = (MapD::SLOTS + 31) / 32 * 32;  // one horizontal-pass item per thread (idle tail lanes when not a warp multiple)
  static constexpr int D_FLOATS = (DH / 2) * PD, V_FLOATS = (TH / 2) * PV, G_FLOATS = (GH / 2) * PG;
  static constexpr int SP_FLOATS = 24 * NT;  // a parked tensor: 3 channels x 4 columns x float2 per thread
  // smem: D (Ix, Iy) | V (3 planes; the gray tile aliases it: dead once the gradient phase is done) | SP1.
  // The HR tensor is parked over D (SP2): dead once the vertical pass is done.
  static constexpr int VG_FLOATS = cmax(3 * V_FLOATS, G_FLOATS);
  static constexpr bool SP2_OVER_D = SP_FLOATS <= 2 * D_FLOATS;        // small radii: D is too small
  static constexpr int SP_OFF = 2 * D_FLOATS + VG_FLOATS;
  static constexpr int SP2_OFF = SP2_OVER_D ? 0 : SP_OFF + SP_FLOATS;
  static constexpr int SMEM_FLOATS = ROLLED ? SP_OFF + SP_FLOATS + (SP2_OVER_D ? 0 : SP_FLOATS) : SP_OFF;
  static constexpr size_t SMEM_BYTES = sizeof(float) * SMEM_FLOATS;
  static_assert((CSB == 4 || CSB == 8) && DW % CSB == 0, "bad gradient segment width");
  static_assert(TH % RS == 0 && RS % 2 == 0 && TH % 2 == 0 && TW % 4 == 0 && RG % 2 == 0 && RK % 2 == 0,
                "bad forward tile");
  static_assert(NT % 32 == 0 && NT <= 1024, "bad forward block size");
  static_assert(CHU == 0 || CHU == 1 || CHU == 2 || CHU == 4, "chain unroll");
};

// Phases A-D for one image of the tile: leaves the smoothed tensor (Jxx,Jyy,Jxy) of this thread's
// 8 pixels (rows 2q, 2q+1; cols 4*seg..4*seg+3 of the tile) in S[3][4] (.x = even row, .y = odd row).
template <class C, bool PX, class Taps>
SRST_DEV void st_unit_tensor(float* smem, const float* __restrict__ base, float* __restrict__ ixy, int b, bool vec4,
                             int H, int W, int y0, int x0, const Taps& tp, int tid, bool dvalid, int dq, int dseg,
                             float2 (&S)[3][4], const float* __restrict__ px_other, float* px_acc,
                             [[maybe_unused]] int stamp0 = 0) {
  float* sD0 = smem;
  float* sD1 = sD0 + C::D_FLOATS;
  float* sV = sD1 + C::D_FLOATS;
  float* sG = sV;

  __syncthreads();  // every thread is done with sV / sD (SP2) of the previous unit
  SRST_STAMP(stamp0 + 0);
  load_gray_tile<C::GH, C::GW, C::PG, C::NT, C::LDEPTH, PX>(sG, base, H, W, y0 - (C::RG + C::RK), x0 - C::HXG, vec4,
                                                            tid, y0, y0 + C::TH, x0, x0 + C::TW, px_other, px_acc);
  __syncthreads();
  SRST_STAMP(stamp0 + 1);

  // Phase B: Ix, Iy on the D region; forced to zero outside the image because the reference
  // zero-pads the *products* for the rho-smoothing (utils.py:225-230).  Tile-interior items also
  // save their values for the backward pass (ixy planes).
  const int Hp = (H + 1) >> 1;
  for (int it = tid; it < C::MapB::SLOTS; it += C::NT) {
    int q, seg;
    if (!C::MapB::decode(it, q, seg)) continue;
    const int dx0 = C::CSB * seg;
    const int gy = y0 - C::RK + 2 * q, gx0 = x0 - C::HXD + dx0;
    float2 Ix[C::CSB], Iy[C::CSB];
    if (gy + 1 >= 0 && gy < H && gx0 + C::CSB - 1 >= 0 && gx0 < W) {
      const float* p = sG + q * C::PG + 2 * (dx0 + C::BW_LO);
      grad_rowpair<C::RG, C::CSB, C::BWIN, C::OFF - C::BW_LO, C::PG, true>(p, p, tp, Ix, Iy);
      if (!(gy >= 0 && gy + 1 < H && gx0 >= 0 && gx0 + C::CSB <= W)) {  // straddles the image border: mask
        const bool r0 = gy >= 0, r1 = gy + 1 < H;  // gy < H and gy + 1 >= 0 hold here
#pragma unroll
        for (int j = 0; j < C::CSB; ++j) {
          const bool ok = (gx0 + j >= 0) && (gx0 + j < W);
          Ix[j].x = (ok && r0) ? Ix[j].x : 0.f;
          Ix[j].y = (ok && r1) ? Ix[j].y : 0.f;
          Iy[j].x = (ok && r0) ? Iy[j].x : 0.f;
          Iy[j].y = (ok && r1) ? Iy[j].y : 0.f;
        }
      }
      if (ixy && gy >= y0 && gy < y0 + C::TH && gx0 >= x0 && gx0 < x0 + C::TW) {  // tile interior, inside the image
        float* ox = ixy + ixy_offset(b, 0, Hp, W, gy >> 1, gx0);
        float* oy = ixy + ixy_offset(b, 1, Hp, W, gy >> 1, gx0);
        if (vec4) {
#pragma unroll
          for (int j = 0; j < C::CSB; j += 2) {
            st4(ox + 2 * j, make_float4(Ix[j].x, Ix[j].y, Ix[j + 1].x, Ix[j + 1].y));
            st4(oy + 2 * j, make_float4(Iy[j].x, Iy[j].y, Iy[j + 1].x, Iy[j + 1].y));
          }
        } else {
#pragma unroll
          for (int j = 0; j < C::CSB; ++j)
            if (gx0 + j < W) { st2(ox + 2 * j, Ix[j]); st2(oy + 2 * j, Iy[j]); }
        }
      }
    } else {
#pragma unroll
      for (int j = 0; j < C::CSB; ++j) { Ix[j] = make_float2(0.f, 0.f); Iy[j] = make_float2(0.f, 0.f); }
    }
    float* o0 = sD0 + q * C::PD + 2 * dx0;
    float* o1 = sD1 + q * C::PD + 2 * dx0;
#pragma unroll
    for (int j = 0; j < C::CSB; j += 2) {
      st4(o0 + 2 * j, make_float4(Ix[j].x, Ix[j].y, Ix[j + 1].x, Ix[j + 1].y));
      st4(o1 + 2 * j, make_float4(Iy[j].x, Iy[j].y, Iy[j + 1].x, Iy[j + 1].y));
    }
  }
  __syncthreads();
  SRST_STAMP(stamp0 + 2);

  // Phase C: vertical rho-pass of the three products; a lane owns one column and RS output rows
  // (RS/2 row pairs).  Columns outside the image hold zeros and are only cleared.
  {
    const int c_lo = max(0, C::HXD - x0), c_hi = min(C::DW, W + C::HXD - x0);  // valid D columns
    const int ncol = c_hi - c_lo;
    const int nclr = C::DW - ncol;
    // it / ncol and it / nclr by multiplication: exact for it < 4096, divisor <= 256 (item counts stay below that)
    const unsigned mg_col = (1048576u + (unsigned)ncol - 1u) / (unsigned)ncol;
    if (nclr > 0) {
      const unsigned mg_clr = (1048576u + (unsigned)nclr - 1u) / (unsigned)nclr;
      for (int it = tid; it < nclr * (C::TH / 2); it += C::NT) {
        const int q = (int)(((unsigned)it * mg_clr) >> 20), u = it - q * nclr;
        const int dx = (u < c_lo) ? u : (c_hi + (u - c_lo));
#pragma unroll
        for (int c = 0; c < 3; ++c) st2(sV + c * C::V_FLOATS + q * C::PV + 2 * dx, make_float2(0.f, 0.f));
      }
    }
    if constexpr (!C::CSPLIT) {
      for (int it = tid; it < ncol * C::NSEG; it += C::NT) {
        const int seg = (int)(((unsigned)it * mg_col) >> 20), dx = c_lo + (it - seg * ncol);
        float2 acc[3][C::RS / 2];
#pragma unroll
        for (int j = 0; j < C::RS / 2; ++j) {
          acc[0][j] = make_float2(0.f, 0.f); acc[1][j] = make_float2(0.f, 0.f); acc[2][j] = make_float2(0.f, 0.f);
        }
        const float* p0 = sD0 + (seg * (C::RS / 2)) * C::PD + 2 * dx;
        const float* p1 = sD1 + (seg * (C::RS / 2)) * C::PD + 2 * dx;
#pragma unroll
        for (int rq = 0; rq < C::RS / 2 + C::RK; ++rq) {
          const float2 ix = ld2(p0 + rq * C::PD), iy = ld2(p1 + rq * C::PD);
          const float2 pxx = mul2(ix, ix), pyy = mul2(iy, iy), pxy = mul2(ix, iy);  // packed FMUL2
#pragma unroll
          for (int jp = 0; jp < C::RS / 2; ++jp) {
            const int u0 = 2 * rq - 2 * jp;  // tap-pair index of input row 2rq for output pair jp
            if (u0 >= 0 && u0 <= 2 * C::RK + 1) {
              acc[0][jp] = ffma2(bcast2(pxx.x), tp.kp[u0], acc[0][jp]);
              acc[1][jp] = ffma2(bcast2(pyy.x), tp.kp[u0], acc[1][jp]);
              acc[2][jp] = ffma2(bcast2(pxy.x), tp.kp[u0], acc[2][jp]);
            }
            if (u0 + 1 >= 0 && u0 + 1 <= 2 * C::RK + 1) {
              acc[0][jp] = ffma2(bcast2(pxx.y), tp.kp[u0 + 1], acc[0][jp]);
              acc[1][jp] = ffma2(bcast2(pyy.y), tp.kp[u0 + 1], acc[1][jp]);
              acc[2][jp] = ffma2(bcast2(pxy.y), tp.kp[u0 + 1], acc[2][jp]);
            }
          }
        }
#pragma unroll
        for (int c = 0; c < 3; ++c) {
          float* o = sV + c * C::V_FLOATS + (seg * (C::RS / 2)) * C::PV + 2 * dx;
#pragma unroll
          for (int jp = 0; jp < C::RS / 2; ++jp) st2(o + jp * C::PV, acc[c][jp]);
        }
      }
    } else {
      // one item = (plane, row segment, column): plane 0 = Ix^2, 1 = Iy^2, 2 = Ix*Iy
      for (int it = tid; it < 3 * ncol * C::NSEG; it += C::NT) {
        const int cs = (int)(((unsigned)it * mg_col) >> 20), dx = c_lo + (it - cs * ncol);
        const int c = cs / C::NSEG, seg = cs - c * C::NSEG;
        float2 acc[C::RS / 2];
#pragma unroll
        for (int j = 0; j < C::RS / 2; ++j) acc[j] = make_float2(0.f, 0.f);
        const float* pa = (c == 1 ? sD1 : sD0) + (seg * (C::RS / 2)) * C::PD + 2 * dx;
        const float* pb = (c == 0 ? sD0 : sD1) + (seg * (C::RS / 2)) * C::PD + 2 * dx;
#pragma unroll
        for (int rq = 0; rq < C::RS / 2 + C::RK; ++rq) {
          const float2 pr = mul2(ld2(pa + rq * C::PD), ld2(pb + rq * C::PD));
#pragma unroll
          for (int jp = 0; jp < C::RS / 2; ++jp) {
            const int u0 = 2 * rq - 2 * jp;
            if (u0 >= 0 && u0 <= 2 * C::RK + 1) acc[jp] = ffma2(bcast2(pr.x), tp.kp[u0], acc[jp]);
            if (u0 + 1 >= 0 && u0 + 1 <= 2 * C::RK + 1) acc[jp] = ffma2(bcast2(pr.y), tp.kp[u0 + 1], acc[jp]);
          }
        }
        float* o = sV + c * C::V_FLOATS + (seg * (C::RS / 2)) * C::PV + 2 * dx;
#pragma unroll
        for (int jp = 0; jp < C::RS / 2; ++jp) st2(o + jp * C::PV, acc[jp]);
      }
    }
  }
  __syncthreads();
  SRST_STAMP(stamp0 + 3);

  // Phase D: horizontal rho-pass; a lane owns 4 consecutive columns of one row pair.
  if (dvalid) {
    const int ox0 = 4 * dseg;
#pragma unroll
    for (int c = 0; c < 3; ++c)
      smooth_h_rowpair_n<C::RK, 4, C::DWIN, C::HXD - C::DW_LO>(sV + c * C::V_FLOATS + dq * C::PV + 2 * (ox0 + C::DW_LO), tp,
                                                              S[c]);
  }
}

// PER_IMG: reduction='none' -- loss_out[b] is the mean over image b's pixels (P.inv_count = 1 / (H W)) instead of
// loss_out[0] over the batch; with PX, loss_out[B + b] is image b's mean squared difference over its 3 H W values.
// MAP: also stores every pixel's distance into P.map_out [B,H,W] (the loss and the other outputs are unchanged).
template <class C, bool PX = false, bool WANT_HR = false, bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(C::NT, C::MINB)
st_forward_kernel(const __grid_constant__ StFwdParamsT<C::RG, C::RK, MAP> P) {
  static_assert(!(MAP && (PX || PER_IMG)), "the distance map comes with the batch loss only");
  SRST_DYN_SMEM(float, smem);
  __shared__ float s_red[32];
  __shared__ unsigned int s_last;
  [[maybe_unused]] __shared__ float s_red_px[PX ? 32 : 1];
  const int tid = threadIdx.x;
  SRST_STAMP(15);
  pdl_wait();     // previous kernel of the stream is complete (it may have produced sr or used the workspace)
  pdl_trigger();  // the next PDL-launched kernel may start launching; it waits for this grid itself

  int t = blockIdx.x;
  const int tx = t % P.tiles_x;
  t /= P.tiles_x;
  const int ty = t % P.tiles_y;
  const int b = t / P.tiles_y;
  const int y0 = ty * C::TH, x0 = tx * C::TW;
  const int H = P.H, W = P.W;
  const size_t img_off = (size_t)b * 3 * H * W;
  const bool vec4 = P.vec4 != 0;
  const bool norm = P.normalize != 0;
  int q, seg;
  const bool dvalid = C::MapD::decode(tid, q, seg);
  float* sp1 = smem + C::SP_OFF + 2 * tid;   // slot (c, j) of this thread: + 2 * NT * (c * 4 + j)
  float* sp2 = smem + C::SP2_OFF + 2 * tid;  // HR tensor, parked over the (dead) D region when it fits there
  [[maybe_unused]] float pxsum = 0.f;

  float lsum = 0.f;
  const int gy0 = y0 + 2 * q, gx0 = x0 + 4 * seg;
  if constexpr (!C::ROLLED) {
    // UNROLLED: two inlined copies of the filter phases; S1 waits in registers while HR is processed
    float2 S1[3][4], S2[3][4];
    st_unit_tensor<C, false>(smem, P.sr + img_off, P.ixy_sr, b, vec4, H, W, y0, x0, P.taps, tid, dvalid, q, seg, S1,
                             nullptr, nullptr, 0);
    st_unit_tensor<C, PX>(smem, P.hr + img_off, P.ixy_hr, b, vec4, H, W, y0, x0, P.taps, tid, dvalid, q, seg, S2,
                          PX ? P.sr + img_off : nullptr, &pxsum, 4);
    SRST_STAMP(8);
    if (dvalid) {
      if constexpr (MAP)
        lsum = st_chain_store<WANT_HR, true>(S1, S2, norm, P.eps, P.ds_sr, P.ds_hr, img_off, H, W, gy0, gx0, vec4,
                                             P.map_out + (size_t)b * H * W);
      else
        lsum = st_chain_store<WANT_HR>(S1, S2, norm, P.eps, P.ds_sr, P.ds_hr, img_off, H, W, gy0, gx0, vec4);
    }
  } else {
    // SR, then HR, through one copy of the filter code
  #pragma unroll 1
    for (int img = 0; img < 2; ++img) {
      float2 S[3][4];
      const float* base = (img ? P.hr : P.sr) + img_off;
      float* ixy = img ? P.ixy_hr : P.ixy_sr;
      st_unit_tensor<C, PX>(smem, base, ixy, b, vec4, H, W, y0, x0, P.taps, tid, dvalid, q, seg, S,
                            (PX && img) ? P.sr + img_off : nullptr, &pxsum, 4 * img);
      if (img) SRST_STAMP(8);
      if (dvalid) {
        {
          float* sp = img ? sp2 : sp1;
  #pragma unroll
          for (int c = 0; c < 3; ++c)
  #pragma unroll
            for (int j = 0; j < 4; ++j) st2(sp + 2 * C::NT * (c * 4 + j), S[c][j]);
        }
      }
    }
    // Per-pixel chain on this thread's 2 x 4 pixels, one pixel pair (two rows of one column) per
    // iteration; operands come from the thread's parked slots and the results go back into them.
    if (dvalid) {
  #pragma unroll C::CHU
      for (int j = 0; j < 4; ++j) {
        float* a1 = sp1 + 2 * C::NT * j;
        float* a2 = sp2 + 2 * C::NT * j;
        StPixelGrad2 G;
        G.da = G.db = G.dc = G.de = G.df = G.dh = make_float2(0.f, 0.f);
        const float2 d = st_pixel2<true, WANT_HR>(ld2(a1), ld2(a1 + 8 * C::NT), ld2(a1 + 16 * C::NT), ld2(a2),
                                                  ld2(a2 + 8 * C::NT), ld2(a2 + 16 * C::NT), norm, P.eps, G);
        const bool okx = gx0 + j < W;
        lsum += (okx && gy0 < H) ? d.x : 0.f;
        lsum += (okx && gy0 + 1 < H) ? d.y : 0.f;
        if constexpr (MAP) {
          float* m = P.map_out + (size_t)b * H * W + (size_t)gy0 * W + gx0 + j;
          if (okx && gy0 < H) m[0] = d.x;
          if (okx && gy0 + 1 < H) m[W] = d.y;
        }
        st2(a1, G.da); st2(a1 + 8 * C::NT, G.db); st2(a1 + 16 * C::NT, G.dc);
        if (WANT_HR) { st2(a2, G.de); st2(a2 + 8 * C::NT, G.df); st2(a2 + 16 * C::NT, G.dh); }
      }
      // ds stores: rows of 4 consecutive columns per channel (STG.128)
      if (gx0 < W && (P.ds_sr || WANT_HR)) {
        const size_t plane = (size_t)H * W;
  #pragma unroll
        for (int c = 0; c < 3; ++c) {
          float2 v[4], w[4];
  #pragma unroll
          for (int j = 0; j < 4; ++j) {
            v[j] = ld2(sp1 + 2 * C::NT * (c * 4 + j));
            if (WANT_HR) w[j] = ld2(sp2 + 2 * C::NT * (c * 4 + j));
          }
  #pragma unroll
          for (int hf = 0; hf < 2; ++hf) {
            if (gy0 + hf >= H) continue;
            const size_t o = img_off + c * plane + (size_t)(gy0 + hf) * W + gx0;
            if (vec4) {
              if (P.ds_sr) st4(P.ds_sr + o, hf ? make_float4(v[0].y, v[1].y, v[2].y, v[3].y)
                                             : make_float4(v[0].x, v[1].x, v[2].x, v[3].x));
              if (WANT_HR) st4(P.ds_hr + o, hf ? make_float4(w[0].y, w[1].y, w[2].y, w[3].y)
                                               : make_float4(w[0].x, w[1].x, w[2].x, w[3].x));
            } else {
  #pragma unroll
              for (int j = 0; j < 4; ++j) {
                if (gx0 + j < W) {
                  if (P.ds_sr) P.ds_sr[o + j] = hf ? v[j].y : v[j].x;
                  if (WANT_HR) P.ds_hr[o + j] = hf ? w[j].y : w[j].x;
                }
              }
            }
          }
        }
      }
    }
  }

  // Deterministic loss reduction: block partial -> workspace; the last block to finish sums all
  // partials in a fixed order (double) and re-zeroes the workspace for the next call.
  SRST_STAMP(9);   // thread 0 is done with its chain + stores
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
  SRST_STAMP(10);  // every warp of the CTA is done
  if constexpr (PER_IMG) {
    if (s_last) {  // image-major grid: image b owns tiles_y * tiles_x consecutive CTAs
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
        if constexpr (PX) P.loss_out[1] = (float)(accp * (double)P.inv_count / 3.0);  // mean over B*3*H*W
        *P.ticket = 0u;
      }
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Structure-tensor features of ONE image tensor: the smoothed tensor itself and its closed-form 2x2
// eigen-decomposition (BASELINE.json north_star: "closed-form 2x2 eigendecomposition giving orientation,
// coherence and eigenvalues").  The reference computes these only in an exploration notebook, with the
// third-party `structure_tensor` package (data-exploration/structure_tensor.ipynb: eig_special_2d, then
// arctan2 of the eigenvector and 1 - val[0]/val[1]); that package is not part of the reference checkout, so
// this output is a diagnostic with its own definition (parity unpinned, DESIGN.md):
//   S = [[Jxx, Jxy], [Jxy, Jyy]]  (Jxx: derivative along H, as utils.py:219-229 names them)
//   lambda_small/large = (Jxx + Jyy)/2 -/+ sqrt(((Jxx - Jyy)/2)^2 + Jxy^2)
//   orientation = 1/2 atan2(2 Jxy, Jxx - Jyy)   angle of the dominant-gradient eigenvector against the H axis,
//                                               in (-pi/2, pi/2]; the coherent structure runs perpendicular to it
//   coherence   = 1 - lambda_small / lambda_large  (0 where lambda_large == 0)
// Same tile phases as the forward kernel (st_unit_tensor); precise math functions: this is not a hot path.
// ------------------------------------------------------------------------------------------------
template <int RG, int RK>
struct StFeatParams {
  const float* img;
  float* J;       // [B,3,H,W] (Jxx, Jyy, Jxy) or null
  float* eig;     // [B,2,H,W] (small, large) or null
  float* orient;  // [B,H,W] or null
  float* coher;   // [B,H,W] or null
  int B, H, W, tiles_x, tiles_y, vec4;
  StTaps<RG, RK> taps;
};

template <class C>
__global__ void __launch_bounds__(C::NT, C::MINB)
st_features_kernel(const __grid_constant__ StFeatParams<C::RG, C::RK> P) {
  SRST_DYN_SMEM(float, smem);
  const int tid = threadIdx.x;
  int t = blockIdx.x;
  const int tx = t % P.tiles_x;
  t /= P.tiles_x;
  const int ty = t % P.tiles_y;
  const int b = t / P.tiles_y;
  const int y0 = ty * C::TH, x0 = tx * C::TW;
  const int H = P.H, W = P.W;
  int q, seg;
  const bool dvalid = C::MapD::decode(tid, q, seg);
  float2 S[3][4];
  st_unit_tensor<C, false>(smem, P.img + (size_t)b * 3 * H * W, nullptr, b, P.vec4 != 0, H, W, y0, x0, P.taps, tid, dvalid, q,
                           seg, S, nullptr, nullptr);
  if (!dvalid) return;
  const size_t plane = (size_t)H * W;
#pragma unroll
  for (int j = 0; j < 4; ++j) {
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      const int gy = y0 + 2 * q + hf, gx = x0 + 4 * seg + j;
      if (gy >= H || gx >= W) continue;
      const float a = hf ? S[0][j].y : S[0][j].x, bb = hf ? S[1][j].y : S[1][j].x, c = hf ? S[2][j].y : S[2][j].x;
      const size_t o = (size_t)gy * W + gx;
      if (P.J) {
        P.J[((size_t)b * 3 + 0) * plane + o] = a;
        P.J[((size_t)b * 3 + 1) * plane + o] = bb;
        P.J[((size_t)b * 3 + 2) * plane + o] = c;
      }
      const float hd = 0.5f * (a - bb), mean = 0.5f * (a + bb);
      const float r = sqrtf(fmaf(hd, hd, c * c));
      const float l_small = mean - r, l_large = mean + r;
      if (P.eig) {
        P.eig[((size_t)b * 2 + 0) * plane + o] = l_small;
        P.eig[((size_t)b * 2 + 1) * plane + o] = l_large;
      }
      if (P.orient) P.orient[(size_t)b * plane + o] = 0.5f * atan2f(2.0f * c, a - bb);
      if (P.coher) P.coher[(size_t)b * plane + o] = l_large > 0.f ? 1.0f - l_small / l_large : 0.f;
    }
  }
}

// ------------------------------------------------------------------------------------------------
// Backward
// ------------------------------------------------------------------------------------------------
template <int TH_, int TW_, int RS_, int NT_, int RG_, int RK_, int MINB_, int CSD_ = 8, bool PIPE_ = false, bool XFULL_ = false>
struct StBwdCfg {
  static constexpr int TH = TH_, TW = TW_, RS = RS_, NT = NT_, RG = RG_, RK = RK_, MINB = MINB_;
  // PIPE: persistent CTAs that loop over tiles and fetch the NEXT tile's ds box as soon as the vertical pass has
  // consumed this one (and its Ix, Iy box as soon as the product rule has), so that the TMA round trip -- a third
  // of the warp time when every CTA waits for its own tile first -- hides behind the rest of the current tile.
  // dIx|dIy then need their own region instead of re-using the ds staging.
  static constexpr bool PIPE = PIPE_;
  // XFULL: for images no wider than the tile (W <= TW, one tile in x, x0 == 0).  Every x-halo column is then outside
  // the image, where ds, Ix and Iy -- and so E, dIx and dIy -- are zero: only the TW image columns of ds and Ix, Iy
  // are staged, the vertical pass and the product rule run on them alone, and the zero columns the horizontal window
  // (RK each side of V) and the adjoint derivative filter (RG each side of dIx|dIy) read are written by the kernel.
  static constexpr bool XFULL = XFULL_;
  static constexpr int CSD = CSD_;  // output columns per phase-D' item: 8 reads a 24-column window per 8 outputs
                                    // (3x shared-memory amplification) instead of 20 per 4 (5x)
  static constexpr int HXE = round_up4(RG);  // x halo of the E region (where dIx, dIy are needed)
  static constexpr int HXK = round_up4(RK);
  static constexpr int EH = TH + 2 * RG, EW = TW + 2 * HXE, PE = smem_pitch(2 * EW);
  static constexpr int VW = (XFULL ? TW : EW) + 2 * HXK, PV = smem_pitch(2 * VW);  // vertical-pass output
  static constexpr int SH = EH + 2 * RK;                            // staged ds rows
  static constexpr int NSEG = EH / RS;
  // x extent of the product rule (E columns EC0..EC0+ECW-1, the rest of the E region is zero), of the staged ds box
  // (SW columns from tile column -SX, landing at V column SX0) and of the saved Ix, Iy box (from tile column -IX)
  static constexpr int EC0 = XFULL ? HXE : 0, ECW = XFULL ? TW : EW;
  static constexpr int SW = XFULL ? TW : VW, SX = XFULL ? 0 : HXE + HXK, SX0 = XFULL ? HXK : 0, IX = XFULL ? 0 : HXE;
  static constexpr int VE = XFULL ? HXE : 0;  // V column of E column e's window start: e - VE
  // saved Ix, Iy tile: TMA box of EH/2 row pairs x EWB columns (x 2 floats); EWB = ECW + 2 makes the
  // pitch 2*EWB == 4 mod 8 floats (conflict-free LDS.128 across row pairs) and a multiple of 16 bytes
  static constexpr int EWB = ECW + 2, PI = 2 * EWB;
  static constexpr int BW_LO = (HXE - RG) / 2 * 2, BW_HI = (HXE + 4 + RG + 1) / 2 * 2, BWIN = BW_HI - BW_LO;
  static constexpr int DW_LO = (HXK - RK) / 2 * 2, DW_HI = (HXK + CSD + RK + 1) / 2 * 2, DWIN = DW_HI - DW_LO;
  using MapD = ItemMap<EH / 2, ECW / CSD, CSD>;  // horizontal pass + product rule
  using MapE = ItemMap<TH / 2, TW / 4, 4>;       // adjoint derivative filters + stores
  // smem: X: staged ds planes [3][SH][SW] row-major (TMA destination), later dIx|dIy (the staging is
  // dead once the vertical pass has consumed it) | I: saved Ix, Iy [2][EH/2][PI] (TMA destination) | V (3 planes)
  static constexpr int V_FLOATS = (EH / 2) * PV, I_FLOATS = (EH / 2) * PI, DI_FLOATS = (EH / 2) * PE;
  static constexpr int S_FLOATS = SH * SW;
  static constexpr int X_FLOATS = PIPE ? 3 * S_FLOATS : cmax(2 * DI_FLOATS, 3 * S_FLOATS);
  static constexpr int I_OFF = (X_FLOATS + 31) / 32 * 32;               // 128-byte aligned (TMA destination)
  static constexpr int V_OFF = (I_OFF + 2 * I_FLOATS + 31) / 32 * 32;
  static constexpr int DI_OFF = PIPE ? V_OFF + 3 * V_FLOATS : 0;
  static constexpr int SMEM_FLOATS = V_OFF + 3 * V_FLOATS + (PIPE ? 2 * DI_FLOATS : 0);
  static constexpr size_t SMEM_BYTES = sizeof(float) * SMEM_FLOATS;
  static_assert(PI % 8 == 4 && PE % 8 == 4 && PV % 8 == 4, "row-pair pitches must be == 4 mod 8");
  static_assert(EH % RS == 0 && RS % 2 == 0 && TH % 2 == 0 && TW % 4 == 0 && RG % 2 == 0 && RK % 2 == 0,
                "bad backward tile");
  static_assert(NT % 32 == 0 && NT <= 1024, "bad backward block size");
  static_assert((CSD == 4 || CSD == 8) && ECW % CSD == 0, "bad phase-D' item width");
  // MINB CTAs per SM: 228 KB of shared memory per SM on sm_100, 1 KB of it reserved per CTA
  static_assert(MINB * (SMEM_BYTES + 1024) <= 228 * 1024, "shared memory does not allow MINB CTAs per SM");
};

// PER_IMG: reduction='none' -- grad_out (and with PX grad_px) is [B] and the tile of image b scales by grad_out[b] / (H W)
// (P.inv_count = 1 / (H W)) instead of grad_out[0] / (B H W)
template <class C, bool PX = false, bool PER_IMG = false>
__global__ void __launch_bounds__(C::NT, C::MINB)
st_backward_kernel(const __grid_constant__ StBwdParams<C::RG, C::RK> P) {
  SRST_DYN_SMEM(float, smem);
  float* sS = smem;                     // staged ds [3][SH][SW]
  float* sdI0 = smem + C::DI_OFF;       // dIx [EH/2][PE]: over the (dead) staging, or its own region when pipelined
  float* sdI1 = sdI0 + C::DI_FLOATS;    // dIy
  float* sI0 = smem + C::I_OFF;         // saved Ix [EH/2][PI]
  float* sI1 = sI0 + C::I_FLOATS;       // saved Iy
  float* sV = smem + C::V_OFF;          // [3][EH/2][PV]  vertical rho-pass of ds
  __shared__ __align__(8) unsigned long long s_mbar;    // ds box (and the Ix, Iy box when not pipelined)
  __shared__ __align__(8) unsigned long long s_mbar_i;  // Ix, Iy box (pipelined kernel)

  const int tid = threadIdx.x;
  const int H = P.H, W = P.W;
  const size_t plane = (size_t)H * W;
  const auto& tp = P.taps;
  const int ntiles = P.B * P.tiles_y * P.tiles_x;
  constexpr unsigned kBytesS = (unsigned)(3 * C::S_FLOATS * sizeof(float)), kBytesI = (unsigned)(2 * C::I_FLOATS * sizeof(float));
  const bool pipe = C::PIPE && P.use_tma;
  // tile -> coordinates of its staged boxes
  auto issue_s = [&](int t) {
    const int tx_ = t % P.tiles_x, r_ = t / P.tiles_x;
    const int ty_ = r_ % P.tiles_y, b_ = r_ / P.tiles_y;
    tma_expect(&s_mbar, pipe ? kBytesS : kBytesS + kBytesI);
    tma_load_3d(&s_mbar, sS, &P.ds_map, tx_ * C::TW - C::SX, ty_ * C::TH - C::RG - C::RK, b_ * 3, C::SW, C::SH, 3);
  };
  auto issue_i = [&](int t) {
    const int tx_ = t % P.tiles_x, r_ = t / P.tiles_x;
    const int ty_ = r_ % P.tiles_y, b_ = r_ / P.tiles_y;
    if (pipe) tma_expect(&s_mbar_i, kBytesI);
    tma_load_3d(pipe ? &s_mbar_i : &s_mbar, sI0, &P.ixy_map, 2 * (tx_ * C::TW - C::IX), (ty_ * C::TH - C::RG) / 2, b_ * 2,
                C::PI, C::EH / 2, 2);
  };

  if (P.use_tma && tid == 0) { tma_barrier_init(&s_mbar); tma_barrier_init(&s_mbar_i); }
  pdl_wait();  // ds and ixy come from the forward kernel, grad_out from the autograd op before this launch
  pdl_trigger();
  if (P.use_tma && tid == 0 && (int)blockIdx.x < ntiles) { issue_s(blockIdx.x); issue_i(blockIdx.x); }
  if (P.use_tma) __syncthreads();  // the barriers are initialised before anyone polls them

  unsigned parity = 0;
#pragma unroll 1
  for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x, parity ^= 1u) {
  const int next = tile + (int)gridDim.x;
  const int tx = tile % P.tiles_x;
  const int trow = tile / P.tiles_x;
  const int ty = trow % P.tiles_y;
  const int b = trow / P.tiles_y;
  const int y0 = ty * C::TH, x0 = tx * C::TW;
  const size_t img_off = (size_t)b * 3 * plane;
  const int xv0 = x0 - C::HXE - C::HXK + C::VE;  // first V column
  const int xs0 = x0 - C::SX;                     // first staged column (V column SX0)
  const int yv0 = y0 - C::RG - C::RK;             // first staged row
  const int xi0 = x0 - C::IX;                     // first staged Ix, Iy column (E column EC0)
  const int qe0 = (y0 - C::RG) / 2;      // first E-region row pair (y0 - RG is even; may be -RG/2)

  // Stage the three ds planes (+halo) and the saved Ix, Iy tile.  Preferred path: two TMA box copies
  // issued by one thread (elements outside the tensors are zero-filled by the hardware = the zero padding
  // of the adjoint smoothing, and Ix = Iy = 0 outside the image); otherwise plain loads.
  if (P.use_tma) {
    tma_wait(&s_mbar, parity);
  } else {
    const float* dsb = P.ds + img_off;
    for (int it = tid; it < 3 * C::SH * C::SW; it += C::NT) {
      const int sx = it % C::SW, rc = it / C::SW;
      const int r = rc % C::SH, c = rc / C::SH;
      const int gy = yv0 + r, gx = xs0 + sx;
      sS[it] = (gy >= 0 && gy < H && gx >= 0 && gx < W) ? __ldg(dsb + c * plane + (size_t)gy * W + gx) : 0.f;
    }
    const int Hp = (H + 1) >> 1;
    for (int it = tid; it < 2 * (C::EH / 2) * C::PI; it += C::NT) {
      const int e = it % C::PI, rc = it / C::PI;
      const int qq = rc % (C::EH / 2), pl = rc / (C::EH / 2);
      const int gp = qe0 + qq, gx = xi0 + (e >> 1);
      sI0[it] = (gp >= 0 && gp < Hp && gx >= 0 && gx < W) ? __ldg(P.ixy + ixy_offset(b, pl, Hp, W, gp, gx) + (e & 1)) : 0.f;
    }
    __syncthreads();
  }

  // Phase C': vertical rho-pass of the three staged ds planes; a lane owns one column and RS rows.
  // The adjoint of the zero-padded symmetric smoothing is the same zero-padded smoothing.
  {
    const int c_lo = max(0, -xv0), c_hi = min(C::SX0 + C::SW, W - xv0);
    const int ncol = c_hi - c_lo;
    const int nclr = C::VW - ncol;
    for (int it = tid; it < nclr * (C::EH / 2); it += C::NT) {
      const int q = it / nclr, u = it - q * nclr;
      const int vx = (u < c_lo) ? u : (c_hi + (u - c_lo));
#pragma unroll
      for (int c = 0; c < 3; ++c) st2(sV + c * C::V_FLOATS + q * C::PV + 2 * vx, make_float2(0.f, 0.f));
    }
    // one item = (plane, row segment, column): the three ds planes are independent, so splitting them
    // over threads costs nothing and keeps every lane busy (ncol * NSEG alone is < NT for most tiles)
    for (int it = tid; it < 3 * ncol * C::NSEG; it += C::NT) {
      const int cs = it / ncol, vx = c_lo + (it - cs * ncol);
      const int c = cs / C::NSEG, seg = cs - c * C::NSEG;
      float2 acc[C::RS / 2];
#pragma unroll
      for (int j = 0; j < C::RS / 2; ++j) acc[j] = make_float2(0.f, 0.f);
      const float* p = sS + (c * C::SH + seg * C::RS) * C::SW + vx - C::SX0;
#pragma unroll
      for (int r = 0; r < C::RS + 2 * C::RK; ++r) {
        const float v = p[r * C::SW];
#pragma unroll
        for (int jp = 0; jp < C::RS / 2; ++jp) {
          const int u = r - 2 * jp;
          if (u >= 0 && u <= 2 * C::RK + 1) acc[jp] = ffma2(bcast2(v), tp.kp[u], acc[jp]);
        }
      }
      float* o = sV + c * C::V_FLOATS + (seg * (C::RS / 2)) * C::PV + 2 * vx;
#pragma unroll
      for (int jp = 0; jp < C::RS / 2; ++jp) st2(o + jp * C::PV, acc[jp]);
    }
  }
  __syncthreads();  // the staging is dead from here on: sdI may overwrite it / the next tile's ds box may land in it
  if (pipe) {
    if (tid == 0 && next < ntiles) { fence_async_smem(); issue_s(next); }
    tma_wait(&s_mbar_i, parity);
  }

  // Phase D': horizontal rho-pass -> E = K*ds at the E-region pixels, then the product rule
  //   dIx = 2 Ix Exx + Iy Exy ,  dIy = 2 Iy Eyy + Ix Exy      (adjoint of utils.py:225-229)
  if constexpr (C::XFULL) {  // the E columns outside the image: dIx = dIy = 0
    constexpr int NZ = C::EW - C::ECW;
    for (int it = tid; it < 2 * NZ * (C::EH / 2); it += C::NT) {
      const int pl = it / (NZ * (C::EH / 2)), r = it - pl * (NZ * (C::EH / 2));
      const int q = r / NZ, u = r - q * NZ;
      const int e = u < C::EC0 ? u : C::ECW + u;
      st2((pl ? sdI1 : sdI0) + q * C::PE + 2 * e, make_float2(0.f, 0.f));
    }
  }
  for (int it = tid; it < C::MapD::SLOTS; it += C::NT) {
    int q, seg;
    if (!C::MapD::decode(it, q, seg)) continue;
    const int ex0 = C::EC0 + C::CSD * seg, ix0 = C::CSD * seg;
    float2 E[3][C::CSD];
#pragma unroll
    for (int c = 0; c < 3; ++c)
      smooth_h_rowpair_n<C::RK, C::CSD, C::DWIN, C::HXK - C::DW_LO>(
          sV + c * C::V_FLOATS + q * C::PV + 2 * (ex0 - C::VE + C::DW_LO), tp, E[c]);
    float* o0 = sdI0 + q * C::PE + 2 * ex0;
    float* o1 = sdI1 + q * C::PE + 2 * ex0;
#pragma unroll
    for (int m = 0; m < C::CSD / 2; ++m) {  // two columns per LDS.128 / STS.128
      const float4 ixv = ld4(sI0 + q * C::PI + 2 * ix0 + 4 * m), iyv = ld4(sI1 + q * C::PI + 2 * ix0 + 4 * m);
      const float2 ix[2] = {make_float2(ixv.x, ixv.y), make_float2(ixv.z, ixv.w)};
      const float2 iy[2] = {make_float2(iyv.x, iyv.y), make_float2(iyv.z, iyv.w)};
      float2 dx[2], dy[2];
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const int j = 2 * m + h;
        const float2 ix2 = make_float2(2.0f * ix[h].x, 2.0f * ix[h].y), iy2 = make_float2(2.0f * iy[h].x, 2.0f * iy[h].y);
        dx[h] = ffma2(ix2, E[0][j], make_float2(iy[h].x * E[2][j].x, iy[h].y * E[2][j].y));
        dy[h] = ffma2(iy2, E[1][j], make_float2(ix[h].x * E[2][j].x, ix[h].y * E[2][j].y));
      }
      st4(o0 + 4 * m, make_float4(dx[0].x, dx[0].y, dx[1].x, dx[1].y));
      st4(o1 + 4 * m, make_float4(dy[0].x, dy[0].y, dy[1].x, dy[1].y));
    }
  }
  __syncthreads();
  if (pipe && tid == 0 && next < ntiles) { fence_async_smem(); issue_i(next); }  // Ix, Iy of this tile are consumed

  // Phase E': adjoint of the derivative filters.  The adjoint of a zero-padded correlation is the
  // correlation with flipped taps; g is symmetric and dg antisymmetric, so
  //   dgray = -[ (dIx * dg|) * g-  +  (dIy * g|) * dg- ]
  // i.e. the forward gradient operators applied to dIx and dIy, negated.
  const float scale = -__ldg(P.grad_out + (PER_IMG ? b : 0)) * P.inv_count;
  [[maybe_unused]] const float px_scale = PX ? __ldg(P.grad_px + (PER_IMG ? b : 0)) * P.inv_count * (2.0f / 3.0f) : 0.f;
  for (int it = tid; it < C::MapE::SLOTS; it += C::NT) {
    int q, seg;
    if (!C::MapE::decode(it, q, seg)) continue;
    const int ox0 = 4 * seg;
    const int gy = y0 + 2 * q, gx0 = x0 + ox0;
    if (gy >= H || gx0 >= W) continue;
    float2 ax[4], ay[4];
    grad_rowpair<C::RG, 4, C::BWIN, C::HXE - C::BW_LO, C::PE, false>(sdI0 + q * C::PE + 2 * (ox0 + C::BW_LO),
                                                                   sdI1 + q * C::PE + 2 * (ox0 + C::BW_LO), tp, ax, ay);
    const float coef[3] = {kGrayR, kGrayG, kGrayB};
#pragma unroll
    for (int hf = 0; hf < 2; ++hf) {
      if (gy + hf >= H) continue;
      float dgr[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) dgr[j] = ((hf ? ax[j].y : ax[j].x) + (hf ? ay[j].y : ay[j].x)) * scale;
      float* o = P.d_img + img_off + (size_t)(gy + hf) * W + gx0;
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        if (P.vec4) {
          float4 r = make_float4(coef[c] * dgr[0], coef[c] * dgr[1], coef[c] * dgr[2], coef[c] * dgr[3]);
          if constexpr (PX) {  // fused Pixel term: d MSE / d img = 2 (img - other) / (3 B H W)
            const size_t e = img_off + (size_t)(gy + hf) * W + gx0 + c * plane;
            const float4 a = ldg4(P.img + e), b4 = ldg4(P.px_other + e);
            r.x = fmaf(px_scale, a.x - b4.x, r.x); r.y = fmaf(px_scale, a.y - b4.y, r.y);
            r.z = fmaf(px_scale, a.z - b4.z, r.z); r.w = fmaf(px_scale, a.w - b4.w, r.w);
          }
          st4(o + c * plane, r);
        } else {
#pragma unroll
          for (int j = 0; j < 4; ++j)
            if (gx0 + j < W) {
              float r = coef[c] * dgr[j];
              if constexpr (PX) {
                const size_t e = img_off + (size_t)(gy + hf) * W + gx0 + j + c * plane;
                r = fmaf(px_scale, __ldg(P.img + e) - __ldg(P.px_other + e), r);
              }
              o[c * plane + j] = r;
            }
        }
      }
    }
  }
    if (!pipe) {
      __syncthreads();  // every thread is done with dIx|dIy (over the staging) and Ix, Iy: the next tile may be staged
      if (P.use_tma && tid == 0 && next < ntiles) { fence_async_smem(); issue_s(next); issue_i(next); }
    }
  }  // tile loop
}

// Backward prepass of the distance map (srst_st_backward_map): out[b][c] = grad_map[b] * ds[b][c] for the three ds
// planes, and *unit = 1.  The unchanged backward then runs on `out` with `unit` as its upstream gradient and a unit
// scale, so d_img is the adjoint of grad_map * ds.  VEC4: W % 4 == 0 and all three pointers 16-byte aligned.
constexpr int kMapNT = 256;
template <bool VEC4>
__global__ void __launch_bounds__(kMapNT) st_map_scale_kernel(const float* __restrict__ ds,
                                                              const float* __restrict__ grad_map, float* __restrict__ out,
                                                              float* __restrict__ unit, int B, size_t plane) {
  pdl_wait();  // grad_map may come from the kernel enqueued just before
  pdl_trigger();
  if (blockIdx.x == 0 && threadIdx.x == 0) *unit = 1.0f;
  constexpr int V = VEC4 ? 4 : 1;
  const size_t n = (size_t)B * plane / V;
  for (size_t i = (size_t)blockIdx.x * kMapNT + threadIdx.x; i < n; i += (size_t)gridDim.x * kMapNT) {
    const size_t p = i * V, b = p / plane, o = p + 2 * b * plane;  // o: channel 0 of pixel p in [B][3][H][W]
    if constexpr (VEC4) {
      const float4 g = ldg4(grad_map + p);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float4 v = ldg4(ds + o + c * plane);
        st4(out + o + c * plane, make_float4(g.x * v.x, g.y * v.y, g.z * v.z, g.w * v.w));
      }
    } else {
      const float g = __ldg(grad_map + p);
#pragma unroll
      for (int c = 0; c < 3; ++c) out[o + c * plane] = g * __ldg(ds + o + c * plane);
    }
  }
}

}  // namespace srst
