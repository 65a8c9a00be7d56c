// Best-Buddy loss kernels for sm_100a.
//
// Reference (loss.py:115-141, utils.py:173-187): unfold 3x3/stride-3 patches of SR and HR, build an
// HR candidate set from three pyramid levels, materialise two [B,N,M] fp32 distance matrices with
// torch.bmm, take torch.min over M, gather, L1.  Here the [B,N,M] matrices never exist:
//
//   bb_pyramid_kernel : bicubic x1/2 and x1/4 levels of HR (same taps as F.interpolate(bicubic,
//                       align_corners=False): t = 0.5 on both levels)                (loss.py:123,127)
//   bb_pack_kernel    : patches -> k-major fp32 matrices Q1 (SR), Q2 (HR), Y (candidates) + norms
//   bb_search_kernel  : register-tiled fp32 distance evaluation fused with a running argmin;
//                       per-thread argmin over its candidates, warp-shuffle argmin across lanes,
//                       shared-memory argmin across warps; first minimal index wins (torch.min)
//   bb_loss_kernel    : mean |sr_patch - cand[idx]| (or squared), deterministic reduction
//   bb_backward_kernel: d_sr = grad/(B*N*27) * sign(sr_patch - cand[idx])  (or 2*diff)
//
// The score is evaluated with exactly the reference's expression and rounding points,
//   alpha * max((xn + yn) - 2*dot1, 0) + beta * max((gn + yn) - 2*dot2, 0),
// with a fixed fp32 order for the 27-term dot products and norms (sequential FMA, k = 0..26;
// oracle/bb_oracle.c restates the same order so indices can be compared bit-exactly).
//
// The same pack / search / loss kernels serve three descriptor MODEs: 0 = raw 27 patch values
// (BestBuddyLoss), 1 = 3x3 Gram matrix (GramLoss, loss.py:146-225), 2 = det-normalised structure
// tensor of the 3x3 grayscale patch (PatchwiseStructureTensorLoss, loss.py:292-375).
#pragma once
#include <cstdint>

#include "srst_device.cuh"

namespace srst {

constexpr int BB_D = 27;   // 3 channels x 3 x 3
constexpr int BB_QT = 128;  // queries per block
constexpr int BB_CT = 128;  // candidates per chunk
constexpr int BB_NT = 256;

struct BbGeom {
  int B, H, W;
  int n0x, N0;          // level 0 patch grid
  int H2, W2, n2x, N2;  // x1/2
  int H4, W4, n4x, N4;  // x1/4
  int N, M, Npad, Mpad;
};

inline BbGeom bb_geom(int B, int H, int W) {
  BbGeom g;
  g.B = B; g.H = H; g.W = W;
  g.n0x = W / 3; g.N0 = (H / 3) * g.n0x;
  g.H2 = H / 2; g.W2 = W / 2; g.n2x = g.W2 / 3; g.N2 = (g.H2 / 3) * g.n2x;
  g.H4 = H / 4; g.W4 = W / 4; g.n4x = g.W4 / 3; g.N4 = (g.H4 / 3) * g.n4x;
  g.N = g.N0;
  g.M = g.N0 + g.N2 + g.N4;
  g.Npad = (g.N + BB_QT - 1) / BB_QT * BB_QT;
  g.Mpad = (g.M + BB_CT - 1) / BB_CT * BB_CT;
  return g;
}

// Workspace carve-up (floats).  Per image: Q1[27][Npad] Q2[27][Npad] Y[27][Mpad] xn[Npad] gn[Npad] yn[Mpad]
struct BbWorkspace {
  unsigned int* ticket;
  float* partials;
  float* mats;
  float* pyr2;
  float* pyr4;
  size_t per_image;  // floats
  size_t total_bytes;
};

inline BbWorkspace bb_carve(void* base, const BbGeom& g, int D = BB_D) {
  BbWorkspace w;
  char* p = reinterpret_cast<char*>(base);
  size_t off = 0;
  w.ticket = reinterpret_cast<unsigned int*>(p + off);
  off += 256;
  const size_t nblk_loss = ((size_t)g.B * g.N + BB_NT - 1) / BB_NT;
  w.partials = reinterpret_cast<float*>(p + off);
  off += (nblk_loss * sizeof(float) + 255) / 256 * 256;
  w.per_image = (size_t)(D + 1) * (2 * (size_t)g.Npad + g.Mpad);
  w.mats = reinterpret_cast<float*>(p + off);
  off += (w.per_image * g.B * sizeof(float) + 255) / 256 * 256;
  w.pyr2 = reinterpret_cast<float*>(p + off);
  off += ((size_t)g.B * 3 * g.H2 * g.W2 * sizeof(float) + 255) / 256 * 256;
  w.pyr4 = reinterpret_cast<float*>(p + off);
  off += ((size_t)g.B * 3 * g.H4 * g.W4 * sizeof(float) + 255) / 256 * 256;
  w.total_bytes = off;
  return w;
}

struct BbPtrs {
  const float* q1; const float* q2; const float* y; const float* xn; const float* gn; const float* yn;
};
SRST_DEV BbPtrs bb_image_ptrs(const float* mats, size_t per_image, int b, int Npad, int Mpad, int D = BB_D) {
  const float* m = mats + per_image * b;
  BbPtrs p;
  p.q1 = m;
  p.q2 = p.q1 + (size_t)D * Npad;
  p.y = p.q2 + (size_t)D * Npad;
  p.xn = p.y + (size_t)D * Mpad;
  p.gn = p.xn + Npad;
  p.yn = p.gn + Npad;
  return p;
}

// ---- HR pyramid ---------------------------------------------------------------------------------
// F.interpolate(gt, scale_factor=s, mode='bicubic', align_corners=False), s = 1/2 and 1/4: the source
// coordinate (dst + 0.5)/s - 0.5 always has fractional part 0.5, so the cubic-convolution (A=-0.75)
// weights are the constants below, applied to rows/cols 2i-1..2i+2 (x1/2) or 4i..4i+3 (x1/4) with
// indices clamped to the image.
SRST_DEV float bb_cubic4(float a, float b, float c, float d) {
  constexpr float w0 = -0.09375f, w1 = 0.59375f;
  return ((a * w0 + b * w1) + c * w1) + d * w0;
}

__global__ void __launch_bounds__(256)
bb_pyramid_kernel(const float* __restrict__ gt, float* __restrict__ o2, float* __restrict__ o4, int planes, int H,
                  int W, int H2, int W2, int H4, int W4) {
  const size_t n2 = (size_t)planes * H2 * W2, n4 = (size_t)planes * H4 * W4;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n2 + n4) return;
  const bool lvl4 = t >= n2;
  const size_t u = lvl4 ? t - n2 : t;
  const int Ho = lvl4 ? H4 : H2, Wo = lvl4 ? W4 : W2;
  const int x = (int)(u % Wo);
  const int y = (int)((u / Wo) % Ho);
  const int pl = (int)(u / ((size_t)Wo * Ho));
  const int sy = lvl4 ? 4 * y : 2 * y - 1;
  const int sx = lvl4 ? 4 * x : 2 * x - 1;
  const float* src = gt + (size_t)pl * H * W;
  float r[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int yy = min(max(sy + i, 0), H - 1);
    const float* row = src + (size_t)yy * W;
    const float a = __ldg(row + min(max(sx, 0), W - 1));
    const float b = __ldg(row + min(max(sx + 1, 0), W - 1));
    const float c = __ldg(row + min(max(sx + 2, 0), W - 1));
    const float d = __ldg(row + min(max(sx + 3, 0), W - 1));
    r[i] = bb_cubic4(a, b, c, d);
  }
  (lvl4 ? o4 : o2)[u] = bb_cubic4(r[0], r[1], r[2], r[3]);
}

// ---- pack ---------------------------------------------------------------------------------------
// Patch vector layout (F.unfold, loss.py:116): element c*9 + ky*3 + kx; patch index py*(W/3) + px.
SRST_DEV void bb_read_patch(const float* __restrict__ img, int H, int W, int nx, int p, float (&v)[BB_D]) {
  const int py = p / nx, px = p - py * nx;
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int ky = 0; ky < 3; ++ky)
#pragma unroll
      for (int kx = 0; kx < 3; ++kx)
        v[c * 9 + ky * 3 + kx] = __ldg(img + ((size_t)c * H + 3 * py + ky) * W + 3 * px + kx);
}
template <int D>
SRST_DEV float bb_norm(const float (&v)[D]) {
  float n = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) n = fmaf(v[k], v[k], n);
  return n;
}

// Gram descriptor of a 3x3x3 patch (reference loss.py:180-184 gram_matrix): features = patch viewed
// as [3 channels][9], G = F F^T / 27, flattened row-major to 9 values.  Fixed order: sequential fma
// over the 9 positions, then a division by 27 (oracle/bb_oracle.c restates the same order).
SRST_DEV void bb_gram(const float (&v)[BB_D], float (&gm)[9]) {
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int b = 0; b < 3; ++b) {
      float s = 0.f;
#pragma unroll
      for (int t = 0; t < 9; ++t) s = fmaf(v[a * 9 + t], v[b * 9 + t], s);
      gm[a * 3 + b] = s / 27.0f;
    }
}


// ---- PatchwiseStructureTensorLoss descriptor (reference loss.py:325-345 s_norm / compute_patches) ----
// Every 3x3x3 patch is treated as a 3x3 IMAGE: Grayscale -> utils.structure_tensor(sigma, rho) with
// zero 'same' padding -> utils.normalize.  On a 3x3 image only the five central taps of each filter
// can touch a pixel, so a separable pass is a 3x3 banded matrix product:
//   vert(w, X)[i][x] = sum_j w[j-i+2] X[j][x]      horz(w, X)[i][x] = sum_j w[j-x+2] X[i][j]
// (cross-correlation like conv2d, utils.py:219-230).  Descriptor element c*9 + i*3 + x with c in
// (Jxx, Jyy, Jxy) / sqrt(det + 1e-12).  Every operation is an explicitly rounded fp32 op in a fixed
// order (oracle/bb_oracle.c restates it), so the search indices are bit-comparable.
struct PstTaps {
  float g[5], dg[5], k[5];  // central taps (offset -2..2) of Gaussian(sigma), its derivative, Gaussian(rho)
};
constexpr float kPstEps = 1e-12f;  // utils.normalize default (utils.py:236)

SRST_DEV void pst_vert(const float (&w)[5], const float (&X)[9], float (&o)[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 3; ++j) s = fmaf(w[j - i + 2], X[j * 3 + x], s);
      o[i * 3 + x] = s;
    }
}
SRST_DEV void pst_horz(const float (&w)[5], const float (&X)[9], float (&o)[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      float s = 0.f;
#pragma unroll
      for (int j = 0; j < 3; ++j) s = fmaf(w[j - x + 2], X[i * 3 + j], s);
      o[i * 3 + x] = s;
    }
}
// adjoints: vertT(w, dO)[j][x] = sum_i w[j-i+2] dO[i][x] ; horzT(w, dO)[i][j] = sum_x w[j-x+2] dO[i][x]
SRST_DEV void pst_vert_t(const float (&w)[5], const float (&dO)[9], float (&o)[9]) {
#pragma unroll
  for (int j = 0; j < 3; ++j)
#pragma unroll
    for (int x = 0; x < 3; ++x) {
      float s = 0.f;
#pragma unroll
      for (int i = 0; i < 3; ++i) s = fmaf(w[j - i + 2], dO[i * 3 + x], s);
      o[j * 3 + x] = s;
    }
}
SRST_DEV void pst_horz_t(const float (&w)[5], const float (&dO)[9], float (&o)[9]) {
#pragma unroll
  for (int i = 0; i < 3; ++i)
#pragma unroll
    for (int j = 0; j < 3; ++j) {
      float s = 0.f;
#pragma unroll
      for (int x = 0; x < 3; ++x) s = fmaf(w[j - x + 2], dO[i * 3 + x], s);
      o[i * 3 + j] = s;
    }
}

// Gradients and raw structure tensor of one patch (v = 27 patch values, element c*9 + y*3 + x).
struct PstState {
  float Ix[9], Iy[9], J[3][9], q[9];  // q = sqrt(det + eps)
};
SRST_DEV void pst_state(const float (&v)[BB_D], const PstTaps& tp, PstState& S) {
  float gray[9], t[9], p[9];
#pragma unroll
  for (int i = 0; i < 9; ++i)
    gray[i] = __fadd_rn(__fadd_rn(__fmul_rn(kGrayR, v[i]), __fmul_rn(kGrayG, v[9 + i])), __fmul_rn(kGrayB, v[18 + i]));
  pst_vert(tp.dg, gray, t); pst_horz(tp.g, t, S.Ix);   // utils.py:219-220
  pst_vert(tp.g, gray, t);  pst_horz(tp.dg, t, S.Iy);  // utils.py:221-222
#pragma unroll
  for (int c = 0; c < 3; ++c) {
#pragma unroll
    for (int i = 0; i < 9; ++i) p[i] = __fmul_rn(c == 1 ? S.Iy[i] : S.Ix[i], c == 0 ? S.Ix[i] : S.Iy[i]);
    pst_vert(tp.k, p, t);
    pst_horz(tp.k, t, S.J[c]);                         // utils.py:225-230
  }
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    const float det = __fsub_rn(__fmul_rn(S.J[0][i], S.J[1][i]), __fmul_rn(S.J[2][i], S.J[2][i]));
    S.q[i] = __fsqrt_rn(__fadd_rn(det, kPstEps));      // utils.py:238-239
  }
}
SRST_DEV void pst_descriptor(const float (&v)[BB_D], const PstTaps& tp, float (&d)[BB_D]) {
  PstState S;
  pst_state(v, tp, S);
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int i = 0; i < 9; ++i) d[c * 9 + i] = __fdiv_rn(S.J[c][i], S.q[i]);
}

// Descriptor of a patch: MODE 0 = the 27 raw values (BestBuddyLoss), MODE 1 = Gram matrix (GramLoss),
// MODE 2 = normalised structure tensor of the patch (PatchwiseStructureTensorLoss).
template <int MODE>
struct BbDesc {
  static constexpr int D = MODE == 1 ? 9 : BB_D;
  SRST_DEV static void make(const float (&v)[BB_D], const PstTaps& tp, float (&d)[D]) {
    if constexpr (MODE == 0) {
#pragma unroll
      for (int k = 0; k < BB_D; ++k) d[k] = v[k];
    } else if constexpr (MODE == 1) {
      bb_gram(v, d);
    } else {
      pst_descriptor(v, tp, d);
    }
  }
};

template <int MODE>
__global__ void __launch_bounds__(256)
bb_pack_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
               const float* __restrict__ gt4, float* __restrict__ mats, size_t per_image, BbGeom g, PstTaps tp) {
  constexpr int D = BbDesc<MODE>::D;
  const int b = blockIdx.y;
  const int t = blockIdx.x * blockDim.x + threadIdx.x;
  float* m = mats + per_image * b;
  float* q1 = m;
  float* q2 = q1 + (size_t)D * g.Npad;
  float* y = q2 + (size_t)D * g.Npad;
  float* xn = y + (size_t)D * g.Mpad;
  float* gn = xn + g.Npad;
  float* yn = gn + g.Npad;
  float v[BB_D], d[D];
  if (t < g.Npad) {  // query t
    if (t < g.N) {
      bb_read_patch(sr + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, t, v);
      BbDesc<MODE>::make(v, tp, d);
#pragma unroll
      for (int k = 0; k < D; ++k) q1[(size_t)k * g.Npad + t] = d[k];
      xn[t] = bb_norm<D>(d);
      bb_read_patch(gt + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, t, v);
      BbDesc<MODE>::make(v, tp, d);
#pragma unroll
      for (int k = 0; k < D; ++k) q2[(size_t)k * g.Npad + t] = d[k];
      gn[t] = bb_norm<D>(d);
    } else {
#pragma unroll
      for (int k = 0; k < D; ++k) { q1[(size_t)k * g.Npad + t] = 0.f; q2[(size_t)k * g.Npad + t] = 0.f; }
      xn[t] = 0.f;
      gn[t] = 0.f;
    }
  }
  if (t < g.Mpad) {  // candidate t: level 0 | level 1/2 | level 1/4 (torch.cat order, loss.py:130)
    if (t < g.M) {
      if (t < g.N0) bb_read_patch(gt + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, t, v);
      else if (t < g.N0 + g.N2) bb_read_patch(gt2 + (size_t)b * 3 * g.H2 * g.W2, g.H2, g.W2, g.n2x, t - g.N0, v);
      else bb_read_patch(gt4 + (size_t)b * 3 * g.H4 * g.W4, g.H4, g.W4, g.n4x, t - g.N0 - g.N2, v);
      BbDesc<MODE>::make(v, tp, d);
#pragma unroll
      for (int k = 0; k < D; ++k) y[(size_t)k * g.Mpad + t] = d[k];
      yn[t] = bb_norm<D>(d);
    } else {
#pragma unroll
      for (int k = 0; k < D; ++k) y[(size_t)k * g.Mpad + t] = 0.f;
      yn[t] = __int_as_float(0x7f800000);  // +inf: a padded candidate never wins
    }
  }
}

// ---- search -------------------------------------------------------------------------------------
SRST_DEV float bb_score(float xn, float gn, float yn, float dot1, float dot2, float alpha, float beta) {
  // utils.py:183-187 with its rounding points: (x_norm + y_norm) - 2*bmm, clamp(0, inf);
  // loss.py:132-133: alpha*d1 + beta*d2 (separate multiply and add roundings).
  float d1 = fmaf(-2.0f, dot1, __fadd_rn(xn, yn));
  float d2 = fmaf(-2.0f, dot2, __fadd_rn(gn, yn));
  d1 = (d1 < 0.0f) ? 0.0f : d1;  // torch.clamp(min=0) keeps NaN (fmaxf would drop it)
  d2 = (d2 < 0.0f) ? 0.0f : d2;
  return __fadd_rn(__fmul_rn(alpha, d1), __fmul_rn(beta, d2));
}

// torch.min order (loss.py:135): a NaN score is "smaller" than every number, the first NaN wins, ties go to the
// lowest index.  (score, index) pairs merge lexicographically under that order.
SRST_DEV bool bb_score_before(float so, int io, float s, int i) {
  const bool nan_o = so != so, nan_s = s != s;
  if (nan_o || nan_s) return nan_o && (!nan_s || io < i);
  return so < s || (so == s && io < i);
}
SRST_DEV void bb_argmin_merge(float& s, int& i, float so, int io) {
  if (bb_score_before(so, io, s, i)) { s = so; i = io; }
}

// Search kernel: a cheap single-dot FILTER in front of the exact score.
//
// With q_i = alpha*x_i + beta*g_i, c_i = alpha*|x_i|^2 + beta*|g_i|^2 and (alpha+beta)*|y_j|^2, the score is, in
// real arithmetic, S_ij = c_i + (alpha+beta)|y_j|^2 - 2 q_i.y_j : ONE 27-term dot product per pair
// instead of the reference's two.  Its fp32 value s'_ij is not the reference's rounding, so it is only
// used to DISCARD candidates: both s'_ij and the exactly-rounded reference score s_ij (bb_score, the
// fixed-order restatement of utils.py:183-187 / loss.py:132-133) lie within
//     tol_ij = kappa * (|alpha|(|x_i|^2+|y_j|^2) + |beta|(|g_i|^2+|y_j|^2)),   kappa = 2e-5  (>= 120 ulp:
// 27-term fp32 dot products and norms accumulate <= 30 ulp each relative to that magnitude) of S_ij.
// Every thread keeps, per query, an upper bound B >= min_j s_ij (seeded with the exact score of the
// co-located HR patch j = i, tightened by every exact score it computes); a candidate whose lower
// bound s'_ij - tol_ij exceeds B cannot be the argmin, nor tie with it, and is skipped.  The few
// that survive are re-scored EXACTLY (two sequential-fma dot products, the oracle's order), in
// ascending j per thread with a strict <, and (score, index) pairs are merged lexicographically, so
// the result is bit-identical to scoring every pair exactly: same indices, same first-minimum rule.
//
// 256 threads as 16 x 16, each owning 8 queries x 8 candidates (two groups of 4 each, 64 apart: a
// quarter-warp reads 128 contiguous bytes per LDS.128): 64 accumulators fed by packed FFMA2 on
// query PAIRS, one byte of shared-memory traffic per FMA (the 4x4 two-dot tile needed 1.5-2 and was
// bound by the shared-memory pipe, profiles/README.md).  Candidate chunks are double-buffered
// through registers; the 16 threads that share a query set sit in one half-warp, so the final
// argmin is four warp-shuffle steps.
constexpr float kBbKappa = 2e-5f;

// The filter compares lo' = yl_j - 2 acc_ij with Bc_i instead of cl_i + lo' with B_i.  With F = fl(B - cl),
// Bc = F + 6e-7 |F| guarantees  lo' > Bc  =>  cl + yl - 2 acc > B  in real arithmetic on the fp32 operands (the two
// roundings involved, of lo' and of F, are each below 1.2e-7 of max(|lo'|, |F|), and |lo'| > |F| only where the margin
// is not needed).  B = -inf (padded queries: nothing is ever evaluated) stays -inf; a NaN bound stays NaN (= always hit).
SRST_DEV float bb_shifted_bound(float B, float cl) {
  const float F = B - cl;
  return (B == __int_as_float(0xff800000)) ? B : fmaf(6e-7f, fabsf(F), F);
}

// Exact reference-order score of (query qi, candidate cj) of one image (the seed of the bound and the survivors' path):
// all 3 D operands are loaded up front (independent loads: one L1/L2 round trip instead of D dependent ones), then the
// two sequential-fma chains run in the oracle's order.
template <int D>
SRST_DEV float bb_exact_score_unrolled(const float* q1, const float* q2, const float* y, const float* xn, const float* gn,
                                       const float* yn, int Npad, int Mpad, int qi, int cj, float alpha, float beta) {
  float a[D], b[D], w[D];
#pragma unroll
  for (int k = 0; k < D; ++k) {
    w[k] = __ldg(y + (size_t)k * Mpad + cj);
    a[k] = __ldg(q1 + (size_t)k * Npad + qi);
    b[k] = __ldg(q2 + (size_t)k * Npad + qi);
  }
  const float xq = __ldg(xn + qi), gq = __ldg(gn + qi), yc = __ldg(yn + cj);
  float dot1 = 0.f, dot2 = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    dot1 = fmaf(a[k], w[k], dot1);
    dot2 = fmaf(b[k], w[k], dot2);
  }
  return bb_score(xq, gq, yc, dot1, dot2, alpha, beta);
}

// SHARE: the 16 threads that own a query also pool their bound -- every chunk early on, every fourth
// later, B_i is lowered to the smallest UPPER bound s'_ij + tol_ij any of them saw in the chunk (four
// shuffle steps).  It costs ~8 % on descriptors whose co-located patch is already a tight seed
// (BestBuddy, Gram) and saves 25 % on PatchwiseST, whose noisy SR descriptors make the seed loose.
// Candidate chunks go through a shared-memory ring guarded by counting mbarriers ("full": every thread's cp.async
// copies of the stage have landed; "empty": every thread is done reading it).  Round 1 used two buffers, register
// staging and one CTA barrier per chunk: ptxas sank the prefetch loads below the FFMA2 block (their L2 latency sat in
// front of every barrier) and a warp with survivors to re-score stalled the other seven (Gram: 21 % of the warp time at
// that barrier).  Now there is no CTA barrier in the loop and warps may drift up to kBbAhead chunks apart.
// Stages: 4 for 27-dimensional descriptors, 8 for 9-dimensional ones (measured: Gram 1.23 -> 1.21 ms with 8,
// BestBuddy / PatchwiseST 1-3 % slower); a thread copies kBbAhead = stages / 2 chunks ahead of the one it scores.
constexpr int kBbMaxStages = 8;
template <int D> struct BbStages { static constexpr int value = D <= 9 ? 8 : 4; };
template <int D>
constexpr size_t bb_search_dyn_smem() { return sizeof(float) * BbStages<D>::value * (D + 1) * BB_CT; }

template <int D, bool SHARE = false>
__global__ void __launch_bounds__(BB_NT, 1)
bb_search_kernel(const float* __restrict__ mats, size_t per_image, BbGeom g, float alpha, float beta,
                 int64_t* __restrict__ idx_out) {
  static_assert(BB_NT == 256 && BB_QT == 128 && BB_CT == 128, "search tile is 16x16 threads x (8 queries x 8 candidates)");
  constexpr int kBbStages = BbStages<D>::value, kBbAhead = kBbStages / 2;
  SRST_DYN_SMEM(float, dyn);                          // [stages][D][BB_CT] candidates, then [stages][BB_CT] |y|^2
  __shared__ __align__(8) unsigned long long mb_full[kBbMaxStages], mb_empty[kBbMaxStages];
  __shared__ __align__(16) float sQ[D][BB_QT];      // alpha*x + beta*g
  // short descriptors (Gram): the survivors' exact re-scoring reads x, g (and y from the chunk buffer) from shared
  // memory -- with 9 dimensions nearly every chunk has a survivor per warp, and its global round trip was the chunk's
  // longest latency
  constexpr bool EXACT_SMEM = D <= 9;   // (PatchwiseST, 27-dim: no gain measured from the shared-memory copy)
  [[maybe_unused]] __shared__ __align__(16) float sX1[EXACT_SMEM ? D : 1][EXACT_SMEM ? BB_QT : 4];
  [[maybe_unused]] __shared__ __align__(16) float sX2[EXACT_SMEM ? D : 1][EXACT_SMEM ? BB_QT : 4];
  [[maybe_unused]] __shared__ __align__(16) float sXn[EXACT_SMEM ? 2 : 1][EXACT_SMEM ? BB_QT : 4];   // |x|^2, |g|^2
  float (*sY)[D][BB_CT] = reinterpret_cast<float (*)[D][BB_CT]>(dyn);
  float (*sYp)[BB_CT] = reinterpret_cast<float (*)[BB_CT]>(dyn + kBbStages * D * BB_CT);   // |y|^2 per stage
  __shared__ __align__(16) float sCl[BB_QT];        // c_i - kappa*(|alpha||x|^2 + |beta||g|^2)
  __shared__ __align__(16) float sB0[BB_QT];        // exact score of the co-located candidate j = i
  // SHARE only: 2*tol of a pair is at most 2 kappa (ca_i + max over the chunk's valid candidates of yt_j)
  [[maybe_unused]] __shared__ __align__(16) float sCa[SHARE ? BB_QT : 4];   // |alpha||x|^2 + |beta||g|^2
  __shared__ int sW[BB_NT / 32][64];   // per warp: queued survivors (tile query << 8 | chunk candidate), then their exact scores

  const int tid = threadIdx.x;
  const int b = blockIdx.y, qt = blockIdx.x;
  const BbPtrs P = bb_image_ptrs(mats, per_image, b, g.Npad, g.Mpad, D);
  const int qbase = qt * BB_QT;
  const float aa = fabsf(alpha), ab = fabsf(beta);

  for (int it = tid; it < D * (BB_QT / 4); it += BB_NT) {
    const int k = it / (BB_QT / 4), c4 = it - k * (BB_QT / 4);
    const float4 x = ldg4(P.q1 + (size_t)k * g.Npad + qbase + 4 * c4);
    const float4 gg = ldg4(P.q2 + (size_t)k * g.Npad + qbase + 4 * c4);
    st4(&sQ[k][4 * c4], make_float4(fmaf(alpha, x.x, beta * gg.x), fmaf(alpha, x.y, beta * gg.y),
                                    fmaf(alpha, x.z, beta * gg.z), fmaf(alpha, x.w, beta * gg.w)));
    if constexpr (EXACT_SMEM) { st4(&sX1[k][4 * c4], x); st4(&sX2[k][4 * c4], gg); }
  }
  if (tid < BB_QT) {
    const int qi = qbase + tid;
    const float xn = __ldg(P.xn + qi), gn = __ldg(P.gn + qi);
    if constexpr (EXACT_SMEM) { sXn[0][tid] = xn; sXn[1][tid] = gn; }
    sCl[tid] = fmaf(alpha, xn, beta * gn) - kBbKappa * fmaf(aa, xn, ab * gn);
    if constexpr (SHARE) sCa[tid] = fmaf(aa, xn, ab * gn);
    // seed of the upper bound; padded queries get -inf so that nothing is ever evaluated for them
    // (unrolled: all operands in flight at once -- the rolled loop paid D dependent L2 round trips, ~8 us per CTA)
    sB0[tid] = (qi < g.N) ? bb_exact_score_unrolled<D>(P.q1, P.q2, P.y, P.xn, P.gn, P.yn, g.Npad, g.Mpad, qi, qi, alpha, beta)
                          : __int_as_float(0xff800000);
  }

  const int ty = tid >> 4, tx = tid & 15;  // 16 x 16 threads; a half-warp shares ty (its queries)
  // local query l (0..7) -> tile query ty*4 + (l&3) + 64*(l>>2); same for candidates with tx

  const int nchunks = g.Mpad / BB_CT;
  // chunk c lives in stage c % kBbStages (its (c / kBbStages)-th use); every thread copies its share of the chunk
  // (D * BB_CT / 4 16-byte pieces over BB_NT threads) and arrives on the stage's "full" barrier once its copies have landed
  auto pipe_load = [&](int c) {
    const int st = c % kBbStages, chunk = c * BB_CT;
    for (int it = tid; it < D * (BB_CT / 4); it += BB_NT) {
      const int k = it / (BB_CT / 4), c4 = it - k * (BB_CT / 4);
      cp_async16(&sY[st][k][4 * c4], P.y + (size_t)k * g.Mpad + chunk + 4 * c4, true);
    }
    if (tid < BB_CT) cp_async4(&sYp[st][tid], P.yn + chunk + tid);
    cp_async_mbar_arrive(&mb_full[st]);
  };
  if (tid == 0)
    for (int st = 0; st < kBbStages; ++st) { mbar_init(&mb_full[st], BB_NT); mbar_init(&mb_empty[st], BB_NT); }
  __syncthreads();  // the barriers are initialised before anyone arrives on them; queries and bounds are in shared memory
  for (int c = 0; c < kBbAhead && c < nchunks; ++c) pipe_load(c);

  float best[8], B[8], Bc[8], clq[8];
  int bidx[8];
  {
    const float4 c0 = ld4(&sCl[4 * ty]), c1 = ld4(&sCl[64 + 4 * ty]);
    const float4 b0 = ld4(&sB0[4 * ty]), b1 = ld4(&sB0[64 + 4 * ty]);
    clq[0] = c0.x; clq[1] = c0.y; clq[2] = c0.z; clq[3] = c0.w; clq[4] = c1.x; clq[5] = c1.y; clq[6] = c1.z; clq[7] = c1.w;
    B[0] = b0.x; B[1] = b0.y; B[2] = b0.z; B[3] = b0.w; B[4] = b1.x; B[5] = b1.y; B[6] = b1.z; B[7] = b1.w;
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) Bc[i] = bb_shifted_bound(B[i], clq[i]);
#pragma unroll
  for (int i = 0; i < 8; ++i) { best[i] = __int_as_float(0x7f800000); bidx[i] = 0x7fffffff; }
  const float2 m2 = make_float2(-2.0f, -2.0f);
  [[maybe_unused]] float ca[8];
  if constexpr (SHARE) {
    const float4 a0 = ld4(&sCa[4 * ty]), a1 = ld4(&sCa[64 + 4 * ty]);
    ca[0] = a0.x; ca[1] = a0.y; ca[2] = a0.z; ca[3] = a0.w; ca[4] = a1.x; ca[5] = a1.y; ca[6] = a1.z; ca[7] = a1.w;
  }

  for (int ci = 0; ci < nchunks; ++ci) {
    const int chunk = ci * BB_CT, buf = ci % kBbStages;
    if (ci + kBbAhead < nchunks) {
      const int c2 = ci + kBbAhead, u2 = c2 / kBbStages;
      if (u2 >= 1) mbar_wait(&mb_empty[c2 % kBbStages], (unsigned)((u2 - 1) & 1));  // chunk c2 - kBbStages has been read by everyone
      pipe_load(c2);
    }
    mbar_wait(&mb_full[buf], (unsigned)((ci / kBbStages) & 1));

    float2 acc[4][8];  // [query pair][candidate]: .x = local query 2p, .y = 2p+1
#pragma unroll
    for (int p = 0; p < 4; ++p)
#pragma unroll
      for (int j = 0; j < 8; ++j) acc[p][j] = make_float2(0.f, 0.f);
#pragma unroll
    for (int k = 0; k < D; ++k) {
      const float4 ua = ld4(&sQ[k][4 * ty]), ub = ld4(&sQ[k][64 + 4 * ty]);
      const float4 wa = ld4(&sY[buf][k][4 * tx]), wb = ld4(&sY[buf][k][64 + 4 * tx]);
      const float2 up[4] = {make_float2(ua.x, ua.y), make_float2(ua.z, ua.w), make_float2(ub.x, ub.y),
                            make_float2(ub.z, ub.w)};
      const float w[8] = {wa.x, wa.y, wa.z, wa.w, wb.x, wb.y, wb.z, wb.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float2 w2 = make_float2(w[j], w[j]);
#pragma unroll
        for (int p = 0; p < 4; ++p) acc[p][j] = __ffma2_rn(up[p], w2, acc[p][j]);
      }
    }
    // Filter: lower bound of the exact score vs the running upper bound; survivors are flagged.  The bound
    // L_ij = cl_i + yl_j - 2 acc_ij is compared in the shifted form  lo'_ij = yl_j - 2 acc_ij  >  Bc_i ~ B_i - cl_i
    // (one FFMA2 per pair, no add), and the per-pair compare is replaced by a per-query minimum (FMNMX3.NAN: a NaN
    // anywhere still reaches the exact path) tested once against Bc_i: the 64 compares + mask updates only run in the
    // rare chunks that hold a survivor.
    unsigned long long hit = 0ull;
    // the per-candidate part of the bound straight from |y|^2; padded candidates (|y|^2 = +inf in the workspace) get a
    // lower bound of exactly +inf (inf - inf would be NaN, which counts as a hit)
    float yl[8];
    [[maybe_unused]] float ytloc = 0.f;   // SHARE: max over this thread's valid candidates of (|alpha|+|beta|)|y|^2
    {
      const float4 na = ld4(&sYp[buf][4 * tx]), nb = ld4(&sYp[buf][64 + 4 * tx]);
      const float yn8[8] = {na.x, na.y, na.z, na.w, nb.x, nb.y, nb.z, nb.w};
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const bool valid = chunk + 4 * tx + (j & 3) + 64 * (j >> 2) < g.M;
        yl[j] = valid ? (alpha + beta) * yn8[j] - kBbKappa * ((aa + ab) * yn8[j]) : __int_as_float(0x7f800000);
        if constexpr (SHARE) ytloc = fmaxf(ytloc, valid ? (aa + ab) * yn8[j] : 0.f);
      }
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float2 y2 = make_float2(yl[j], yl[j]);
#pragma unroll
      for (int p = 0; p < 4; ++p) acc[p][j] = __ffma2_rn(m2, acc[p][j], y2);
    }
    float mq[8];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      float mx = min3_nan(acc[p][0].x, acc[p][1].x, acc[p][2].x), my = min3_nan(acc[p][0].y, acc[p][1].y, acc[p][2].y);
      mx = min3_nan(mx, acc[p][3].x, acc[p][4].x); my = min3_nan(my, acc[p][3].y, acc[p][4].y);
      mx = min3_nan(mx, acc[p][5].x, acc[p][6].x); my = min3_nan(my, acc[p][5].y, acc[p][6].y);
      mq[2 * p] = min3_nan(mx, acc[p][7].x, acc[p][7].x);
      mq[2 * p + 1] = min3_nan(my, acc[p][7].y, acc[p][7].y);
    }
    if constexpr (SHARE) {
      // an upper bound of a pair is L_ij + 2 tol_ij <= L_ij + delta_i with delta_i = 2 kappa (ca_i + max over the
      // chunk of yt): pool min_j L_ij + delta_i over the half-warp into B_i before the test
      const int cidx = chunk / BB_CT;
      if (cidx < 4 || (cidx & 3) == 0) {
        float ytmax = ytloc;   // the 16 lanes of a half-warp hold all 128 candidates of the chunk between them
#pragma unroll
        for (int o = 1; o <= 8; o <<= 1) ytmax = fmaxf(ytmax, __shfl_xor_sync(0xffffffffu, ytmax, o));
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          float m = mq[i];
#pragma unroll
          for (int o = 1; o <= 8; o <<= 1) m = fminf(m, __shfl_xor_sync(0xffffffffu, m, o));
          // the fp32 roundings of this expression stay far inside the slack of kappa
          B[i] = fminf(B[i], (m + clq[i]) + 2.0002f * kBbKappa * (ca[i] + ytmax));
          Bc[i] = bb_shifted_bound(B[i], clq[i]);
        }
      }
    }
    bool any = false;
#pragma unroll
    for (int i = 0; i < 8; ++i) any |= !(mq[i] > Bc[i]);
    if (any) {
#pragma unroll
      for (int j = 0; j < 8; ++j)
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          // !(lo' > Bc): a NaN bound or a NaN candidate is a hit, so NaN inputs reach the exact path below
          if (!(acc[p][j].x > Bc[2 * p])) hit |= 1ull << (8 * j + 2 * p);
          if (!(acc[p][j].y > Bc[2 * p + 1])) hit |= 1ull << (8 * j + 2 * p + 1);
        }
    }
    // Survivors: exact re-scoring, warp-cooperative.  The survivors of all 32 lanes are numbered by a warp prefix sum
    // (a lane's own ones in ascending bit order = ascending candidate order per query, which the first-minimum rule
    // needs) and queued 64 at a time; every lane scores queue slots lane and lane+32, then each owner folds the results
    // of its slots into its running minima in slot order.  Round 1 let every lane score its own survivors inside a
    // divergent branch: the warp then serialised the UNION of all lanes' survivors (PatchwiseST: 15 % of the kernel's
    // samples there and 27 % waiting for it at the chunk barrier; Gram likewise on its 9-dimensional descriptors).
    {
      constexpr int QCAP = 64;
      const int lane = tid & 31, wrp = tid >> 5;
      const int cnt = __popcll(hit);
      int pre = cnt;
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const int up = __shfl_up_sync(0xffffffffu, pre, o);
        if (lane >= o) pre += up;
      }
      const int total = __shfl_sync(0xffffffffu, pre, 31);
      const int first = pre - cnt;  // queue slot of this lane's first survivor
      for (int w0 = 0; w0 < total; w0 += QCAP) {
        {
          unsigned long long h = hit;
          for (int slot = first - w0; h; ++slot) {
            const int e = __ffsll((long long)h) - 1;
            h &= h - 1ull;
            if (slot >= 0 && slot < QCAP) {
              const int i = e & 7, j = e >> 3;
              sW[wrp][slot] = ((4 * ty + (i & 3) + 64 * (i >> 2)) << 8) | (4 * tx + (j & 3) + 64 * (j >> 2));
            }
          }
        }
        __syncwarp();
        const int n = min(QCAP, total - w0);
        float sc[QCAP / 32];
#pragma unroll
        for (int u = 0; u < QCAP / 32; ++u) {
          const int s0 = lane + 32 * u;
          sc[u] = 0.f;
          if (s0 < n) {
            const int ent = sW[wrp][s0];
            if constexpr (EXACT_SMEM) {
              const int q = ent >> 8, c = ent & 255;
              float dot1 = 0.f, dot2 = 0.f;
#pragma unroll
              for (int k = 0; k < D; ++k) {
                const float w = sY[buf][k][c];
                dot1 = fmaf(sX1[k][q], w, dot1);
                dot2 = fmaf(sX2[k][q], w, dot2);
              }
              sc[u] = bb_score(sXn[0][q], sXn[1][q], __ldg(P.yn + chunk + c), dot1, dot2, alpha, beta);
            } else {
              sc[u] = bb_exact_score_unrolled<D>(P.q1, P.q2, P.y, P.xn, P.gn, P.yn, g.Npad, g.Mpad, qbase + (ent >> 8),
                                                 chunk + (ent & 255), alpha, beta);
            }
          }
        }
        __syncwarp();  // every entry has been read
#pragma unroll
        for (int u = 0; u < QCAP / 32; ++u)
          if (lane + 32 * u < n) sW[wrp][lane + 32 * u] = __float_as_int(sc[u]);
        __syncwarp();
        {
          unsigned long long h = hit;
          for (int slot = first - w0; h; ++slot) {
            const int e = __ffsll((long long)h) - 1;
            h &= h - 1ull;
            if (slot >= 0 && slot < QCAP) {
              const float s = __int_as_float(sW[wrp][slot]);
              const int iq = e & 7, j = e >> 3;
              const int cj = chunk + 4 * tx + (j & 3) + 64 * (j >> 2);
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                if (i == iq) {
                  // ascending cj per thread: first minimum kept; the first NaN beats every number (torch.min)
                  if (s < best[i] || (s != s && best[i] == best[i])) { best[i] = s; bidx[i] = cj; }
                  B[i] = fminf(B[i], s);
                  Bc[i] = bb_shifted_bound(B[i], clq[i]);
                }
              }
            }
          }
        }
        __syncwarp();  // the queue is reused by the next window
      }
    }
    mbar_arrive(&mb_empty[buf]);  // this thread is done with the stage
  }

  // argmin across the 16 threads (one half-warp) that share these queries: four shuffle steps
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int o = 1; o <= 8; o <<= 1) {
      const float so = __shfl_xor_sync(0xffffffffu, best[i], o);
      const int io = __shfl_xor_sync(0xffffffffu, bidx[i], o);
      bb_argmin_merge(best[i], bidx[i], so, io);
    }
    const int qi = qbase + 4 * ty + (i & 3) + 64 * (i >> 2);
    // no comparison ever passed (every score +inf): torch.min returns index 0; never emit an out-of-range index
    if (tx == 0 && qi < g.N) idx_out[(size_t)b * g.N + qi] = (int64_t)(bidx[i] == 0x7fffffff ? 0 : bidx[i]);
  }
}

// ---- search, dist_norm = 'l1' (utils.py:166-172) ------------------------------------------------------
// score_ij = alpha * sum_k |x_ik - y_jk| + beta * sum_k |g_ik - y_jk|.  No dot-product form exists, so every pair is
// scored exactly: the sums run over k = 0..D-1 in fp32 (the C oracle restates this order; torch's reduction order over
// the last axis is unspecified, so against the reference itself the near-tie protocol of the tests applies), then
// (alpha * d1) + (beta * d2) with the reference's rounding points (loss.py:132-133).  The reference materialises a
// [B,N,M,d] tensor here (64 x 4096 x 5376 x 27 floats at configs[3]: it cannot run); this kernel keeps nothing.
// Tile: 128 queries x 64 candidates per chunk, 256 threads as 16 x 16, 8 queries x 4 candidates per thread
// (64 accumulators: d1, d2 per pair), 4 FADD per term and pair (the |.| is an operand modifier).
template <int D>
__global__ void __launch_bounds__(BB_NT, 1)
bb_search_l1_kernel(const float* __restrict__ mats, size_t per_image, BbGeom g, float alpha, float beta,
                    int64_t* __restrict__ idx_out) {
  constexpr int CT = 64;
  __shared__ __align__(16) float sX[D][BB_QT];
  __shared__ __align__(16) float sG[D][BB_QT];
  __shared__ __align__(16) float sY[D][CT];
  const int tid = threadIdx.x;
  const int b = blockIdx.y, qbase = blockIdx.x * BB_QT;
  const BbPtrs P = bb_image_ptrs(mats, per_image, b, g.Npad, g.Mpad, D);
  for (int it = tid; it < D * (BB_QT / 4); it += BB_NT) {
    const int k = it / (BB_QT / 4), c4 = it - k * (BB_QT / 4);
    st4(&sX[k][4 * c4], ldg4(P.q1 + (size_t)k * g.Npad + qbase + 4 * c4));
    st4(&sG[k][4 * c4], ldg4(P.q2 + (size_t)k * g.Npad + qbase + 4 * c4));
  }
  const int ty = tid >> 4, tx = tid & 15;  // queries 8*ty .. +7, candidates 4*tx .. +3 of the chunk
  float best[8];
  int bidx[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) { best[i] = __int_as_float(0x7f800000); bidx[i] = 0x7fffffff; }
  for (int chunk = 0; chunk < g.Mpad; chunk += CT) {
    __syncthreads();  // the previous chunk has been consumed (first pass: queries are staged)
    for (int it = tid; it < D * (CT / 4); it += BB_NT) {
      const int k = it / (CT / 4), c4 = it - k * (CT / 4);
      st4(&sY[k][4 * c4], ldg4(P.y + (size_t)k * g.Mpad + chunk + 4 * c4));
    }
    __syncthreads();
    float d1[8][4], d2[8][4];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) { d1[i][j] = 0.f; d2[i][j] = 0.f; }
#pragma unroll
    for (int k = 0; k < D; ++k) {
      const float4 xa = ld4(&sX[k][8 * ty]), xb = ld4(&sX[k][8 * ty + 4]);
      const float4 ga = ld4(&sG[k][8 * ty]), gb = ld4(&sG[k][8 * ty + 4]);
      const float4 yv = ld4(&sY[k][4 * tx]);
      const float x[8] = {xa.x, xa.y, xa.z, xa.w, xb.x, xb.y, xb.z, xb.w};
      const float gg[8] = {ga.x, ga.y, ga.z, ga.w, gb.x, gb.y, gb.z, gb.w};
      const float y[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          d1[i][j] = __fadd_rn(d1[i][j], fabsf(__fsub_rn(x[i], y[j])));
          d2[i][j] = __fadd_rn(d2[i][j], fabsf(__fsub_rn(gg[i], y[j])));
        }
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int cj = chunk + 4 * tx + j;
      if (cj >= g.M) continue;  // padding candidates
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float s = __fadd_rn(__fmul_rn(alpha, d1[i][j]), __fmul_rn(beta, d2[i][j]));
        // ascending cj per thread: first minimum kept; the first NaN beats every number (torch.min)
        if (s < best[i] || (s != s && best[i] == best[i])) { best[i] = s; bidx[i] = cj; }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i) {
#pragma unroll
    for (int o = 1; o <= 8; o <<= 1) {
      const float so = __shfl_xor_sync(0xffffffffu, best[i], o);
      const int io = __shfl_xor_sync(0xffffffffu, bidx[i], o);
      bb_argmin_merge(best[i], bidx[i], so, io);
    }
    const int qi = qbase + 8 * ty + i;
    if (tx == 0 && qi < g.N) idx_out[(size_t)b * g.N + qi] = (int64_t)(bidx[i] == 0x7fffffff ? 0 : bidx[i]);
  }
}

// ---- loss ---------------------------------------------------------------------------------------
// criterion term (sum over the D descriptor elements) of query i of image b against its selected candidate j
template <int D>
SRST_DEV float bb_loss_term(const float* mats, size_t per_image, const BbGeom& g, int b, int i, int j, int criterion) {
  const BbPtrs P = bb_image_ptrs(mats, per_image, b, g.Npad, g.Mpad, D);
  float acc = 0.f;
#pragma unroll
  for (int k = 0; k < D; ++k) {
    const float d = __ldg(P.q1 + (size_t)k * g.Npad + i) - __ldg(P.y + (size_t)k * g.Mpad + j);
    acc += (criterion == 0) ? fabsf(d) : d * d;
  }
  return acc;
}

// Criterion-gradient scale of a term of query i of image b over `D` elements: grad_out[0] / (B N D) for the batch
// mean, grad_out[b] / (N D) per image (reduction='none': grad_out is [B]), grad_out[b N + i] / D per patch (MAP, the
// loss map: grad_out is [B][N]).
template <bool PER_IMG, bool MAP = false>
SRST_DEV float patch_grad_scale(const float* __restrict__ grad_out, int b, int B, int N, float D, int i = 0) {
  if constexpr (MAP) return __ldg(grad_out + (size_t)b * N + i) / D;
  else return __ldg(grad_out + (PER_IMG ? b : 0)) / ((float)(PER_IMG ? 1 : B) * (float)N * D);
}

// PER_IMG: reduction='none' -- ceil(N / BB_NT) CTAs per image, image-major, so no CTA spans two images;
// loss_out[b] = the mean over image b's N*D terms.
// MAP: the scalar grid and reduction (loss_out[0] keeps its bits), and every query's term / D also goes to map_out[B][N].
template <int D, bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(BB_NT)
bb_loss_kernel(const float* __restrict__ mats, size_t per_image, BbGeom g, const int64_t* __restrict__ idx,
               int criterion, float* partials, unsigned int* ticket, float* loss_out, float* __restrict__ map_out = nullptr) {
  static_assert(!(MAP && PER_IMG), "the loss map comes with the batch loss");
  __shared__ float s_red[BB_NT / 32];
  __shared__ unsigned int s_last;
  const int tid = threadIdx.x;
  const size_t t = (size_t)blockIdx.x * BB_NT + tid;
  float acc = 0.f;
  if constexpr (PER_IMG) {
    const unsigned int per = gridDim.x / g.B, b = blockIdx.x / per;
    const int i = (int)(blockIdx.x - b * per) * BB_NT + tid;
    if (i < g.N) acc = bb_loss_term<D>(mats, per_image, g, (int)b, i, (int)idx[(size_t)b * g.N + i], criterion);
  } else if (t < (size_t)g.B * g.N) {
    const int b = (int)(t / g.N), i = (int)(t - (size_t)b * g.N);
    acc = bb_loss_term<D>(mats, per_image, g, b, i, (int)idx[t], criterion);
    if constexpr (MAP) map_out[t] = acc / (float)D;
  }
  acc = warp_sum(acc);
  if ((tid & 31) == 0) s_red[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    float bs = 0.f;
    for (int w = 0; w < BB_NT / 32; ++w) bs += s_red[w];
    partials[blockIdx.x] = bs;
    __threadfence();
    s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if constexpr (PER_IMG) {
    if (s_last) {
      __threadfence();
      reduce_partials_per_image(partials, g.B, gridDim.x / g.B, 1.0 / ((double)g.N * D), loss_out);
      if (tid == 0) *ticket = 0u;
    }
  } else if (s_last && tid < 32) {
    __threadfence();
    double tot = 0.0;
    for (unsigned int i = tid; i < gridDim.x; i += 32) { tot += (double)__ldcg(partials + i); partials[i] = 0.f; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    if (tid == 0) {
      loss_out[0] = (float)(tot / ((double)g.B * g.N * D));
      *ticket = 0u;
    }
  }
}

// ---- backward -----------------------------------------------------------------------------------
SRST_DEV float bb_candidate_value(const float* gt, const float* gt2, const float* gt4, const BbGeom& g, int b,
                                  int j, int c, int ky, int kx) {
  const float* img; int H, W, nx, p;
  if (j < g.N0) { img = gt + (size_t)b * 3 * g.H * g.W; H = g.H; W = g.W; nx = g.n0x; p = j; }
  else if (j < g.N0 + g.N2) { img = gt2 + (size_t)b * 3 * g.H2 * g.W2; H = g.H2; W = g.W2; nx = g.n2x; p = j - g.N0; }
  else { img = gt4 + (size_t)b * 3 * g.H4 * g.W4; H = g.H4; W = g.W4; nx = g.n4x; p = j - g.N0 - g.N2; }
  const int py = p / nx, px = p - py * nx;
  return __ldg(img + ((size_t)c * H + 3 * py + ky) * W + 3 * px + kx);
}

// PER_IMG: reduction='none', grad_out is [B]; MAP: the loss map, grad_out is [B][N] (patch_grad_scale)
template <bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(256)
bb_backward_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
                   const float* __restrict__ gt4, const int64_t* __restrict__ idx, const float* __restrict__ grad_out,
                   BbGeom g, int criterion, float* __restrict__ d_sr) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t total = (size_t)g.B * 3 * g.H * g.W;
  if (t >= total) return;
  const int x = (int)(t % g.W);
  const int y = (int)((t / g.W) % g.H);
  const int c = (int)((t / ((size_t)g.W * g.H)) % 3);
  const int b = (int)(t / ((size_t)3 * g.W * g.H));
  const int py = y / 3, px = x / 3;
  float out = 0.f;
  if (py < g.H / 3 && px < g.n0x) {
    const int i = py * g.n0x + px;
    const int j = (int)idx[(size_t)b * g.N + i];
    const float sel = bb_candidate_value(gt, gt2, gt4, g, b, j, c, y - 3 * py, x - 3 * px);
    const float d = __ldg(sr + t) - sel;
    const float scale = patch_grad_scale<PER_IMG, MAP>(grad_out, b, g.B, g.N, (float)BB_D, i);
    out = (criterion == 0) ? ((d > 0.f) ? scale : ((d < 0.f) ? -scale : 0.f)) : 2.0f * d * scale;
  }
  d_sr[t] = out;
}

// ---- gradient w.r.t. gt (loss.py:136-139: the gather of the selected candidates is differentiable in p2_cat) ----
// The final criterion is symmetric in its two arguments, so d/d(candidate) is the SR-side formula with the roles of
// the SR patch and the selected candidate swapped.  Several queries may select the same candidate: the 27 values of a
// query are accumulated with atomicAdd into the gradient image of the candidate's pyramid level (level 0 = d_gt
// itself), and bb_pyramid_adjoint_kernel then folds the two coarse levels back through the bicubic taps.
struct BbLevel { float* img; int H, W, nx, p; };
SRST_DEV BbLevel bb_locate(const BbGeom& g, int b, int j, float* d0, float* d2, float* d4) {
  BbLevel L;
  if (j < g.N0) { L.img = d0 + (size_t)b * 3 * g.H * g.W; L.H = g.H; L.W = g.W; L.nx = g.n0x; L.p = j; }
  else if (j < g.N0 + g.N2) { L.img = d2 + (size_t)b * 3 * g.H2 * g.W2; L.H = g.H2; L.W = g.W2; L.nx = g.n2x; L.p = j - g.N0; }
  else { L.img = d4 + (size_t)b * 3 * g.H4 * g.W4; L.H = g.H4; L.W = g.W4; L.nx = g.n4x; L.p = j - g.N0 - g.N2; }
  return L;
}
SRST_DEV void bb_read_candidate(const float* gt, const float* gt2, const float* gt4, const BbGeom& g, int b, int j,
                                float (&w)[BB_D]) {
  if (j < g.N0) bb_read_patch(gt + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, j, w);
  else if (j < g.N0 + g.N2) bb_read_patch(gt2 + (size_t)b * 3 * g.H2 * g.W2, g.H2, g.W2, g.n2x, j - g.N0, w);
  else bb_read_patch(gt4 + (size_t)b * 3 * g.H4 * g.W4, g.H4, g.W4, g.n4x, j - g.N0 - g.N2, w);
}
// element c*9 + ky*3 + kx of `v` is added to pixel (c, 3 py + ky, 3 px + kx) of the level image
SRST_DEV void bb_scatter_add_patch(const BbLevel& L, const float (&v)[BB_D]) {
  const int py = L.p / L.nx, px = L.p - py * L.nx;
#pragma unroll
  for (int e = 0; e < BB_D; ++e) {
    const int c = e / 9, ky = (e % 9) / 3, kx = e % 3;
    atomicAdd(L.img + ((size_t)c * L.H + 3 * py + ky) * L.W + 3 * px + kx, v[e]);
  }
}

__global__ void __launch_bounds__(256) bb_fill_zero_kernel(float* __restrict__ p, size_t n) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) p[i] = 0.f;
}

// BestBuddyLoss: one thread per query patch (PER_IMG: grad_out is [B]; MAP: [B][N]; patch_grad_scale)
template <bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(256)
bb_backward_gt_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
                      const float* __restrict__ gt4, const int64_t* __restrict__ idx, const float* __restrict__ grad_out,
                      BbGeom g, int criterion, float* __restrict__ d0, float* __restrict__ d2, float* __restrict__ d4) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)g.B * g.N) return;
  const int b = (int)(t / g.N), i = (int)(t - (size_t)b * g.N);
  const int j = (int)idx[t];
  float v[BB_D], w[BB_D];
  bb_read_patch(sr + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, i, v);
  bb_read_candidate(gt, gt2, gt4, g, b, j, w);
  const float scale = patch_grad_scale<PER_IMG, MAP>(grad_out, b, g.B, g.N, (float)BB_D, i);
#pragma unroll
  for (int e = 0; e < BB_D; ++e) {
    const float d = w[e] - v[e];
    w[e] = (criterion == 0) ? ((d > 0.f) ? scale : ((d < 0.f) ? -scale : 0.f)) : 2.0f * d * scale;
  }
  bb_scatter_add_patch(bb_locate(g, b, j, d0, d2, d4), w);
}

// Adjoint of bb_pyramid_kernel: every element of the two coarse gradient images is spread over its 4x4 source
// taps (same constants, same clamped indices) into d_gt.
__global__ void __launch_bounds__(256)
bb_pyramid_adjoint_kernel(const float* __restrict__ d2, const float* __restrict__ d4, float* __restrict__ d_gt, int planes,
                          int H, int W, int H2, int W2, int H4, int W4) {
  const size_t n2 = (size_t)planes * H2 * W2, n4 = (size_t)planes * H4 * W4;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= n2 + n4) return;
  const bool lvl4 = t >= n2;
  const size_t u = lvl4 ? t - n2 : t;
  const float gv = lvl4 ? d4[u] : d2[u];
  if (gv == 0.f) return;
  const int Ho = lvl4 ? H4 : H2, Wo = lvl4 ? W4 : W2;
  const int x = (int)(u % Wo);
  const int y = (int)((u / Wo) % Ho);
  const int pl = (int)(u / ((size_t)Wo * Ho));
  const int sy = lvl4 ? 4 * y : 2 * y - 1;
  const int sx = lvl4 ? 4 * x : 2 * x - 1;
  float* dst = d_gt + (size_t)pl * H * W;
  const float wt[4] = {-0.09375f, 0.59375f, 0.59375f, -0.09375f};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int yy = min(max(sy + i, 0), H - 1);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int xx = min(max(sx + k, 0), W - 1);
      atomicAdd(dst + (size_t)yy * W + xx, gv * (wt[i] * wt[k]));
    }
  }
}

// ---- GramLoss backward --------------------------------------------------------------------------
// loss = mean over B*N*9 of |G1 - Gsel| (or squared); G1 = F F^T / 27 of the SR patch.
//   dL/dG1[a][b] = scale * sign(G1 - Gsel)[a][b]                 (or 2*diff)
//   dL/dF[a][s]  = sum_b (dG[a][b] + dG[b][a]) F[b][s] / 27
// One thread per patch; every pixel covered by a patch belongs to exactly one, the rest stay 0.
// TO_GT: the same formula with the roles swapped (v = the selected candidate, differentiated; w = the SR patch), the
// result accumulated into the candidate's level image (d_sr = level 0 = d_gt, d2, d4).
// PER_IMG: reduction='none', grad_out is [B]; MAP: the loss map, grad_out is [B][N] (patch_grad_scale)
template <bool TO_GT = false, bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(256)
gram_backward_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
                     const float* __restrict__ gt4, const int64_t* __restrict__ idx, const float* __restrict__ grad_out,
                     BbGeom g, int criterion, float* __restrict__ d_sr, float* __restrict__ d2 = nullptr,
                     float* __restrict__ d4 = nullptr) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)g.B * g.N) return;
  const int b = (int)(t / g.N), i = (int)(t - (size_t)b * g.N);
  float v[BB_D], w[BB_D], g1[9], gs[9];
  const int j = (int)idx[t];
  if constexpr (TO_GT) {
    bb_read_candidate(gt, gt2, gt4, g, b, j, v);
    bb_read_patch(sr + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, i, w);
  } else {
    bb_read_patch(sr + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, i, v);
    bb_read_candidate(gt, gt2, gt4, g, b, j, w);
  }
  bb_gram(v, g1);
  bb_gram(w, gs);
  const float scale = patch_grad_scale<PER_IMG, MAP>(grad_out, b, g.B, g.N, 9.0f, i);
  float dG[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) {
    const float d = g1[k] - gs[k];
    dG[k] = (criterion == 0) ? ((d > 0.f) ? scale : ((d < 0.f) ? -scale : 0.f)) : 2.0f * d * scale;
  }
  const int py = i / g.n0x, px = i - py * g.n0x;
  float* o = d_sr + (size_t)b * 3 * g.H * g.W;
  [[maybe_unused]] float outv[BB_D];
#pragma unroll
  for (int a = 0; a < 3; ++a)
#pragma unroll
    for (int s9 = 0; s9 < 9; ++s9) {
      float acc = 0.f;
#pragma unroll
      for (int c = 0; c < 3; ++c) acc = fmaf(dG[a * 3 + c] + dG[c * 3 + a], v[c * 9 + s9], acc);
      if constexpr (TO_GT) outv[a * 9 + s9] = acc / 27.0f;
      else o[((size_t)a * g.H + 3 * py + s9 / 3) * g.W + 3 * px + s9 % 3] = acc / 27.0f;
    }
  if constexpr (TO_GT) bb_scatter_add_patch(bb_locate(g, b, j, d_sr, d2, d4), outv);
}

// ---- PatchwiseStructureTensorLoss backward ------------------------------------------------------
// loss = mean over B*N*27 of |D1 - Dsel| (or squared), D1 = descriptor of the SR patch.  Per pixel of
// the patch, through utils.normalize (q = sqrt(det+eps), s = <J, dD>, ddet = -s/(2 q^3)):
//   dJxx = dDxx/q + ddet*Jyy , dJyy = dDyy/q + ddet*Jxx , dJxy = dDxy/q - 2 ddet*Jxy
// then the adjoint 3x3 smoothing, the product rule dIx = 2 Ix dPxx + Iy dPxy, dIy = 2 Iy dPyy + Ix dPxy,
// the adjoint derivative filters and the grayscale weights.  One thread per patch.
// TO_GT: roles swapped and scatter-add into the candidate's level image, as in gram_backward_kernel; PER_IMG, MAP: as
// there
template <bool TO_GT = false, bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(128)
pst_backward_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
                    const float* __restrict__ gt4, const int64_t* __restrict__ idx, const float* __restrict__ grad_out,
                    BbGeom g, PstTaps tp, int criterion, float* __restrict__ d_sr, float* __restrict__ d2 = nullptr,
                    float* __restrict__ d4 = nullptr) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)g.B * g.N) return;
  const int b = (int)(t / g.N), i = (int)(t - (size_t)b * g.N);
  float v[BB_D], w[BB_D], dsel[BB_D];
  const int j = (int)idx[t];
  if constexpr (TO_GT) {
    bb_read_patch(sr + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, i, w);
    bb_read_candidate(gt, gt2, gt4, g, b, j, v);
  } else {
    bb_read_candidate(gt, gt2, gt4, g, b, j, w);
    bb_read_patch(sr + (size_t)b * 3 * g.H * g.W, g.H, g.W, g.n0x, i, v);
  }
  pst_descriptor(w, tp, dsel);
  PstState S;
  pst_state(v, tp, S);
  const float scale = patch_grad_scale<PER_IMG, MAP>(grad_out, b, g.B, g.N, (float)BB_D, i);
  float dJ[3][9];
#pragma unroll
  for (int p = 0; p < 9; ++p) {
    float dd[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) {
      const float d = __fdiv_rn(S.J[c][p], S.q[p]) - dsel[c * 9 + p];
      dd[c] = (criterion == 0) ? ((d > 0.f) ? scale : ((d < 0.f) ? -scale : 0.f)) : 2.0f * d * scale;
    }
    const float iq = 1.0f / S.q[p];
    const float s = fmaf(S.J[0][p], dd[0], fmaf(S.J[1][p], dd[1], S.J[2][p] * dd[2]));
    const float ddet = (-0.5f * s) * (iq * iq) * iq;
    dJ[0][p] = fmaf(dd[0], iq, ddet * S.J[1][p]);
    dJ[1][p] = fmaf(dd[1], iq, ddet * S.J[0][p]);
    dJ[2][p] = fmaf(dd[2], iq, -2.0f * ddet * S.J[2][p]);
  }
  float dP[3][9], tmp[9];
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    pst_horz_t(tp.k, dJ[c], tmp);
    pst_vert_t(tp.k, tmp, dP[c]);
  }
  float dIx[9], dIy[9], ga[9], gb[9];
#pragma unroll
  for (int p = 0; p < 9; ++p) {
    dIx[p] = fmaf(2.0f * S.Ix[p], dP[0][p], S.Iy[p] * dP[2][p]);
    dIy[p] = fmaf(2.0f * S.Iy[p], dP[1][p], S.Ix[p] * dP[2][p]);
  }
  pst_horz_t(tp.g, dIx, tmp);  pst_vert_t(tp.dg, tmp, ga);
  pst_horz_t(tp.dg, dIy, tmp); pst_vert_t(tp.g, tmp, gb);
  const int py = i / g.n0x, px = i - py * g.n0x;
  float* o = d_sr + (size_t)b * 3 * g.H * g.W;
  const float coef[3] = {kGrayR, kGrayG, kGrayB};
  [[maybe_unused]] float outv[BB_D];
#pragma unroll
  for (int c = 0; c < 3; ++c)
#pragma unroll
    for (int p = 0; p < 9; ++p) {
      if constexpr (TO_GT) outv[c * 9 + p] = coef[c] * (ga[p] + gb[p]);
      else o[((size_t)c * g.H + 3 * py + p / 3) * g.W + 3 * px + p % 3] = coef[c] * (ga[p] + gb[p]);
    }
  if constexpr (TO_GT) bb_scatter_add_patch(bb_locate(g, b, j, d_sr, d2, d4), outv);
}

}  // namespace srst
