// Best-Buddy loss for an ARBITRARY patch geometry (ksize, pad, stride) on sm_100a.
//
// The reference's BestBuddyLoss takes ksize / pad / stride (loss.py:86, used at :116-129); its training entry point only
// ever builds the default (3, 0, 3), which has the tuned kernels of bb_kernels.cuh.  Every other geometry runs here:
//
//   bbg_search_kernel   : every (query, candidate) pair scored EXACTLY with the reference's expression and rounding
//                         points (bb_score, utils.py:183-187 / loss.py:132-133; l1: utils.py:166-172), patch elements
//                         accumulated in ascending order e = c*k*k + ky*k + kx (F.unfold's layout, zero outside the
//                         image = its padding); first minimal index wins (torch.min).  bbg_pack_kernel gathers the
//                         candidate patches of an image once (element-major matrix + norms); the query tile of a CTA
//                         is gathered straight from the images.
//   bbg_loss_kernel     : mean |sr_patch - cand[idx]| (or squared) over B*N*D, deterministic reduction
//   bbg_backward_kernel : d_sr in GATHER form -- a pixel sums, in a fixed order, the criterion gradients of the
//                         ceil(k/s)^2 patches that cover it (overlapping patches when stride < ksize; no atomics)
//   bbg_backward_gt_kernel : d_gt through the gather of the selected candidates (loss.py:136-139): scattered with
//                         atomicAdd into per-level gradient images, folded back by bb_pyramid_adjoint_kernel
//
// A 64-query x 64-candidate tile per CTA step, four queries x four candidates per thread: 3 LDS.128 per 32 FMA
// (the first version, one query x four candidates, was bound by the shared-memory pipe: 14 TFLOP/s algorithmic at
// (3, 0, 3), profiles/r02_bb_geometry.log).  Both dot products of every pair are evaluated -- no filter as in the
// tuned (3, 0, 3) search.
// oracle/bbg_oracle.c restates the same order; tests/test_bb_geometry.py pins both on outputs of the reference.
#pragma once
#include "bb_kernels.cuh"

namespace srst {

constexpr int BBG_MAXK = 8;                 // ksize 1..8: D = 3 k^2 <= 192
constexpr int BBG_QT = 64, BBG_CT = 64, BBG_NT = 256;

struct BbgLevel { int H, W, ny, nx, n; };
struct BbgGeom {
  int B, k, p, s, D;
  BbgLevel L[3];  // gt, gt x1/2, gt x1/4
  int N, M;
};

inline int bbg_npatch(int size, int k, int p, int s) {
  const long long span = (long long)size + 2LL * p - k;
  return span < 0 ? 0 : (int)(span / s) + 1;  // F.unfold: floor((size + 2p - k) / s) + 1
}
inline BbgGeom bbg_geom(int B, int H, int W, int k, int p, int s) {
  BbgGeom g;
  g.B = B; g.k = k; g.p = p; g.s = s; g.D = 3 * k * k;
  const int hs[3] = {H, H / 2, H / 4}, ws[3] = {W, W / 2, W / 4};
  for (int l = 0; l < 3; ++l) {
    g.L[l].H = hs[l]; g.L[l].W = ws[l];
    g.L[l].ny = bbg_npatch(hs[l], k, p, s); g.L[l].nx = bbg_npatch(ws[l], k, p, s);
    g.L[l].n = g.L[l].ny * g.L[l].nx;
  }
  g.N = g.L[0].n;
  g.M = g.L[0].n + g.L[1].n + g.L[2].n;
  return g;
}
inline bool bbg_geom_ok(int B, int H, int W, int k, int p, int s) {
  if (B <= 0 || B > 65535 || k < 1 || k > BBG_MAXK || p < 0 || p > 64 || s < 1 || s > 4096) return false;
  if (H < 4 || W < 4 || H > 32768 || W > 32768) return false;
  const BbgGeom g = bbg_geom(B, H, W, k, p, s);
  if (g.L[0].n <= 0 || g.L[1].n <= 0 || g.L[2].n <= 0) return false;  // F.unfold raises on an empty level
  return (long long)g.L[0].ny * g.L[0].nx < 0x3fffffffLL;
}

struct BbgWorkspace {
  unsigned int* ticket;
  float* partials;
  float *pyr2, *pyr4;  // the two coarse levels of gt when the caller does not pass them
  float *d2, *d4;      // their gradient images (gradient w.r.t. gt)
  float* ymat;         // per image: candidate patches Y[D][Mpad] (element-major) followed by their norms yn[Mpad]
  size_t y_per_image;  // floats
  int Mpad;
  size_t total_bytes;
};
inline BbgWorkspace bbg_carve(void* base, const BbgGeom& g) {
  BbgWorkspace w;
  char* p = reinterpret_cast<char*>(base);
  size_t off = 0;
  auto take = [&](size_t bytes) { char* q = p + off; off += (bytes + 255) / 256 * 256; return q; };
  w.ticket = reinterpret_cast<unsigned int*>(take(256));
  w.partials = reinterpret_cast<float*>(take((((size_t)g.B * g.N + BBG_NT - 1) / BBG_NT) * sizeof(float)));
  const size_t n2 = (size_t)g.B * 3 * g.L[1].H * g.L[1].W, n4 = (size_t)g.B * 3 * g.L[2].H * g.L[2].W;
  w.pyr2 = reinterpret_cast<float*>(take(n2 * sizeof(float)));
  w.pyr4 = reinterpret_cast<float*>(take(n4 * sizeof(float)));
  w.d2 = reinterpret_cast<float*>(take((n2 + 3) / 4 * 4 * sizeof(float) + n4 * sizeof(float)));  // d4 follows d2: one fill
  w.d4 = w.d2 + (n2 + 3) / 4 * 4;
  w.Mpad = (g.M + BBG_CT - 1) / BBG_CT * BBG_CT;
  w.y_per_image = (size_t)(g.D + 1) * w.Mpad;
  w.ymat = reinterpret_cast<float*>(take(w.y_per_image * g.B * sizeof(float)));
  w.total_bytes = off;
  return w;
}

// A patch of a level image: top-left corner (may lie in the zero padding) and the image
struct BbgPatch { const float* img; int H, W, y0, x0; };
SRST_DEV BbgPatch bbg_patch_of(const float* img_b, const BbgLevel& L, int p, int s, int n) {
  const int py = n / L.nx, px = n - py * L.nx;
  BbgPatch P;
  P.img = img_b; P.H = L.H; P.W = L.W; P.y0 = py * s - p; P.x0 = px * s - p;
  return P;
}
SRST_DEV BbgPatch bbg_candidate(const float* gt, const float* gt2, const float* gt4, const BbgGeom& g, int b, int j) {
  int l = 0;
  if (j >= g.L[0].n) { j -= g.L[0].n; l = 1; }
  if (l == 1 && j >= g.L[1].n) { j -= g.L[1].n; l = 2; }
  const float* base = l == 0 ? gt : (l == 1 ? gt2 : gt4);
  return bbg_patch_of(base + (size_t)b * 3 * g.L[l].H * g.L[l].W, g.L[l], g.p, g.s, j);
}
// element (c, ky, kx): F.unfold zero-pads
SRST_DEV float bbg_value(const BbgPatch& P, int c, int ky, int kx) {
  const int y = P.y0 + ky, x = P.x0 + kx;
  return (y >= 0 && y < P.H && x >= 0 && x < P.W) ? __ldg(P.img + ((size_t)c * P.H + y) * P.W + x) : 0.f;
}

// Candidate patches of one image, gathered ONCE: Y[e][j] (element-major, Mpad columns, zeros beyond M) and the norms
// yn[j] (fmaf over e ascending).  The search then stages its chunks with coalesced 16-byte copies; gathering them from
// the images inside the search cost 41 % of its time (every CTA repeated the index arithmetic for all M candidates).
__global__ void __launch_bounds__(256)
bbg_pack_kernel(const float* __restrict__ gt, const float* __restrict__ gt2, const float* __restrict__ gt4, BbgGeom g,
                float* __restrict__ ymat, size_t y_per_image, int Mpad) {
  const int j = blockIdx.x * blockDim.x + threadIdx.x, b = blockIdx.y;
  if (j >= Mpad) return;
  float* Y = ymat + y_per_image * b;
  const bool ok = j < g.M;
  const BbgPatch Pc = bbg_candidate(gt, gt2, gt4, g, b, ok ? j : 0);
  float yn = 0.f;
  int e = 0;
  for (int c = 0; c < 3; ++c)
    for (int ky = 0; ky < g.k; ++ky)
      for (int kx = 0; kx < g.k; ++kx, ++e) {
        const float v = ok ? bbg_value(Pc, c, ky, kx) : 0.f;
        Y[(size_t)e * Mpad + j] = v;
        yn = fmaf(v, v, yn);
      }
  Y[(size_t)g.D * Mpad + j] = yn;
}

inline size_t bbg_search_smem(int D) { return sizeof(float) * ((size_t)D * (2 * BBG_QT + BBG_CT)) + sizeof(int) * (size_t)D; }

__global__ void __launch_bounds__(BBG_NT)
bbg_search_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ ymat,
                  size_t y_per_image, int Mpad, BbgGeom g, float alpha, float beta, int dist_l1,
                  int64_t* __restrict__ idx_out) {
  SRST_DYN_SMEM(float, smem);
  constexpr int NQG = BBG_QT / 4, NCG = BBG_CT / 4;  // 16 x 16 threads, each 4 queries x 4 candidates
  static_assert(NQG * NCG == BBG_NT && BBG_QT == BBG_CT && BBG_NT % BBG_QT == 0, "bbg: tile");
  constexpr int NEG = BBG_NT / BBG_QT;               // element groups of the gather (a thread owns one patch)
  const int D = g.D;
  float* sX = smem;                         // [D][QT]  SR query patches
  float* sG = sX + (size_t)D * BBG_QT;      // [D][QT]  gt query patches
  float* sY = sG + (size_t)D * BBG_QT;      // [D][CT]  candidate chunk
  int* sE = reinterpret_cast<int*>(sY + (size_t)D * BBG_CT);  // element e -> c << 16 | ky << 8 | kx
  __shared__ float s_xn[BBG_QT], s_gn[BBG_QT], s_yn[BBG_CT];
  __shared__ float s_best[NCG][BBG_QT];
  __shared__ int s_bidx[NCG][BBG_QT];
  const int tid = threadIdx.x;
  const int pslot = tid % BBG_QT, egrp = tid / BBG_QT;  // gather: patch slot, element group
  const int qg = tid % NQG, cg = tid / NQG;             // scoring: queries 4 qg .., candidates 4 cg .. of the chunk
  const int b = blockIdx.y, qbase = blockIdx.x * BBG_QT;
  const float* __restrict__ Y = ymat + y_per_image * b;   // [D][Mpad], then yn[Mpad]
  const int kk = g.k * g.k;
  for (int e = tid; e < D; e += BBG_NT) {
    const int c = e / kk, r = e - c * kk, ky = r / g.k;
    sE[e] = (c << 16) | (ky << 8) | (r - ky * g.k);
  }
  __syncthreads();
  {
    // queries: this thread gathers elements egrp, egrp + NEG, .. of query `pslot` (SR and gt patch at the same place)
    const int i = qbase + pslot;
    const bool ok = i < g.N;
    const BbgPatch P1 = bbg_patch_of(sr + (size_t)b * 3 * g.L[0].H * g.L[0].W, g.L[0], g.p, g.s, ok ? i : 0);
    BbgPatch P2 = P1;
    P2.img = gt + (size_t)b * 3 * g.L[0].H * g.L[0].W;
    for (int e = egrp; e < D; e += NEG) {
      const int code = sE[e];
      const int c = code >> 16, ky = (code >> 8) & 255, kx = code & 255;
      sX[e * BBG_QT + pslot] = ok ? bbg_value(P1, c, ky, kx) : 0.f;
      sG[e * BBG_QT + pslot] = ok ? bbg_value(P2, c, ky, kx) : 0.f;
    }
  }
  __syncthreads();
  if (tid < BBG_QT) {
    float xn = 0.f, gn = 0.f;
    for (int e = 0; e < D; ++e) {
      const float x = sX[e * BBG_QT + tid], q = sG[e * BBG_QT + tid];
      xn = fmaf(x, x, xn);
      gn = fmaf(q, q, gn);
    }
    s_xn[tid] = xn;
    s_gn[tid] = gn;
  }
  float best[4];
  int bidx[4];
#pragma unroll
  for (int i = 0; i < 4; ++i) { best[i] = __int_as_float(0x7f800000); bidx[i] = 0x7fffffff; }
  for (int chunk = 0; chunk < g.M; chunk += BBG_CT) {
    __syncthreads();  // the previous chunk has been consumed (first pass: query norms are in place)
    for (int it = tid; it < D * (BBG_CT / 4); it += BBG_NT) {   // packed candidates: coalesced 16-byte copies
      const int e = it / (BBG_CT / 4), c4 = it - e * (BBG_CT / 4);
      st4(sY + e * BBG_CT + 4 * c4, ldg4(Y + (size_t)e * Mpad + chunk + 4 * c4));
    }
    if (tid < BBG_CT) s_yn[tid] = __ldg(Y + (size_t)D * Mpad + chunk + tid);
    __syncthreads();
    float d1[4][4], d2[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int u = 0; u < 4; ++u) { d1[i][u] = 0.f; d2[i][u] = 0.f; }
    if (dist_l1) {
#pragma unroll 2
      for (int e = 0; e < D; ++e) {
        const float4 xv = ld4(sX + e * BBG_QT + 4 * qg), qv = ld4(sG + e * BBG_QT + 4 * qg);
        const float4 yv = ld4(sY + e * BBG_CT + 4 * cg);
        const float x[4] = {xv.x, xv.y, xv.z, xv.w}, q[4] = {qv.x, qv.y, qv.z, qv.w}, y[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            d1[i][u] = __fadd_rn(d1[i][u], fabsf(__fsub_rn(x[i], y[u])));
            d2[i][u] = __fadd_rn(d2[i][u], fabsf(__fsub_rn(q[i], y[u])));
          }
      }
    } else {
#pragma unroll 2
      for (int e = 0; e < D; ++e) {
        const float4 xv = ld4(sX + e * BBG_QT + 4 * qg), qv = ld4(sG + e * BBG_QT + 4 * qg);
        const float4 yv = ld4(sY + e * BBG_CT + 4 * cg);
        const float x[4] = {xv.x, xv.y, xv.z, xv.w}, q[4] = {qv.x, qv.y, qv.z, qv.w}, y[4] = {yv.x, yv.y, yv.z, yv.w};
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            d1[i][u] = fmaf(x[i], y[u], d1[i][u]);
            d2[i][u] = fmaf(q[i], y[u], d2[i][u]);
          }
      }
    }
#pragma unroll
    for (int u = 0; u < 4; ++u) {   // ascending candidate index per thread
      const int cj = chunk + 4 * cg + u;
      if (cj >= g.M) continue;
      const float yn = s_yn[4 * cg + u];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float sc = dist_l1 ? __fadd_rn(__fmul_rn(alpha, d1[i][u]), __fmul_rn(beta, d2[i][u]))
                                 : bb_score(s_xn[4 * qg + i], s_gn[4 * qg + i], yn, d1[i][u], d2[i][u], alpha, beta);
        if (bb_score_before(sc, cj, best[i], bidx[i])) { best[i] = sc; bidx[i] = cj; }
      }
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    s_best[cg][4 * qg + i] = best[i];
    s_bidx[cg][4 * qg + i] = bidx[i];
  }
  __syncthreads();
  if (tid < BBG_QT && qbase + tid < g.N) {
    float sb = s_best[0][tid];
    int ib = s_bidx[0][tid];
    for (int w = 1; w < NCG; ++w) bb_argmin_merge(sb, ib, s_best[w][tid], s_bidx[w][tid]);
    if (ib < 0 || ib >= g.M) ib = 0;  // unreachable (M >= 1 and (score, index) order is total); keeps later reads in range
    idx_out[(size_t)b * g.N + qbase + tid] = ib;
  }
}

// criterion term (sum over the D patch elements) of query i of image b against its selected candidate
SRST_DEV float bbg_loss_term(const float* sr, const float* gt, const float* gt2, const float* gt4, const BbgGeom& g,
                             int criterion, int b, int i, int j) {
  j = min(max(j, 0), g.M - 1);
  const BbgPatch P1 = bbg_patch_of(sr + (size_t)b * 3 * g.L[0].H * g.L[0].W, g.L[0], g.p, g.s, i);
  const BbgPatch Pc = bbg_candidate(gt, gt2, gt4, g, b, j);
  float acc = 0.f;
  for (int c = 0; c < 3; ++c)
    for (int ky = 0; ky < g.k; ++ky)
      for (int kx = 0; kx < g.k; ++kx) {
        const float d = bbg_value(P1, c, ky, kx) - bbg_value(Pc, c, ky, kx);
        acc += (criterion == 0) ? fabsf(d) : d * d;
      }
  return acc;
}

// one thread per query patch.  PER_IMG: reduction='none' -- ceil(N / BBG_NT) CTAs per image, image-major, so no CTA
// spans two images; loss_out[b] = the mean over image b's N*D terms.
// MAP: the scalar grid and reduction (loss_out[0] keeps its bits), and every query's term / D also goes to map_out[B][N].
template <bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(BBG_NT)
bbg_loss_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
                const float* __restrict__ gt4, BbgGeom g, const int64_t* __restrict__ idx, int criterion, float* partials,
                unsigned int* ticket, float* loss_out, float* __restrict__ map_out = nullptr) {
  static_assert(!(MAP && PER_IMG), "the loss map comes with the batch loss");
  __shared__ float s_red[BBG_NT / 32];
  __shared__ unsigned int s_last;
  const int tid = threadIdx.x;
  const size_t t = (size_t)blockIdx.x * BBG_NT + tid;
  float acc = 0.f;
  if constexpr (PER_IMG) {
    const unsigned int per = gridDim.x / g.B, b = blockIdx.x / per;
    const int i = (int)(blockIdx.x - b * per) * BBG_NT + tid;
    if (i < g.N) acc = bbg_loss_term(sr, gt, gt2, gt4, g, criterion, (int)b, i, (int)idx[(size_t)b * g.N + i]);
  } else if (t < (size_t)g.B * g.N) {
    const int b = (int)(t / g.N), i = (int)(t - (size_t)b * g.N);
    acc = bbg_loss_term(sr, gt, gt2, gt4, g, criterion, b, i, (int)idx[t]);
    if constexpr (MAP) map_out[t] = acc / (float)g.D;
  }
  acc = warp_sum(acc);
  if ((tid & 31) == 0) s_red[tid >> 5] = acc;
  __syncthreads();
  if (tid == 0) {
    float bs = 0.f;
    for (int w = 0; w < BBG_NT / 32; ++w) bs += s_red[w];
    partials[blockIdx.x] = bs;
    __threadfence();
    s_last = (atomicAdd(ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if constexpr (PER_IMG) {
    if (s_last) {
      __threadfence();
      reduce_partials_per_image(partials, g.B, gridDim.x / g.B, 1.0 / ((double)g.N * g.D), loss_out);
      if (tid == 0) *ticket = 0u;
    }
  } else if (s_last && tid < 32) {
    __threadfence();
    double tot = 0.0;
    for (unsigned int i = tid; i < gridDim.x; i += 32) { tot += (double)__ldcg(partials + i); partials[i] = 0.f; }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) tot += __shfl_xor_sync(0xffffffffu, tot, o);
    if (tid == 0) {
      loss_out[0] = (float)(tot / ((double)g.B * g.N * g.D));
      *ticket = 0u;
    }
  }
}

SRST_DEV float bbg_crit_grad(float d, int criterion, float scale) {
  return (criterion == 0) ? ((d > 0.f) ? scale : ((d < 0.f) ? -scale : 0.f)) : 2.0f * d * scale;
}

// one thread per SR pixel: the patches py in [ceil((y + p - k + 1)/s), floor((y + p)/s)] x likewise px cover it.
// PER_IMG: reduction='none', grad_out is [B] and image b scales by grad_out[b] / (N D).
// MAP: the loss map, grad_out is [B][N]: every covering patch q scales by its own grad_out[b N + q] / D, in the same
// fixed order.
template <bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(256)
bbg_backward_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
                    const float* __restrict__ gt4, const int64_t* __restrict__ idx, const float* __restrict__ grad_out,
                    BbgGeom g, int criterion, float* __restrict__ d_sr) {
  const int H = g.L[0].H, W = g.L[0].W;
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)g.B * 3 * H * W) return;
  const int x = (int)(t % W);
  const int y = (int)((t / W) % H);
  const int c = (int)((t / ((size_t)W * H)) % 3);
  const int b = (int)(t / ((size_t)3 * W * H));
  float scale = 0.f;
  if constexpr (!MAP)
    scale = __ldg(grad_out + (PER_IMG ? b : 0)) / ((float)(PER_IMG ? 1 : g.B) * (float)g.N * (float)g.D);
  const float v = __ldg(sr + t);
  const int ylo = y + g.p - g.k + 1, xlo = x + g.p - g.k + 1;
  const int py0 = ylo <= 0 ? 0 : (ylo + g.s - 1) / g.s, py1 = min((y + g.p) / g.s, g.L[0].ny - 1);
  const int px0 = xlo <= 0 ? 0 : (xlo + g.s - 1) / g.s, px1 = min((x + g.p) / g.s, g.L[0].nx - 1);
  float out = 0.f;
  for (int py = py0; py <= py1; ++py)
    for (int px = px0; px <= px1; ++px) {
      const size_t q = (size_t)b * g.N + py * g.L[0].nx + px;
      int j = (int)idx[q];
      j = min(max(j, 0), g.M - 1);
      const BbgPatch Pc = bbg_candidate(gt, gt2, gt4, g, b, j);
      const float sel = bbg_value(Pc, c, y + g.p - py * g.s, x + g.p - px * g.s);
      if constexpr (MAP) scale = __ldg(grad_out + q) / (float)g.D;
      out += bbg_crit_grad(v - sel, criterion, scale);
    }
  d_sr[t] = out;
}

// one thread per (query patch, channel): minus the SR-side gradient lands on the selected candidate's pixels
// (PER_IMG: reduction='none', grad_out is [B] and image b scales by grad_out[b] / (N D); MAP: the loss map, grad_out
// is [B][N] and query i of image b scales by grad_out[b N + i] / D)
template <bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(256)
bbg_backward_gt_kernel(const float* __restrict__ sr, const float* __restrict__ gt, const float* __restrict__ gt2,
                       const float* __restrict__ gt4, const int64_t* __restrict__ idx, const float* __restrict__ grad_out,
                       BbgGeom g, int criterion, float* __restrict__ d0, float* __restrict__ d2, float* __restrict__ d4) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= (size_t)g.B * g.N * 3) return;
  const int c = (int)(t % 3);
  const size_t bi = t / 3;
  const int b = (int)(bi / g.N), i = (int)(bi - (size_t)b * g.N);
  int j = (int)idx[bi];
  j = min(max(j, 0), g.M - 1);
  const float scale = MAP ? __ldg(grad_out + bi) / (float)g.D
                          : __ldg(grad_out + (PER_IMG ? b : 0)) / ((float)(PER_IMG ? 1 : g.B) * (float)g.N * (float)g.D);
  const BbgPatch P1 = bbg_patch_of(sr + (size_t)b * 3 * g.L[0].H * g.L[0].W, g.L[0], g.p, g.s, i);
  const BbgPatch Pc = bbg_candidate(gt, gt2, gt4, g, b, j);
  const int l = j < g.L[0].n ? 0 : (j < g.L[0].n + g.L[1].n ? 1 : 2);
  float* dimg = (l == 0 ? d0 : (l == 1 ? d2 : d4)) + (size_t)b * 3 * Pc.H * Pc.W;
  for (int ky = 0; ky < g.k; ++ky)
    for (int kx = 0; kx < g.k; ++kx) {
      const int yy = Pc.y0 + ky, xx = Pc.x0 + kx;
      if (yy < 0 || yy >= Pc.H || xx < 0 || xx >= Pc.W) continue;  // padding carries no gradient
      const float d = bbg_value(Pc, c, ky, kx) - bbg_value(P1, c, ky, kx);
      const float gv = bbg_crit_grad(d, criterion, scale);
      if (gv != 0.f) atomicAdd(dimg + ((size_t)c * Pc.H + yy) * Pc.W + xx, gv);
    }
}

}  // namespace srst
