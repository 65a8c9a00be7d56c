// Structure-tensor loss for filter radii OUTSIDE the compiled classes (r_sigma > 4 or r_rho > 12, up to 64 each:
// sigma, rho <= 16.1).  The reference's radius max(int(4 sigma + 0.5), 1) is unbounded (utils.py:198); the tiled and
// marching kernels keep whole halos in shared memory and are compiled per radius class, so large radii take this
// path instead: the same separable passes (utils.py:212-233) and the same per-pixel chain (st_pixel2_raw), one
// thread per pixel, intermediates in global scratch planes supplied through the workspace argument.  It is a
// correctness path for hyper-parameter sweeps, not a tuned one: every pass is a coalesced 1-D correlation that reads
// its (2r+1)-tap window through L1/L2.
//
//   forward, per image:   RGB -> gray -> T1 = Ch(dg) gray, T2 = Ch(g) gray       (gen_gray_v)
//                         Ix = Cw(g) T1, Iy = Cw(dg) T2                          (gen_grad_h; saved for the backward)
//                         V = Ch(k) [Ix^2, Iy^2, Ix Iy]                          (gen_prod_v)
//                         S = Cw(k) V                                            (gen_smooth_h)
//            both images: chain + adjoint -> loss partials, ds_sr, ds_hr         (gen_chain)
//   backward:             V = Ch(k) ds ; E = Cw(k) V ; dIx = 2 Ix Exx + Iy Exy, dIy = 2 Iy Eyy + Ix Exy
//                         U1 = Cw(g) dIx, U2 = Cw(dg) dIy ; dgray = -(Ch(dg) U1 + Ch(g) U2) ; d_img = w_c dgray
// C(k) is the zero-padded cross-correlation of conv2d(padding='same'); h = along H (vertical), w = along W.
// In this path the saved "ixy" buffer is PLANAR: [B][2][H][W] (it fits: srst_st_ixy_floats >= 2 B H W).
#pragma once
#include "st_kernels.cuh"
#include "st_march.cuh"

namespace srst {

constexpr int kGenMaxR = 64;
constexpr int kGenNT = 256;
constexpr int kGenMaxPartials = 1024;

struct StGenTaps {
  int rs, rk;
  float g[2 * kGenMaxR + 1], dg[2 * kGenMaxR + 1], k[2 * kGenMaxR + 1];
};

struct StGenParams {
  const float* in0;   // pass input (image, plane set, ...)
  const float* in1;
  const float* in2;
  float* out0;
  float* out1;
  int B, H, W;
  float scale;
  StGenTaps taps;
};

// pixel index -> (b, y, x); returns false past the end
SRST_DEV bool gen_pixel(const StGenParams& P, size_t i, int& b, int& y, int& x) {
  const size_t plane = (size_t)P.H * P.W;
  if (i >= (size_t)P.B * plane) return false;
  b = (int)(i / plane);
  const size_t r = i - (size_t)b * plane;
  y = (int)(r / P.W);
  x = (int)(r - (size_t)y * P.W);
  return true;
}

// in0 = img [B,3,H,W] -> out0 = T1 = Ch(dg) gray, out1 = T2 = Ch(g) gray   ([B,H,W] each)
__global__ void __launch_bounds__(kGenNT) gen_gray_v_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const float* img = P.in0 + (size_t)b * 3 * plane + x;
  const int r = P.taps.rs;
  float t1 = 0.f, t2 = 0.f;
  for (int t = max(-r, -y); t <= min(r, P.H - 1 - y); ++t) {
    const float* p = img + (size_t)(y + t) * P.W;
    const float gv = gray_of(__ldg(p), __ldg(p + plane), __ldg(p + 2 * plane));
    t1 = fmaf(P.taps.dg[t + r], gv, t1);
    t2 = fmaf(P.taps.g[t + r], gv, t2);
  }
  P.out0[i] = t1;
  P.out1[i] = t2;
}

// in0 = T1, in1 = T2 -> out0 = planar ixy [B][2][H][W]: Ix = Cw(g) T1, Iy = Cw(dg) T2
__global__ void __launch_bounds__(kGenNT) gen_grad_h_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const int r = P.taps.rs;
  float ix = 0.f, iy = 0.f;
  for (int t = max(-r, -x); t <= min(r, P.W - 1 - x); ++t) {
    ix = fmaf(P.taps.g[t + r], __ldg(P.in0 + i + t), ix);
    iy = fmaf(P.taps.dg[t + r], __ldg(P.in1 + i + t), iy);
  }
  float* o = P.out0 + (size_t)b * 2 * plane + (size_t)y * P.W + x;
  o[0] = ix;
  o[plane] = iy;
}

// in0 = planar ixy -> out0 = V [B][3][H][W] = Ch(k) of the products (zero outside the image: utils.py:225-230)
__global__ void __launch_bounds__(kGenNT) gen_prod_v_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const float* pix = P.in0 + (size_t)b * 2 * plane + x;
  const int r = P.taps.rk;
  float vxx = 0.f, vyy = 0.f, vxy = 0.f;
  for (int t = max(-r, -y); t <= min(r, P.H - 1 - y); ++t) {
    const float ix = __ldg(pix + (size_t)(y + t) * P.W), iy = __ldg(pix + plane + (size_t)(y + t) * P.W);
    const float w = P.taps.k[t + r];
    vxx = fmaf(w, ix * ix, vxx);
    vyy = fmaf(w, iy * iy, vyy);
    vxy = fmaf(w, ix * iy, vxy);
  }
  float* o = P.out0 + (size_t)b * 3 * plane + (size_t)y * P.W + x;
  o[0] = vxx;
  o[plane] = vyy;
  o[2 * plane] = vxy;
}

// in0 = [B][3][H][W] -> out0 = Cw(k) in0, plane by plane (forward: S from V)
__global__ void __launch_bounds__(kGenNT) gen_smooth_h_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const size_t o = (size_t)b * 3 * plane + (size_t)y * P.W + x;
  const int r = P.taps.rk;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f;
  for (int t = max(-r, -x); t <= min(r, P.W - 1 - x); ++t) {
    const float w = P.taps.k[t + r];
    s0 = fmaf(w, __ldg(P.in0 + o + t), s0);
    s1 = fmaf(w, __ldg(P.in0 + o + plane + t), s1);
    s2 = fmaf(w, __ldg(P.in0 + o + 2 * plane + t), s2);
  }
  P.out0[o] = s0;
  P.out0[o + plane] = s1;
  P.out0[o + 2 * plane] = s2;
}

struct StGenChainParams {
  const float* s1;   // [B][3][H][W] raw SR tensor
  const float* s2;
  float* ds_sr;      // or null
  float* ds_hr;      // or null
  float* partials;   // [gridDim.x]
  unsigned int* ticket;
  float* loss_out;
  int B, H, W, normalize;
  float eps, inv_count;
};
// MAP: the distance map [B,H,W] (see StFwdMapParams)
struct StGenChainMapParams : StGenChainParams {
  float* map_out;
};

// chain of pixel i (flat over [B][H][W]): adds its distance to lsum, writes its ds_sr / ds_hr (and with MAP its
// distance to map[i])
template <bool MAP = false>
SRST_DEV void gen_chain_pixel(const StGenChainParams& P, size_t i, size_t plane, float& lsum, float* map = nullptr) {
  const size_t b = i / plane, o = b * 3 * plane + (i - b * plane);
  const float a = __ldg(P.s1 + o), bb = __ldg(P.s1 + o + plane), c = __ldg(P.s1 + o + 2 * plane);
  const float e = __ldg(P.s2 + o), f = __ldg(P.s2 + o + plane), h = __ldg(P.s2 + o + 2 * plane);
  StPixelGrad2 G;
  G.da = G.db = G.dc = G.de = G.df = G.dh = make_float2(0.f, 0.f);
  const float2 d = st_pixel2_raw<true, true>(bcast2(a), bcast2(bb), bcast2(c), bcast2(e), bcast2(f), bcast2(h),
                                            P.normalize != 0, P.eps, G);
  lsum += d.x;
  if constexpr (MAP) map[i] = d.x;
  if (P.ds_sr) { P.ds_sr[o] = G.da.x; P.ds_sr[o + plane] = G.db.x; P.ds_sr[o + 2 * plane] = G.dc.x; }
  if (P.ds_hr) { P.ds_hr[o] = G.de.x; P.ds_hr[o + plane] = G.df.x; P.ds_hr[o + 2 * plane] = G.dh.x; }
}

// per-pixel chain (utils.py:236-279) and its adjoint on both tensors; deterministic loss reduction (CTA partial ->
// workspace, last CTA sums in a fixed order in double and hands the ticket back zeroed).
// PER_IMG: reduction='none' -- the grid is gridDim.x / B CTAs per image, image-major, each striding over its own
// image only; loss_out[b] = the mean over image b's pixels (P.inv_count = 1 / (H W)).
// MAP: also stores every pixel's distance into P.map_out [B,H,W] (the loss and the other outputs are unchanged).
template <bool PER_IMG = false, bool MAP = false>
__global__ void __launch_bounds__(kGenNT)
gen_chain_kernel(const __grid_constant__ std::conditional_t<MAP, StGenChainMapParams, StGenChainParams> P) {
  static_assert(!(MAP && PER_IMG), "the distance map comes with the batch loss only");
  __shared__ float s_red[kGenNT / 32];
  __shared__ unsigned int s_last;
  const size_t plane = (size_t)P.H * P.W, npix = (size_t)P.B * plane;
  float lsum = 0.f;
  if constexpr (PER_IMG) {
    const unsigned int per = gridDim.x / P.B, b = blockIdx.x / per;
    const size_t end = (size_t)(b + 1) * plane;
    for (size_t i = (size_t)b * plane + (size_t)(blockIdx.x - b * per) * kGenNT + threadIdx.x; i < end; i += (size_t)per * kGenNT)
      gen_chain_pixel(P, i, plane, lsum);
  } else {
    for (size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x; i < npix; i += (size_t)gridDim.x * kGenNT) {
      if constexpr (MAP) gen_chain_pixel<true>(P, i, plane, lsum, P.map_out);
      else gen_chain_pixel(P, i, plane, lsum);
    }
  }
  lsum = warp_sum(lsum);
  if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = lsum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float bs = 0.f;
    for (int w = 0; w < kGenNT / 32; ++w) bs += s_red[w];
    P.partials[blockIdx.x] = bs;
    __threadfence();
    const unsigned int tk = atomicAdd(P.ticket, 1u);
    s_last = (tk == gridDim.x - 1) ? 1u : 0u;
  }
  __syncthreads();
  if constexpr (PER_IMG) {
    if (s_last) {
      __threadfence();
      reduce_partials_per_image(P.partials, P.B, gridDim.x / P.B, (double)P.inv_count, P.loss_out);
      if (threadIdx.x == 0) *P.ticket = 0u;
    }
  } else if (s_last && threadIdx.x < 32) {
    __threadfence();
    double acc = 0.0;
    for (unsigned int i = threadIdx.x; i < gridDim.x; i += 32) acc += (double)__ldcg(P.partials + i);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (threadIdx.x == 0) {
      P.loss_out[0] = (float)(acc * (double)P.inv_count);
      *P.ticket = 0u;
    }
  }
}

// backward: in0 = ds [B][3][H][W] -> out0 = Ch(k) ds  (the adjoint of the zero-padded symmetric smoothing is itself)
__global__ void __launch_bounds__(kGenNT) gen_smooth_v_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const float* p = P.in0 + (size_t)b * 3 * plane + x;
  const int r = P.taps.rk;
  float s0 = 0.f, s1 = 0.f, s2 = 0.f;
  for (int t = max(-r, -y); t <= min(r, P.H - 1 - y); ++t) {
    const float w = P.taps.k[t + r];
    const float* q = p + (size_t)(y + t) * P.W;
    s0 = fmaf(w, __ldg(q), s0);
    s1 = fmaf(w, __ldg(q + plane), s1);
    s2 = fmaf(w, __ldg(q + 2 * plane), s2);
  }
  float* o = P.out0 + (size_t)b * 3 * plane + (size_t)y * P.W + x;
  o[0] = s0;
  o[plane] = s1;
  o[2 * plane] = s2;
}

// backward: in0 = V = Ch(k) ds, in1 = planar ixy -> out0 = [B][2][H][W]: dIx, dIy  (adjoint of utils.py:225-229)
__global__ void __launch_bounds__(kGenNT) gen_bwd_prod_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const size_t o3 = (size_t)b * 3 * plane + (size_t)y * P.W + x, o2 = (size_t)b * 2 * plane + (size_t)y * P.W + x;
  const int r = P.taps.rk;
  float exx = 0.f, eyy = 0.f, exy = 0.f;
  for (int t = max(-r, -x); t <= min(r, P.W - 1 - x); ++t) {
    const float w = P.taps.k[t + r];
    exx = fmaf(w, __ldg(P.in0 + o3 + t), exx);
    eyy = fmaf(w, __ldg(P.in0 + o3 + plane + t), eyy);
    exy = fmaf(w, __ldg(P.in0 + o3 + 2 * plane + t), exy);
  }
  const float ix = __ldg(P.in1 + o2), iy = __ldg(P.in1 + o2 + plane);
  P.out0[o2] = fmaf(2.0f * ix, exx, iy * exy);
  P.out0[o2 + plane] = fmaf(2.0f * iy, eyy, ix * exy);
}

// backward: in0 = [B][2][H][W] dIx, dIy -> out0 = [B][2][H][W]: U1 = Cw(g) dIx, U2 = Cw(dg) dIy
__global__ void __launch_bounds__(kGenNT) gen_bwd_gh_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const size_t o2 = (size_t)b * 2 * plane + (size_t)y * P.W + x;
  const int r = P.taps.rs;
  float u1 = 0.f, u2 = 0.f;
  for (int t = max(-r, -x); t <= min(r, P.W - 1 - x); ++t) {
    u1 = fmaf(P.taps.g[t + r], __ldg(P.in0 + o2 + t), u1);
    u2 = fmaf(P.taps.dg[t + r], __ldg(P.in0 + o2 + plane + t), u2);
  }
  P.out0[o2] = u1;
  P.out0[o2 + plane] = u2;
}

// backward: in0 = U1, U2; in1 = grad_out (device scalar) -> out0 = d_img [B,3,H,W]:
// dgray = -(Ch(dg) U1 + Ch(g) U2) (g symmetric, dg antisymmetric: the adjoint flips the taps), times the upstream
// gradient / (B H W), spread over the channels with the grayscale weights.
// PER_IMG: in1 = grad_out [B]; pixel of image b scales by grad_out[b] (P.scale = 1 / (H W))
template <bool PER_IMG = false>
__global__ void __launch_bounds__(kGenNT) gen_bwd_gv_kernel(const __grid_constant__ StGenParams P) {
  const size_t i = (size_t)blockIdx.x * kGenNT + threadIdx.x;
  int b, y, x;
  if (!gen_pixel(P, i, b, y, x)) return;
  const size_t plane = (size_t)P.H * P.W;
  const float* p = P.in0 + (size_t)b * 2 * plane + x;
  const int r = P.taps.rs;
  float acc = 0.f;
  for (int t = max(-r, -y); t <= min(r, P.H - 1 - y); ++t) {
    const float* q = p + (size_t)(y + t) * P.W;
    acc = fmaf(P.taps.dg[t + r], __ldg(q), acc);
    acc = fmaf(P.taps.g[t + r], __ldg(q + plane), acc);
  }
  const float dgr = acc * (-__ldg(P.in1 + (PER_IMG ? b : 0)) * P.scale);
  float* o = P.out0 + (size_t)b * 3 * plane + (size_t)y * P.W + x;
  o[0] = kGrayR * dgr;
  o[plane] = kGrayG * dgr;
  o[2 * plane] = kGrayB * dgr;
}

}  // namespace srst
