/* srst.h -- C ABI of libsrst.so: the B200-native structure-tensor / Best-Buddy loss hot path.
 *
 * This is the drop-in boundary for the loss hot path of SebastianBitsch/SRGAN-ST.  The reference
 * has no native code: the hot path is a chain of ATen calls behind two nn.Modules
 * (loss.py:380-413 StructureTensorLoss, loss.py:78-141 BestBuddyLoss).  Each entry point below
 * names the reference code it replaces.  The Python host (srgan_st_b200/loss.py) binds these with
 * ctypes from inside a torch.autograd.Function; INTEGRATION.md shows the binding.
 *
 * Conventions
 *   - every function returns int: 0 = ok, >0 = a cudaError_t value, <0 = an SRST_E_* code.
 *   - image/gradient buffers are DEVICE pointers to contiguous fp32 NCHW tensors owned by the
 *     caller; filter taps are HOST pointers (they are copied into kernel parameters).
 *   - no function allocates, synchronises or keeps state: all work is enqueued on `stream`
 *     (a cudaStream_t passed as void*) and every scratch buffer comes in through `workspace`.
 *     The library is re-entrant across streams and devices as long as workspaces differ.
 *   - there is no CPU fallback anywhere behind this ABI.
 */
#ifndef SRST_H_
#define SRST_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define SRST_VERSION 208 /* major*100 + minor: the major number changes whenever an argument list changes */

#define SRST_E_INVALID (-1)     /* null pointer / non-positive size / bad enum */
#define SRST_E_UNSUPPORTED (-2) /* filter radius or patch geometry not compiled in */
#define SRST_E_WORKSPACE (-3)   /* workspace missing, misaligned or too small */
#define SRST_E_SHAPE (-4)       /* image shape not usable by this entry point */

int srst_version(void);
const char* srst_error_string(int code);

/* ---------------------------------------------------------------------------------------------
 * Structure-tensor loss.   Replaces, fused into one kernel per direction:
 *   torchvision Grayscale                        (loss.py:400-401)
 *   utils.structure_tensor  (10 conv2d / image)  (utils.py:212-233)
 *   utils.normalize / compute_invS1xS2           (utils.py:236-254)
 *   utils.compute_eigenvalues / compute_distance (utils.py:257-279)
 *   .mean() over pixels and batch                (loss.py:409,413)
 * and the autograd backward of that chain.
 *
 * g, dg: 2*r_sigma+1 host floats (utils.get_gaussian_kernel(sigma, also_dg=True), utils.py:194-208)
 * k    : 2*r_rho+1   host floats (utils.get_gaussian_kernel(rho))
 * Radii are padded with zero taps to the compiled classes r_sigma in {2,4}, r_rho in {4,8,12} (shared-memory
 * kernels; the reference default sigma=0.5, rho=2.0 is (2, 8)).  Larger radii, up to 64 each -- the reference's
 * radius max(int(4 sigma + 0.5), 1) is unbounded, utils.py:198 -- run on the generic-radius path: the same passes,
 * one thread per pixel, intermediates in global scratch planes (srst_st_workspace_bytes_r,
 * srst_st_backward_workspace_bytes, srst_st_backward_ws).
 * ------------------------------------------------------------------------------------------- */

/* 1 if the (r_sigma, r_rho) pair fits a compiled radius class, 2 if it takes the generic-radius path
 * (srst_st_forward + srst_st_backward_ws only; not the fused Pixel variant, not srst_st_features), else 0. */
int srst_st_supported(int r_sigma, int r_rho);

/* Tile-shape override for tests and tuning sweeps: force compiled forward / backward tile configuration
 * fwd_cfg / bwd_cfg (0 .. srst_st_num_cfgs(0|1) - 1) for the default radius class, -1 = the library's own
 * choice.  Process-wide; the environment variables SRST_ST_FWD_CFG / SRST_ST_BWD_CFG set the initial value
 * (read once). */
int srst_st_num_cfgs(int backward);
int srst_st_force_cfg(int fwd_cfg, int bwd_cfg);
/* Forward cfgs 0-2 are tiled shapes (32x64, 24x96 with two or three CTAs per SM), 3 and 4 the row-marching kernel
 * (96- / 112-column strips); backward cfgs: 0 = 28x56 tiles, 1 = 12x96 strips (both persistent).  The marching kernel cuts a strip into row chunks so
 * that small batches fill the machine; `blocks` > 0 forces the chunk height to blocks*16 rows (tests), <= 0 hands
 * the choice back to the library.  Process-wide; SRST_ST_CHUNK_BLOCKS sets the initial value. */
int srst_st_force_chunk_blocks(int blocks);

/* Scratch bytes srst_st_forward / srst_stpx_forward need for a [B,3,H,W] problem (per-CTA partial sums + ticket).
 * The workspace must be 16-byte aligned; its first 16 bytes (the ticket counter) must be ZERO before the
 * first use.  Every launch writes its partial sums before reading them and hands the ticket back zeroed,
 * so the buffer can be reused by later calls on the same stream; do not share one buffer between
 * streams, or between this entry point and the patch-loss entry points (they lay it out differently). */
size_t srst_st_workspace_bytes(int B, int H, int W);
/* Same, for a given radius pair: equal to srst_st_workspace_bytes() for the compiled classes; the generic-radius
 * path adds eleven [B,H,W] fp32 scratch planes (smoothed tensors of both images, one pass buffer, Ix/Iy when they
 * are not saved).  0 if the pair is not supported at all. */
size_t srst_st_workspace_bytes_r(int B, int H, int W, int r_sigma, int r_rho);
/* Scratch bytes srst_st_backward_ws needs: 0 for the compiled classes, five [B,H,W] fp32 planes on the
 * generic-radius path (no zero-initialisation required). */
size_t srst_st_backward_workspace_bytes(int B, int H, int W, int r_sigma, int r_rho);

/* Number of floats of a saved-gradient buffer ("ixy") for a [B,3,H,W] problem: [B][2][ceil(H/2)][W][2],
 * plane 0 = Ix (derivative along H), plane 1 = Iy, rows 2p / 2p+1 of a column interleaved (the layout the
 * kernels use in shared memory, so the backward fetches its tile with one TMA box copy). */
size_t srst_st_ixy_floats(int B, int H, int W);

/* Forward.  sr, hr: device [B,3,H,W] fp32.  Writes
 *   loss_out[0]  = mean over B*H*W pixels of the Riemannian distance   (device, 1 float)
 *   ds_sr        = d(sum of distances)/d(Jxx,Jyy,Jxy of SR), device [B,3,H,W], or NULL to skip
 *   ds_hr        = same w.r.t. the HR tensor, or NULL (only needed when hr requires grad)
 *   ixy_sr/_hr   = the Gaussian-derivative gradients Ix, Iy of the grayscale image (utils.py:219-222),
 *                  srst_st_ixy_floats() floats each, or NULL; required next to the matching ds_*
 * ds_* and ixy_* are the "saved intermediates" the backward pass consumes (20 B/pixel); ds is unscaled
 * (neither 1/(B*H*W) nor the upstream gradient is applied yet). */
int srst_st_forward(const float* sr, const float* hr, int B, int H, int W,
                    const float* g, const float* dg, int r_sigma,
                    const float* k, int r_rho,
                    int normalize, float eps,
                    float* loss_out, float* ds_sr, float* ds_hr, float* ixy_sr, float* ixy_hr,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Backward for one image tensor (sr or hr): ixy, ds = the matching ixy_* / ds_* buffers the forward
 * wrote; grad_out: device pointer to the upstream scalar gradient.  The image itself is not read again.
 * Writes d_img[B,3,H,W] = grad_out/(B*H*W) * dLoss_sum/dimg (adjoint smoothing, product rule,
 * adjoint Gaussian-derivative filters, grayscale weights).
 * Ordering: plain stream order -- every input may be produced by the kernel enqueued immediately before
 * this call on `stream` (the kernel waits for its predecessor before its first global read). */
int srst_st_backward(const float* ixy, const float* ds, const float* grad_out,
                     int B, int H, int W,
                     const float* g, const float* dg, int r_sigma,
                     const float* k, int r_rho,
                     float* d_img, void* stream);
/* Same with a scratch buffer: the only backward entry point of the generic-radius path (srst_st_backward returns
 * SRST_E_WORKSPACE there); for the compiled classes `workspace` is ignored and may be NULL.  On the generic path
 * the saved ixy buffer is planar [B][2][H][W] (written by srst_st_forward with the same radii). */
int srst_st_backward_ws(const float* ixy, const float* ds, const float* grad_out,
                        int B, int H, int W,
                        const float* g, const float* dg, int r_sigma,
                        const float* k, int r_rho,
                        float* d_img, void* workspace, size_t workspace_bytes, void* stream);

/* Per-image reduction (reduction='none'; the reference's vmap(st_loss)(x, gt) before its .mean(), loss.py:411-413).
 * Same arguments, checks, return codes, workspace and saved buffers as srst_st_forward / srst_st_backward_ws, for the
 * compiled radius classes and the generic-radius path alike, but
 *   srst_st_forward_per_image:  loss_out[b] = mean over the H*W pixels of image b   (device, B floats)
 *   srst_st_backward_per_image: grad_out = device [B], the upstream gradient of each loss_out[b] (any values, e.g.
 *                               all equal after .sum()); d_img of image b = grad_out[b]/(H*W) * dLoss_b/dimg
 * The tile shapes are the ones srst_st_forward / srst_st_backward pick, and each image's pixels are reduced in double
 * in a fixed order, so results are deterministic; d_img of image b is bit-identical to srst_st_backward_ws on that
 * image alone (B = 1) with grad_out[b]. */
int srst_st_forward_per_image(const float* sr, const float* hr, int B, int H, int W,
                              const float* g, const float* dg, int r_sigma,
                              const float* k, int r_rho,
                              int normalize, float eps,
                              float* loss_out, float* ds_sr, float* ds_hr, float* ixy_sr, float* ixy_hr,
                              void* workspace, size_t workspace_bytes, void* stream);
int srst_st_backward_per_image(const float* ixy, const float* ds, const float* grad_out,
                               int B, int H, int W,
                               const float* g, const float* dg, int r_sigma,
                               const float* k, int r_rho,
                               float* d_img, void* workspace, size_t workspace_bytes, void* stream);

/* Per-pixel distance map (the element-wise form of the loss: the map d = utils.compute_distance(L) that st_loss builds
 * before its .mean(), loss.py:408-409, utils.py:269-279), e.g. for spatial weighting or masking of the loss and for
 * loss heat maps.
 *   srst_st_forward_map: the arguments of srst_st_forward with map_out (device [B,H,W] fp32, required) after loss_out.
 *     Same checks, return codes and workspace (srst_st_workspace_bytes_r); compiled radius classes and the generic-radius
 *     path.  map_out[b,y,x] = the distance of pixel (y, x) of image b.  loss_out[0], ds_* and ixy_* are bit-identical to
 *     srst_st_forward on the same inputs (the same tile shapes are picked), so loss_out[0] = mean(map_out) up to the
 *     order of the summation.
 *   srst_st_backward_map: d_img = sum over pixels p of grad_map[p] * d(map_out[p])/d(img), for one image tensor.
 *     ixy, ds as for srst_st_backward (the unscaled buffers the forward wrote; they are only read, so the call can be
 *     repeated); grad_map: device [B,H,W], any values.  A prepass writes grad_map * ds into the workspace, then the
 *     srst_st_backward kernels run on it with a unit upstream gradient.  The workspace is always required
 *     (srst_st_backward_map_workspace_bytes; no zero-initialisation needed).  Ordering as for srst_st_backward.
 *   srst_st_backward_map_workspace_bytes: the weighted ds planes (12 B/px) plus a 256-byte slot, plus
 *     srst_st_backward_workspace_bytes on the generic-radius path; 0 for unsupported radii or non-positive sizes. */
int srst_st_forward_map(const float* sr, const float* hr, int B, int H, int W,
                        const float* g, const float* dg, int r_sigma,
                        const float* k, int r_rho,
                        int normalize, float eps,
                        float* loss_out, float* map_out, float* ds_sr, float* ds_hr, float* ixy_sr, float* ixy_hr,
                        void* workspace, size_t workspace_bytes, void* stream);
size_t srst_st_backward_map_workspace_bytes(int B, int H, int W, int r_sigma, int r_rho);
int srst_st_backward_map(const float* ixy, const float* ds, const float* grad_map,
                         int B, int H, int W,
                         const float* g, const float* dg, int r_sigma,
                         const float* k, int r_rho,
                         float* d_img, void* workspace, size_t workspace_bytes, void* stream);

/* Structure-tensor FEATURES of one image tensor (diagnostic output; BASELINE.json north_star: "closed-form 2x2
 * eigendecomposition giving orientation, coherence and eigenvalues").  The reference computes these only in an
 * exploration notebook through the third-party `structure_tensor` package (data-exploration/structure_tensor.ipynb,
 * cells 12-18: eig_special_2d, arctan2 of the eigenvector, 1 - val[0]/val[1]), which is not part of its checkout:
 * the definitions below are this library's own (parity unpinned).
 *   J_out      [B,3,H,W]  Jxx, Jyy, Jxy: the smoothed tensor of utils.structure_tensor (utils.py:212-233)
 *   eig_out    [B,2,H,W]  lambda_small, lambda_large = (Jxx+Jyy)/2 -/+ sqrt(((Jxx-Jyy)/2)^2 + Jxy^2)
 *   orient_out [B,H,W]    1/2 atan2(2 Jxy, Jxx - Jyy): angle of the dominant-gradient eigenvector against the H axis
 *   coher_out  [B,H,W]    1 - lambda_small / lambda_large (0 where lambda_large == 0)
 * Any output may be NULL (at least one must be given).  No gradient. */
int srst_st_features(const float* img, int B, int H, int W,
                     const float* g, const float* dg, int r_sigma,
                     const float* k, int r_rho,
                     float* J_out, float* eig_out, float* orient_out, float* coher_out, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Structure-tensor loss with the "Pixel" MSE criterion fused in (SURVEY.md 8f rank 4).  The warm-up
 * and training loops evaluate MSELoss(sr, gt) and StructureTensorLoss(sr, gt) on the same two
 * tensors one after the other (warmup.py:88-96, train.py:131-144, criteria registered in
 * config.py:71-93); here the squared RGB difference is accumulated while the forward kernel has
 * the HR tile in registers, and the backward kernel adds 2 (sr - hr) / (3 B H W) * grad_px to d_sr
 * in its final store -- no extra pass over either tensor.
 *   loss2_out[0] = structure-tensor loss (as srst_st_forward), loss2_out[1] = mean((sr - hr)^2)
 *   grad_st, grad_px: device scalars, the upstream gradients of the two terms.
 * Workspace: srst_st_workspace_bytes.
 * ------------------------------------------------------------------------------------------- */
int srst_stpx_forward(const float* sr, const float* hr, int B, int H, int W,
                      const float* g, const float* dg, int r_sigma,
                      const float* k, int r_rho,
                      int normalize, float eps,
                      float* loss2_out, float* ds_sr, float* ixy_sr,
                      void* workspace, size_t workspace_bytes, void* stream);
int srst_stpx_backward(const float* sr, const float* hr, const float* ixy, const float* ds,
                       const float* grad_st, const float* grad_px,
                       int B, int H, int W,
                       const float* g, const float* dg, int r_sigma,
                       const float* k, int r_rho,
                       float* d_sr, void* stream);

/* Per-image reduction (reduction='none') of the fused criterion.  Same arguments, checks, return codes, workspace and
 * saved buffers as srst_stpx_forward / srst_stpx_backward (generic radii: SRST_E_UNSUPPORTED), but
 *   srst_stpx_forward_per_image:  loss2_out = device [2][B]: loss2_out[b] = mean of the ST distance over image b's
 *                                 H*W pixels (as srst_st_forward_per_image), loss2_out[B + b] = mean((sr_b - hr_b)^2)
 *                                 over its 3*H*W values
 *   srst_stpx_backward_per_image: grad_st, grad_px = device [B] each (any values); d_sr of image b =
 *                                 grad_st[b]/(H*W) * dST_b/dsr + grad_px[b] * 2 (sr_b - hr_b) / (3*H*W)
 * The tile shapes are the ones the scalar entry points pick and each image's terms are reduced in double in a fixed
 * order; d_sr of image b is bit-identical to srst_stpx_backward on that image alone with (grad_st[b], grad_px[b]). */
int srst_stpx_forward_per_image(const float* sr, const float* hr, int B, int H, int W,
                                const float* g, const float* dg, int r_sigma,
                                const float* k, int r_rho,
                                int normalize, float eps,
                                float* loss2_out, float* ds_sr, float* ixy_sr,
                                void* workspace, size_t workspace_bytes, void* stream);
int srst_stpx_backward_per_image(const float* sr, const float* hr, const float* ixy, const float* ds,
                                 const float* grad_st, const float* grad_px,
                                 int B, int H, int W,
                                 const float* g, const float* dg, int r_sigma,
                                 const float* k, int r_rho,
                                 float* d_sr, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Best-Buddy loss.   Replaces
 *   F.unfold x4, torch.cat                        (loss.py:116-130)
 *   utils.batch_pairwise_distance(...,'l2') x2    (utils.py:173-187; two torch.bmm)
 *   torch.min(score, dim=2), torch.gather         (loss.py:135-137)
 *   L1Loss / MSELoss                              (loss.py:139)
 * for ksize=3, stride=3, pad=0 (27-dim patches).  gt2 / gt4 are the bicubic x1/2 and x1/4
 * levels of gt ([B,3,H/2,W/2], [B,3,H/4,W/4]); pass NULL to have the library compute them with
 * the same taps F.interpolate(mode='bicubic', align_corners=False) uses (loss.py:123,127),
 * in which case `workspace` must also hold them (see srst_bb_workspace_bytes).
 * H, W >= 12; sizes that are not multiples of 3 / 12 follow the floor semantics of F.unfold and
 * F.interpolate(scale_factor=...).
 * ------------------------------------------------------------------------------------------- */
#define SRST_BB_L1 0
#define SRST_BB_L2 1
/* OR-ed into `criterion` of the three *_forward entry points below: search with dist_norm='l1'
 * (utils.py:166-172: alpha * sum|x - y| + beta * sum|g - y|) instead of the default squared l2 distance.  Every pair is
 * scored exactly then (no filter); the backward entry points ignore the flag (they only need the indices). */
#define SRST_BB_DIST_L1 0x100

size_t srst_bb_workspace_bytes(int B, int H, int W);

/* Forward: idx_out[B, N] int64 (N = (H/3)*(W/3)) = argmin over the M = N + N/4 + N/16 candidate
 * patches of alpha*d(sr_i, cand_j) + beta*d(gt_i, cand_j), first minimal index on ties
 * (torch.min rule); loss_out[0] = mean |sr_patch - cand[idx]| (L1) or mean square (L2). */
int srst_bb_forward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                    int B, int H, int W, float alpha, float beta, int criterion,
                    int64_t* idx_out, float* loss_out,
                    void* workspace, size_t workspace_bytes, void* stream);

/* Backward: only the final criterion is differentiable w.r.t. sr (loss.py:139; argmin is not).
 * d_sr[B,3,H,W] = grad_out/(B*N*27) * sign(sr_patch - cand[idx])           (L1)
 *               = grad_out/(B*N*27) * 2*(sr_patch - cand[idx])             (L2)     */
int srst_bb_backward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                     const int64_t* idx, const float* grad_out,
                     int B, int H, int W, int criterion,
                     float* d_sr, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Gram loss (reference loss.py:146-225): the same three-level best-buddy search, but every 3x3x3
 * patch is replaced by its 3x3 Gram matrix (features [3][9], G = F F^T / 27; 9-dim descriptor) for
 * both the search and the final L1/MSE criterion.  Workspace: srst_bb_workspace_bytes.
 *   d_sr = through the criterion and the Gram descriptor of the SR patch (argmin is not differentiated).
 * ------------------------------------------------------------------------------------------- */
int srst_gram_forward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                      int B, int H, int W, float alpha, float beta, int criterion,
                      int64_t* idx_out, float* loss_out,
                      void* workspace, size_t workspace_bytes, void* stream);
int srst_gram_backward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                       const int64_t* idx, const float* grad_out,
                       int B, int H, int W, int criterion,
                       float* d_sr, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Patchwise structure-tensor loss (reference loss.py:292-375): the same three-level best-buddy
 * search, but every 3x3x3 patch is replaced by the det-normalised structure tensor of the patch
 * seen as a 3x3 image (Grayscale -> utils.structure_tensor(sigma, rho) with zero 'same' padding
 * -> utils.normalize; 27-dim descriptor c*9 + y*3 + x, c in Jxx,Jyy,Jxy), replacing
 *   vmap(vmap(s_norm)) over [B,N,3,3,3]            (loss.py:325-345)
 *   batch_pairwise_distance x2, torch.min, gather  (loss.py:361-369)
 *   L1Loss / MSELoss on the descriptors            (loss.py:371)
 * g, dg, k: host taps as for srst_st_forward; any radius >= 1 is accepted (a 3x3 image only sees
 * the five central taps).  Workspace: srst_bb_workspace_bytes.
 *   d_sr = through the criterion, utils.normalize and the structure tensor of the SR patch
 *          (argmin is not differentiated).
 * ------------------------------------------------------------------------------------------- */
int srst_pst_forward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                     int B, int H, int W,
                     const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                     float alpha, float beta, int criterion,
                     int64_t* idx_out, float* loss_out,
                     void* workspace, size_t workspace_bytes, void* stream);
int srst_pst_backward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                      const int64_t* idx, const float* grad_out,
                      int B, int H, int W,
                      const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                      int criterion,
                      float* d_sr, void* workspace, size_t workspace_bytes, void* stream);

/* Gradient w.r.t. gt of the three patch losses: the reference's gather of the selected candidates is differentiable
 * in p2_cat (loss.py:136-139, :219-222, :369-371), so a gt that requires grad receives, per query, minus the SR-side
 * criterion gradient pushed through the descriptor of the SELECTED candidate, accumulated over the queries that chose
 * it, and folded back through the bicubic pyramid taps for candidates of the two coarse levels.
 *   mode: 0 = BestBuddyLoss, 1 = GramLoss, 2 = PatchwiseStructureTensorLoss (g, dg, k as for srst_pst_forward;
 *         ignored, may be NULL, for modes 0 and 1).
 *   d_gt [B,3,H,W] is overwritten.  Workspace: srst_bb_workspace_bytes (always required).  Sums over queries use
 *   atomicAdd: the result can differ in the last bits from run to run. */
int srst_patch_backward_gt(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                           const int64_t* idx, const float* grad_out,
                           int B, int H, int W,
                           const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                           int criterion,
                           float* d_gt, void* workspace, size_t workspace_bytes, void* stream);

/* Per-image reduction (reduction='none') of the three default-geometry patch losses.
 *   mode: 0 = BestBuddyLoss, 1 = GramLoss, 2 = PatchwiseStructureTensorLoss (g, dg, k as for srst_pst_forward;
 *         ignored, may be NULL, for modes 0 and 1); any other mode: SRST_E_INVALID.
 * srst_patch_forward_per_image: the arguments of srst_bb_forward / srst_gram_forward / srst_pst_forward (criterion with
 *   SRST_BB_DIST_L1, gt2 / gt4, workspace: srst_bb_workspace_bytes), but loss_out[b] = the mean over image b's N*D
 *   criterion terms (device, B floats): the reference module applied to image b alone.  idx_out is the same as there.
 * srst_patch_backward_per_image: grad_out = device [B]; d_sr = the srst_*_backward result with image b scaled by
 *   grad_out[b]/(N*D) instead of grad_out[0]/(B*N*D) (bit-identical to the scalar entry point on image b alone), d_gt
 *   = the srst_patch_backward_gt result likewise (atomicAdd: last bits may vary).  Either of d_sr / d_gt may be NULL,
 *   not both.  The workspace is required whenever d_gt is given or gt2 / gt4 are NULL.
 * Return codes as the scalar entry points; the per-image forward may overwrite the x1/2 pyramid level it built in the
 * workspace (the backward entry points rebuild it). */
int srst_patch_forward_per_image(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                                 int B, int H, int W,
                                 const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                                 float alpha, float beta, int criterion,
                                 int64_t* idx_out, float* loss_out,
                                 void* workspace, size_t workspace_bytes, void* stream);
int srst_patch_backward_per_image(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                                  const int64_t* idx, const float* grad_out,
                                  int B, int H, int W,
                                  const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                                  int criterion,
                                  float* d_sr, float* d_gt, void* workspace, size_t workspace_bytes, void* stream);

/* Per-patch loss map (the element-wise form of the three patch losses: one criterion value per query patch, the
 * `L1Loss()(p1, sel_p2)` / MSELoss terms of loss.py:139, :222, :371 before their mean), e.g. for spatial weighting or
 * masking of the loss and for heat maps of the patches that found no good buddy.
 *   srst_patch_forward_map: the arguments of srst_patch_forward_per_image with map_out (device [B][N] fp32, required)
 *     after loss_out.  map_out[b*N + n] = the mean over the D criterion terms of query patch n of image b against its
 *     selected candidate (D = 27 for modes 0 and 2, 9 for mode 1).  loss_out[0] and idx_out are bit-identical to
 *     srst_bb_forward / srst_gram_forward / srst_pst_forward on the same inputs (same search, same loss grid, same
 *     reduction order), so loss_out[0] = mean(map_out) up to the order of the summation.
 *   srst_patch_backward_map: the arguments of srst_patch_backward_per_image with grad_map (device [B][N], any values)
 *     in place of grad_out: query n of image b contributes with scale grad_map[b*N + n] / D, so d_sr / d_gt = the
 *     gradient of sum(grad_map * map_out).  Either of d_sr / d_gt may be NULL, not both; d_gt sums with atomicAdd (last
 *     bits may vary, as for srst_patch_backward_gt).
 * A NULL map_out / grad_map returns SRST_E_INVALID; every other check, return code and workspace rule is that of the
 * per-image twins. */
int srst_patch_forward_map(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                           int B, int H, int W,
                           const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                           float alpha, float beta, int criterion,
                           int64_t* idx_out, float* loss_out, float* map_out,
                           void* workspace, size_t workspace_bytes, void* stream);
int srst_patch_backward_map(int mode, const float* sr, const float* gt, const float* gt2, const float* gt4,
                            const int64_t* idx, const float* grad_map,
                            int B, int H, int W,
                            const float* g, const float* dg, int r_sigma, const float* k, int r_rho,
                            int criterion,
                            float* d_sr, float* d_gt, void* workspace, size_t workspace_bytes, void* stream);

/* ---------------------------------------------------------------------------------------------
 * Best-Buddy loss with an arbitrary patch geometry: BestBuddyLoss(ksize, pad, stride) of the reference
 * (loss.py:86; F.unfold(kernel_size=ksize, padding=pad, stride=stride) at loss.py:116-129) for everything
 * but the default (3, 0, 3), which the tuned entry points above serve.  1 <= ksize <= 8, 0 <= pad <= 64, 1 <= stride <= 4096
 * (srst_bbg_supported);
 * patches may overlap (stride < ksize), leave gaps (stride > ksize) and reach into the zero padding.
 *   N = ny*nx, ny = (H + 2 pad - ksize)/stride + 1 (srst_bbg_num_patches); every pyramid level must hold at least
 *   one patch (F.unfold raises otherwise): SRST_E_SHAPE.  D = 3*ksize*ksize elements per patch.
 * Every (query, candidate) pair is scored exactly (no filter); criterion / SRST_BB_DIST_L1, gt2 / gt4 and the
 * first-minimum rule as for srst_bb_forward.  Workspace: srst_bbg_workspace_bytes (always required; 0 = geometry or
 * shape not usable).
 * Backward: d_sr [B,3,H,W] sums, per pixel and in a fixed order, the criterion gradients grad_out/(B*N*D) *
 * sign(sr_patch - cand[idx]) (or 2*diff) of the patches that cover the pixel; d_gt [B,3,H,W] is the gradient through
 * the gather of the selected candidates (loss.py:136-139; atomicAdd, then the bicubic pyramid adjoint).  Either of
 * d_sr / d_gt may be NULL.
 * ------------------------------------------------------------------------------------------- */
int srst_bbg_supported(int ksize, int pad, int stride);
size_t srst_bbg_workspace_bytes(int B, int H, int W, int ksize, int pad, int stride);
long long srst_bbg_num_patches(int H, int W, int ksize, int pad, int stride);
int srst_bbg_forward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                     int B, int H, int W, int ksize, int pad, int stride,
                     float alpha, float beta, int criterion,
                     int64_t* idx_out, float* loss_out,
                     void* workspace, size_t workspace_bytes, void* stream);
int srst_bbg_backward(const float* sr, const float* gt, const float* gt2, const float* gt4,
                      const int64_t* idx, const float* grad_out,
                      int B, int H, int W, int ksize, int pad, int stride, int criterion,
                      float* d_sr, float* d_gt,
                      void* workspace, size_t workspace_bytes, void* stream);

/* Per-image reduction (reduction='none') of the arbitrary-geometry path: the arguments, checks and workspace of
 * srst_bbg_forward / srst_bbg_backward, but loss_out[b] = the mean over image b's N*D terms (device, B floats) and
 * grad_out = device [B] (image b's gradients scaled by grad_out[b]/(N*D)). */
int srst_bbg_forward_per_image(const float* sr, const float* gt, const float* gt2, const float* gt4,
                               int B, int H, int W, int ksize, int pad, int stride,
                               float alpha, float beta, int criterion,
                               int64_t* idx_out, float* loss_out,
                               void* workspace, size_t workspace_bytes, void* stream);
int srst_bbg_backward_per_image(const float* sr, const float* gt, const float* gt2, const float* gt4,
                                const int64_t* idx, const float* grad_out,
                                int B, int H, int W, int ksize, int pad, int stride, int criterion,
                                float* d_sr, float* d_gt,
                                void* workspace, size_t workspace_bytes, void* stream);

/* Per-patch loss map of the arbitrary-geometry path: the arguments, checks and workspace of srst_bbg_forward_per_image /
 * srst_bbg_backward_per_image, with map_out (device [B][N] fp32, required) after loss_out and grad_map (device [B][N])
 * in place of grad_out, as for srst_patch_forward_map / srst_patch_backward_map.  D = 3*ksize*ksize, N and the
 * row-major patch order as F.unfold.  loss_out[0] and idx_out are bit-identical to srst_bbg_forward.  d_sr stays
 * deterministic: a pixel sums the gradients of the patches that cover it, each with its own weight, in a fixed order.
 * A NULL map_out / grad_map returns SRST_E_INVALID. */
int srst_bbg_forward_map(const float* sr, const float* gt, const float* gt2, const float* gt4,
                         int B, int H, int W, int ksize, int pad, int stride,
                         float alpha, float beta, int criterion,
                         int64_t* idx_out, float* loss_out, float* map_out,
                         void* workspace, size_t workspace_bytes, void* stream);
int srst_bbg_backward_map(const float* sr, const float* gt, const float* gt2, const float* gt4,
                          const int64_t* idx, const float* grad_map,
                          int B, int H, int W, int ksize, int pad, int stride, int criterion,
                          float* d_sr, float* d_gt,
                          void* workspace, size_t workspace_bytes, void* stream);

/* The HR pyramid on its own (exposed for tests): out2 [B,3,H/2,W/2], out4 [B,3,H/4,W/4]. */
int srst_bb_pyramid(const float* gt, int B, int H, int W, float* out2, float* out4, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* SRST_H_ */
