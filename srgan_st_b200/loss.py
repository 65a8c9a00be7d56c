"""Drop-in loss modules backed by the sm_100a kernels in libsrst.so.

``StructureTensorLoss``, ``BestBuddyLoss``, ``GramLoss`` and ``PatchwiseStructureTensorLoss`` keep the reference's constructor signatures,
attributes and ``criterion(sr, gt) -> 0-dim fp32 tensor`` contract (reference loss.py:380-413 and
loss.py:78-141; called from train.py:138 and warmup.py:91), so they register through
``config.add_g_criterion(name, module, weight)`` (config.py:122-125) unchanged.  With the extra keyword
``reduction='none'`` they return the per-image losses ``[B]`` instead, reduced on the device by the same kernels.  Underneath, each is
a ``torch.autograd.Function`` whose forward/backward enqueue hand-written CUDA kernels on the
current stream through the C ABI of ``include/srst.h``.

No CPU path, no PyTorch fallback: CPU tensors, non-fp32 dtypes and unsupported filter radii raise.
"""
from __future__ import annotations

from typing import Dict, Tuple

import torch
from torch import nn
from torch.autograd.function import once_differentiable

from . import _cabi, taps as _taps

_WORKSPACES: Dict[Tuple[str, int, int], torch.Tensor] = {}
_DIST_L1 = 0x100  # SRST_BB_DIST_L1 (include/srst.h): OR-ed into the criterion argument, search with dist_norm='l1' (utils.py:166-172)


def _workspace(kind: str, device: torch.device, stream_ptr: int, nbytes: int) -> torch.Tensor:
    """Scratch for one family of entry points (`kind`: "st" or "bb" -- they lay the buffer out differently,
    so they never share one), cached per (kind, device, stream).  Only the 16-byte ticket header has to be
    zero before the first launch; the kernels hand it back zeroed (srst.h, srst_st_workspace_bytes).
    Nothing is cached while a CUDA graph is being captured: an allocation made then belongs to the graph's
    private pool and must not be handed to eager code later."""
    key = (kind, device.index if device.index is not None else torch.cuda.current_device(), stream_ptr)
    ws = _WORKSPACES.get(key)
    if ws is not None and ws.numel() >= nbytes:
        return ws
    ws = torch.zeros(max(nbytes, 4096), dtype=torch.uint8, device=device)
    if not torch.cuda.is_current_stream_capturing():
        _WORKSPACES[key] = ws
    return ws


def _check_pair(x: torch.Tensor, gt: torch.Tensor, who: str) -> None:
    if not (isinstance(x, torch.Tensor) and isinstance(gt, torch.Tensor)):
        raise TypeError(f"{who}: expected two tensors")
    if not (x.is_cuda and gt.is_cuda):
        raise RuntimeError(f"{who}: inputs must be CUDA tensors (this build has no CPU fallback)")
    if x.device != gt.device:
        raise RuntimeError(f"{who}: inputs are on different devices ({x.device} vs {gt.device})")
    if x.dtype != torch.float32 or gt.dtype != torch.float32:
        raise TypeError(f"{who}: inputs must be float32 (got {x.dtype}, {gt.dtype})")
    if x.dim() != 4 or x.shape[1] != 3:
        raise ValueError(f"{who}: expected [B,3,H,W] input, got {tuple(x.shape)}")
    if x.shape != gt.shape:
        raise ValueError(f"{who}: shape mismatch {tuple(x.shape)} vs {tuple(gt.shape)}")


def _no_gt_grad(gt: torch.Tensor, who: str) -> None:
    """The reference would send a gradient into gt through the gathered candidates (loss.py:137-139);
    the training loops never ask for it (gt comes from the data loader) and libsrst has no kernel for it."""
    if gt.requires_grad and torch.is_grad_enabled():
        raise NotImplementedError(f"{who}: gradient w.r.t. gt is not implemented (pass gt.detach())")


def _check_reduction(reduction, who: str) -> str:
    """'mean' (the reference's batch mean) or 'none' (one loss per image, [B]); anything else raises."""
    if reduction not in ("mean", "none"):
        raise ValueError(f"{who}: reduction must be 'mean' or 'none' (got {reduction!r})")
    return reduction


def _reduction_repr(reduction: str) -> str:
    return "" if reduction == "mean" else f"reduction='{reduction}'"


def _ptr(t):
    return t.data_ptr() if t is not None else None


def _raw_stream(device: torch.device) -> int:
    """cudaStream_t of torch's current stream on `device` as an integer.  torch.cuda.current_stream() builds a
    Stream object (~5 us); the raw getter behind it is a plain C call."""
    return torch._C._cuda_getCurrentRawStream(device.index if device.index is not None else torch.cuda.current_device())


_SIZES: Dict[Tuple[int, int, int, int, int], Tuple[int, int, int, int]] = {}


def _st_sizes(B: int, H: int, W: int, rs: int = 2, rk: int = 8) -> Tuple[int, int, int, int]:
    """(ds floats padded to 16 bytes, ixy floats, forward workspace bytes, backward workspace bytes) of a
    [B,3,H,W] problem with filter radii (rs, rk), cached per shape.  The last one is 0 for the compiled classes."""
    key = (B, H, W, rs, rk)
    v = _SIZES.get(key)
    if v is None:
        lib = _cabi.lib()
        v = ((B * 3 * H * W + 3) // 4 * 4, lib.srst_st_ixy_floats(B, H, W), lib.srst_st_workspace_bytes_r(B, H, W, rs, rk),
             lib.srst_st_backward_workspace_bytes(B, H, W, rs, rk))
        _SIZES[key] = v
    return v


class _on_device:
    """`with torch.cuda.device(d)` costs ~10 us per call even when d is already current (the normal case in a
    training loop); this enters the context only when the tensor lives on another device."""
    __slots__ = ("_ctx",)

    def __init__(self, device: torch.device):
        self._ctx = None if device.index == torch.cuda.current_device() else torch.cuda.device(device)

    def __enter__(self):
        if self._ctx is not None:
            self._ctx.__enter__()

    def __exit__(self, *exc):
        if self._ctx is not None:
            self._ctx.__exit__(*exc)
        return False


_ST_TAPS: Dict[Tuple[float, float], tuple] = {}


def _st_taps(sigma: float, rho: float, who: str, compiled_only: bool = False):
    """(g*, dg*, r_sigma, k*, r_rho, arrays, generic) as ready-made ctypes arguments, cached per (sigma, rho).
    `generic` is True for radii beyond the compiled shared-memory classes (r_sigma > 4 or r_rho > 12, i.e.
    sigma > 1.1 or rho > 3.1): they run on the library's generic-radius path, which needs scratch planes in the
    workspace and has no fused Pixel / feature variant (`compiled_only`).  Radii above 64 raise."""
    key = (float(sigma), float(rho))
    t = _ST_TAPS.get(key)
    if t is None:
        g, dg = _taps.gaussian_taps(key[0])
        k, _ = _taps.gaussian_taps(key[1])
        rs, rk = len(g) // 2, len(k) // 2
        sup = _cabi.lib().srst_st_supported(rs, rk)
        if not sup:
            raise NotImplementedError(
                f"{who}: filter radii (sigma={sigma} -> {rs}, rho={rho} -> {rk}) exceed what libsrst.so handles (64)")
        t = (_taps.as_c(g), _taps.as_c(dg), rs, _taps.as_c(k), rk, (g, dg, k), sup == 2)  # keep the arrays alive
        _ST_TAPS[key] = t
    if compiled_only and t[6]:
        raise NotImplementedError(
            f"{who}: filter radii (sigma={sigma} -> {t[2]}, rho={rho} -> {t[4]}) are outside the compiled radius classes; "
            "only StructureTensorLoss has a generic-radius path")
    return t


class _StructureTensorLossFn(torch.autograd.Function):
    """autograd boundary of the fused ST loss (the reference lets autograd differentiate ~100
    ATen ops instead; loss.py:399-413).  Saved for backward: per image that needs a gradient, ONE buffer
    holding the ds planes (12 B/px) followed by the Ix, Iy planes (8 B/px); the images themselves are not.
    `per_image`: reduction='none' -- the loss is [B] and the upstream gradient [B] (the *_per_image entry points)."""

    @staticmethod
    def forward(ctx, sr, hr, sigma, rho, normalize, per_image=False):
        lib = _cabi.lib()
        sr = sr.contiguous()
        hr = hr.contiguous()
        B, _, H, W = sr.shape
        tp = _st_taps(sigma, rho, "StructureTensorLoss")
        need = ctx.needs_input_grad
        n_ds, n_ixy, ws_bytes, bws_bytes = _st_sizes(B, H, W, tp[2], tp[4])   # n_ds is padded: the ixy part stays 16-byte aligned
        with _on_device(sr.device):
            stream = _raw_stream(sr.device)
            loss = torch.empty((B,) if per_image else (), dtype=torch.float32, device=sr.device)
            saved = [torch.empty(n_ds + n_ixy, dtype=torch.float32, device=sr.device) if n else None for n in need[:2]]
            ds = [t.data_ptr() if t is not None else None for t in saved]
            ixy = [p + 4 * n_ds if p is not None else None for p in ds]
            ws = _workspace("st", sr.device, stream, ws_bytes)
            fwd = lib.srst_st_forward_per_image if per_image else lib.srst_st_forward
            rc = fwd(sr.data_ptr(), hr.data_ptr(), B, H, W, tp[0], tp[1], tp[2], tp[3], tp[4],
                     int(bool(normalize)), 1e-12, loss.data_ptr(), ds[0], ds[1], ixy[0], ixy[1],
                     ws.data_ptr(), ws.numel(), stream)
        if rc:
            _cabi.check(rc, "srst_st_forward_per_image" if per_image else "srst_st_forward")
        ctx.save_for_backward(saved[0], saved[1])
        ctx.meta = (tp, B, H, W, n_ds, bws_bytes, per_image)
        return loss

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out):
        lib = _cabi.lib()
        tp, B, H, W, n_ds, bws_bytes, per_image = ctx.meta
        if grad_out.dtype != torch.float32 or not grad_out.is_contiguous():   # also the stride-0 [B] of .sum() / .mean()
            grad_out = grad_out.to(torch.float32).contiguous()
        outs = [None, None]
        dev = grad_out.device
        with _on_device(dev):
            stream = _raw_stream(dev)
            for i, saved in enumerate(ctx.saved_tensors):
                if saved is None or not ctx.needs_input_grad[i]:
                    continue
                d_img = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
                if per_image:  # one entry point for both paths; the compiled classes need no workspace
                    ws = _workspace("st_bwd", dev, stream, bws_bytes) if bws_bytes else None
                    rc = lib.srst_st_backward_per_image(saved.data_ptr() + 4 * n_ds, saved.data_ptr(), grad_out.data_ptr(), B,
                                                        H, W, tp[0], tp[1], tp[2], tp[3], tp[4], d_img.data_ptr(), _ptr(ws),
                                                        ws.numel() if ws is not None else 0, stream)
                elif bws_bytes:  # generic-radius path: five scratch planes
                    ws = _workspace("st_bwd", dev, stream, bws_bytes)
                    rc = lib.srst_st_backward_ws(saved.data_ptr() + 4 * n_ds, saved.data_ptr(), grad_out.data_ptr(), B, H, W,
                                                 tp[0], tp[1], tp[2], tp[3], tp[4], d_img.data_ptr(), ws.data_ptr(),
                                                 ws.numel(), stream)
                else:
                    rc = lib.srst_st_backward(saved.data_ptr() + 4 * n_ds, saved.data_ptr(), grad_out.data_ptr(), B, H, W,
                                              tp[0], tp[1], tp[2], tp[3], tp[4], d_img.data_ptr(), stream)
                if rc:
                    _cabi.check(rc, "srst_st_backward")
                outs[i] = d_img
        return outs[0], outs[1], None, None, None, None


class StructureTensorLoss(nn.Module):
    """Structure-tensor loss; same signature and semantics as reference loss.py:380-413.

    ``forward(x, gt)``: x = SR ``[B,3,H,W]``, gt = HR, both fp32 CUDA; returns the mean over all
    pixels of the affine-invariant distance between the det-normalised structure tensors.
    ``reduction='none'`` returns the ``[B]`` per-image means instead (the reference's ``vmap(st_loss)(x, gt)``
    before its ``.mean()``, loss.py:411-413), differentiable w.r.t. x and gt.
    """

    def __init__(self, sigma: float = 0.5, rho: float = 2.0, normalize: bool = True, reduction: str = "mean"):
        super().__init__()
        self.sigma = sigma
        self.rho = rho
        self.normalize = normalize
        self.reduction = _check_reduction(reduction, "StructureTensorLoss")
        _cabi.lib()  # fail at construction time if the CUDA library is missing

    def st_loss(self, x, gt):
        """Single-sample form (reference loss.py:399-409): x, gt are [3,H,W]."""
        return self.forward(x.unsqueeze(0), gt.unsqueeze(0))

    def forward(self, x, gt):
        _check_pair(x, gt, "StructureTensorLoss")
        if self.reduction == "none":
            return _StructureTensorLossFn.apply(x, gt, self.sigma, self.rho, self.normalize, True)
        return _StructureTensorLossFn.apply(x, gt, self.sigma, self.rho, self.normalize)

    def extra_repr(self) -> str:
        r = f"sigma={self.sigma}, rho={self.rho}, normalize={self.normalize}"
        return r if self.reduction == "mean" else f"{r}, {_reduction_repr(self.reduction)}"


class _StructureTensorDistanceFn(torch.autograd.Function):
    """autograd boundary of the per-pixel distance map (srst_st_forward_map / srst_st_backward_map).  Saves what
    `_StructureTensorLossFn` saves: per image that needs a gradient, ONE buffer of ds planes followed by Ix, Iy.  The
    upstream gradient is any [B,H,W] tensor."""

    @staticmethod
    def forward(ctx, sr, hr, sigma, rho, normalize):
        lib = _cabi.lib()
        sr = sr.contiguous()
        hr = hr.contiguous()
        B, _, H, W = sr.shape
        tp = _st_taps(sigma, rho, "structure_tensor_distance")
        need = ctx.needs_input_grad
        n_ds, n_ixy, ws_bytes, _ = _st_sizes(B, H, W, tp[2], tp[4])
        with _on_device(sr.device):
            stream = _raw_stream(sr.device)
            loss = torch.empty((), dtype=torch.float32, device=sr.device)
            dmap = torch.empty((B, H, W), dtype=torch.float32, device=sr.device)
            saved = [torch.empty(n_ds + n_ixy, dtype=torch.float32, device=sr.device) if n else None for n in need[:2]]
            ds = [t.data_ptr() if t is not None else None for t in saved]
            ixy = [p + 4 * n_ds if p is not None else None for p in ds]
            ws = _workspace("st", sr.device, stream, ws_bytes)
            rc = lib.srst_st_forward_map(sr.data_ptr(), hr.data_ptr(), B, H, W, tp[0], tp[1], tp[2], tp[3], tp[4],
                                         int(bool(normalize)), 1e-12, loss.data_ptr(), dmap.data_ptr(), ds[0], ds[1],
                                         ixy[0], ixy[1], ws.data_ptr(), ws.numel(), stream)
        if rc:
            _cabi.check(rc, "srst_st_forward_map")
        ctx.save_for_backward(saved[0], saved[1])
        ctx.meta = (tp, B, H, W, n_ds)
        return dmap

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_map):
        lib = _cabi.lib()
        tp, B, H, W, n_ds = ctx.meta
        if grad_map.dtype != torch.float32 or not grad_map.is_contiguous():   # also the stride-0 ones of .sum() / .mean()
            grad_map = grad_map.to(torch.float32).contiguous()
        outs = [None, None]
        dev = grad_map.device
        with _on_device(dev):
            stream = _raw_stream(dev)
            ws = None
            for i, saved in enumerate(ctx.saved_tensors):
                if saved is None or not ctx.needs_input_grad[i]:
                    continue
                if ws is None:   # weighted ds planes + unit slot (+ the generic path's planes); the two calls run in order
                    ws = _workspace("st_map_bwd", dev, stream,
                                    lib.srst_st_backward_map_workspace_bytes(B, H, W, tp[2], tp[4]))
                d_img = torch.empty((B, 3, H, W), dtype=torch.float32, device=dev)
                rc = lib.srst_st_backward_map(saved.data_ptr() + 4 * n_ds, saved.data_ptr(), grad_map.data_ptr(), B, H, W,
                                              tp[0], tp[1], tp[2], tp[3], tp[4], d_img.data_ptr(), ws.data_ptr(),
                                              ws.numel(), stream)
                if rc:
                    _cabi.check(rc, "srst_st_backward_map")
                outs[i] = d_img
        return outs[0], outs[1], None, None, None


def structure_tensor_distance(x: torch.Tensor, gt: torch.Tensor, sigma: float = 0.5, rho: float = 2.0,
                              normalize: bool = True) -> torch.Tensor:
    """Per-pixel structure-tensor distance between x (SR) and gt (HR), both ``[B,3,H,W]`` fp32 CUDA: the ``[B,H,W]``
    fp32 map whose mean is ``StructureTensorLoss(sigma, rho, normalize)(x, gt)`` (the map ``compute_distance`` builds
    before ``st_loss`` takes its mean, reference loss.py:408-409, utils.py:269-279).  Differentiable w.r.t. x, and w.r.t.
    gt when gt requires grad, under any upstream gradient, e.g. a spatial weighting ``(d * w).sum() / w.sum()``."""
    _check_pair(x, gt, "structure_tensor_distance")
    return _StructureTensorDistanceFn.apply(x, gt, sigma, rho, normalize)


def structure_tensor_features(img: torch.Tensor, sigma: float = 0.5, rho: float = 2.0):
    """Diagnostic structure-tensor features of ``img`` ``[B,3,H,W]`` (fp32 CUDA), no gradient: a dict with
    ``J`` ``[B,3,H,W]`` (Jxx, Jyy, Jxy as reference utils.py:212-233 names them), ``eigenvalues`` ``[B,2,H,W]`` (small,
    large), ``orientation`` ``[B,H,W]`` (angle of the dominant-gradient eigenvector against the H axis, radians in
    (-pi/2, pi/2]; the coherent structure runs perpendicular to it) and ``coherence`` ``[B,H,W]``
    (``1 - lambda_small / lambda_large``).  The reference derives orientation / anisotropy only in an exploration
    notebook via the third-party ``structure_tensor`` package; see ``include/srst.h`` (srst_st_features)."""
    if not (isinstance(img, torch.Tensor) and img.is_cuda and img.dtype == torch.float32 and img.dim() == 4
            and img.shape[1] == 3):
        raise TypeError("structure_tensor_features: expected a float32 CUDA tensor [B,3,H,W] (no CPU fallback)")
    lib = _cabi.lib()
    img = img.detach().contiguous()
    B, _, H, W = img.shape
    tp = _st_taps(sigma, rho, "structure_tensor_features", compiled_only=True)
    with _on_device(img.device):
        stream = _raw_stream(img.device)
        J = torch.empty((B, 3, H, W), dtype=torch.float32, device=img.device)
        eig = torch.empty((B, 2, H, W), dtype=torch.float32, device=img.device)
        orient = torch.empty((B, H, W), dtype=torch.float32, device=img.device)
        coher = torch.empty((B, H, W), dtype=torch.float32, device=img.device)
        rc = lib.srst_st_features(img.data_ptr(), B, H, W, tp[0], tp[1], tp[2], tp[3], tp[4], J.data_ptr(), eig.data_ptr(),
                                  orient.data_ptr(), coher.data_ptr(), stream)
    if rc:
        _cabi.check(rc, "srst_st_features")
    return {"J": J, "eigenvalues": eig, "orientation": orient, "coherence": coher}


class _StructureTensorPixelLossFn(torch.autograd.Function):
    """ST loss and the "Pixel" MSE criterion from ONE pass over (sr, gt) per direction (SURVEY 8f rank 4).
    Returns the two unweighted terms as one 2-vector [st, mse]; gt carries no gradient.
    `per_image`: reduction='none' -- the terms are [2, B] (row 0 ST, row 1 MSE) and so is the upstream gradient
    (the *_per_image entry points)."""

    @staticmethod
    def forward(ctx, sr, hr, sigma, rho, normalize, per_image=False):
        lib = _cabi.lib()
        sr = sr.contiguous()
        hr = hr.contiguous()
        B, _, H, W = sr.shape
        tp = _st_taps(sigma, rho, "StructureTensorPixelLoss", compiled_only=True)
        need_sr = ctx.needs_input_grad[0]
        n_ds, n_ixy, ws_bytes, _ = _st_sizes(B, H, W)
        with _on_device(sr.device):
            stream = _raw_stream(sr.device)
            both = torch.empty((2, B) if per_image else 2, dtype=torch.float32, device=sr.device)
            saved = torch.empty(n_ds + n_ixy, dtype=torch.float32, device=sr.device) if need_sr else None
            p = saved.data_ptr() if need_sr else None
            ws = _workspace("st", sr.device, stream, ws_bytes)
            fwd = lib.srst_stpx_forward_per_image if per_image else lib.srst_stpx_forward
            rc = fwd(sr.data_ptr(), hr.data_ptr(), B, H, W, tp[0], tp[1], tp[2], tp[3], tp[4],
                     int(bool(normalize)), 1e-12, both.data_ptr(), p,
                     p + 4 * n_ds if need_sr else None, ws.data_ptr(), ws.numel(), stream)
        if rc:
            _cabi.check(rc, "srst_stpx_forward_per_image" if per_image else "srst_stpx_forward")
        ctx.save_for_backward(sr, hr, saved)
        ctx.meta = (tp, n_ds, per_image)
        return both

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_both):
        lib = _cabi.lib()
        sr, hr, saved = ctx.saved_tensors
        tp, n_ds, per_image = ctx.meta
        if saved is None or not ctx.needs_input_grad[0]:
            return None, None, None, None, None, None
        B, _, H, W = sr.shape
        with _on_device(sr.device):
            stream = _raw_stream(sr.device)
            if grad_both.dtype != torch.float32 or not grad_both.is_contiguous():   # also the stride-0 one of .sum()
                grad_both = grad_both.to(torch.float32).contiguous()
            d_sr = torch.empty_like(sr)
            g = grad_both.data_ptr()   # [d/d st, d/d mse]: two adjacent device scalars, or two adjacent [B] rows
            bwd = lib.srst_stpx_backward_per_image if per_image else lib.srst_stpx_backward
            rc = bwd(sr.data_ptr(), hr.data_ptr(), saved.data_ptr() + 4 * n_ds, saved.data_ptr(),
                     g, g + 4 * (B if per_image else 1), B, H, W, tp[0], tp[1], tp[2], tp[3], tp[4], d_sr.data_ptr(),
                     stream)
        if rc:
            _cabi.check(rc, "srst_stpx_backward_per_image" if per_image else "srst_stpx_backward")
        return d_sr, None, None, None, None, None


class StructureTensorPixelLoss(nn.Module):
    """``st_weight * StructureTensorLoss(sigma, rho, normalize)(x, gt) + pixel_weight * MSELoss()(x, gt)``
    from one fused pass per direction.

    The reference's warm-up / training loops register "Pixel" (``nn.MSELoss``) and "ST" as two criteria
    and evaluate them one after the other on the same two tensors (config.py:71-93, warmup.py:88-96,
    train.py:131-144).  Registering this module once, with weight 1.0, gives the same generator loss
    and gradient; the two unweighted terms of the last call stay on the device in ``last_terms`` for
    logging without a synchronisation.

    ``reduction='none'`` returns the ``[B]`` per-image losses ``st_weight * st[b] + pixel_weight * mse[b]`` instead:
    ``st[b]`` is ``StructureTensorLoss(reduction='none')`` of image b, ``mse[b]`` the mean of ``(x[b] - gt[b])**2``.
    It is differentiable w.r.t. x, still from one fused pass per direction."""

    def __init__(self, sigma: float = 0.5, rho: float = 2.0, normalize: bool = True, st_weight: float = 1.0,
                 pixel_weight: float = 1.0, reduction: str = "mean"):
        super().__init__()
        self.sigma = sigma
        self.rho = rho
        self.normalize = normalize
        self.st_weight = st_weight
        self.pixel_weight = pixel_weight
        self.reduction = _check_reduction(reduction, "StructureTensorPixelLoss")
        self._last = None
        self._w = None   # (device, st_weight, pixel_weight, tensor): the weights as a device 2-vector
        _cabi.lib()

    @property
    def last_terms(self):
        """(st, mse) of the most recent call as two device tensors (detached), or None: 0-dim, or [B] each with
        reduction='none'."""
        return None if self._last is None else (self._last[0], self._last[1])

    def forward(self, x, gt):
        _check_pair(x, gt, "StructureTensorPixelLoss")
        _no_gt_grad(gt, "StructureTensorPixelLoss")
        per_image = self.reduction == "none"
        if per_image:
            both = _StructureTensorPixelLossFn.apply(x, gt, self.sigma, self.rho, self.normalize, True)
        else:
            both = _StructureTensorPixelLossFn.apply(x, gt, self.sigma, self.rho, self.normalize)
        self._last = both.detach()
        w = self._w
        if w is None or w[0] != x.device or w[1] != self.st_weight or w[2] != self.pixel_weight:
            w = (x.device, self.st_weight, self.pixel_weight,
                 torch.tensor([self.st_weight, self.pixel_weight], dtype=torch.float32, device=x.device))
            self._w = w
        return w[3] @ both if per_image else torch.dot(both, w[3])

    def extra_repr(self) -> str:
        r = (f"sigma={self.sigma}, rho={self.rho}, normalize={self.normalize}, st_weight={self.st_weight}, "
             f"pixel_weight={self.pixel_weight}")
        return r if self.reduction == "mean" else f"{r}, {_reduction_repr(self.reduction)}"


def _hr_pyramid(gt, pyramid: str):
    """(gt2, gt4), the x1/2 and x1/4 HR levels of the patch losses: the reference's own op for "aten" (loss.py:123,127,
    :353,356); None, None for "fused", where libsrst builds them (srst_bb_pyramid taps)."""
    if pyramid != "aten":
        return None, None
    with torch.no_grad():
        return tuple(torch.nn.functional.interpolate(gt, scale_factor=s, mode="bicubic", align_corners=False).contiguous()
                     for s in (0.5, 0.25))


_PST_TAPS: Dict[Tuple[float, float], tuple] = {}


def _pst_taps(sigma: float, rho: float):
    """(g*, dg*, r_sigma, k*, r_rho, arrays) of PatchwiseStructureTensorLoss as ready-made ctypes arguments, cached per
    (sigma, rho).  No radius limit as in _st_taps: a 3x3 patch image only sees the five central taps, and the PST entry
    points take radii up to 4096."""
    key = (float(sigma), float(rho))
    t = _PST_TAPS.get(key)
    if t is None:
        g, dg = _taps.gaussian_taps(key[0])
        k, _ = _taps.gaussian_taps(key[1])
        t = (_taps.as_c(g), _taps.as_c(dg), len(g) // 2, _taps.as_c(k), len(k) // 2, (g, dg, k))  # keep the arrays alive
        _PST_TAPS[key] = t
    return t


_NO_TAPS = (None, None, 0, None, 0)


def _patch_backward_gt(mode: int, sr, gt, gt2, gt4, idx, grad_out, taps, criterion: int, d_gt, ws, stream: int):
    """d loss / d gt of a default-geometry patch loss (include/srst.h, srst_patch_backward_gt): the reference's gather of
    the selected candidates is differentiable in p2_cat (loss.py:136-139), so a gt that requires grad gets one."""
    B, _, H, W = sr.shape
    rc = _cabi.lib().srst_patch_backward_gt(mode, _ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx), _ptr(grad_out), B, H,
                                            W, *taps[:5], criterion, _ptr(d_gt), _ptr(ws), ws.numel(), stream)
    _cabi.check(rc, "srst_patch_backward_gt")


class _PatchLossFn(torch.autograd.Function):
    """autograd boundary of the three patch losses.  Only the final criterion is differentiable: w.r.t. the SR patches
    and, through the gather of the selected candidates, w.r.t. gt (reference loss.py:135-139, :219-222, :369-371); the
    argmin is not.  `loss_cls` is the module class: its _plan / _fwd / _bwd make the C ABI calls that differ per loss.
    `args` holds what they take from the module (weights, criterion, taps, geometry), fixed at forward time: a module
    changed between forward and backward does not change the gradient.  `form` is the output: "mean" (a 0-dim batch
    mean), "none" (reduction='none': the loss and the upstream gradient are [B], _fwd_none / _bwd_none make the calls)
    or "map" (loss_map: one value per query patch, [B,N], _fwd_map / _bwd_map)."""

    @staticmethod
    def forward(ctx, sr, gt, loss_cls, args, pyramid, form="mean"):
        sr = sr.contiguous()
        gt = gt.contiguous()
        B, _, H, W = sr.shape
        n, kind, nbytes = loss_cls._plan(args, B, H, W)
        with _on_device(sr.device):
            stream = _raw_stream(sr.device)
            gt2, gt4 = _hr_pyramid(gt, pyramid)
            idx = torch.empty((B, n), dtype=torch.int64, device=sr.device)
            ws = _workspace(kind, sr.device, stream, nbytes)
            if form == "map":
                out = torch.empty((B, n), dtype=torch.float32, device=sr.device)
                loss_cls._fwd_map(args, sr, gt, gt2, gt4, idx, torch.empty((), dtype=torch.float32, device=sr.device),
                                  out, ws, stream)
            else:
                out = torch.empty((B,) if form == "none" else (), dtype=torch.float32, device=sr.device)
                fwd = loss_cls._fwd_none if form == "none" else loss_cls._fwd
                fwd(args, sr, gt, gt2, gt4, idx, out, ws, stream)
        ctx.save_for_backward(sr, gt, gt2, gt4, idx)
        ctx.meta = (loss_cls, args, kind, nbytes, form)
        ctx.mark_non_differentiable(idx)
        return out, idx

    @staticmethod
    @once_differentiable
    def backward(ctx, grad_out, _grad_idx):
        need_sr, need_gt = ctx.needs_input_grad[:2]
        if not (need_sr or need_gt):
            return None, None, None, None, None, None
        sr, gt, gt2, gt4, idx = ctx.saved_tensors
        loss_cls, args, kind, nbytes, form = ctx.meta
        grad_out = grad_out.to(torch.float32).contiguous()   # also the stride-0 [B] / [B,N] of .sum() / .mean()
        with _on_device(sr.device):
            stream = _raw_stream(sr.device)
            d_sr = torch.empty_like(sr) if need_sr else None
            d_gt = torch.empty_like(gt) if need_gt else None
            bwd = {"mean": loss_cls._bwd, "none": loss_cls._bwd_none, "map": loss_cls._bwd_map}[form]
            bwd(args, sr, gt, gt2, gt4, idx, grad_out, d_sr, d_gt, _workspace(kind, sr.device, stream, nbytes), stream)
        return d_sr, d_gt, None, None, None, None


class _PatchLoss(nn.Module):
    """What BestBuddyLoss, GramLoss and PatchwiseStructureTensorLoss share: the reference's constructor arguments
    `alpha`, `beta`, `ksize`, `dist_norm`, `criterion`, the `pyramid` and `reduction` choices, the call through
    _PatchLossFn, and ``last_indices``, the argmin indices ``[B,N]`` (int64) of the most recent call.  A subclass supplies
    the C ABI calls (_args, _fwd, _bwd; _MODE and _taps_of for the per-image and loss-map entry points) and checks its
    patch geometry (_check_geometry).

    ``reduction='none'`` returns ``[B]``: entry b is the mean over image b's criterion terms, i.e. the reference module
    applied to ``(x[b:b+1], gt[b:b+1])``; the search and ``last_indices`` are the same as with 'mean'.

    ``loss_map(x, gt)`` returns the element-wise form, one value per query patch (see there)."""

    _criterion_error = "%s criterion has not been implmented."   # the reference's message (loss.py:113, :178)
    _MODE = 0   # `mode` of the srst_patch_*_per_image / srst_patch_*_map entry points

    def __init__(self, alpha, beta, ksize, dist_norm, criterion, pyramid, pad=0, stride=3, reduction="mean"):
        super().__init__()
        self.reduction = _check_reduction(reduction, type(self).__name__)
        self.alpha = alpha
        self.beta = beta
        self.ksize = ksize
        self.dist_norm = dist_norm
        if criterion == "l1":
            self.criterion = torch.nn.L1Loss()   # kept for repr/config parity (config.py:133-139)
            self._crit = 0
        elif criterion == "l2" or criterion == "mse":
            self.criterion = torch.nn.MSELoss()
            self._crit = 1
        else:
            raise NotImplementedError(self._criterion_error % criterion)
        if dist_norm not in ("l1", "l2"):
            raise NotImplementedError("%s norm has not been supported." % dist_norm)        # utils.py:189
        self._check_geometry(ksize, pad, stride)
        if dist_norm == "l1":
            self._crit |= _DIST_L1
        if pyramid not in ("aten", "fused"):
            raise ValueError("pyramid must be 'aten' or 'fused'")
        self.pyramid = pyramid
        self.last_indices = None
        _cabi.lib()

    def _check_geometry(self, ksize, pad, stride):
        if ksize != 3:
            raise NotImplementedError(f"{type(self).__name__}: libsrst.so implements ksize=3 only")

    def forward(self, x, gt):
        _check_pair(x, gt, type(self).__name__)
        if self.reduction == "none":
            loss, idx = _PatchLossFn.apply(x, gt, type(self), self._args(), self.pyramid, "none")
        else:
            loss, idx = _PatchLossFn.apply(x, gt, type(self), self._args(), self.pyramid)
        self.last_indices = idx
        return loss

    def loss_map(self, x, gt):
        """The per-patch loss map, an fp32 ``[B, ny, nx]`` tensor on the query patch grid (F.unfold's row-major order;
        ``ny, nx = H // 3, W // 3`` for the default 3x3 / stride-3 geometry).  Entry ``[b, i, j]`` is the mean over the
        D criterion terms of query patch (i, j) of image b against its selected candidate: the reference's
        ``criterion(reduction='none')(p1, sel_p2).mean(-1)`` (loss.py:139, :222, :371) before its mean.  So
        ``loss_map(x, gt).mean()`` is the 'mean' loss and its per-image means are the 'none' losses, whatever
        ``self.reduction`` says.  Differentiable w.r.t. x, and w.r.t. gt when gt requires grad, under any ``[B, ny, nx]``
        upstream gradient: spatial weighting or masking of the loss, heat maps of the patches without a good buddy.
        The search, its checks and errors and ``last_indices`` are those of ``forward``."""
        _check_pair(x, gt, type(self).__name__)
        args = self._args()
        m, idx = _PatchLossFn.apply(x, gt, type(self), args, self.pyramid, "map")
        self.last_indices = idx
        return m.view(x.shape[0], *self._grid(args, x.shape[2], x.shape[3]))

    def extra_repr(self) -> str:
        return _reduction_repr(self.reduction)

    @staticmethod
    def _taps_of(args):
        return _NO_TAPS

    @classmethod
    def _fwd_none(cls, args, sr, gt, gt2, gt4, idx, loss, ws, stream):
        """reduction='none' forward of the default 3x3 / stride-3 patch grid: loss is [B]."""
        alpha, beta, crit = args[:3]
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_patch_forward_per_image(cls._MODE, _ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W,
                                                      *cls._taps_of(args)[:5], alpha, beta, crit, _ptr(idx), _ptr(loss),
                                                      _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_patch_forward_per_image")

    @classmethod
    def _bwd_none(cls, args, sr, gt, gt2, gt4, idx, grad_out, d_sr, d_gt, ws, stream):
        """reduction='none' backward: grad_out is [B]; one call fills d_sr and d_gt, either of which may be None."""
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_patch_backward_per_image(cls._MODE, _ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx),
                                                       _ptr(grad_out), B, H, W, *cls._taps_of(args)[:5], args[2], _ptr(d_sr),
                                                       _ptr(d_gt), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_patch_backward_per_image")

    @classmethod
    def _fwd_map(cls, args, sr, gt, gt2, gt4, idx, loss, out, ws, stream):
        """loss_map forward of the default 3x3 / stride-3 patch grid: out is [B,N], loss the (unused) batch mean."""
        alpha, beta, crit = args[:3]
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_patch_forward_map(cls._MODE, _ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W,
                                                *cls._taps_of(args)[:5], alpha, beta, crit, _ptr(idx), _ptr(loss), _ptr(out),
                                                _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_patch_forward_map")

    @classmethod
    def _bwd_map(cls, args, sr, gt, gt2, gt4, idx, grad_map, d_sr, d_gt, ws, stream):
        """loss_map backward: grad_map is [B,N]; one call fills d_sr and d_gt, either of which may be None."""
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_patch_backward_map(cls._MODE, _ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx),
                                                 _ptr(grad_map), B, H, W, *cls._taps_of(args)[:5], args[2], _ptr(d_sr),
                                                 _ptr(d_gt), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_patch_backward_map")

    @classmethod
    def _grid(cls, args, H, W):
        """(ny, nx), the query patch grid of the default 3x3 / stride-3 geometry."""
        return H // 3, W // 3

    @classmethod
    def _plan(cls, args, B, H, W):
        """(patches per image, workspace kind, workspace bytes) of the default 3x3 / stride-3 patch grid."""
        if H < 12 or W < 12:
            raise ValueError(f"{cls.__name__}: images must be at least 12x12 (got {H}x{W})")
        return (H // 3) * (W // 3), "bb", _cabi.lib().srst_bb_workspace_bytes(B, H, W)


class BestBuddyLoss(_PatchLoss):
    """Best-Buddy loss; same signature and semantics as reference loss.py:78-141.

    ``forward(x, gt)``: for every 3x3 SR patch pick the HR candidate patch (three pyramid levels)
    minimising ``alpha*|sr-cand|^2 + beta*|gt-cand|^2`` and return the L1 (or MSE) distance to it.
    The reference's default patch geometry (ksize=3, pad=0, stride=3) runs the tuned filter + exact re-scoring search;
    any other ``ksize`` (1..8), ``pad`` and ``stride`` -- overlapping patches, gaps, zero padding (F.unfold semantics,
    loss.py:116-129) -- runs an exact all-pairs search kernel.  ``dist_norm='l1'`` (utils.py:166-172) scores every pair
    exactly with
    ``alpha*sum|sr-cand| + beta*sum|gt-cand|`` (the reference materialises a [B,N,M,27] tensor for it).

    ``pyramid``: "fused" (default) lets libsrst build the two HR pyramid levels with the cubic taps of
    ``F.interpolate(mode='bicubic', align_corners=False)`` (equal to 2e-7; 0.03 ms instead of 0.43 ms at
    batch 64 x 192x192); "aten" calls the reference's own op.
    ``last_indices`` holds the argmin indices ``[B,N]`` (int64) of the most recent call.
    ``reduction='none'`` returns the ``[B]`` per-image losses (every geometry).
    """

    def __init__(self, alpha: float = 1.0, beta: float = 1.0, ksize: int = 3, pad: int = 0, stride: int = 3,
                 dist_norm: str = "l2", criterion: str = "l1", pyramid: str = "fused", reduction: str = "mean"):
        super().__init__(alpha, beta, ksize, dist_norm, criterion, pyramid, pad, stride, reduction)
        self.pad = pad
        self.stride = stride

    def _check_geometry(self, ksize, pad, stride):
        self._geom = None   # None: the tuned (3, 0, 3) kernels; else the generic-geometry path
        if (ksize, pad, stride) != (3, 0, 3):
            if not all(isinstance(v, int) and not isinstance(v, bool) for v in (ksize, pad, stride)):
                raise TypeError("BestBuddyLoss: ksize, pad and stride must be ints")
            if not _cabi.lib().srst_bbg_supported(ksize, pad, stride):
                raise NotImplementedError(
                    f"BestBuddyLoss: libsrst.so has kernels for 1 <= ksize <= 8, pad >= 0, stride >= 1 "
                    f"(got ksize={ksize}, pad={pad}, stride={stride})")
            self._geom = (ksize, pad, stride)

    def _args(self):
        return float(self.alpha), float(self.beta), int(self._crit), self._geom

    @classmethod
    def _plan(cls, args, B, H, W):
        if args[3] is None:
            return super()._plan(args, B, H, W)
        lib = _cabi.lib()
        ks, pad, st = args[3]
        n = lib.srst_bbg_num_patches(H, W, ks, pad, st)
        nbytes = lib.srst_bbg_workspace_bytes(B, H, W, ks, pad, st)
        if n <= 0 or nbytes == 0:
            raise ValueError(f"BestBuddyLoss: a {H}x{W} image has a pyramid level without a single "
                             f"ksize={ks}, pad={pad}, stride={st} patch (F.unfold would raise too)")
        return n, "bbg", nbytes

    @classmethod
    def _grid(cls, args, H, W):
        if args[3] is None:
            return super()._grid(args, H, W)
        ks, pad, st = args[3]
        return (H + 2 * pad - ks) // st + 1, (W + 2 * pad - ks) // st + 1   # F.unfold

    @staticmethod
    def _fwd(args, sr, gt, gt2, gt4, idx, loss, ws, stream):
        alpha, beta, crit, geom = args
        lib = _cabi.lib()
        B, _, H, W = sr.shape
        if geom is None:
            rc = lib.srst_bb_forward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W, alpha, beta, crit, _ptr(idx),
                                     _ptr(loss), _ptr(ws), ws.numel(), stream)
            _cabi.check(rc, "srst_bb_forward")
        else:
            rc = lib.srst_bbg_forward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W, *geom, alpha, beta, crit,
                                      _ptr(idx), _ptr(loss), _ptr(ws), ws.numel(), stream)
            _cabi.check(rc, "srst_bbg_forward")

    @staticmethod
    def _bwd(args, sr, gt, gt2, gt4, idx, grad_out, d_sr, d_gt, ws, stream):
        crit, geom = args[2:]
        lib = _cabi.lib()
        B, _, H, W = sr.shape
        if geom is not None:   # one call fills d_sr and d_gt, either of which may be None
            rc = lib.srst_bbg_backward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx), _ptr(grad_out), B, H, W, *geom,
                                       crit, _ptr(d_sr), _ptr(d_gt), _ptr(ws), ws.numel(), stream)
            _cabi.check(rc, "srst_bbg_backward")
            return
        if d_sr is not None:
            rc = lib.srst_bb_backward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx), _ptr(grad_out), B, H, W, crit,
                                      _ptr(d_sr), _ptr(ws), ws.numel(), stream)
            _cabi.check(rc, "srst_bb_backward")
        if d_gt is not None:
            _patch_backward_gt(0, sr, gt, gt2, gt4, idx, grad_out, _NO_TAPS, crit, d_gt, ws, stream)

    @classmethod
    def _fwd_none(cls, args, sr, gt, gt2, gt4, idx, loss, ws, stream):
        alpha, beta, crit, geom = args
        if geom is None:
            return super()._fwd_none(args, sr, gt, gt2, gt4, idx, loss, ws, stream)
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_bbg_forward_per_image(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W, *geom, alpha, beta,
                                                    crit, _ptr(idx), _ptr(loss), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_bbg_forward_per_image")

    @classmethod
    def _bwd_none(cls, args, sr, gt, gt2, gt4, idx, grad_out, d_sr, d_gt, ws, stream):
        crit, geom = args[2:]
        if geom is None:
            return super()._bwd_none(args, sr, gt, gt2, gt4, idx, grad_out, d_sr, d_gt, ws, stream)
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_bbg_backward_per_image(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx), _ptr(grad_out), B,
                                                     H, W, *geom, crit, _ptr(d_sr), _ptr(d_gt), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_bbg_backward_per_image")

    @classmethod
    def _fwd_map(cls, args, sr, gt, gt2, gt4, idx, loss, out, ws, stream):
        alpha, beta, crit, geom = args
        if geom is None:
            return super()._fwd_map(args, sr, gt, gt2, gt4, idx, loss, out, ws, stream)
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_bbg_forward_map(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W, *geom, alpha, beta, crit,
                                              _ptr(idx), _ptr(loss), _ptr(out), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_bbg_forward_map")

    @classmethod
    def _bwd_map(cls, args, sr, gt, gt2, gt4, idx, grad_map, d_sr, d_gt, ws, stream):
        crit, geom = args[2:]
        if geom is None:
            return super()._bwd_map(args, sr, gt, gt2, gt4, idx, grad_map, d_sr, d_gt, ws, stream)
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_bbg_backward_map(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx), _ptr(grad_map), B, H, W,
                                               *geom, crit, _ptr(d_sr), _ptr(d_gt), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_bbg_backward_map")


class GramLoss(_PatchLoss):
    """Gram loss; same signature and semantics as reference loss.py:146-225: the best-buddy search
    and the final criterion run on the 3x3 Gram matrix of every 3x3x3 patch instead of its pixels.
    Only ``ksize=3`` has kernels (the reference's default); ``dist_norm`` may be 'l2' or 'l1'.
    ``reduction='none'`` returns the ``[B]`` per-image losses."""

    _MODE = 1

    def __init__(self, alpha: float = 1.0, beta: float = 1.0, ksize: int = 3, dist_norm: str = "l2",
                 criterion: str = "l1", pyramid: str = "fused", reduction: str = "mean"):
        super().__init__(alpha, beta, ksize, dist_norm, criterion, pyramid, reduction=reduction)

    def _args(self):
        return float(self.alpha), float(self.beta), int(self._crit)

    @staticmethod
    def _fwd(args, sr, gt, gt2, gt4, idx, loss, ws, stream):
        alpha, beta, crit = args
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_gram_forward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W, alpha, beta, crit, _ptr(idx),
                                           _ptr(loss), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_gram_forward")

    @staticmethod
    def _bwd(args, sr, gt, gt2, gt4, idx, grad_out, d_sr, d_gt, ws, stream):
        crit = args[2]
        B, _, H, W = sr.shape
        if d_sr is not None:
            rc = _cabi.lib().srst_gram_backward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx), _ptr(grad_out), B, H, W,
                                                crit, _ptr(d_sr), _ptr(ws), ws.numel(), stream)
            _cabi.check(rc, "srst_gram_backward")
        if d_gt is not None:
            _patch_backward_gt(1, sr, gt, gt2, gt4, idx, grad_out, _NO_TAPS, crit, d_gt, ws, stream)


class PatchwiseStructureTensorLoss(_PatchLoss):
    """Patchwise structure-tensor loss; same signature and semantics as reference loss.py:292-375:
    the best-buddy search and the final criterion run on the det-normalised structure tensor of
    every 3x3 patch (seen as a 3x3 image, zero 'same' padding) instead of its pixels.
    Only ``ksize=3`` has kernels (the reference's default); ``dist_norm`` may be 'l2' or 'l1'.
    ``reduction='none'`` returns the ``[B]`` per-image losses."""

    _criterion_error = "%s criterion has not been supported."   # loss.py:323
    _MODE = 2

    def __init__(self, sigma: float = 0.5, rho: float = 2, alpha: float = 1.0, beta: float = 1.0, ksize: int = 3,
                 dist_norm: str = "l2", criterion: str = "l1", pyramid: str = "fused", reduction: str = "mean"):
        super().__init__(alpha, beta, ksize, dist_norm, criterion, pyramid, reduction=reduction)
        self.sigma = sigma
        self.rho = rho

    def _args(self):
        return float(self.alpha), float(self.beta), int(self._crit), _pst_taps(self.sigma, self.rho)

    @staticmethod
    def _taps_of(args):
        return args[3]

    @staticmethod
    def _fwd(args, sr, gt, gt2, gt4, idx, loss, ws, stream):
        alpha, beta, crit, taps = args
        B, _, H, W = sr.shape
        rc = _cabi.lib().srst_pst_forward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), B, H, W, *taps[:5], alpha, beta, crit,
                                          _ptr(idx), _ptr(loss), _ptr(ws), ws.numel(), stream)
        _cabi.check(rc, "srst_pst_forward")

    @staticmethod
    def _bwd(args, sr, gt, gt2, gt4, idx, grad_out, d_sr, d_gt, ws, stream):
        crit, taps = args[2:]
        B, _, H, W = sr.shape
        if d_sr is not None:
            rc = _cabi.lib().srst_pst_backward(_ptr(sr), _ptr(gt), _ptr(gt2), _ptr(gt4), _ptr(idx), _ptr(grad_out), B, H, W,
                                               *taps[:5], crit, _ptr(d_sr), _ptr(ws), ws.numel(), stream)
            _cabi.check(rc, "srst_pst_backward")
        if d_gt is not None:
            _patch_backward_gt(2, sr, gt, gt2, gt4, idx, grad_out, taps, crit, d_gt, ws, stream)
