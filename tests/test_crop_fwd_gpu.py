"""GPU: the crop layout of the marching forward, which the library picks for images no wider than 96 columns.  It
stages no x halo and skips the warps whose rows are all outside the image, but moves no per-pixel operation, so ds,
ixy, the distance map and the gradients must be bit-identical to those of the 112-column halo strips (forward cfg 4)
on the same input.  The losses are reduced from differently shaped CTAs, so they are held to 1e-6."""
import ctypes

import pytest
import torch

from srgan_st_b200 import StructureTensorLoss, StructureTensorPixelLoss, _cabi, structure_tensor_distance
from srgan_st_b200 import taps as T

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
HALO = 4   # forward cfg id of the 112-column strips


def _pair(B, H, W, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    hr = torch.rand(B, 3, H, W, generator=g)
    sr = (hr + 0.05 * torch.randn(B, 3, H, W, generator=g)).clamp(0, 1)
    return sr.to(DEV), hr.to(DEV)


def _forced(fwd_cfg, fn):
    lib = _cabi.lib()
    assert lib.srst_st_force_cfg(fwd_cfg, -1) == 0
    try:
        out = fn()
        torch.cuda.synchronize()
        return out
    finally:
        lib.srst_st_force_cfg(-1, -1)


def _cabi_forward(sr, hr):
    """srst_st_forward with ds and ixy of both images."""
    lib = _cabi.lib()
    B, _, H, W = sr.shape
    vp = lambda t: ctypes.c_void_p(t.data_ptr())
    g, dg = T.gaussian_taps(0.5)
    k, _ = T.gaussian_taps(2.0)
    loss = torch.zeros((), device=DEV)
    ds = [torch.full_like(sr, float("nan")) for _ in range(2)]
    ixy = [torch.full((lib.srst_st_ixy_floats(B, H, W),), float("nan"), device=DEV) for _ in range(2)]
    ws = torch.zeros(lib.srst_st_workspace_bytes(B, H, W), dtype=torch.uint8, device=DEV)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
    _cabi.check(lib.srst_st_forward(vp(sr), vp(hr), B, H, W, T.as_c(g), T.as_c(dg), 2, T.as_c(k), 8, 1, 1e-12, vp(loss),
                                    vp(ds[0]), vp(ds[1]), vp(ixy[0]), vp(ixy[1]), vp(ws), ws.numel(), stream), "fwd")
    return loss, ds, ixy


def _grads(module, sr, hr, w=None, gt_grad=True):
    x = sr.clone().requires_grad_(True)
    y = hr.clone().requires_grad_(gt_grad)
    loss = module(x, y)
    (loss if w is None else (w * loss).sum()).backward()
    return loss.detach(), x.grad, y.grad


def _close(a, b, tol=1e-6):
    return bool(((a.double() - b.double()).abs() <= tol * b.double().abs()).all())


@pytest.mark.parametrize("shape", [(16, 96, 96), (64, 96, 96), (1024, 96, 96), (64, 90, 92)],
                         ids=lambda s: "x".join(map(str, s)))
def test_crop_forward_matches_halo_strips(shape):
    sr, hr = _pair(*shape, seed=sum(shape))
    loss, ds, ixy = _forced(-1, lambda: _cabi_forward(sr, hr))
    r_loss, r_ds, r_ixy = _forced(HALO, lambda: _cabi_forward(sr, hr))
    for a, b in zip(ds + ixy, r_ds + r_ixy):
        assert torch.isfinite(a).all() and torch.equal(a, b)
    assert _close(loss, r_loss)
    l, d_sr, d_hr = _forced(-1, lambda: _grads(StructureTensorLoss(), sr, hr))
    rl, r_sr, r_hr = _forced(HALO, lambda: _grads(StructureTensorLoss(), sr, hr))
    assert torch.equal(d_sr, r_sr) and torch.equal(d_hr, r_hr)
    assert _close(l, rl) and torch.equal(l, loss)


def test_crop_forward_reductions_and_map():
    sr, hr = _pair(64, 96, 96, seed=11)
    w = torch.empty(64).uniform_(-2.0, 2.0, generator=torch.Generator().manual_seed(5)).to(DEV)
    for module in (StructureTensorLoss(reduction="none"), StructureTensorPixelLoss(),
                   StructureTensorPixelLoss(reduction="none")):
        wi = w if module.reduction == "none" else None
        gt_grad = isinstance(module, StructureTensorLoss)
        l, d_sr, _ = _forced(-1, lambda: _grads(module, sr, hr, wi, gt_grad))
        rl, r_sr, _ = _forced(HALO, lambda: _grads(module, sr, hr, wi, gt_grad))
        assert torch.equal(d_sr, r_sr), module
        assert _close(l, rl), module
    wm = torch.rand(64, 96, 96, generator=torch.Generator().manual_seed(9)).to(DEV)
    dist = lambda x, y: structure_tensor_distance(x, y)
    m, d_sr, d_hr = _forced(-1, lambda: _grads(dist, sr, hr, wm))
    rm, r_sr, r_hr = _forced(HALO, lambda: _grads(dist, sr, hr, wm))
    assert torch.equal(m, rm) and torch.equal(d_sr, r_sr) and torch.equal(d_hr, r_hr)
