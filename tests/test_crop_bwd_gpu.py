"""GPU: the crop-width backward picks its strip height from the batch (12 rows at 16 x 96x96, 24 rows at 64 and
1024 x 96x96).  Neither the strip height nor the missing x halo changes a per-pixel operation, so the gradients must
be bit-identical to those of the 28x56 tiles (cfg 0, which stage the x halo) and, per image, to one-image calls."""
import pytest
import torch

from srgan_st_b200 import StructureTensorLoss, _cabi

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _pair(B, H, W, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    hr = torch.rand(B, 3, H, W, generator=g)
    sr = (hr + 0.05 * torch.randn(B, 3, H, W, generator=g)).clamp(0, 1)
    return sr.to(DEV), hr.to(DEV)


def _grads(module, sr, hr, w=None, bwd_cfg=-1):
    lib = _cabi.lib()
    assert lib.srst_st_force_cfg(-1, bwd_cfg) == 0
    try:
        x = sr.clone().requires_grad_(True)
        y = hr.clone().requires_grad_(True)
        loss = module(x, y)
        (loss if w is None else (w * loss).sum()).backward()
        torch.cuda.synchronize()
    finally:
        lib.srst_st_force_cfg(-1, -1)
    return x.grad, y.grad


@pytest.mark.parametrize("B", [16, 64, 1024])
def test_crop_strips_match_halo_tiles(B):
    sr, hr = _pair(B, 96, 96, seed=B)
    d_sr, d_hr = _grads(StructureTensorLoss(), sr, hr)
    r_sr, r_hr = _grads(StructureTensorLoss(), sr, hr, bwd_cfg=0)
    assert torch.equal(d_sr, r_sr) and torch.equal(d_hr, r_hr)
    assert torch.isfinite(d_sr).all()


def test_crop_strips_per_image_match_one_image_calls():
    B = 64
    sr, hr = _pair(B, 96, 96, seed=7)
    w = torch.empty(B).uniform_(-2.0, 2.0, generator=torch.Generator().manual_seed(3)).to(DEV)
    d_sr, d_hr = _grads(StructureTensorLoss(reduction="none"), sr, hr, w)
    for b in (0, 17, B - 1):
        o_sr, o_hr = _grads(StructureTensorLoss(), sr[b:b + 1], hr[b:b + 1], w[b:b + 1])
        assert torch.equal(d_sr[b], o_sr[0]) and torch.equal(d_hr[b], o_hr[0])
