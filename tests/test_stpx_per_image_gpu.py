"""GPU: reduction='none' of StructureTensorPixelLoss, the fused ST + "Pixel" (MSE) criterion, through the module.

Entry b must be st_weight * StructureTensorLoss(reduction='none')(x, gt)[b] + pixel_weight * mean((x[b] - gt[b])**2),
computed in one fused pass per direction, with last_terms holding the two [B] rows.  Held to the golden fixtures of
tests/test_stpx.py per image, and to the unfused modules (loss 1e-6, x.grad 1e-5 max-norm) at the warm-up batch
shape, at full-size DIV2K crops and at a ragged shape, for weighted and stride-0 (.sum()) upstream gradients.
reduction='mean' gives the bits of a module built without the keyword, and a fused 'none' step captured into a CUDA
graph replays with the bits of the eager step."""
import numpy as np
import pytest
import torch

from oracle import st_oracle as O
from tests.helpers import golden, maxnorm_err, rel_err

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
CASES = ["st_rand_2x24x36", "st_srlike_2x40x52", "st_rand_ragged_1x37x53"]   # those of tests/test_stpx.py


def _pair(B, H, W, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    hr = torch.randint(0, 256, (B, 3, H, W), generator=g).float() / 255
    sr = (hr + 0.05 * torch.randn(B, 3, H, W, generator=g)).clamp(0, 1)
    return sr.to(DEV), hr.to(DEV)


def _grad_of(loss_fn, sr, hr, reduce):
    x = sr.clone().requires_grad_(True)
    loss = loss_fn(x, hr)
    reduce(loss).backward()
    torch.cuda.synchronize()
    return loss.detach(), x.grad


@pytest.mark.parametrize("name", CASES)
def test_golden_per_image(name):
    from srgan_st_b200 import StructureTensorPixelLoss
    z = golden(name)
    taps = (z["g"], z["dg"], z["k"])
    w_st, w_px = 1.0 / 3.0, 1.7
    m = StructureTensorPixelLoss(st_weight=w_st, pixel_weight=w_px, reduction="none")
    sr, hr = torch.from_numpy(z["sr"]).to(DEV), torch.from_numpy(z["hr"]).to(DEV)
    loss, d_sr = _grad_of(m, sr, hr, lambda t: t.mean())
    B = z["sr"].shape[0]
    st, px = m.last_terms
    assert loss.shape == st.shape == px.shape == (B,) and loss.dtype == torch.float32
    assert not st.requires_grad and not px.requires_grad
    assert rel_err(st.double().mean().item(), z["loss"]) < 1e-5     # the reference's own ST loss of the batch
    d = z["sr"].astype(np.float64) - z["hr"].astype(np.float64)
    for b in range(B):
        ref = O.st_loss(z["sr"][b:b + 1], z["hr"][b:b + 1], taps=taps, want_grad=False)
        assert rel_err(st[b].item(), ref["loss"]) < 1e-5
        assert rel_err(px[b].item(), (d[b] ** 2).mean()) < 1e-6
        assert rel_err(loss[b].item(), w_st * st[b].item() + w_px * px[b].item()) < 1e-6
    # .mean() over the images is the batch mean: the golden ST gradient plus the MSE gradient 2 d / n
    want = w_st * z["d_sr"].astype(np.float64) + w_px * 2.0 * d / d.size
    ref64 = O.st_loss(z["sr"], z["hr"], taps=taps)
    tol = 1e-4 + maxnorm_err(z["d_sr"], ref64["d_sr"])     # the reference's own fp32 noise (DESIGN.md section 6)
    assert maxnorm_err(d_sr.cpu().numpy(), want) < tol


def _unfused(w_st, w_px):
    from srgan_st_b200 import StructureTensorLoss
    st = StructureTensorLoss(reduction="none")
    return lambda x, gt: w_st * st(x, gt) + w_px * ((x - gt) ** 2).mean((1, 2, 3))


@pytest.mark.parametrize("shape", [(64, 96, 96), (2, 1356, 2040), (3, 37, 53)], ids=["configs1", "div2k", "ragged"])
def test_matches_unfused_modules(shape):
    from srgan_st_b200 import StructureTensorPixelLoss
    B, H, W = shape
    sr, hr = _pair(B, H, W, seed=B + H)
    w_st, w_px = 0.5, 2.0
    v = torch.empty(B).uniform_(-2.0, 2.0, generator=torch.Generator().manual_seed(B)).to(DEV)
    fused = StructureTensorPixelLoss(st_weight=w_st, pixel_weight=w_px, reduction="none")
    ref = _unfused(w_st, w_px)
    for reduce in (lambda t: (t * v).sum(), lambda t: t.sum()):   # per-sample weights; the stride-0 [B] of .sum()
        lf, gf = _grad_of(fused, sr, hr, reduce)
        lr, gr = _grad_of(ref, sr, hr, reduce)
        assert lf.shape == (B,)
        assert float((lf.double() - lr.double()).abs().max() / lr.double().abs().max()) < 1e-6
        assert maxnorm_err(gf.cpu().numpy(), gr.cpu().numpy()) < 1e-5
    assert rel_err(fused.last_terms[1].double().mean().item(), torch.nn.functional.mse_loss(sr, hr).item()) < 1e-6


def test_mean_keyword_is_bit_identical_and_repr():
    from srgan_st_b200 import StructureTensorPixelLoss
    sr, hr = _pair(4, 96, 96, seed=5)
    kw = dict(st_weight=0.5, pixel_weight=2.0)
    a, b = StructureTensorPixelLoss(**kw), StructureTensorPixelLoss(reduction="mean", **kw)
    assert repr(a) == repr(b) and "reduction" not in repr(a)
    assert repr(StructureTensorPixelLoss(reduction="none", **kw)).count("reduction='none'") == 1
    (la, ga), (lb, gb) = _grad_of(a, sr, hr, lambda t: t), _grad_of(b, sr, hr, lambda t: t)
    assert la.shape == () and torch.equal(la, lb) and torch.equal(ga, gb)
    assert a.last_terms[0].shape == () and torch.equal(a.last_terms[0], b.last_terms[0])
    assert torch.equal(a.last_terms[1], b.last_terms[1])
    with pytest.raises(ValueError):
        StructureTensorPixelLoss(reduction="sum")


def test_limits_are_unchanged():
    from srgan_st_b200 import StructureTensorPixelLoss
    a = torch.rand(2, 3, 32, 32, device=DEV)
    with pytest.raises(NotImplementedError):
        StructureTensorPixelLoss(rho=4.0, reduction="none")(a, a)   # compiled radius classes only
    with pytest.raises(NotImplementedError):
        StructureTensorPixelLoss(reduction="none")(a.clone().requires_grad_(True), a.clone().requires_grad_(True))


def test_none_step_replays_from_a_cuda_graph():
    from srgan_st_b200 import StructureTensorPixelLoss
    torch.manual_seed(2)
    crit = StructureTensorPixelLoss(st_weight=0.5, pixel_weight=2.0, reduction="none")
    gen = torch.nn.Conv2d(3, 3, 3, padding=1).to(DEV)
    opt = torch.optim.SGD(gen.parameters(), lr=1e-3)
    gt = torch.rand(4, 3, 48, 48, device=DEV)
    lr = (gt + 0.1 * torch.randn_like(gt)).clamp(0, 1)
    w = torch.tensor([1.0, 0.0, 2.0, 0.5], device=DEV)   # per-sample weights, one masked out

    def step():
        sr = gen(lr).clamp(0, 1)
        per = crit(sr, gt)
        opt.zero_grad(set_to_none=False)
        (per * w).sum().backward()
        return torch.cat([per.detach(), *crit.last_terms])

    for _ in range(2):
        step()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(2):
            step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        static = step()
    with torch.no_grad():
        snapshot = [p.detach().clone() for p in gen.parameters()]
    graph.replay()
    torch.cuda.synchronize()
    replayed, grads = static.clone(), [p.grad.clone() for p in gen.parameters()]
    with torch.no_grad():
        for p, q in zip(gen.parameters(), snapshot):
            p.copy_(q)
    eager = step()
    torch.cuda.synchronize()
    assert torch.isfinite(replayed).all() and replayed.shape == (12,)
    assert torch.equal(replayed, eager)
    for a, p in zip(grads, gen.parameters()):
        assert torch.allclose(a, p.grad, rtol=1e-5, atol=1e-8)   # conv backward may reorder
