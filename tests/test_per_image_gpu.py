"""GPU: reduction='none' of StructureTensorLoss and the three patch losses, through the modules.

Per image, the [B] losses and the gradients of (w * loss).sum() are held to the float64 oracles run on that image
alone (loss 1e-5, gradients 1e-4 max-norm, the bounds of the scalar tests).  reduction='mean' gives the bits of a
module built without the keyword, w = 1/B reproduces the mean path's gradients to 1e-6, and a reduction='none' step
captured into a CUDA graph replays with the bits of the eager step."""
import numpy as np
import pytest
import torch

from oracle import bb_oracle as BO
from oracle import st_oracle as O
from tests.helpers import maxnorm_err, rel_err

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")


def _pair(B, H, W, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    hr = torch.randint(0, 256, (B, 3, H, W), generator=g).float() / 255
    sr = (hr + 0.05 * torch.randn(B, 3, H, W, generator=g)).clamp(0, 1)
    return sr.to(DEV), hr.to(DEV)


def _weights(B, seed):
    return torch.empty(B).uniform_(-2.0, 2.0, generator=torch.Generator().manual_seed(seed)).to(DEV)


def _run(module, sr, hr, w=None, want_gt=True):
    x = sr.clone().requires_grad_(True)
    y = hr.clone().requires_grad_(want_gt)
    loss = module(x, y)
    (loss if w is None else (w * loss).sum()).backward()
    torch.cuda.synchronize()
    return loss.detach(), x.grad, (y.grad if want_gt else None), getattr(module, "last_indices", None)


@pytest.mark.parametrize("shape", [(64, 96, 96), (2, 1356, 2040)], ids=["configs1", "div2k"])
def test_st_none_matches_per_image_oracle(shape):
    from srgan_st_b200 import StructureTensorLoss
    B, H, W = shape
    sr, hr = _pair(B, H, W, seed=B)
    w = _weights(B, seed=1)
    loss, d_sr, d_hr, _ = _run(StructureTensorLoss(reduction="none"), sr, hr, w)
    assert loss.shape == (B,) and loss.dtype == torch.float32
    check = range(B) if B <= 4 else (0, 17, B - 1)
    srn, hrn, wn = sr.cpu().numpy(), hr.cpu().numpy(), w.cpu().numpy()
    for b in check:
        ref = O.st_loss(srn[b:b + 1], hrn[b:b + 1], want_hr_grad=True)
        assert rel_err(loss[b].item(), ref["loss"]) < 1e-5
        assert maxnorm_err(d_sr[b].cpu().numpy(), wn[b] * ref["d_sr"][0]) < 1e-4
        assert maxnorm_err(d_hr[b].cpu().numpy(), wn[b] * ref["d_hr"][0]) < 1e-4
    # the mean path: same loss on average, same gradients with w = 1/B
    mean, m_sr, m_hr, _ = _run(StructureTensorLoss(), sr, hr)
    assert rel_err(loss.double().mean().item(), mean.item()) < 1e-6
    _, n_sr, n_hr, _ = _run(StructureTensorLoss(reduction="none"), sr, hr, torch.full((B,), 1.0 / B, device=DEV))
    assert maxnorm_err(n_sr.cpu().numpy(), m_sr.cpu().numpy()) < 1e-6
    assert maxnorm_err(n_hr.cpu().numpy(), m_hr.cpu().numpy()) < 1e-6


def test_st_generic_radius_none():
    from srgan_st_b200 import StructureTensorLoss
    sr, hr = _pair(3, 40, 52, seed=3)
    w = _weights(3, seed=2)
    loss, d_sr, _, _ = _run(StructureTensorLoss(sigma=1.5, rho=4.0, reduction="none"), sr, hr, w, want_gt=False)
    taps = (*O.gaussian_taps(1.5, True), O.gaussian_taps(4.0))
    for b in range(3):
        ref = O.st_loss(sr[b:b + 1].cpu().numpy(), hr[b:b + 1].cpu().numpy(), taps=taps)
        assert rel_err(loss[b].item(), ref["loss"]) < 1e-5
        assert maxnorm_err(d_sr[b].cpu().numpy(), w[b].item() * ref["d_sr"][0]) < 1e-4


def _patch_oracle(mode, sr, gt, idx, crit, taps):
    """float64 loss, d_sr, d_gt of one image [1,3,H,W] given its indices [1,N] (the library's own pyramid levels)."""
    gt2, gt4 = BO.pyramid_c(gt)
    desc = {"patch": BO.unfold3, "gram": BO.gram_descriptors, "pst": lambda t: BO.pst_descriptors(t, taps)}[mode]
    cat = np.concatenate([desc(t) for t in (gt, gt2, gt4)], 1)
    sel = np.take_along_axis(cat, idx[..., None], 1)
    diff = desc(sr).astype(np.float64) - sel
    loss = np.abs(diff).mean() if crit == "l1" else (diff ** 2).mean()
    if mode == "patch":
        d_sr = BO.bb_backward(sr, sel, crit)
    elif mode == "gram":
        d_sr = BO.gram_backward(sr, sel, crit)
    else:
        d_sr = BO.pst_backward(sr, sel, taps, crit)
    d_gt = BO.patch_backward_gt(sr, gt, gt2, gt4, idx, mode, taps, crit)
    return loss, d_sr, d_gt


@pytest.mark.parametrize("mode", ["patch", "gram", "pst"])
@pytest.mark.parametrize("crit", ["l1", "l2"])
def test_patch_none_matches_per_image_oracle(mode, crit):
    from srgan_st_b200 import BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss
    cls = {"patch": BestBuddyLoss, "gram": GramLoss, "pst": PatchwiseStructureTensorLoss}[mode]
    B, H, W = 4, 192, 192
    sr, hr = _pair(B, H, W, seed=len(mode) + (crit == "l2"))
    w = _weights(B, seed=3)
    loss, d_sr, d_gt, idx = _run(cls(criterion=crit, reduction="none"), sr, hr, w)
    mean, m_sr, m_gt, m_idx = _run(cls(criterion=crit), sr, hr)
    assert torch.equal(idx, m_idx)                          # the search is untouched
    assert rel_err(loss.double().mean().item(), mean.item()) < 1e-6
    taps = (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0)) if mode == "pst" else None
    for b in range(B):
        s, t = sr[b:b + 1].cpu().numpy(), hr[b:b + 1].cpu().numpy()
        ref_loss, ref_sr, ref_gt = _patch_oracle(mode, s, t, idx[b:b + 1].cpu().numpy(), crit, taps)
        assert rel_err(loss[b].item(), ref_loss) < 1e-5
        assert maxnorm_err(d_sr[b].cpu().numpy(), w[b].item() * ref_sr[0]) < 1e-4
        assert maxnorm_err(d_gt[b].cpu().numpy(), w[b].item() * ref_gt[0]) < 1e-4
    _, n_sr, n_gt, _ = _run(cls(criterion=crit, reduction="none"), sr, hr, torch.full((B,), 1.0 / B, device=DEV))
    assert maxnorm_err(n_sr.cpu().numpy(), m_sr.cpu().numpy()) < 1e-6
    assert maxnorm_err(n_gt.cpu().numpy(), m_gt.cpu().numpy()) < 1e-6


def test_bbg_none_matches_one_image_calls():
    """A non-default geometry: entry b equals the reference module on image b alone (here: the scalar path on
    x[b:b+1], which tests/test_bb_geometry.py holds to the float64 restatement); d_sr of image b is bit-identical to
    that call with its upstream gradient w[b]."""
    from srgan_st_b200 import BestBuddyLoss
    B, H, W = 3, 60, 66
    sr, hr = _pair(B, H, W, seed=9)
    w = _weights(B, seed=4)
    kw = dict(ksize=4, pad=1, stride=2, criterion="l2")
    loss, d_sr, d_gt, idx = _run(BestBuddyLoss(reduction="none", **kw), sr, hr, w)
    for b in range(B):
        one = BestBuddyLoss(**kw)
        x, y = sr[b:b + 1].clone().requires_grad_(True), hr[b:b + 1].clone().requires_grad_(True)
        lb = one(x, y)
        (w[b] * lb).backward()
        assert torch.equal(one.last_indices[0], idx[b])
        assert rel_err(loss[b].item(), lb.item()) < 1e-6
        assert torch.equal(d_sr[b], x.grad[0])
        assert maxnorm_err(d_gt[b].cpu().numpy(), y.grad[0].cpu().numpy()) < 1e-6


def test_mean_keyword_is_bit_identical_and_repr():
    from srgan_st_b200 import BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss, StructureTensorLoss
    sr, hr = _pair(4, 96, 96, seed=5)
    for cls, kw in ((StructureTensorLoss, {}), (BestBuddyLoss, {}), (BestBuddyLoss, dict(ksize=4, pad=1, stride=2)),
                    (GramLoss, {}), (PatchwiseStructureTensorLoss, {})):
        a, b = cls(**kw), cls(reduction="mean", **kw)
        assert repr(a) == repr(b) and "reduction" not in repr(a)
        assert repr(cls(reduction="none", **kw)).count("reduction='none'") == 1
        (la, sa, ga, ia), (lb, sb, gb, ib) = _run(a, sr, hr), _run(b, sr, hr)
        assert torch.equal(la, lb) and torch.equal(sa, sb) and (ia is None and ib is None or torch.equal(ia, ib))
        if cls is StructureTensorLoss:
            assert torch.equal(ga, gb)
        else:   # the gradient w.r.t. gt sums with atomicAdd
            assert maxnorm_err(ga.cpu().numpy(), gb.cpu().numpy()) < 1e-6
        with pytest.raises(ValueError):
            cls(reduction="sum", **kw)


def test_none_step_replays_from_a_cuda_graph():
    from srgan_st_b200 import BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss, StructureTensorLoss
    torch.manual_seed(2)
    crits = [StructureTensorLoss(reduction="none"), BestBuddyLoss(reduction="none"), GramLoss(reduction="none"),
             PatchwiseStructureTensorLoss(reduction="none"), BestBuddyLoss(ksize=4, pad=1, stride=2, reduction="none")]
    gen = torch.nn.Conv2d(3, 3, 3, padding=1).to(DEV)
    opt = torch.optim.SGD(gen.parameters(), lr=1e-3)
    gt = torch.rand(4, 3, 48, 48, device=DEV)
    lr = (gt + 0.1 * torch.randn_like(gt)).clamp(0, 1)
    w = torch.tensor([1.0, 0.0, 2.0, 0.5], device=DEV)   # per-sample weights, one masked out

    def step():
        sr = gen(lr).clamp(0, 1)
        per = torch.stack([m(sr, gt) for m in crits])    # [5, B]
        total = (per * w).sum()
        opt.zero_grad(set_to_none=False)
        total.backward()
        return per.detach()

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
    assert torch.isfinite(replayed).all() and replayed.shape == (5, 4)
    assert torch.equal(replayed, eager)
    for a, p in zip(grads, gen.parameters()):
        assert torch.allclose(a, p.grad, rtol=1e-5, atol=1e-8)   # d_gt-free here, but conv backward may reorder
