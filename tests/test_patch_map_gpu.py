"""GPU: the per-patch loss map (``loss_map``) of BestBuddyLoss, GramLoss and PatchwiseStructureTensorLoss.

The golden fixtures (outputs of the reference): the map recomputed in float64 from the fixture's indices, and its mean
against the fixture's loss.  Agreement with ``forward`` ('mean' and 'none') at training-crop sizes, the gradients of a
border-masked and of a random-weight ``(m * w).sum()`` against float64, both pyramids, CUDA-graph replay, 0xFF-poisoned
allocations and the errors of ``forward``."""
import numpy as np
import pytest
import torch

from oracle import bbg_oracle as GO
from oracle import st_oracle as O
from tests import patch_map_ref as R
from tests.helpers import golden, golden_names, maxnorm_err, rel_err

pytestmark = pytest.mark.gpu
DEV = torch.device("cuda:0")
MODES = ("patch", "gram", "pst")


def _cls(mode):
    from srgan_st_b200 import BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss
    return {"patch": BestBuddyLoss, "gram": GramLoss, "pst": PatchwiseStructureTensorLoss}[mode]


def _pair(B, H, W, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    hr = torch.randint(0, 256, (B, 3, H, W), generator=g).float() / 255
    sr = (hr + 0.05 * torch.randn(B, 3, H, W, generator=g)).clamp(0, 1)
    return sr.to(DEV), hr.to(DEV)


def _map_grads(module, sr, hr, w, want_gt=True):
    """(map, d_sr, d_gt, idx) of (module.loss_map(x, y) * w).sum()."""
    x = sr.clone().requires_grad_(True)
    y = hr.clone().requires_grad_(want_gt)
    m = module.loss_map(x, y)
    (m * w).sum().backward()
    torch.cuda.synchronize()
    return m.detach(), x.grad, (y.grad if want_gt else None), module.last_indices


def _taps_of(d):
    return (d["g"], d["dg"], d["k"]) if "g" in d.files else (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0))


# ---- golden fixtures ---------------------------------------------------------------------------------------------
def _fixtures():
    out = []
    for prefix, mode in (("bb_", "patch"), ("bbl1_", None), ("gram", "gram"), ("pst", "pst"), ("bbg_", "patch")):
        for n in golden_names(prefix):
            d = golden(n)
            m = mode or {"bb": "patch", "gram": "gram", "pst": "pst"}[str(d["which"])]
            out.append((n, m))
    return out


@pytest.mark.parametrize("name,mode", _fixtures(), ids=[n for n, _ in _fixtures()])
def test_golden_fixture_map(name, mode):
    d = golden(name)
    crit = str(d["criterion"])
    dist = "l1" if name.startswith(("bbl1", "graml1", "pstl1")) else (str(d["dist_norm"]) if "dist_norm" in d.files else "l2")
    kw = dict(alpha=float(d["alpha"]), beta=float(d["beta"]), criterion=crit, dist_norm=dist, pyramid="aten")
    geom = (int(d["ksize"]), int(d["pad"]), int(d["stride"])) if "ksize" in d.files else None
    if mode == "pst":
        kw.update(sigma=float(d["sigma"]) if "sigma" in d.files else 0.5, rho=float(d["rho"]) if "rho" in d.files else 2.0)
    if geom is not None:
        kw.update(ksize=geom[0], pad=geom[1], stride=geom[2])
    module = _cls(mode)(**kw)
    sr, hr = (torch.from_numpy(np.ascontiguousarray(d[k], np.float32)).to(DEV) for k in ("sr", "hr"))
    m = module.loss_map(sr, hr)
    torch.cuda.synchronize()
    B, _, H, W = sr.shape
    ny, nx = (H // 3, W // 3) if geom is None else (GO.npatch(H, *geom), GO.npatch(W, *geom))
    assert m.shape == (B, ny, nx) and m.dtype == torch.float32
    ind = d["ind"]

    def f64(idx):
        if geom is None:
            return R.patch_map(d["sr"], d["hr"], idx, mode, _taps_of(d) if mode == "pst" else None, crit, d["hr2"], d["hr4"])
        return R.bbg_map(d["sr"], d["hr"], idx, *geom, crit, d["hr2"], d["hr4"])

    ref = f64(ind)
    assert rel_err(float(ref.mean()), float(d["loss"])) < 1e-5 or float(d["loss"]) == 0.0
    # the indices may differ from the reference's on near-ties (and, with dist_norm='l1', on the exact ties of the Gram
    # and PatchwiseST descriptors: tests/test_dist_l1.py): the fixture's loss holds when every index agrees; entry by
    # entry, the fixture's map holds where they agree, and the map of the indices this call chose holds everywhere
    own = module.last_indices.cpu().numpy()
    if (own == ind).all():
        assert rel_err(m.double().mean().item(), float(d["loss"])) < 1e-5 or abs(m.double().mean().item()) < 1e-7
    same = (own == ind).reshape(B, ny, nx)
    got = m.cpu().numpy()
    scale = max(np.abs(ref).max(), 1e-30)
    assert np.abs(got[same] - ref.reshape(B, ny, nx)[same]).max(initial=0.0) <= 1e-5 * scale
    assert np.abs(got.reshape(B, -1) - f64(own)).max() <= 1e-5 * scale


# ---- agreement with forward --------------------------------------------------------------------------------------
CASES = [(m, s) for m in MODES for s in ((64, 96, 96), (64, 192, 192))] + [("bbg", (16, 96, 96))]


@pytest.mark.parametrize("mode,shape", CASES, ids=[f"{m}-{s[0]}x{s[1]}x{s[2]}" for m, s in CASES])
def test_map_agrees_with_forward(mode, shape):
    B, H, W = shape
    kw = dict(ksize=4, pad=0, stride=4) if mode == "bbg" else {}
    cls = _cls("patch" if mode == "bbg" else mode)
    sr, hr = _pair(B, H, W, seed=B + H + len(mode))
    a, b, c = cls(**kw), cls(reduction="none", **kw), cls(**kw)
    mean = a(sr, hr)
    none = b(sr, hr)
    m = c.loss_map(sr, hr)
    torch.cuda.synchronize()
    assert m.shape == ((B, H // 4, W // 4) if mode == "bbg" else (B, H // 3, W // 3))
    assert torch.equal(c.last_indices, a.last_indices) and torch.equal(c.last_indices, b.last_indices)
    assert rel_err(m.double().mean().item(), mean.item()) < 1e-6
    per = m.double().mean(dim=(1, 2))
    assert (per - none.double()).abs().max().item() <= 1e-6 * none.abs().max().item()
    # the map's upstream gradient 1/(B N) is the gradient of the mean: same d_sr and d_gt as forward
    x, y = sr.clone().requires_grad_(True), hr.clone().requires_grad_(True)
    cls(**kw)(x, y).backward()
    _, d_sr, d_gt, _ = _map_grads(cls(**kw), sr, hr, 1.0 / m.numel())
    assert maxnorm_err(d_sr.cpu().numpy(), x.grad.cpu().numpy()) < 1e-6
    assert maxnorm_err(d_gt.cpu().numpy(), y.grad.cpu().numpy()) < 1e-6
    # and .mean() of the map (a stride-0 upstream gradient) too
    x2, y2 = sr.clone().requires_grad_(True), hr.clone().requires_grad_(True)
    cls(**kw).loss_map(x2, y2).mean().backward()
    assert maxnorm_err(x2.grad.cpu().numpy(), x.grad.cpu().numpy()) < 1e-6


# ---- weighted gradients against float64 ---------------------------------------------------------------------------
def _border_mask(B, ny, nx):
    w = torch.zeros(B, ny, nx, device=DEV)
    w[:, 2:-2, 2:-2] = 1
    return w


def _random_weight(B, ny, nx, seed):
    return torch.empty(B, ny, nx).uniform_(-2.0, 2.0, generator=torch.Generator().manual_seed(seed)).to(DEV)


@pytest.mark.parametrize("mode", list(MODES) + ["bbg"])
@pytest.mark.parametrize("weight", ["border", "random"])
@pytest.mark.parametrize("pyramid", ["fused", "aten"])
def test_weighted_gradients_against_float64(mode, weight, pyramid):
    B, H, W = 3, 50, 61   # H % 3 != 0, W % 3 != 0
    geom = (4, 1, 2) if mode == "bbg" else None
    kw = dict(criterion="l2" if mode == "gram" else "l1", pyramid=pyramid)
    if geom:
        kw.update(ksize=4, pad=1, stride=2)
    module = _cls("patch" if geom else mode)(**kw)
    sr, hr = _pair(B, H, W, seed=7 + len(mode))
    ny, nx = (H // 3, W // 3) if geom is None else (GO.npatch(H, *geom), GO.npatch(W, *geom))
    w = _border_mask(B, ny, nx) if weight == "border" else _random_weight(B, ny, nx, 5)
    m, d_sr, d_gt, idx = _map_grads(module, sr, hr, w)
    s, t, i, wn = sr.cpu().numpy(), hr.cpu().numpy(), idx.cpu().numpy(), w.cpu().numpy().reshape(B, -1)
    gt2 = gt4 = None
    if pyramid == "aten":
        gt2, gt4 = (torch.nn.functional.interpolate(hr, scale_factor=f, mode="bicubic", align_corners=False).cpu().numpy()
                    for f in (0.5, 0.25))
    crit = kw["criterion"]
    if geom is None:
        taps = (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0)) if mode == "pst" else None
        ref_map = R.patch_map(s, t, i, mode, taps, crit, gt2, gt4)
        r_sr, r_gt = R.patch_grads(s, t, i, wn, mode, taps, crit, gt2, gt4)
    else:
        ref_map = R.bbg_map(s, t, i, *geom, crit, gt2, gt4)
        r_sr, r_gt = R.bbg_grads(s, t, i, *geom, crit, wn)
    assert maxnorm_err(m.cpu().numpy().reshape(B, -1), ref_map) < 1e-5
    assert maxnorm_err(d_sr.cpu().numpy(), r_sr) < 1e-4
    assert maxnorm_err(d_gt.cpu().numpy(), r_gt) < 1e-4


# ---- CUDA graph ----------------------------------------------------------------------------------------------------
def test_map_step_replays_from_a_cuda_graph():
    from srgan_st_b200 import BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss
    torch.manual_seed(2)
    crits = [BestBuddyLoss(), GramLoss(), PatchwiseStructureTensorLoss(), BestBuddyLoss(ksize=4, pad=1, stride=2)]
    gen = torch.nn.Conv2d(3, 3, 3, padding=1).to(DEV)
    opt = torch.optim.SGD(gen.parameters(), lr=1e-3)
    gt = torch.rand(4, 3, 48, 48, device=DEV)
    lr = (gt + 0.1 * torch.randn_like(gt)).clamp(0, 1)
    ws = [_border_mask(4, 16, 16), _border_mask(4, 16, 16), _random_weight(4, 16, 16, 1), _random_weight(4, 24, 24, 2)]

    def step():
        sr = gen(lr).clamp(0, 1)
        maps = [c.loss_map(sr, gt) for c in crits]
        total = sum((m * w).sum() for m, w in zip(maps, ws))
        opt.zero_grad(set_to_none=False)
        total.backward()
        return torch.cat([m.detach().reshape(-1) for m in maps])

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
    assert torch.isfinite(replayed).all()
    assert torch.equal(replayed, eager)
    for a, p in zip(grads, gen.parameters()):
        assert torch.allclose(a, p.grad, rtol=1e-5, atol=1e-8)   # the conv's own backward may reorder


# ---- poisoned allocations ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", list(MODES) + ["bbg"])
def test_poisoned_allocations_same_bits(monkeypatch, mode):
    from srgan_st_b200 import loss as L
    from tests.test_st_map_gpu import _PoisonedTorch   # empty / empty_like hand out 0xFF bytes (NaN as a float)
    kw = dict(ksize=3, pad=1, stride=1) if mode == "bbg" else {}
    module = _cls("patch" if mode == "bbg" else mode)(**kw)
    sr, hr = _pair(2, 37, 44, seed=11)
    shape = module.loss_map(sr, hr).shape
    w = _random_weight(*shape, 3)
    clean = _map_grads(module, sr, hr, w)
    with monkeypatch.context() as m:
        m.setattr(L, "torch", _PoisonedTorch())
        dirty = _map_grads(module, sr, hr, w)
    assert torch.equal(clean[0], dirty[0]) and torch.equal(clean[1], dirty[1]) and torch.equal(clean[3], dirty[3])
    assert not torch.isnan(dirty[2]).any()
    assert maxnorm_err(dirty[2].cpu().numpy(), clean[2].cpu().numpy()) < 1e-6   # d_gt sums with atomicAdd


# ---- errors --------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode", list(MODES) + ["bbg"])
def test_errors_match_forward(mode):
    kw = dict(ksize=5, pad=0, stride=5) if mode == "bbg" else {}
    module = _cls("patch" if mode == "bbg" else mode)(**kw)
    x = torch.rand(1, 3, 24, 24, device=DEV)
    bad = [((x.cpu(), x.cpu()), RuntimeError), ((x.double(), x.double()), TypeError), ((x[:, :2], x[:, :2]), ValueError),
           ((x, x[:, :, :12]), ValueError), ((x[:, :, :9, :9], x[:, :, :9, :9]), ValueError), ((x, "gt"), TypeError)]
    for args, exc in bad:
        with pytest.raises(exc) as e_fwd:
            module(*args)
        with pytest.raises(exc) as e_map:
            module.loss_map(*args)
        assert str(e_fwd.value) == str(e_map.value)
