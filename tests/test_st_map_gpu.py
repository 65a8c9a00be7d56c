"""GPU: structure_tensor_distance, the per-pixel structure-tensor distance map [B,H,W] and its gradient under any
per-pixel weighting, against the golden fixtures, the float64 oracle and StructureTensorLoss (mean and
reduction='none') at training-crop and full-image sizes; CUDA-graph replay, 0xFF-poisoned allocations and the errors."""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests.helpers import golden, golden_names, maxnorm_err, rel_err
from tests.test_emu_st_map import oracle_map_backward

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")
DEV = "cuda:0"


def _weights(B, H, W, seed, band=10):
    """Random upstream gradient with zeros and negative values, times a mask that zeroes the border band where the
    zero 'same' padding acts (r_sigma + r_rho = 10 pixels deep at the default sigma / rho)."""
    g = torch.Generator().manual_seed(seed)
    G = torch.empty(B, H, W).uniform_(-2.0, 2.0, generator=g)
    G[torch.rand(B, H, W, generator=g) < 0.2] = 0.0
    mask = torch.zeros(H, W)
    mask[band:H - band, band:W - band] = 1.0
    return (G * mask).to(DEV)


def _map_grads(x, y, G, **kw):
    from srgan_st_b200 import structure_tensor_distance
    xs = x.detach().clone().requires_grad_(True)
    ys = y.detach().clone().requires_grad_(True)
    d = structure_tensor_distance(xs, ys, **kw)
    (d * G).sum().backward()
    torch.cuda.synchronize()
    return d.detach(), xs.grad, ys.grad


@pytest.mark.parametrize("name", golden_names("st_"))
def test_golden_fixtures(name):
    z = golden(name)
    norm, sigma, rho = bool(z["normalize"]), float(z["sigma"]), float(z["rho"])
    taps = (z["g"], z["dg"], z["k"])
    x, y = (torch.from_numpy(np.ascontiguousarray(z[k])).to(DEV) for k in ("sr", "hr"))
    B, _, H, W = x.shape
    G = _weights(B, H, W, B * H + W, band=2)
    d, gx, gy = _map_grads(x, y, G, sigma=sigma, rho=rho, normalize=norm)
    assert d.shape == (B, H, W) and d.dtype == torch.float32
    # sr == hr: every pixel at the sqrt(eps) floor, held as tests/test_st_gpu.py holds this fixture's loss
    assert rel_err(d.double().mean().item(), z["loss"]) < (2e-2 if "same" in name else 1e-5)
    if "same" in name or "nonorm" in name:
        return
    ref = O.st_loss(z["sr"], z["hr"], normalize=norm, taps=taps, want_hr_grad=True)
    o_sr, o_hr = oracle_map_backward(z["sr"], z["hr"], taps, G.cpu().numpy(), norm)
    # 1e-4 widened by the reference's own distance from float64 on this fixture (tests/test_st_gpu.py)
    for ours, orc, refg, orcg in ((gx, o_sr, z["d_sr"], ref["d_sr"]), (gy, o_hr, z["d_hr"], ref["d_hr"])):
        assert maxnorm_err(ours.cpu().numpy(), orc) < 1e-4 + maxnorm_err(refg, orcg)


@pytest.mark.parametrize("shape", [(64, 96, 96), (1, 1356, 2040), (3, 101, 150)])
def test_matches_the_loss_modules(shape):
    from srgan_st_b200 import StructureTensorLoss, structure_tensor_distance
    B, H, W = shape
    torch.manual_seed(B + H)
    y = torch.rand(B, 3, H, W, device=DEV)
    x = (y + 0.05 * torch.randn_like(y)).clamp(0, 1)

    xs = x.clone().requires_grad_(True)
    ys = y.clone().requires_grad_(True)
    d = structure_tensor_distance(xs, ys)
    m = d.mean()
    m.backward()
    xl = x.clone().requires_grad_(True)
    yl = y.clone().requires_grad_(True)
    loss = StructureTensorLoss()(xl, yl)
    loss.backward()
    per = StructureTensorLoss(reduction="none")(x, y)
    torch.cuda.synchronize()
    assert rel_err(m.item(), loss.item()) < 1e-6
    assert torch.allclose(d.double().mean((1, 2)), per.double(), rtol=1e-6, atol=0)
    assert maxnorm_err(xs.grad.cpu().numpy(), xl.grad.cpu().numpy()) < 1e-6
    assert maxnorm_err(ys.grad.cpu().numpy(), yl.grad.cpu().numpy()) < 1e-6

    # a border-masked, weighted loss against the float64 oracle (two images at most).  Independent images, as in
    # tests/test_st_gpu.py: where SR and HR nearly coincide, fp32 itself sits up to ~4e-4 from float64 (DESIGN.md §6).
    n = min(B, 2)
    G = _weights(n, H, W, H)
    xr, yr = torch.rand(n, 3, H, W, device=DEV), torch.rand(n, 3, H, W, device=DEV)
    _, gx, gy = _map_grads(xr, yr, G)
    o_sr, o_hr = oracle_map_backward(xr.cpu().numpy(), yr.cpu().numpy(),
                                     tuple(np.float32(t) for t in (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0))),
                                     G.cpu().numpy())
    assert maxnorm_err(gx.cpu().numpy(), o_sr) < 1e-4
    assert maxnorm_err(gy.cpu().numpy(), o_hr) < 1e-4


def test_generic_radius_and_stride0_gradients():
    from srgan_st_b200 import StructureTensorLoss, structure_tensor_distance
    torch.manual_seed(3)
    y = torch.rand(2, 3, 40, 52, device=DEV)
    x = (y + 0.05 * torch.randn_like(y)).clamp(0, 1).requires_grad_(True)
    d = structure_tensor_distance(x, y, sigma=1.5, rho=4.0)
    d.sum().backward()                          # stride-0 upstream gradient
    xl = x.detach().clone().requires_grad_(True)
    (StructureTensorLoss(sigma=1.5, rho=4.0)(xl, y) * (2 * 40 * 52)).backward()
    torch.cuda.synchronize()
    assert maxnorm_err(x.grad.cpu().numpy(), xl.grad.cpu().numpy()) < 1e-6


def test_loss_bits_unchanged_around_map_calls():
    """The map and the loss share the "st" workspace: the loss must give the same bits before and after map calls."""
    from srgan_st_b200 import StructureTensorLoss, structure_tensor_distance
    torch.manual_seed(4)
    y = torch.rand(8, 3, 96, 96, device=DEV)
    x = (y + 0.05 * torch.randn_like(y)).clamp(0, 1)

    def loss_and_grad():
        xs = x.clone().requires_grad_(True)
        loss = StructureTensorLoss()(xs, y)
        loss.backward()
        return loss.detach().clone(), xs.grad.clone()

    before = loss_and_grad()
    for _ in range(2):
        xs = x.clone().requires_grad_(True)
        (structure_tensor_distance(xs, y) * 0.5).sum().backward()
    after = loss_and_grad()
    torch.cuda.synchronize()
    assert torch.equal(before[0], after[0]) and torch.equal(before[1], after[1])


def test_weighted_step_replays_from_a_cuda_graph():
    from srgan_st_b200 import structure_tensor_distance
    torch.manual_seed(5)
    gen = torch.nn.Conv2d(3, 3, 3, padding=1).to(DEV)
    gt = torch.rand(4, 3, 96, 96, device=DEV)
    lr = (gt + 0.1 * torch.randn_like(gt)).clamp(0, 1)
    w = _weights(4, 96, 96, 9).abs()

    def step():
        sr = gen(lr).clamp(0, 1)
        sr.retain_grad()
        d = structure_tensor_distance(sr, gt)
        total = (d * w).mean()
        for p in gen.parameters():
            p.grad = None
        total.backward()
        return d.detach(), sr.grad, [p.grad for p in gen.parameters()]

    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        for _ in range(3):
            step()
    torch.cuda.current_stream().wait_stream(s)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        static_d, static_dsr, static_g = step()
    graph.replay()
    torch.cuda.synchronize()
    replayed_d, replayed_dsr, replayed_g = static_d.clone(), static_dsr.clone(), [g.clone() for g in static_g]
    eager_d, eager_dsr, eager_g = step()
    torch.cuda.synchronize()
    assert torch.isfinite(replayed_d).all()
    assert torch.equal(replayed_d, eager_d) and torch.equal(replayed_dsr, eager_dsr)
    for a, b in zip(replayed_g, eager_g):   # the conv's own backward may pick another algorithm or order
        assert torch.allclose(a, b, rtol=1e-5, atol=1e-8)


class _PoisonedTorch:
    """Delegates to torch, except that empty / empty_like hand out 0xFF-filled memory (NaN as a float)."""

    def __getattr__(self, name):
        return getattr(torch, name)

    @staticmethod
    def empty(*args, **kwargs):
        t = torch.empty(*args, **kwargs)
        t.reshape(-1).view(torch.uint8).fill_(0xFF)
        return t

    @staticmethod
    def empty_like(*args, **kwargs):
        t = torch.empty_like(*args, **kwargs)
        t.reshape(-1).view(torch.uint8).fill_(0xFF)
        return t


@pytest.fixture
def poisoned(monkeypatch):
    """Every torch.empty / torch.empty_like inside srgan_st_b200.loss returns 0xFF bytes."""
    from srgan_st_b200 import loss as L

    def run(fn):
        with monkeypatch.context() as m:
            m.setattr(L, "torch", _PoisonedTorch())
            out = fn()
        torch.cuda.synchronize()
        return out

    return run


@pytest.mark.parametrize("shape,sigma,rho", [((4, 96, 96), 0.5, 2.0), ((2, 37, 53), 0.5, 2.0), ((1, 30, 44), 1.5, 4.0)])
def test_poisoned_allocations_same_bits(poisoned, shape, sigma, rho):
    B, H, W = shape
    torch.manual_seed(6)
    y = torch.rand(B, 3, H, W, device=DEV)
    x = (y + 0.05 * torch.randn_like(y)).clamp(0, 1)
    G = _weights(B, H, W, 6, band=3)
    clean = _map_grads(x, y, G, sigma=sigma, rho=rho)
    dirty = poisoned(lambda: _map_grads(x, y, G, sigma=sigma, rho=rho))
    for a, b in zip(clean, dirty):
        assert torch.equal(a, b)


def test_errors():
    from srgan_st_b200 import structure_tensor_distance
    x = torch.rand(1, 3, 16, 16, device=DEV)
    with pytest.raises(RuntimeError):
        structure_tensor_distance(x.cpu(), x.cpu())
    with pytest.raises(TypeError):
        structure_tensor_distance(x.double(), x.double())
    with pytest.raises(ValueError):
        structure_tensor_distance(x[:, :2], x[:, :2])
    with pytest.raises(ValueError):
        structure_tensor_distance(x, x[:, :, :8])
    with pytest.raises(NotImplementedError):
        structure_tensor_distance(x, x, sigma=20.0)
