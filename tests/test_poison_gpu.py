"""GPU: no kernel may depend on global memory it did not write.

The loss modules take their outputs and saved buffers from torch.empty / torch.empty_like, and the caching allocator
hands back whatever an earlier step left there -- after a diverged GAN step that is NaN / Inf.  Their workspaces are
only promised a zeroed 16-byte ticket header (include/srst.h).  Here every call runs twice: once normally, once with
every torch.empty / torch.empty_like made inside srgan_st_b200.loss filled with 0xFF bytes (NaN as a float, -1 as an
int) and with fresh workspaces that are 0xFF everywhere but the ticket header.  Loss, d_sr, d_hr and the indices must
come back bit for bit; d_gt (summed with atomics) is held to the float64 oracle.  After every poisoned call the
workspace header must be zero again."""
import ctypes
import os
import subprocess

import numpy as np
import pytest

from oracle import bb_oracle as OB
from tests.helpers import maxnorm_err

pytestmark = pytest.mark.gpu

torch = pytest.importorskip("torch")


def _fill_ff(t):
    t.reshape(-1).view(torch.uint8).fill_(0xFF)
    return t


class _PoisonedTorch:
    """Delegates to torch, except that empty / empty_like hand out 0xFF-filled memory."""

    def __getattr__(self, name):
        return getattr(torch, name)

    @staticmethod
    def empty(*args, **kwargs):
        return _fill_ff(torch.empty(*args, **kwargs))

    @staticmethod
    def empty_like(*args, **kwargs):
        return _fill_ff(torch.empty_like(*args, **kwargs))


@pytest.fixture
def poison(monkeypatch):
    """poison(fn) runs fn() with poisoned allocations and workspaces and returns its result."""
    from srgan_st_b200 import loss as L
    issued = []

    def workspace(kind, device, stream_ptr, nbytes):
        ws = torch.full((max(nbytes, 4096),), 0xFF, dtype=torch.uint8, device=device)
        ws[:16].zero_()
        issued.append((kind, ws))
        return ws

    def run(fn):
        issued.clear()
        with monkeypatch.context() as m:
            m.setattr(L, "torch", _PoisonedTorch())
            m.setattr(L, "_workspace", workspace)
            out = fn()
        torch.cuda.synchronize()
        assert issued, "the call used no workspace"
        for kind, ws in issued:
            if kind != "st_bwd":   # the generic-radius backward's scratch planes have no ticket (srst.h)
                assert not ws[:16].any().item(), f"{kind} workspace: ticket header not handed back zeroed"
        return out

    return run


def _same_bits(a, b):
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _compare(clean, poisoned, keys):
    for k in keys:
        assert _same_bits(clean[k], poisoned[k]), f"{k} differs after poisoning"
        if clean[k].dtype.kind == "f":
            assert np.isfinite(clean[k]).all(), k


def _np(t):
    return t.detach().cpu().numpy() if t is not None else None


def _inputs(shape, seed, offset=False):
    g = torch.Generator(device="cuda").manual_seed(seed)
    gt = torch.rand(shape, device="cuda", generator=g)
    sr = (gt + 0.1 * (torch.rand(shape, device="cuda", generator=g) - 0.5)).clamp(0, 1)
    if offset:   # contiguous but 4 bytes past a 16-byte boundary: no TMA, no vec4
        n = int(np.prod(shape))
        sr, gt = [torch.empty(n + 1, device="cuda")[1:].view(shape).copy_(t) for t in (sr, gt)]
        assert sr.data_ptr() % 16 and gt.data_ptr() % 16 and sr.is_contiguous()
    return sr, gt


def _run_module(make, sr, gt, want=("sr", "gt"), scale=0.75):
    x = sr.detach().requires_grad_("sr" in want)   # detach() keeps the storage offset of the input
    y = gt.detach().requires_grad_("gt" in want)
    m = make()
    loss = m(x, y)
    (loss * scale).backward()
    torch.cuda.synchronize()
    out = dict(loss=_np(loss).reshape(-1), d_sr=_np(x.grad), d_gt=_np(y.grad))
    if getattr(m, "last_indices", None) is not None:
        out["idx"] = _np(m.last_indices)
    return out


# ---- structure tensor ---------------------------------------------------------------------------------------------
ST_SHAPES = [(4, 96, 96), (2, 64, 112), (2, 48, 200),   # default dispatch: march96 / march112 by W
             (1, 333, 517), (1, 37, 53),                # odd H, W % 4 != 0
             (128, 96, 96)]                             # persistent backward: three and more tiles per CTA


@pytest.mark.parametrize("shape", ST_SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_st_default_dispatch(poison, shape):
    import srgan_st_b200 as S
    sr, gt = _inputs((shape[0], 3, shape[1], shape[2]), sum(shape))
    run = lambda: _run_module(S.StructureTensorLoss, sr, gt)
    clean = run()
    _compare(clean, poison(run), ["loss", "d_sr", "d_gt"])   # d_gt here is d_hr: no atomics, bit for bit


@pytest.mark.parametrize("cfg", [(0, 0), (1, 1), (2, 0), (3, 1), (4, 0)], ids=lambda p: f"fwd{p[0]}-bwd{p[1]}")
@pytest.mark.parametrize("shape", [(2, 67, 100), (1, 37, 52)], ids=lambda s: "x".join(map(str, s)))
def test_st_forced_cfgs(poison, cfg, shape):
    import srgan_st_b200 as S
    from srgan_st_b200 import _cabi
    sr, gt = _inputs((shape[0], 3, shape[1], shape[2]), 3 * sum(shape))
    assert _cabi.lib().srst_st_force_cfg(*cfg) == 0
    try:
        run = lambda: _run_module(S.StructureTensorLoss, sr, gt)
        clean = run()
        poisoned = poison(run)
    finally:
        _cabi.lib().srst_st_force_cfg(-1, -1)
    _compare(clean, poisoned, ["loss", "d_sr", "d_gt"])


@pytest.mark.parametrize("shape", [(2, 96, 96), (1, 37, 53)], ids=lambda s: "x".join(map(str, s)))
def test_st_storage_offset_inputs(poison, shape):
    import srgan_st_b200 as S
    sr, gt = _inputs((shape[0], 3, shape[1], shape[2]), 11, offset=True)
    run = lambda: _run_module(S.StructureTensorLoss, sr, gt)
    clean = run()
    _compare(clean, poison(run), ["loss", "d_sr", "d_gt"])


@pytest.mark.parametrize("shape", [(2, 64, 80), (1, 37, 53)], ids=lambda s: "x".join(map(str, s)))
def test_st_generic_radius(poison, shape):
    """sigma 1.5, rho 4 (radii 6, 16): the generic path, scratch planes in the forward and the st_bwd workspace."""
    import srgan_st_b200 as S
    sr, gt = _inputs((shape[0], 3, shape[1], shape[2]), 5 + sum(shape))
    run = lambda: _run_module(lambda: S.StructureTensorLoss(sigma=1.5, rho=4.0), sr, gt)
    clean = run()
    _compare(clean, poison(run), ["loss", "d_sr", "d_gt"])


@pytest.mark.parametrize("shape", [(4, 96, 96), (2, 64, 200), (1, 37, 53)], ids=lambda s: "x".join(map(str, s)))
def test_stpx(poison, shape):
    import srgan_st_b200 as S
    sr, gt = _inputs((shape[0], 3, shape[1], shape[2]), 17 + sum(shape))
    run = lambda: _run_module(lambda: S.StructureTensorPixelLoss(st_weight=0.5, pixel_weight=2.0), sr, gt, want=("sr",))
    clean = run()
    _compare(clean, poison(run), ["loss", "d_sr"])


@pytest.mark.parametrize("shape", [(2, 96, 96), (1, 333, 517)], ids=lambda s: "x".join(map(str, s)))
def test_st_features(shape):
    from srgan_st_b200 import structure_tensor_features
    img, _ = _inputs((shape[0], 3, shape[1], shape[2]), 23)

    def run():
        f = structure_tensor_features(img)
        torch.cuda.synchronize()
        return {k: _np(v) for k, v in f.items()}

    clean = run()
    from srgan_st_b200 import loss as L
    with pytest.MonkeyPatch.context() as m:   # features use no workspace: poison the outputs only
        m.setattr(L, "torch", _PoisonedTorch())
        poisoned = run()
    _compare(clean, poisoned, list(clean))


# ---- Best-Buddy, Gram, patchwise structure tensor ------------------------------------------------------------------
def _patch_module(mode, pyramid, dist, crit):
    import srgan_st_b200 as S
    cls = {"patch": S.BestBuddyLoss, "gram": S.GramLoss, "pst": S.PatchwiseStructureTensorLoss}[mode]
    return lambda: cls(alpha=0.7, beta=1.3, dist_norm=dist, criterion=crit, pyramid=pyramid)


@pytest.mark.parametrize("mode", ["patch", "gram", "pst"])
@pytest.mark.parametrize("pyramid", ["fused", "aten"])
@pytest.mark.parametrize("dist,crit", [("l2", "l1"), ("l1", "l2")], ids=["dist_l2-l1", "dist_l1-l2"])
@pytest.mark.parametrize("shape", [(3, 12, 12), (2, 50, 77), (1, 192, 192)], ids=lambda s: "x".join(map(str, s)))
def test_patch_losses(poison, mode, pyramid, dist, crit, shape):
    B, H, W = shape
    sr, gt = _inputs((B, 3, H, W), H * W + len(mode))
    run = lambda: _run_module(_patch_module(mode, pyramid, dist, crit), sr, gt)
    clean = run()
    poisoned = poison(run)
    _compare(clean, poisoned, ["loss", "d_sr", "idx"])
    M = (H // 3) * (W // 3) + (H // 6) * (W // 6) + (H // 12) * (W // 12)
    assert poisoned["idx"].min() >= 0 and poisoned["idx"].max() < M
    # d gt: the float64 oracle on the kernel's own indices and the pyramid the loss used
    g = gt.cpu().numpy()
    if pyramid == "fused":
        g2, g4 = OB.pyramid_c(g)
    else:
        g2, g4 = [torch.nn.functional.interpolate(gt, scale_factor=f, mode="bicubic", align_corners=False).cpu().numpy()
                  for f in (0.5, 0.25)]
    taps = None
    if mode == "pst":
        from oracle import st_oracle as O
        taps = (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0))
    ref = 0.75 * OB.patch_backward_gt(sr.cpu().numpy(), g, g2, g4, poisoned["idx"], mode, taps, crit)
    for out in (clean, poisoned):
        assert np.isfinite(out["d_gt"]).all() and maxnorm_err(out["d_gt"], ref) < 1e-4


@pytest.mark.parametrize("k,p,s", [(4, 1, 2), (8, 4, 7), (1, 0, 1)])
@pytest.mark.parametrize("pyramid", ["fused", "aten"])
def test_bb_geometry(poison, k, p, s, pyramid):
    import srgan_st_b200 as S
    sr, gt = _inputs((2, 3, 50, 77), 100 * k + s)
    make = lambda: S.BestBuddyLoss(ksize=k, pad=p, stride=s, criterion="l2", dist_norm="l1" if k == 8 else "l2",
                                   pyramid=pyramid)
    run = lambda: _run_module(make, sr, gt)
    clean = run()
    poisoned = poison(run)
    _compare(clean, poisoned, ["loss", "d_sr", "idx"])
    # d gt is summed with atomics: the clean run's value (held to the reference by test_bb_geometry.py) up to ordering
    assert np.isfinite(poisoned["d_gt"]).all() and maxnorm_err(poisoned["d_gt"], clean["d_gt"]) < 1e-5


# ---- shared memory ------------------------------------------------------------------------------------------------
# Before each single-kernel entry point (called directly through the C ABI, with explicit gt2 / gt4 where that removes
# the pyramid launch), tests/poison/smem_poison.cu fills the shared memory of every SM, on the same stream; the results
# after a 0xFFFFFFFF fill must equal those after a zero fill bit for bit.  Assumption: the pack kernel that
# srst_bb_forward / srst_gram_forward / srst_pst_forward launch before their search kernel uses no dynamic and little
# static shared memory, so the search kernel's mbarrier ring and staging buffers still see the fill.
SMEM_SRC = os.path.join(os.path.dirname(os.path.abspath(__file__)), "poison", "smem_poison.cu")


@pytest.fixture(scope="module")
def smem_fill(tmp_path_factory):
    """fill(value, stream) -> 0 on success.  Skips when shared memory does not keep the fill until the next kernel."""
    from srgan_st_b200 import build as B
    try:
        nvcc = B._nvcc()
    except RuntimeError as e:
        pytest.skip(f"shared-memory poison helper cannot be built: {e}")
    so = str(tmp_path_factory.mktemp("smem_poison") / "libsmem_poison.so")
    subprocess.run([nvcc, "-gencode", "arch=compute_100a,code=sm_100a", "-O2", "-std=c++17", "--shared", "-Xcompiler",
                    "-fPIC", "-o", so, SMEM_SRC], check=True, capture_output=True)
    lib = ctypes.CDLL(so)
    lib.smem_poison_fill.argtypes = [ctypes.c_uint, ctypes.c_void_p]
    lib.smem_poison_probe.argtypes = [ctypes.c_uint, ctypes.c_void_p, ctypes.c_void_p]
    nblk, words = lib.smem_poison_blocks(), lib.smem_poison_words()
    assert nblk > 0 and words > 0
    stream = torch.cuda.current_stream().cuda_stream
    counts = torch.zeros(nblk, dtype=torch.int32, device="cuda")
    assert lib.smem_poison_fill(0xFFFFFFFF, stream) == 0
    assert lib.smem_poison_probe(0xFFFFFFFF, counts.data_ptr(), stream) == 0
    torch.cuda.synchronize()
    full = int((counts.cpu().numpy() == words).sum())
    if full != nblk:
        pytest.skip(f"shared memory does not keep its contents from one kernel to the next here: {full} of {nblk} "
                    "probe CTAs found the whole fill")
    return lib.smem_poison_fill


def _smem_twice(fill, outputs, launch):
    """outputs(): fresh NaN-filled output tensors; launch(outs, stream) enqueues one entry point and returns its code."""
    res = []
    for value in (0, 0xFFFFFFFF):
        outs = outputs()
        torch.cuda.synchronize()
        stream = torch.cuda.current_stream().cuda_stream
        assert fill(value, stream) == 0
        assert launch(outs, stream) == 0
        torch.cuda.synchronize()
        res.append([_np(t) for t in outs])
    for i, (a, b) in enumerate(zip(*res)):
        assert _same_bits(a, b), f"output {i} differs after the shared-memory fill"
        if a.dtype.kind == "f":
            assert np.isfinite(a).all(), f"output {i}"
    return res[1]


def _nan(*shape, dtype=torch.float32):
    return torch.full(shape, float("nan") if dtype.is_floating_point else -1, dtype=dtype, device="cuda")


def _st_taps():
    from srgan_st_b200 import taps as T
    g, dg = T.gaussian_taps(0.5)
    k, _ = T.gaussian_taps(2.0)
    return (T.as_c(g), T.as_c(dg), len(g) // 2, T.as_c(k), len(k) // 2)


def _st_forward(lib, sr, hr, outs, stream):
    B, _, H, W = sr.shape
    loss, ds_sr, ds_hr, ixy_sr, ixy_hr, ws = outs
    return lib.srst_st_forward(sr.data_ptr(), hr.data_ptr(), B, H, W, *_st_taps(), 1, 1e-12, loss.data_ptr(),
                               ds_sr.data_ptr(), ds_hr.data_ptr(), ixy_sr.data_ptr(), ixy_hr.data_ptr(), ws.data_ptr(),
                               ws.numel(), stream)


def _st_outputs(lib, B, H, W):
    n_ixy = lib.srst_st_ixy_floats(B, H, W)
    return lambda: (_nan(1), _nan(B, 3, H, W), _nan(B, 3, H, W), _nan(n_ixy), _nan(n_ixy),
                    torch.zeros(lib.srst_st_workspace_bytes(B, H, W), dtype=torch.uint8, device="cuda"))


@pytest.mark.parametrize("cfg,shape", [(3, (4, 96, 96)), (4, (2, 37, 112)), (0, (2, 67, 100)), (1, (1, 37, 53))],
                         ids=["march96", "march112", "tiled-32x64", "tiled-24x96-unaligned"])
def test_smem_st_forward(smem_fill, cfg, shape):
    from srgan_st_b200 import _cabi
    lib = _cabi.lib()
    B, H, W = shape
    sr, hr = _inputs((B, 3, H, W), 31 + cfg)
    assert lib.srst_st_force_cfg(cfg, -1) == 0
    try:
        _smem_twice(smem_fill, _st_outputs(lib, B, H, W), lambda o, s: _st_forward(lib, sr, hr, o, s))
    finally:
        lib.srst_st_force_cfg(-1, -1)


@pytest.mark.parametrize("bwd,shape", [(1, (64, 96, 96)), (0, (2, 67, 200)), (0, (1, 37, 53)), (1, (2, 37, 94))],
                         ids=["tma-12x96", "tma-28x56", "plain-odd", "plain-94"])
def test_smem_st_backward(smem_fill, bwd, shape):
    """With TMA (aligned, W % 4 == 0; the persistent CTAs loop over several tiles) and with plain staging loads."""
    from srgan_st_b200 import _cabi
    lib = _cabi.lib()
    B, H, W = shape
    sr, hr = _inputs((B, 3, H, W), 41 + W)
    fwd = _st_outputs(lib, B, H, W)()
    assert _st_forward(lib, sr, hr, fwd, torch.cuda.current_stream().cuda_stream) == 0
    _, ds, _, ixy, _, _ = fwd
    go = torch.full((1,), 0.75, device="cuda")
    assert lib.srst_st_force_cfg(-1, bwd) == 0
    try:
        _smem_twice(smem_fill, lambda: (_nan(B, 3, H, W),),
                    lambda o, s: lib.srst_st_backward(ixy.data_ptr(), ds.data_ptr(), go.data_ptr(), B, H, W, *_st_taps(),
                                                      o[0].data_ptr(), s))
    finally:
        lib.srst_st_force_cfg(-1, -1)


@pytest.mark.parametrize("shape", [(2, 50, 77), (1, 192, 192)], ids=lambda s: "x".join(map(str, s)))
def test_smem_bb_pyramid(smem_fill, shape):
    from srgan_st_b200 import _cabi
    lib = _cabi.lib()
    B, H, W = shape
    _, gt = _inputs((B, 3, H, W), 53)
    out = _smem_twice(smem_fill, lambda: (_nan(B, 3, H // 2, W // 2), _nan(B, 3, H // 4, W // 4)),
                      lambda o, s: lib.srst_bb_pyramid(gt.data_ptr(), B, H, W, o[0].data_ptr(), o[1].data_ptr(), s))
    r2, r4 = OB.pyramid_c(gt.cpu().numpy())
    assert np.abs(out[0] - r2).max() < 1e-6 and np.abs(out[1] - r4).max() < 1e-6


@pytest.mark.parametrize("mode", ["patch", "gram", "pst"])
@pytest.mark.parametrize("crit", [0, 0x101], ids=["l1-dist_l2", "l2-dist_l1"])
@pytest.mark.parametrize("shape", [(2, 50, 77), (1, 192, 192)], ids=lambda s: "x".join(map(str, s)))
def test_smem_patch_forward(smem_fill, mode, crit, shape):
    """srst_bb_forward / srst_gram_forward / srst_pst_forward with a given pyramid: pack, search, loss."""
    from srgan_st_b200 import _cabi
    lib = _cabi.lib()
    B, H, W = shape
    sr, gt = _inputs((B, 3, H, W), 59 + crit)
    gt2, gt4 = [torch.from_numpy(a).cuda() for a in OB.pyramid_c(gt.cpu().numpy())]
    N = (H // 3) * (W // 3)
    nbytes = lib.srst_bb_workspace_bytes(B, H, W)
    common = (sr.data_ptr(), gt.data_ptr(), gt2.data_ptr(), gt4.data_ptr(), B, H, W)

    def launch(o, s):
        idx, loss, ws = o
        tail = (idx.data_ptr(), loss.data_ptr(), ws.data_ptr(), ws.numel(), s)
        if mode == "pst":
            return lib.srst_pst_forward(*common, *_st_taps(), 0.7, 1.3, crit, *tail)
        fwd = lib.srst_bb_forward if mode == "patch" else lib.srst_gram_forward
        return fwd(*common, 0.7, 1.3, crit, *tail)

    out = _smem_twice(smem_fill, lambda: (_nan(B, N, dtype=torch.int64), _nan(1),
                                          torch.zeros(nbytes, dtype=torch.uint8, device="cuda")), launch)
    M = N + (H // 6) * (W // 6) + (H // 12) * (W // 12)
    assert out[0].min() >= 0 and out[0].max() < M
