"""CPU: the per-image (reduction='none') entry points of include/srst.h, run on the emulation library.

For every path -- each compiled forward shape, a short marching chunk, ragged shapes, a generic radius, the three patch
losses with both search norms and both criteria, and one non-default Best-Buddy geometry -- the [B] losses must match
the float64 oracles run on each image alone and average to the scalar entry point's loss.  With a random upstream
gradient g[B], image b's d_sr must be bit-identical to the scalar entry point run on image b alone with grad_out =
g[b] (the tile choice of the backward does not depend on B, and the patch scale is the same expression with B = 1);
d_gt, which sums with atomics, is held to 1e-6.  The indices are those of the scalar path, bit for bit."""
import numpy as np
import pytest

from oracle import bb_oracle as BO
from oracle import bbg_oracle as GO
from oracle import st_oracle as O
from tests.helpers import _fp, _p, _workspace, emu_bb, emu_bbg, emu_lib, emu_patch_gt, emu_st, maxnorm_err, rel_err

DIST_L1 = 0x100   # SRST_BB_DIST_L1


@pytest.fixture(scope="module")
def lib():
    return emu_lib()


def _taps(sigma=0.5, rho=2.0):
    return tuple(np.ascontiguousarray(t, np.float32) for t in (*O.gaussian_taps(sigma, True), O.gaussian_taps(rho)))


def emu_st_per_image(lib, sr, hr, taps, grad_out, want_hr=False):
    """srst_st_forward_per_image + srst_st_backward_per_image on host arrays."""
    B, _, H, W = sr.shape
    g, dg, k = taps
    rs, rk = len(g) // 2, len(k) // 2
    nb = lib.srst_st_workspace_bytes_r(B, H, W, rs, rk)
    ws = _workspace(nb)
    nbb = lib.srst_st_backward_workspace_bytes(B, H, W, rs, rk)
    bws = np.full(nbb // 4 + 4, np.nan, np.float32)
    loss = np.full(B, np.nan, np.float32)
    n_ixy = lib.srst_st_ixy_floats(B, H, W)
    ds = [np.full_like(sr, np.nan), np.full_like(sr, np.nan) if want_hr else None]
    ixy = [np.full(n_ixy, np.nan, np.float32), np.full(n_ixy, np.nan, np.float32) if want_hr else None]
    rc = lib.srst_st_forward_per_image(_p(sr), _p(hr), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, 1, 1e-12, _p(loss),
                                       _p(ds[0]), _p(ds[1]), _p(ixy[0]), _p(ixy[1]), _p(ws), nb, None)
    assert rc == 0, rc
    go = np.ascontiguousarray(grad_out, np.float32)
    out = dict(loss=loss, header=ws[:4].copy())
    for name, s, d in zip(("d_sr", "d_hr"), ixy, ds):
        if s is None:
            continue
        grad = np.full_like(sr, np.nan)
        rc = lib.srst_st_backward_per_image(_p(s), _p(d), _p(go), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, _p(grad),
                                            _p(bws) if nbb else None, nbb, None)
        assert rc == 0, rc
        out[name] = grad
    return out


def _check_st(lib, sr, hr, taps, want_hr=False):
    B = sr.shape[0]
    go = np.random.default_rng(B + sr.shape[2]).uniform(-2.0, 2.0, B).astype(np.float32)
    out = emu_st_per_image(lib, sr, hr, taps, go, want_hr)
    assert np.all(out["header"] == 0)                       # ticket handed back zeroed
    whole = emu_st(lib, sr, hr, taps)
    assert rel_err(float(np.mean(out["loss"].astype(np.float64))), whole["loss"]) < 1e-6
    for b in range(B):
        ref = O.st_loss(sr[b:b + 1], hr[b:b + 1], taps=taps, want_grad=False)
        assert rel_err(float(out["loss"][b]), ref["loss"]) < 1e-5
        one = emu_st(lib, sr[b:b + 1], hr[b:b + 1], taps, want_hr=want_hr, grad_out=float(go[b]))
        assert out["d_sr"][b].tobytes() == one["d_sr"][0].tobytes()
        if want_hr:
            assert out["d_hr"][b].tobytes() == one["d_hr"][0].tobytes()


@pytest.mark.parametrize("fwd_cfg", [0, 1, 2, 3, 4])
def test_st_per_image_every_compiled_forward_shape(lib, fwd_cfg):
    assert lib.srst_st_force_cfg(fwd_cfg, -1) == 0
    try:
        rng = np.random.default_rng(fwd_cfg)
        sr, hr = (rng.random((3, 3, 40, 52), dtype=np.float32) for _ in range(2))
        _check_st(lib, sr, hr, _taps(), want_hr=fwd_cfg == 3)
    finally:
        lib.srst_st_force_cfg(-1, -1)


def test_st_per_image_short_march_chunks(lib):
    """16-row chunks of the marching forward: an image's partials are several chunks x strips."""
    assert lib.srst_st_force_cfg(3, -1) == 0 and lib.srst_st_force_chunk_blocks(1) == 0
    try:
        rng = np.random.default_rng(11)
        sr, hr = (rng.random((2, 3, 50, 100), dtype=np.float32) for _ in range(2))
        _check_st(lib, sr, hr, _taps())
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)


@pytest.mark.parametrize("shape", [(2, 37, 53), (3, 21, 30), (2, 17, 98)])
def test_st_per_image_ragged_shapes(lib, shape):
    """W % 4 != 0 (no TMA: tiled shapes, plain loads) and odd H / W."""
    rng = np.random.default_rng(sum(shape))
    sr, hr = (rng.random((shape[0], 3, shape[1], shape[2]), dtype=np.float32) for _ in range(2))
    _check_st(lib, sr, hr, _taps(), want_hr=True)


def test_st_per_image_padded_radius_class(lib):
    rng = np.random.default_rng(5)
    sr, hr = (rng.random((2, 3, 24, 36), dtype=np.float32) for _ in range(2))
    _check_st(lib, sr, hr, _taps(1.0, 3.0))


def test_st_per_image_generic_radius(lib):
    taps = _taps(1.5, 3.5)
    assert lib.srst_st_supported(len(taps[0]) // 2, len(taps[2]) // 2) == 2
    rng = np.random.default_rng(6)
    sr, hr = (rng.random((3, 3, 20, 28), dtype=np.float32) for _ in range(2))
    _check_st(lib, sr, hr, taps, want_hr=True)


MODES = {"patch": 0, "gram": 1, "pst": 2}


def emu_patch_per_image(lib, mode, sr, gt, criterion, grad_out, taps=None):
    """srst_patch_forward_per_image + srst_patch_backward_per_image (d_sr and d_gt in one call) on host arrays."""
    B, _, H, W = sr.shape
    N = (H // 3) * (W // 3)
    nb = lib.srst_bb_workspace_bytes(B, H, W)
    ws = _workspace(nb)
    tp = (_fp(taps[0]), _fp(taps[1]), len(taps[0]) // 2, _fp(taps[2]), len(taps[2]) // 2) if taps else (None, None, 0, None, 0)
    idx = np.full((B, N), -1, np.int64)
    loss = np.full(B, np.nan, np.float32)
    rc = lib.srst_patch_forward_per_image(MODES[mode], _p(sr), _p(gt), None, None, B, H, W, *tp, 1.0, 0.5, criterion,
                                          _p(idx), _p(loss), _p(ws), nb, None)
    assert rc == 0, rc
    header = ws[:4].copy()
    go = np.ascontiguousarray(grad_out, np.float32)
    d_sr, d_gt = np.full_like(sr, np.nan), np.full_like(gt, np.nan)
    rc = lib.srst_patch_backward_per_image(MODES[mode], _p(sr), _p(gt), None, None, _p(idx), _p(go), B, H, W, *tp,
                                           criterion, _p(d_sr), _p(d_gt), _p(ws), nb, None)
    assert rc == 0, rc
    return dict(loss=loss, idx=idx, d_sr=d_sr, d_gt=d_gt, header=header)


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("dist_norm", ["l2", "l1"])
@pytest.mark.parametrize("criterion", ["l1", "l2"])
def test_patch_per_image(lib, mode, dist_norm, criterion):
    rng = np.random.default_rng(len(mode) + 3 * len(dist_norm) + (criterion == "l2"))
    B, H, W = 3, 24, 28   # N = 8 * 9 = 72: every image's CTA is partly empty
    sr, gt = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    taps = _taps() if mode == "pst" else None
    crit = (0 if criterion == "l1" else 1) | (DIST_L1 if dist_norm == "l1" else 0)
    go = rng.uniform(-2.0, 2.0, B).astype(np.float32)
    out = emu_patch_per_image(lib, mode, sr, gt, crit, go, taps)
    assert np.all(out["header"] == 0)
    whole = emu_bb(lib, sr, gt, alpha=1.0, beta=0.5, criterion=crit, mode=mode, taps=taps)
    assert out["idx"].tobytes() == whole["idx"].tobytes()
    assert rel_err(float(np.mean(out["loss"].astype(np.float64))), whole["loss"]) < 1e-6
    for b in range(B):
        s, t = sr[b:b + 1], gt[b:b + 1]
        ref = BO.bb_forward_c(s, t, alpha=1.0, beta=0.5, criterion=criterion, mode=mode, taps=taps, dist_norm=dist_norm)
        assert rel_err(float(out["loss"][b]), ref["loss"]) < 1e-5
        one = emu_bb(lib, s, t, alpha=1.0, beta=0.5, criterion=crit, grad_out=float(go[b]), mode=mode, taps=taps)
        assert out["d_sr"][b].tobytes() == one["d_sr"][0].tobytes()
        d_gt = emu_patch_gt(lib, s, t, one["idx"], criterion=crit, grad_out=float(go[b]), mode=mode, taps=taps)
        assert maxnorm_err(out["d_gt"][b], d_gt[0]) < 1e-6


@pytest.mark.parametrize("criterion", ["l1", "l2"])
def test_bbg_per_image(lib, criterion):
    ksize, pad, stride = 4, 1, 2
    rng = np.random.default_rng(21 + (criterion == "l2"))
    B, H, W = 3, 20, 26
    sr, gt = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    crit = 0 if criterion == "l1" else 1
    go = rng.uniform(-2.0, 2.0, B).astype(np.float32)
    N = lib.srst_bbg_num_patches(H, W, ksize, pad, stride)
    nb = lib.srst_bbg_workspace_bytes(B, H, W, ksize, pad, stride)
    ws = _workspace(nb)
    idx = np.full((B, N), -1, np.int64)
    loss = np.full(B, np.nan, np.float32)
    assert lib.srst_bbg_forward_per_image(_p(sr), _p(gt), None, None, B, H, W, ksize, pad, stride, 1.0, 0.5, crit, _p(idx),
                                          _p(loss), _p(ws), nb, None) == 0
    assert np.all(ws[:4] == 0)
    d_sr, d_gt = np.full_like(sr, np.nan), np.full_like(gt, np.nan)
    assert lib.srst_bbg_backward_per_image(_p(sr), _p(gt), None, None, _p(idx), _p(go), B, H, W, ksize, pad, stride, crit,
                                           _p(d_sr), _p(d_gt), _p(ws), nb, None) == 0
    whole = emu_bbg(lib, sr, gt, ksize, pad, stride, alpha=1.0, beta=0.5, criterion=crit)
    assert idx.tobytes() == whole["idx"].tobytes()
    assert rel_err(float(np.mean(loss.astype(np.float64))), whole["loss"]) < 1e-6
    for b in range(B):
        s, t = sr[b:b + 1], gt[b:b + 1]
        ref = GO.bbg_forward_c(s, t, ksize=ksize, pad=pad, stride=stride, alpha=1.0, beta=0.5, criterion=criterion)
        assert rel_err(float(loss[b]), ref["loss"]) < 1e-5
        one = emu_bbg(lib, s, t, ksize, pad, stride, alpha=1.0, beta=0.5, criterion=crit, grad_out=float(go[b]),
                      want_gt=True)
        assert d_sr[b].tobytes() == one["d_sr"][0].tobytes()
        assert maxnorm_err(d_gt[b], one["d_gt"][0]) < 1e-6
