"""CPU: the crop layout of the marching forward (cfg 3 on images no wider than its 96-column strip) under the host
emulation.

The crop layout stages no x halo: its raw box and gray rows cover the image columns only, the zero columns the edge
windows read are written once per CTA, and its gradient and horizontal items give each warp 4 consecutive row pairs,
so that the warps whose rows are all outside the image skip their arithmetic.  No per-pixel operation moves, so ds,
ixy and the distance map must be bit-identical to the 112-column halo strips (cfg 4) on the same input.  The heights
put the image bottom at different row-pair offsets inside a 16-row block and inside a warp's 4 row pairs; the chunk
sizes put the out-of-image rows at the top and the bottom of different chunks.  Each result is also held to the
float64 oracle, and a run with 0xFF (NaN) in shared memory and in the workspace must give the same bytes: a zero
column or a ring row that is never written would show there."""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests import helpers
from tests.helpers import _fp, _p, _workspace, emu_lib, emu_stpx, maxnorm_err, rel_err
from tests.test_emu_per_image import emu_st_per_image
from tests.test_emu_stpx_per_image import emu_stpx_per_image

POISON = 0xFF
CROP, HALO = 3, 4   # forward cfg ids: 96-column strips (the crop layout here), 112-column strips
SHAPES = [(B, H, W) for W in (52, 96) for H in (23, 37, 61, 90, 96) for B in ((1, 3) if H in (37, 90) else (3,))]
CHUNKS = [1, 2, 3, 0]   # row blocks per chunk; 0: the library's choice


@pytest.fixture(scope="module")
def lib():
    lib = emu_lib()
    yield lib
    lib.srst_emu_set_poison(0xCD)
    lib.srst_st_force_cfg(-1, -1)
    lib.srst_st_force_chunk_blocks(0)


def _taps():
    return tuple(np.ascontiguousarray(t, np.float32) for t in (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0)))


def _pair(shape, seed):
    rng = np.random.default_rng(seed)
    B, H, W = shape
    hr = rng.random((B, 3, H, W), dtype=np.float32)
    sr = np.clip(hr + 0.1 * rng.standard_normal((B, 3, H, W), dtype=np.float32), 0, 1).astype(np.float32)
    return sr, hr


def _poisoned(lib, run):
    helpers.WORKSPACE_FILL = POISON
    lib.srst_emu_set_poison(POISON)
    try:
        return run()
    finally:
        lib.srst_emu_set_poison(0xCD)
        helpers.WORKSPACE_FILL = None
        helpers.FILLED_WORKSPACES.clear()


def _forward(lib, sr, hr, taps, with_map):
    """srst_st_forward (or srst_st_forward_map) with both ds and both ixy buffers, NaN-prefilled."""
    B, _, H, W = sr.shape
    g, dg, k = taps
    nb = lib.srst_st_workspace_bytes(B, H, W)
    ws = _workspace(nb)
    loss = np.full(1, np.nan, np.float32)
    n_ixy = lib.srst_st_ixy_floats(B, H, W)
    out = dict(ds_sr=np.full_like(sr, np.nan), ds_hr=np.full_like(sr, np.nan),
               ixy_sr=np.full(n_ixy, np.nan, np.float32), ixy_hr=np.full(n_ixy, np.nan, np.float32))
    args = (_p(sr), _p(hr), B, H, W, _fp(g), _fp(dg), len(g) // 2, _fp(k), len(k) // 2, 1, 1e-12, _p(loss))
    outs = (_p(out["ds_sr"]), _p(out["ds_hr"]), _p(out["ixy_sr"]), _p(out["ixy_hr"]), _p(ws), nb, None)
    if with_map:
        out["map"] = np.full((B, H, W), np.nan, np.float32)
        rc = lib.srst_st_forward_map(*args, _p(out["map"]), *outs)
    else:
        rc = lib.srst_st_forward(*args, *outs)
    assert rc == 0, rc
    out["loss"] = loss
    return out


def _backward(lib, taps, ixy, ds, shape):
    B, _, H, W = shape
    g, dg, k = taps
    go = np.ones(1, np.float32)
    d = np.full(shape, np.nan, np.float32)
    rc = lib.srst_st_backward(_p(ixy), _p(ds), _p(go), B, H, W, _fp(g), _fp(dg), len(g) // 2, _fp(k), len(k) // 2, _p(d),
                              None)
    assert rc == 0, rc
    return d


def _run(lib, cfg, chunk, fn):
    assert lib.srst_st_force_cfg(cfg, -1) == 0 and lib.srst_st_force_chunk_blocks(chunk) == 0
    try:
        return fn()
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)


def _same(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.mark.parametrize("chunk", CHUNKS, ids=lambda c: f"chunk{c}" if c else "chunkdefault")
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_crop_forward_matches_halo_strips(lib, shape, chunk):
    """ds, ixy and the map bit-identical to the 112-column strips; loss and gradients against the oracle."""
    sr, hr = _pair(shape, sum(shape) + chunk)
    taps = _taps()
    crop = _run(lib, CROP, chunk, lambda: _forward(lib, sr, hr, taps, with_map=True))
    halo = _run(lib, HALO, chunk, lambda: _forward(lib, sr, hr, taps, with_map=True))
    bad = _run(lib, CROP, chunk, lambda: _poisoned(lib, lambda: _forward(lib, sr, hr, taps, with_map=True)))
    for key in ("ds_sr", "ds_hr", "ixy_sr", "ixy_hr", "map"):
        assert not np.isnan(crop[key]).any(), key
        assert _same(crop[key], halo[key]), key
        assert _same(crop[key], bad[key]), key
    assert _same(crop["loss"], bad["loss"])
    assert rel_err(crop["loss"][0], halo["loss"][0]) < 1e-6
    ref = O.st_loss(sr, hr, taps=taps, want_hr_grad=True)
    assert rel_err(crop["loss"][0], ref["loss"]) < 1e-5
    assert rel_err(float(np.mean(crop["map"].astype(np.float64))), ref["loss"]) < 1e-5
    for img in ("sr", "hr"):
        d = _backward(lib, taps, crop["ixy_" + img], crop["ds_" + img], sr.shape)
        assert maxnorm_err(d, ref["d_" + img]) < 1e-4, img


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_crop_forward_per_image_and_pixel_term(lib, shape):
    """reduction='none' and the fused Pixel term (scalar and per image) through the crop layout."""
    sr, hr = _pair(shape, 7 * sum(shape))
    taps = _taps()
    B = shape[0]
    go = np.random.default_rng(shape[1]).uniform(-2.0, 2.0, B).astype(np.float32)
    grad = np.random.default_rng(shape[2]).uniform(-2.0, 2.0, (2, B)).astype(np.float32)

    def run():
        return (emu_st_per_image(lib, sr, hr, taps, go, want_hr=True), emu_stpx(lib, sr, hr, taps, grad_st=0.5, grad_px=1.5),
                emu_stpx_per_image(lib, sr, hr, taps, grad))

    none, px, px_none = _run(lib, CROP, 0, run)
    bad = _run(lib, CROP, 0, lambda: _poisoned(lib, run))
    halo = _run(lib, HALO, 0, run)
    for k in ("loss", "d_sr", "d_hr"):
        assert _same(none[k], bad[0][k]), k
    assert _same(px["d_sr"], bad[1]["d_sr"]) and px["st"] == bad[1]["st"] and px["px"] == bad[1]["px"]
    assert _same(px_none["both"], bad[2]["both"]) and _same(px_none["d_sr"], bad[2]["d_sr"])
    # the fused backward reads the forward's ds / ixy only: bit-identical to the halo strips
    assert _same(none["d_sr"], halo[0]["d_sr"]) and _same(none["d_hr"], halo[0]["d_hr"])
    assert _same(px["d_sr"], halo[1]["d_sr"]) and _same(px_none["d_sr"], halo[2]["d_sr"])
    # the Pixel term's partial sums may be spread differently over the threads: 1e-6
    assert rel_err(px["px"], halo[1]["px"]) < 1e-6 and rel_err(px["st"], halo[1]["st"]) < 1e-6
    np.testing.assert_allclose(px_none["both"], halo[2]["both"], rtol=1e-6, atol=0)
    np.testing.assert_allclose(none["loss"], halo[0]["loss"], rtol=1e-6, atol=0)
    ref = O.st_loss(sr, hr, taps=taps, want_hr_grad=True)
    mse = np.mean((sr.astype(np.float64) - hr) ** 2, axis=(1, 2, 3))
    assert rel_err(px["st"], ref["loss"]) < 1e-5 and rel_err(px["px"], mse.mean()) < 1e-5
    d_px = 2.0 * (sr.astype(np.float64) - hr) / sr.size
    assert maxnorm_err(px["d_sr"], 0.5 * ref["d_sr"] + 1.5 * d_px) < 1e-4
    for b in range(B):
        one = O.st_loss(sr[b:b + 1], hr[b:b + 1], taps=taps, want_hr_grad=True)
        assert rel_err(none["loss"][b], one["loss"]) < 1e-5 and rel_err(px_none["both"][0, b], one["loss"]) < 1e-5
        assert rel_err(px_none["both"][1, b], mse[b]) < 1e-5
        for k in ("d_sr", "d_hr"):
            assert maxnorm_err(none[k][b], go[b] * one[k][0]) < 1e-4, (k, b)
