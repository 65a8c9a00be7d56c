"""CPU: the crop-width backward (cfg 1, images no wider than its 96-column strips) under the host emulation.

The strips stage no x halo: the zero columns the horizontal rho window and the adjoint derivative filter read are
written by the kernel itself.  The strip height follows the batch (12 rows while those fit one round of resident CTAs,
24 rows beyond).  The emulation has 2 SMs, i.e. 4 CTA slots, so B=3 x H=23 and B=1 x H=61 take the 24-row strips
and B=1 x H=37 the 12-row ones.  Each case is held to the float64 oracle, run a second time with 0xFF (NaN) in all
shared memory, and compared with one-image calls (12-row strips for H=23), bit for bit where the scale is the same:
the tile height changes no per-pixel operation order."""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests import helpers
from tests.helpers import emu_lib, emu_st, emu_stpx, maxnorm_err, rel_err
from tests.test_emu_per_image import emu_st_per_image
from tests.test_emu_stpx_per_image import emu_stpx_per_image

POISON = 0xFF
SHAPES = [(3, 23, 52), (3, 23, 96), (1, 61, 52), (1, 61, 96), (1, 37, 96)]


@pytest.fixture(scope="module")
def lib():
    lib = emu_lib()
    yield lib
    lib.srst_emu_set_poison(0xCD)
    lib.srst_st_force_cfg(-1, -1)


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


def _same(a, b):
    return a.shape == b.shape and a.tobytes() == b.tobytes()


@pytest.mark.parametrize("forced", [-1, 1], ids=["default", "cfg1"])
@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_crop_backward_matches_oracle(lib, shape, forced):
    sr, hr = _pair(shape, sum(shape))
    taps = _taps()
    assert lib.srst_st_force_cfg(-1, forced) == 0
    try:
        out = emu_st(lib, sr, hr, taps, want_hr=True)
        bad = _poisoned(lib, lambda: emu_st(lib, sr, hr, taps, want_hr=True))
        ones = [emu_st(lib, sr[b:b + 1], hr[b:b + 1], taps, want_hr=True) for b in range(shape[0])]
    finally:
        lib.srst_st_force_cfg(-1, -1)
    ref = O.st_loss(sr, hr, taps=taps, want_hr_grad=True)
    assert rel_err(out["loss"], ref["loss"]) < 1e-5
    assert maxnorm_err(out["d_sr"], ref["d_sr"]) < 1e-4 and maxnorm_err(out["d_hr"], ref["d_hr"]) < 1e-4
    for k in ("d_sr", "d_hr"):
        assert _same(out[k], bad[k]), f"{k}: {np.isnan(bad[k]).sum()} NaN with poisoned shared memory"
        # one-image calls scale by 1 / (H W) instead of 1 / (B H W): compare the unscaled gradients
        for b, one in enumerate(ones):
            np.testing.assert_allclose(out[k][b] * shape[0], one[k][0], rtol=1e-6, atol=1e-9)


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_crop_backward_per_image(lib, shape):
    """reduction='none': image b's d_sr / d_hr bit-identical to a one-image call with grad_out = g[b]."""
    sr, hr = _pair(shape, 3 * sum(shape))
    taps = _taps()
    go = np.random.default_rng(shape[1]).uniform(-2.0, 2.0, shape[0]).astype(np.float32)
    out = emu_st_per_image(lib, sr, hr, taps, go, want_hr=True)
    bad = _poisoned(lib, lambda: emu_st_per_image(lib, sr, hr, taps, go, want_hr=True))
    for b in range(shape[0]):
        one = emu_st(lib, sr[b:b + 1], hr[b:b + 1], taps, want_hr=True, grad_out=float(go[b]))
        for k in ("d_sr", "d_hr"):
            assert out[k][b].tobytes() == one[k][0].tobytes(), (k, b)
    for k in ("d_sr", "d_hr"):
        assert _same(out[k], bad[k]), k
        assert not np.isnan(out[k]).any()


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: "x".join(map(str, s)))
def test_crop_backward_fused_pixel_term(lib, shape):
    """The fused ST + Pixel backward, scalar and per image, against the oracle and one-image calls."""
    sr, hr = _pair(shape, 5 * sum(shape))
    taps = _taps()
    out = emu_stpx(lib, sr, hr, taps, grad_st=0.5, grad_px=1.5)
    bad = _poisoned(lib, lambda: emu_stpx(lib, sr, hr, taps, grad_st=0.5, grad_px=1.5))
    assert _same(out["d_sr"], bad["d_sr"])
    ref = O.st_loss(sr, hr, taps=taps)
    d_px = 2.0 * (sr.astype(np.float64) - hr) / sr.size
    assert maxnorm_err(out["d_sr"], 0.5 * ref["d_sr"] + 1.5 * d_px) < 1e-4
    grad = np.random.default_rng(shape[2]).uniform(-2.0, 2.0, (2, shape[0])).astype(np.float32)
    per = emu_stpx_per_image(lib, sr, hr, taps, grad)
    bad = _poisoned(lib, lambda: emu_stpx_per_image(lib, sr, hr, taps, grad))
    assert _same(per["d_sr"], bad["d_sr"]) and not np.isnan(per["d_sr"]).any()
    for b in range(shape[0]):
        one = emu_stpx(lib, sr[b:b + 1], hr[b:b + 1], taps, grad_st=float(grad[0, b]), grad_px=float(grad[1, b]))
        assert per["d_sr"][b].tobytes() == one["d_sr"][0].tobytes(), b
