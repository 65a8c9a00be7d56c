"""CPU: the per-image (reduction='none') entry points of the fused ST + Pixel criterion, run on the emulation library.

For every forward shape the fused path can take -- both marching strips, both fused tile shapes, a padded radius
class, a short marching chunk and ragged shapes -- row 0 of the [2][B] output must match the float64 ST oracle run on
each image alone and row 1 the float64 per-image MSE, and each row must average to the scalar entry point's term.
With a random [2][B] upstream gradient, image b's d_sr must be bit-identical to srst_stpx_backward run on image b
alone with (grad_st[b], grad_px[b]), and the workspace (both partial arrays and the ticket) must come back zeroed.

The argument contract follows tests/test_per_image_contract.py: each argument that is bad on its own gets its
documented code, and a run with 0xFF (NaN as a float) in shared memory and in every workspace byte but the ticket
header gives the same bytes."""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests import helpers
from tests.helpers import _fp, _p, _workspace, emu_lib, emu_stpx, rel_err

E_INVALID, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -3
POISON = 0xFF


@pytest.fixture(scope="module")
def lib():
    lib = emu_lib()
    yield lib
    lib.srst_emu_set_poison(0xCD)
    lib.srst_st_force_cfg(-1, -1)
    lib.srst_st_force_chunk_blocks(0)


def _taps(sigma=0.5, rho=2.0):
    return tuple(np.ascontiguousarray(t, np.float32) for t in (*O.gaussian_taps(sigma, True), O.gaussian_taps(rho)))


def emu_stpx_per_image(lib, sr, hr, taps, grad):
    """srst_stpx_forward_per_image + srst_stpx_backward_per_image on host arrays; grad is the [2][B] upstream
    gradient (row 0 for the ST terms, row 1 for the MSE terms)."""
    B, _, H, W = sr.shape
    g, dg, k = taps
    rs, rk = len(g) // 2, len(k) // 2
    nb = lib.srst_st_workspace_bytes(B, H, W)
    ws = _workspace(nb)
    both = np.full((2, B), np.nan, np.float32)
    ds = np.full_like(sr, np.nan)
    ixy = np.full(lib.srst_st_ixy_floats(B, H, W), np.nan, np.float32)
    rc = lib.srst_stpx_forward_per_image(_p(sr), _p(hr), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, 1, 1e-12, _p(both),
                                         _p(ds), _p(ixy), _p(ws), nb, None)
    assert rc == 0, rc
    grad = np.ascontiguousarray(grad, np.float32)
    d_sr = np.full_like(sr, np.nan)
    rc = lib.srst_stpx_backward_per_image(_p(sr), _p(hr), _p(ixy), _p(ds), _p(grad[0]), _p(grad[1]), B, H, W, _fp(g),
                                          _fp(dg), rs, _fp(k), rk, _p(d_sr), None)
    assert rc == 0, rc
    return dict(both=both, d_sr=d_sr, ws=ws[:nb // 4])


def _pair(shape, seed):
    rng = np.random.default_rng(seed)
    B, H, W = shape
    hr = rng.random((B, 3, H, W), dtype=np.float32)
    sr = np.clip(hr + 0.1 * rng.standard_normal((B, 3, H, W), dtype=np.float32), 0, 1).astype(np.float32)
    return sr, hr, rng.uniform(-2.0, 2.0, (2, B)).astype(np.float32)


def _check(lib, shape, taps, seed):
    sr, hr, grad = _pair(shape, seed)
    B = shape[0]
    out = emu_stpx_per_image(lib, sr, hr, taps, grad)
    assert np.all(out["ws"] == 0), "workspace must come back zeroed (both partial arrays and the ticket)"
    whole = emu_stpx(lib, sr, hr, taps)
    st, px = out["both"].astype(np.float64)
    assert rel_err(st.mean(), whole["st"]) < 1e-6
    assert rel_err(px.mean(), whole["px"]) < 1e-6
    for b in range(B):
        ref = O.st_loss(sr[b:b + 1], hr[b:b + 1], taps=taps, want_grad=False)
        assert rel_err(float(out["both"][0, b]), ref["loss"]) < 1e-5
        d = sr[b].astype(np.float64) - hr[b].astype(np.float64)
        assert rel_err(float(out["both"][1, b]), (d * d).mean()) < 1e-6
        one = emu_stpx(lib, sr[b:b + 1], hr[b:b + 1], taps, grad_st=float(grad[0, b]), grad_px=float(grad[1, b]))
        assert out["d_sr"][b].tobytes() == one["d_sr"][0].tobytes(), b


@pytest.mark.parametrize("fwd_cfg", [3, 4, 0, 1], ids=["march96", "march112", "tiled0", "tiled1"])
def test_every_fused_forward_shape(lib, fwd_cfg):
    assert lib.srst_st_force_cfg(fwd_cfg, -1) == 0
    try:
        _check(lib, (3, 40, 52), _taps(), seed=fwd_cfg)
    finally:
        lib.srst_st_force_cfg(-1, -1)


def test_padded_radius_class(lib):
    _check(lib, (2, 24, 36), _taps(1.0, 3.0), seed=5)


def test_short_march_chunks(lib):
    """16-row chunks of the marching forward: an image's partials are several chunks x strips; W > 96 takes the
    28x56 backward tiles."""
    assert lib.srst_st_force_cfg(3, -1) == 0 and lib.srst_st_force_chunk_blocks(1) == 0
    try:
        _check(lib, (2, 50, 100), _taps(), seed=11)
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)


@pytest.mark.parametrize("shape", [(3, 21, 30), (2, 37, 53)])
def test_ragged_shapes(lib, shape):
    """W % 4 != 0 and odd H: no TMA, the tiled shapes with plain loads."""
    _check(lib, shape, _taps(), seed=sum(shape))


# ---- argument contract -------------------------------------------------------------------------------------------
def _call(lib, fwd, taps=None, **over):
    B, H, W = 2, 20, 24
    g, dg, k = taps or _taps()
    rng = np.random.default_rng(1)
    sr, hr = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    nb = lib.srst_st_workspace_bytes(B, H, W)
    ws = np.zeros(nb // 4 + 8, np.float32)
    v = dict(sr=sr, hr=hr, B=B, H=H, W=W, g=g, dg=dg, k=k, rs=len(g) // 2, rk=len(k) // 2,
             loss=np.zeros((2, B), np.float32), ds=np.zeros_like(sr), ixy=np.zeros(lib.srst_st_ixy_floats(B, H, W), np.float32),
             grad_st=np.ones(B, np.float32), grad_px=np.ones(B, np.float32), d_sr=np.zeros_like(sr), ws=ws.ctypes.data,
             nbytes=nb)
    v.update(over)
    a = {n: (x.ctypes.data if isinstance(x, np.ndarray) else x) for n, x in v.items()}
    for t in ("g", "dg", "k"):
        a[t] = _fp(v[t]) if v[t] is not None else None
    if fwd:
        return lib.srst_stpx_forward_per_image(a["sr"], a["hr"], v["B"], v["H"], v["W"], a["g"], a["dg"], v["rs"], a["k"],
                                               v["rk"], 1, 1e-12, a["loss"], a["ds"], a["ixy"], a["ws"], v["nbytes"], None)
    return lib.srst_stpx_backward_per_image(a["sr"], a["hr"], a["ixy"], a["ds"], a["grad_st"], a["grad_px"], v["B"],
                                            v["H"], v["W"], a["g"], a["dg"], v["rs"], a["k"], v["rk"], a["d_sr"], None)


@pytest.mark.parametrize("fwd", [True, False], ids=["forward", "backward"])
def test_contract(lib, fwd):
    assert _call(lib, fwd) == 0
    ptrs = ("sr", "hr", "g", "dg", "k") + (("loss",) if fwd else ("ixy", "ds", "grad_st", "grad_px", "d_sr"))
    bad = [({p: None}, E_INVALID) for p in ptrs]
    bad += [({"B": 0}, E_INVALID), ({"H": 0}, E_INVALID), ({"W": -1}, E_INVALID)]
    bad += [({"taps": _taps(1.5, 3.5)}, E_UNSUPPORTED), ({"rs": 65}, E_UNSUPPORTED)]   # generic radius: no fused variant
    if fwd:
        nb = lib.srst_st_workspace_bytes(2, 20, 24)
        ws = np.zeros(nb // 4 + 8, np.float32)
        bad += [({"ws": None}, E_WORKSPACE), ({"nbytes": nb - 4}, E_WORKSPACE),
                ({"ws": ws.ctypes.data + 4}, E_WORKSPACE)]   # unaligned
    wrong = [(o, rc, want) for o, want in bad if (rc := _call(lib, fwd, **o)) != want]
    assert not wrong, f"(bad argument, returned, expected): {wrong}"


# ---- poison ------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["march-chunk", "tiled-ragged", "padded"])
def test_poison(lib, case):
    shape, taps = {"march-chunk": ((2, 40, 100), _taps()), "tiled-ragged": ((3, 21, 30), _taps()),
                   "padded": ((2, 24, 36), _taps(1.0, 3.0))}[case]
    sr, hr, grad = _pair(shape, seed=3)
    if case == "march-chunk":
        assert lib.srst_st_force_cfg(3, -1) == 0 and lib.srst_st_force_chunk_blocks(1) == 0
    try:
        clean = emu_stpx_per_image(lib, sr, hr, taps, grad)
        helpers.WORKSPACE_FILL = POISON
        helpers.FILLED_WORKSPACES.clear()
        lib.srst_emu_set_poison(POISON)
        try:
            poisoned = emu_stpx_per_image(lib, sr, hr, taps, grad)
        finally:
            lib.srst_emu_set_poison(0xCD)
            helpers.WORKSPACE_FILL = None
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)
    assert len(helpers.FILLED_WORKSPACES) == 1
    assert np.all(helpers.FILLED_WORKSPACES[0].view(np.uint32)[:4] == 0), "ticket header not handed back zeroed"
    helpers.FILLED_WORKSPACES.clear()
    for key in ("both", "d_sr"):
        assert clean[key].tobytes() == poisoned[key].tobytes(), key
        assert not np.isnan(clean[key]).any(), key
