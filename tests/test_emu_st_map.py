"""CPU: the per-pixel distance map (srst_st_forward_map / srst_st_backward_map of include/srst.h) on the emulation
library.

For every forward path -- each compiled forward shape, a one-block marching chunk (chunk seams and filler rows), odd H
and W % 4 != 0, a padded radius class and the generic-radius path, with and without ds_hr -- the map must match the
float64 oracle's per-pixel distance, and loss_out, ds_* and ixy_* must be bit-identical to srst_st_forward on the same
inputs.  The backward, under a random per-pixel upstream gradient with zeros, negative values and a border-band mask,
must match the float64 oracle composed from st_distance_backward and _st_image_backward; under a constant or a
per-image constant gradient it must agree with srst_st_backward / srst_st_backward_per_image.  The saved buffers are
only read, so a second backward gives the same bits.  The argument contract and the independence from memory the
kernels did not write (0xFF workspaces and shared memory, NaN-prefilled outputs) are pinned as well."""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests import helpers
from tests.helpers import _fp, _p, _workspace, emu_lib, golden, maxnorm_err, rel_err

E_INVALID, E_UNSUPPORTED, E_WORKSPACE = -1, -2, -3
POISON = 0xFF


@pytest.fixture(scope="module")
def lib():
    lib = emu_lib()
    assert lib.srst_emu_set_poison(0xCD) == 0xCD
    yield lib
    lib.srst_emu_set_poison(0xCD)
    lib.srst_st_force_cfg(-1, -1)
    lib.srst_st_force_chunk_blocks(0)


def _taps(sigma=0.5, rho=2.0):
    return tuple(np.ascontiguousarray(t, np.float32) for t in (*O.gaussian_taps(sigma, True), O.gaussian_taps(rho)))


def oracle_map_backward(sr, hr, taps, G, normalize=True):
    """float64 (d_sr, d_hr) of sum(G * map): st_distance_backward(gd=G), then the adjoint of the image chain."""
    sr, hr = np.asarray(sr, np.float64), np.asarray(hr, np.float64)
    g, dg, k = (np.asarray(t, np.float64) for t in taps)
    Ix1, Iy1, a, b, c = O.structure_tensor(O.grayscale(sr), g, dg, k)
    Ix2, Iy2, e, f, h = O.structure_tensor(O.grayscale(hr), g, dg, k)
    F = O.st_distance_fields((a, b, c), (e, f, h), normalize)
    dS1, dS2 = O.st_distance_backward((a, b, c), (e, f, h), F, np.asarray(G, np.float64), normalize, want_hr=True)
    coef = np.array([O.GRAY_R, O.GRAY_G, O.GRAY_B], np.float64).reshape(1, 3, 1, 1)
    return (coef * O._st_image_backward(Ix1, Iy1, dS1, g, dg, k)[:, None],
            coef * O._st_image_backward(Ix2, Iy2, dS2, g, dg, k)[:, None])


def _weights(B, H, W, seed, band=3):
    """Random per-pixel upstream gradient with zeros and negative values, times a mask that zeroes a border band."""
    rng = np.random.default_rng(seed)
    G = rng.uniform(-2.0, 2.0, (B, H, W)).astype(np.float32)
    G[rng.random((B, H, W)) < 0.2] = 0.0
    mask = np.zeros((H, W), np.float32)
    mask[band:H - band, band:W - band] = 1.0
    return np.ascontiguousarray(G * mask)


def _forward(lib, sr, hr, taps, want_hr, map_out=None):
    """srst_st_forward_map (map_out given: a NaN-prefilled [B,H,W]) or srst_st_forward on host arrays."""
    B, _, H, W = sr.shape
    g, dg, k = taps
    rs, rk = len(g) // 2, len(k) // 2
    nb = lib.srst_st_workspace_bytes_r(B, H, W, rs, rk)
    ws = _workspace(nb)
    loss = np.full(1, np.nan, np.float32)
    n_ixy = lib.srst_st_ixy_floats(B, H, W)
    ds = [np.full_like(sr, np.nan), np.full_like(sr, np.nan) if want_hr else None]
    ixy = [np.full(n_ixy, np.nan, np.float32), np.full(n_ixy, np.nan, np.float32) if want_hr else None]
    args = (_p(sr), _p(hr), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, 1, 1e-12, _p(loss))
    outs = (_p(ds[0]), _p(ds[1]), _p(ixy[0]), _p(ixy[1]), _p(ws), nb, None)
    rc = lib.srst_st_forward_map(*args, _p(map_out), *outs) if map_out is not None else lib.srst_st_forward(*args, *outs)
    assert rc == 0, rc
    return dict(loss=loss, ds=ds, ixy=ixy, header=ws[:4].copy())


def _backward_map(lib, taps, ixy, ds, G):
    B, H, W = G.shape
    g, dg, k = taps
    rs, rk = len(g) // 2, len(k) // 2
    nb = lib.srst_st_backward_map_workspace_bytes(B, H, W, rs, rk)
    assert nb > 0
    ws = _workspace(nb)
    d = np.full((B, 3, H, W), np.nan, np.float32)
    rc = lib.srst_st_backward_map(_p(ixy), _p(ds), _p(G), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, _p(d), _p(ws), nb,
                                  None)
    assert rc == 0, rc
    return d


def _backward_scalar(lib, taps, ixy, ds, shape, grad_out, per_image=False):
    B, _, H, W = shape
    g, dg, k = taps
    rs, rk = len(g) // 2, len(k) // 2
    nbb = lib.srst_st_backward_workspace_bytes(B, H, W, rs, rk)
    bws = np.full(nbb // 4 + 4, np.nan, np.float32)
    go = np.ascontiguousarray(grad_out, np.float32)
    d = np.full(shape, np.nan, np.float32)
    fn = lib.srst_st_backward_per_image if per_image else lib.srst_st_backward_ws
    rc = fn(_p(ixy), _p(ds), _p(go), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, _p(d), _p(bws) if nbb else None, nbb,
            None)
    assert rc == 0, rc
    return d


def emu_st_map(lib, sr, hr, taps, G, want_hr=True):
    """srst_st_forward_map + srst_st_backward_map (upstream gradient G [B,H,W]) on host arrays."""
    sr, hr = np.ascontiguousarray(sr, np.float32), np.ascontiguousarray(hr, np.float32)
    B, _, H, W = sr.shape
    dmap = np.full((B, H, W), np.nan, np.float32)
    out = _forward(lib, sr, hr, taps, want_hr, dmap)
    out["map"] = dmap
    for name, s, d in zip(("d_sr", "d_hr"), out["ixy"], out["ds"]):
        if s is not None:
            out[name] = _backward_map(lib, taps, s, d, G)
    return out


def _check(lib, sr, hr, taps, want_hr, map_tol=1e-5, seed=0):
    sr, hr = np.ascontiguousarray(sr, np.float32), np.ascontiguousarray(hr, np.float32)
    B, _, H, W = sr.shape
    G = _weights(B, H, W, seed)
    out = emu_st_map(lib, sr, hr, taps, G, want_hr)
    assert np.all(out["header"] == 0)                       # ticket handed back zeroed
    ref = O.st_loss(sr, hr, taps=taps, want_grad=False)
    assert maxnorm_err(out["map"], ref["d"]) < map_tol
    # loss, ds and ixy: the bits of srst_st_forward
    plain = _forward(lib, sr, hr, taps, want_hr)
    assert out["loss"].tobytes() == plain["loss"].tobytes()
    for a, b in zip(out["ds"] + out["ixy"], plain["ds"] + plain["ixy"]):
        assert (a is None) == (b is None) and (a is None or a.tobytes() == b.tobytes())
    assert rel_err(out["map"].astype(np.float64).sum() / (B * H * W), out["loss"][0]) < 1e-6
    # backward against the float64 oracle
    o_sr, o_hr = oracle_map_backward(sr, hr, taps, G)
    assert maxnorm_err(out["d_sr"], o_sr) < 1e-4
    if want_hr:
        assert maxnorm_err(out["d_hr"], o_hr) < 1e-4
    # a constant gradient is the batch mean's, a per-image constant the per-image mean's
    c = -0.75
    w = np.random.default_rng(seed + 1).uniform(-2.0, 2.0, B).astype(np.float32)
    for i, (s, d) in enumerate(zip(out["ixy"], out["ds"])):
        if s is None:
            continue
        ds_bits, ixy_bits = d.tobytes(), s.tobytes()
        const = _backward_map(lib, taps, s, d, np.full((B, H, W), c, np.float32))
        assert maxnorm_err(const, _backward_scalar(lib, taps, s, d, sr.shape, [c * B * H * W])) < 1e-6
        Gw = np.ascontiguousarray(np.broadcast_to((w / (H * W))[:, None, None], (B, H, W)), np.float32)
        per = _backward_map(lib, taps, s, d, Gw)
        assert maxnorm_err(per, _backward_scalar(lib, taps, s, d, sr.shape, w, per_image=True)) < 1e-6
        again = _backward_map(lib, taps, s, d, G)
        assert again.tobytes() == out[("d_sr", "d_hr")[i]].tobytes()     # the saved buffers are only read
        assert d.tobytes() == ds_bits and s.tobytes() == ixy_bits
    return out


@pytest.mark.parametrize("fwd_cfg", [0, 1, 2, 3, 4, -1])
def test_map_every_forward_shape(lib, fwd_cfg):
    assert lib.srst_st_force_cfg(fwd_cfg, -1) == 0
    try:
        rng = np.random.default_rng(20 + fwd_cfg)
        sr, hr = (rng.random((2, 3, 40, 52), dtype=np.float32) for _ in range(2))
        _check(lib, sr, hr, _taps(), want_hr=fwd_cfg in (-1, 0, 3), seed=fwd_cfg + 10)
    finally:
        lib.srst_st_force_cfg(-1, -1)


def test_map_one_block_march_chunks(lib):
    """16-row chunks: every chunk seam is crossed, and the last chunk's filler rows (odd H) must not be stored."""
    assert lib.srst_st_force_cfg(3, -1) == 0 and lib.srst_st_force_chunk_blocks(1) == 0
    try:
        rng = np.random.default_rng(31)
        sr, hr = (rng.random((2, 3, 45, 100), dtype=np.float32) for _ in range(2))
        _check(lib, sr, hr, _taps(), want_hr=True, seed=31)
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)


@pytest.mark.parametrize("shape,want_hr", [((2, 37, 53), True), ((1, 21, 30), False)])
def test_map_ragged_shapes(lib, shape, want_hr):
    """Odd H and W % 4 != 0: no TMA, the tiled fall-back with scalar stores."""
    rng = np.random.default_rng(sum(shape))
    sr, hr = (rng.random((shape[0], 3, shape[1], shape[2]), dtype=np.float32) for _ in range(2))
    _check(lib, sr, hr, _taps(), want_hr=want_hr, seed=sum(shape))


@pytest.mark.parametrize("name,want_hr", [("st_rand_s1_r25_1x32x40", True), ("st_rand_s15_r4_1x40x52", True),
                                          ("st_srlike_s2_r5_2x33x45", False)])
def test_map_padded_and_generic_radii(lib, name, want_hr):
    z = golden(name)
    _check(lib, z["sr"], z["hr"], tuple(np.ascontiguousarray(z[t], np.float32) for t in ("g", "dg", "k")), want_hr)


def test_map_identical_images(lib):
    """sr == hr: every distance sits at the sqrt(eps) = 1e-6 floor, where the fp32 rounding of the eigenvalue logs
    (|L| ~ 1e-7) is a large part of each pixel's value: measured 0.104 max-norm, 1.2e-7 absolute.  The map's mean is
    held to the 2e-2 that tests/test_st_gpu.py uses for this fixture's loss (measured 9.5e-3), each pixel to 2e-7."""
    z = golden("st_same_1x24x24")
    taps = tuple(np.ascontiguousarray(z[t], np.float32) for t in ("g", "dg", "k"))
    sr, hr = np.ascontiguousarray(z["sr"], np.float32), np.ascontiguousarray(z["hr"], np.float32)
    out = emu_st_map(lib, sr, hr, taps, _weights(1, 24, 24, 5))
    d = O.st_loss(sr, hr, taps=taps, want_grad=False)["d"]
    assert rel_err(out["map"].astype(np.float64).mean(), d.mean()) < 2e-2
    assert np.abs(out["map"] - d).max() < 2e-7
    assert rel_err(out["map"].astype(np.float64).mean(), out["loss"][0]) < 1e-6


# ---- memory the kernels did not write ----------------------------------------------------------------------------
@pytest.mark.parametrize("case", ["default", "tiled", "chunks", "ragged", "generic"])
def test_map_poison(lib, case):
    """0xFF in shared memory and in every workspace byte but the ticket header: the same bits."""
    cfg, chunk, shape, taps = {"default": (-1, 0, (2, 40, 52), _taps()), "tiled": (1, 0, (2, 33, 48), _taps()),
                               "chunks": (4, 1, (1, 45, 120), _taps()), "ragged": (-1, 0, (2, 37, 53), _taps()),
                               "generic": (-1, 0, (1, 30, 44), _taps(1.5, 4.0))}[case]
    rng = np.random.default_rng(len(case))
    sr, hr = (rng.random((shape[0], 3, shape[1], shape[2]), dtype=np.float32) for _ in range(2))
    G = _weights(*shape, seed=7)
    assert lib.srst_st_force_cfg(cfg, -1) == 0 and lib.srst_st_force_chunk_blocks(chunk) == 0
    try:
        clean = emu_st_map(lib, sr, hr, taps, G)
        helpers.WORKSPACE_FILL = POISON
        helpers.FILLED_WORKSPACES.clear()
        lib.srst_emu_set_poison(POISON)
        try:
            poisoned = emu_st_map(lib, sr, hr, taps, G)
        finally:
            lib.srst_emu_set_poison(0xCD)
            helpers.WORKSPACE_FILL = None
        # the forward workspace and the two backward ones; only the forward's has a ticket header
        assert len(helpers.FILLED_WORKSPACES) == 3
        assert np.all(helpers.FILLED_WORKSPACES[0].view(np.uint32)[:4] == 0)
        helpers.FILLED_WORKSPACES.clear()
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)
    for key in ("loss", "map", "d_sr", "d_hr"):
        assert clean[key].tobytes() == poisoned[key].tobytes(), key
    for a, b in zip(clean["ds"] + clean["ixy"], poisoned["ds"] + poisoned["ixy"]):
        assert a.tobytes() == b.tobytes()


# ---- argument contract -------------------------------------------------------------------------------------------
def test_map_argument_contract(lib):
    B, H, W = 2, 20, 24
    g, dg, k = _taps()
    rs, rk = len(g) // 2, len(k) // 2
    rng = np.random.default_rng(3)
    sr, hr = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    nb = lib.srst_st_workspace_bytes_r(B, H, W, rs, rk)
    ws = np.zeros(nb // 4 + 4, np.float32)
    loss = np.zeros(1, np.float32)
    dmap = np.zeros((B, H, W), np.float32)
    ds = np.zeros_like(sr)
    ixy = np.zeros(lib.srst_st_ixy_floats(B, H, W), np.float32)

    def fwd(map_out=dmap, rs_=rs, ws_=ws, nb_=nb):
        return lib.srst_st_forward_map(_p(sr), _p(hr), B, H, W, _fp(g), _fp(dg), rs_, _fp(k), rk, 1, 1e-12, _p(loss),
                                       _p(map_out), _p(ds), None, _p(ixy), None, _p(ws_), nb_, None)

    assert fwd() == 0
    assert fwd(map_out=None) == E_INVALID
    assert fwd(rs_=65) == E_UNSUPPORTED
    assert fwd(ws_=None) == E_WORKSPACE
    assert fwd(nb_=nb - 1) == E_WORKSPACE

    nbb = lib.srst_st_backward_map_workspace_bytes(B, H, W, rs, rk)
    assert nbb >= ((B * 3 * H * W * 4 + 255) // 256) * 256
    bws = np.zeros(nbb // 4 + 4, np.float32)
    G = np.ones((B, H, W), np.float32)
    d = np.zeros_like(sr)

    def bwd(grad_map=G, rs_=rs, ws_=bws, nb_=nbb):
        return lib.srst_st_backward_map(_p(ixy), _p(ds), _p(grad_map), B, H, W, _fp(g), _fp(dg), rs_, _fp(k), rk, _p(d),
                                        _p(ws_), nb_, None)

    assert bwd() == 0
    assert bwd(grad_map=None) == E_INVALID
    assert bwd(rs_=65) == E_UNSUPPORTED
    assert bwd(ws_=None) == E_WORKSPACE
    assert bwd(nb_=nbb - 1) == E_WORKSPACE
    # the generic-radius path needs its own scratch planes on top
    assert lib.srst_st_backward_map_workspace_bytes(B, H, W, 6, 16) == nbb + lib.srst_st_backward_workspace_bytes(
        B, H, W, 6, 16)
    for bad in ((0, H, W, rs, rk), (B, -1, W, rs, rk), (B, H, 0, rs, rk), (B, H, W, 65, rk), (B, H, W, rs, 65),
                (B, H, W, 0, rk)):
        assert lib.srst_st_backward_map_workspace_bytes(*bad) == 0
