"""CPU: no emulated kernel may depend on memory it did not write.

Every case runs twice under the host emulation (tests/emu): once with the default 0xCD shared-memory fill (the
finite float -4.3e8) and zeroed workspaces, once with 0xFF in all shared memory -- dynamic and static arrays, before
every block -- and in every workspace byte but the 16-byte ticket header, the only part srst.h promises to be zero.
0xFF is a NaN as a float and -1 as an int, so a never-written value that is multiplied by a zero weight, padded over
or summed into a reduction turns the result NaN instead of hiding.  Outputs are NaN-filled before both runs (the
emu_* helpers do that).  Deterministic outputs must come back bit for bit; the gradients w.r.t. gt are summed with
atomics in a thread-order-dependent order and are held to the float64 oracle instead."""
import ctypes

import numpy as np
import pytest

from oracle import bb_oracle as OB
from oracle import bbg_oracle as OG
from oracle import st_oracle as O
from tests import helpers
from tests.helpers import emu_bb, emu_bbg, emu_lib, emu_patch_gt, emu_st, emu_stpx, golden, maxnorm_err, rel_err

DIST_L1 = 0x100   # SRST_BB_DIST_L1
POISON = 0xFF


@pytest.fixture(scope="module")
def lib():
    lib = emu_lib()
    assert lib.srst_emu_set_poison(0xCD) == 0xCD
    yield lib
    lib.srst_emu_set_poison(0xCD)
    lib.srst_st_force_cfg(-1, -1)
    lib.srst_st_force_chunk_blocks(0)


def _twice(lib, run):
    """(clean, poisoned) results of run(); checks that every poisoned workspace got its ticket header back zeroed."""
    clean = run()
    helpers.WORKSPACE_FILL = POISON
    helpers.FILLED_WORKSPACES.clear()
    lib.srst_emu_set_poison(POISON)
    try:
        poisoned = run()
    finally:
        lib.srst_emu_set_poison(0xCD)
        helpers.WORKSPACE_FILL = None
    assert helpers.FILLED_WORKSPACES, "the poisoned run must have used a workspace"
    for ws in helpers.FILLED_WORKSPACES:
        assert np.all(ws.view(np.uint32)[:4] == 0), "ticket header not handed back zeroed"
    helpers.FILLED_WORKSPACES.clear()
    return clean, poisoned


def _same_bits(a, b):
    a, b = np.asarray(a), np.asarray(b)
    return a.shape == b.shape and a.dtype == b.dtype and a.tobytes() == b.tobytes()


def _assert_identical(clean, poisoned, keys):
    for k in keys:
        if isinstance(clean[k], float):
            assert np.float32(clean[k]).tobytes() == np.float32(poisoned[k]).tobytes(), (k, clean[k], poisoned[k])
            assert np.isfinite(clean[k]), k
        else:
            assert _same_bits(clean[k], poisoned[k]), f"{k} differs: {np.isnan(poisoned[k]).sum()} NaN in the poisoned run"
            assert not np.isnan(clean[k]).any(), k


def _rand(shape, seed):
    rng = np.random.default_rng(seed)
    return rng.random(shape, dtype=np.float32), rng.random(shape, dtype=np.float32)


TAPS = (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0))


# ---- structure tensor ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("cfg", [(0, 0), (1, 1), (2, 0), (3, 1), (4, 0)], ids=lambda p: f"fwd{p[0]}-bwd{p[1]}")
@pytest.mark.parametrize("shape", [(1, 37, 52), (1, 37, 53), (2, 30, 100)])
def test_st_every_tile_shape(lib, cfg, shape):
    """Every compiled forward / backward shape; odd H (the filler row of the interleaved Ix, Iy pairs) and W % 4 != 0
    (no vec4, no TMA: the marching cfgs fall back to tiles)."""
    sr, hr = _rand((shape[0], 3, shape[1], shape[2]), sum(shape))
    assert lib.srst_st_force_cfg(*cfg) == 0
    try:
        clean, poisoned = _twice(lib, lambda: emu_st(lib, sr, hr, TAPS, want_hr=True))
    finally:
        lib.srst_st_force_cfg(-1, -1)
    _assert_identical(clean, poisoned, ["loss", "d_sr", "d_hr"])
    ref = O.st_loss(sr, hr, taps=TAPS)
    assert rel_err(clean["loss"], ref["loss"]) < 1e-5


@pytest.mark.parametrize("cfg", [3, 4])
@pytest.mark.parametrize("chunk_blocks", [1, 2])
def test_st_marching_chunk_seams(lib, cfg, chunk_blocks):
    sr, hr = _rand((1, 3, 70, 204), 7 + chunk_blocks)
    assert lib.srst_st_force_cfg(cfg, -1) == 0 and lib.srst_st_force_chunk_blocks(chunk_blocks) == 0
    try:
        clean, poisoned = _twice(lib, lambda: emu_st(lib, sr, hr, TAPS, want_hr=True))
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)
    _assert_identical(clean, poisoned, ["loss", "d_sr", "d_hr"])


@pytest.mark.parametrize("sigma,rho,shape", [(0.3, 1.0, (1, 37, 52)), (1.0, 2.5, (1, 33, 45)),   # zero-padded taps
                                             (2.0, 2.0, (1, 20, 28)), (0.5, 4.0, (2, 17, 19))])  # generic radius
def test_st_other_radii(lib, sigma, rho, shape):
    """Radii padded with zero taps into a compiled class, and the generic-radius path (scratch planes in both
    workspaces: the forward's beyond the ticket header, the backward's entirely)."""
    sr, hr = _rand((shape[0], 3, shape[1], shape[2]), int(10 * sigma + rho))
    taps = (*O.gaussian_taps(sigma, True), O.gaussian_taps(rho))
    clean, poisoned = _twice(lib, lambda: emu_st(lib, sr, hr, taps, want_hr=True, grad_out=-0.5))
    _assert_identical(clean, poisoned, ["loss", "d_sr", "d_hr"])
    assert rel_err(clean["loss"], O.st_loss(sr, hr, taps=taps)["loss"]) < 1e-5


@pytest.mark.parametrize("cfg", [-1, 0, 1])
@pytest.mark.parametrize("name", ["st_rand_2x24x36", "st_rand_ragged_1x37x53"])
def test_stpx(lib, cfg, name):
    z = golden(name)
    assert lib.srst_st_force_cfg(cfg, cfg) == 0
    try:
        clean, poisoned = _twice(lib, lambda: emu_stpx(lib, z["sr"], z["hr"], TAPS, grad_st=0.5, grad_px=1.5))
    finally:
        lib.srst_st_force_cfg(-1, -1)
    _assert_identical(clean, poisoned, ["st", "px", "d_sr"])


@pytest.mark.parametrize("shape", [(1, 37, 53), (2, 40, 72)])
def test_st_features(lib, shape):
    B, H, W = shape
    img = _rand((B, 3, H, W), H)[0]
    g, dg, k = TAPS
    fp = lambda a: a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))
    vp = lambda a: ctypes.c_void_p(a.ctypes.data)

    def run():
        out = dict(J=np.full((B, 3, H, W), np.nan, np.float32), eig=np.full((B, 2, H, W), np.nan, np.float32),
                   orient=np.full((B, H, W), np.nan, np.float32), coher=np.full((B, H, W), np.nan, np.float32))
        assert lib.srst_st_features(vp(img), B, H, W, fp(g), fp(dg), len(g) // 2, fp(k), len(k) // 2, vp(out["J"]),
                                    vp(out["eig"]), vp(out["orient"]), vp(out["coher"]), None) == 0
        return out

    clean = run()
    lib.srst_emu_set_poison(POISON)
    try:
        poisoned = run()
    finally:
        lib.srst_emu_set_poison(0xCD)
    _assert_identical(clean, poisoned, ["J", "eig", "orient", "coher"])


# ---- Best-Buddy, Gram, patchwise structure tensor ------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["patch", "gram", "pst"])
@pytest.mark.parametrize("own_pyramid", [True, False], ids=["own-pyramid", "given-pyramid"])
@pytest.mark.parametrize("crit", [0, 1 | DIST_L1], ids=["l1-dist_l2", "l2-dist_l1"])
@pytest.mark.parametrize("shape", [(1, 26, 31), (2, 24, 36), (1, 13, 40)])
def test_patch_losses(lib, mode, own_pyramid, crit, shape):
    """H, W not multiples of 3 or 12 (padded query / candidate columns of the descriptor matrices, pixels outside
    every patch), the library's own pyramid (in the workspace) and a given one, both search norms and criteria."""
    B, H, W = shape
    gt, noise = _rand((B, 3, H, W), H * W + crit)
    sr = np.clip(gt + 0.1 * (noise - 0.5), 0, 1).astype(np.float32)
    gt2, gt4 = (None, None) if own_pyramid else OB.pyramid_c(gt)
    clean, poisoned = _twice(lib, lambda: emu_bb(lib, sr, gt, gt2, gt4, 0.7, 1.3, crit, 0.75, mode, TAPS))
    _assert_identical(clean, poisoned, ["loss", "d_sr"])
    assert np.array_equal(clean["idx"], poisoned["idx"])
    M = (H // 3) * (W // 3) + (H // 6) * (W // 6) + (H // 12) * (W // 12)
    assert poisoned["idx"].min() >= 0 and poisoned["idx"].max() < M


@pytest.mark.parametrize("mode", ["patch", "gram", "pst"])
@pytest.mark.parametrize("own_pyramid", [True, False], ids=["own-pyramid", "given-pyramid"])
@pytest.mark.parametrize("shape", [(1, 26, 31), (2, 24, 24)])
def test_patch_gt_gradient(lib, mode, own_pyramid, shape):
    """d loss / d gt: the zero-filled coarse-level gradient images d2 / d4 live in the (poisoned) workspace."""
    B, H, W = shape
    gt, noise = _rand((B, 3, H, W), 3 * H + W)
    sr = np.clip(gt + 0.1 * (noise - 0.5), 0, 1).astype(np.float32)
    o2, o4 = OB.pyramid_c(gt)
    idx = emu_bb(lib, sr, gt, o2, o4, mode=mode, taps=TAPS)["idx"]
    gt2, gt4 = (None, None) if own_pyramid else (o2, o4)
    taps = TAPS if mode == "pst" else None
    clean, poisoned = _twice(lib, lambda: emu_patch_gt(lib, sr, gt, idx, gt2, gt4, 1, -1.5, mode, taps))
    ref = -1.5 * OB.patch_backward_gt(sr, gt, o2, o4, idx, mode, taps, "l2")
    for d in (clean, poisoned):
        assert not np.isnan(d).any()
        assert maxnorm_err(d, ref) < 1e-4


@pytest.mark.parametrize("k,p,s", [(4, 1, 2), (3, 2, 5), (8, 4, 7), (1, 0, 1)])
@pytest.mark.parametrize("own_pyramid", [True, False], ids=["own-pyramid", "given-pyramid"])
def test_bb_geometry(lib, k, p, s, own_pyramid):
    """Non-default patch geometries: padding, stride > ksize (gaps), stride < ksize (overlap), 3-element patches."""
    gt, noise = _rand((2, 3, 33, 35), 10 * k + s)
    sr = np.clip(gt + 0.1 * (noise - 0.5), 0, 1).astype(np.float32)
    gt2, gt4 = (None, None) if own_pyramid else OB.pyramid_c(gt)
    crit = 1 if k % 2 else DIST_L1
    clean, poisoned = _twice(lib, lambda: emu_bbg(lib, sr, gt, k, p, s, gt2, gt4, 1.0, 1.0, crit, 1.0, want_gt=True))
    _assert_identical(clean, poisoned, ["loss", "d_sr"])
    assert np.array_equal(clean["idx"], poisoned["idx"])
    orc = OG.bbg_forward_c(sr, gt, gt2, gt4, k, p, s, 1.0, 1.0, "l2" if crit & 1 else "l1", "l1" if crit & DIST_L1 else "l2")
    assert np.array_equal(poisoned["idx"], orc["idx"])
    assert not np.isnan(poisoned["d_gt"]).any() and maxnorm_err(poisoned["d_gt"], clean["d_gt"]) < 1e-5
