"""CPU: the argument contract of the per-image (reduction='none') entry points of include/srst.h, and their
independence from memory they did not write, on the emulation library.

Each argument that is bad on its own gets the code of the matching scalar entry point (the good call it starts from
succeeds).  The poisoned run fills shared memory and every workspace byte but the 16-byte ticket header with 0xFF (NaN
as a float), as tests/test_emu_poison.py does for the scalar paths: losses, indices and d_sr must come back bit for
bit, the ticket header zeroed, and d_gt (summed with atomics) within 1e-6."""
import ctypes

import numpy as np
import pytest

from tests import helpers
from tests.helpers import _fp, _p, emu_lib, maxnorm_err
from tests.test_emu_per_image import _taps, emu_patch_per_image, emu_st_per_image

E_INVALID, E_UNSUPPORTED, E_WORKSPACE, E_SHAPE = -1, -2, -3, -4
DIST_L1 = 0x100
POISON = 0xFF


@pytest.fixture(scope="module")
def lib():
    lib = emu_lib()
    assert lib.srst_emu_set_poison(0xCD) == 0xCD
    yield lib
    lib.srst_emu_set_poison(0xCD)
    lib.srst_st_force_cfg(-1, -1)
    lib.srst_st_force_chunk_blocks(0)


# ---- argument contract -------------------------------------------------------------------------------------------
def _st_call(lib, fwd, taps=None, **over):
    B, H, W = 2, 20, 24
    g, dg, k = taps or _taps()
    rs, rk = len(g) // 2, len(k) // 2
    rng = np.random.default_rng(1)
    sr, hr = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    nb = lib.srst_st_workspace_bytes_r(B, H, W, rs, rk)
    nbb = lib.srst_st_backward_workspace_bytes(B, H, W, rs, rk)
    v = dict(sr=sr, hr=hr, B=B, H=H, W=W, rs=rs, rk=rk, loss=np.zeros(B, np.float32), ds=np.zeros_like(sr),
             ixy=np.zeros(lib.srst_st_ixy_floats(B, H, W), np.float32), grad_out=np.ones(B, np.float32),
             d_img=np.zeros_like(sr), ws=np.zeros(max(nb, nbb) // 4 + 8, np.float32), nbytes=nb if fwd else nbb)
    v.update(over)
    a = {n: (x.ctypes.data if isinstance(x, np.ndarray) else x) for n, x in v.items()}
    if fwd:
        return lib.srst_st_forward_per_image(a["sr"], a["hr"], v["B"], v["H"], v["W"], _fp(g), _fp(dg), v["rs"], _fp(k),
                                             v["rk"], 1, 1e-12, a["loss"], a["ds"], None, a["ixy"], None, a["ws"],
                                             v["nbytes"], None)
    return lib.srst_st_backward_per_image(a["ixy"], a["ds"], a["grad_out"], v["B"], v["H"], v["W"], _fp(g), _fp(dg),
                                          v["rs"], _fp(k), v["rk"], a["d_img"], a["ws"], v["nbytes"], None)


def test_st_per_image_contract(lib):
    generic = _taps(1.5, 3.5)
    assert _st_call(lib, True) == 0 and _st_call(lib, False) == 0
    assert _st_call(lib, True, taps=generic) == 0 and _st_call(lib, False, taps=generic) == 0
    for fwd in (True, False):
        for a in (("sr", "loss") if fwd else ("ixy", "ds", "grad_out", "d_img")):
            assert _st_call(lib, fwd, **{a: None}) == E_INVALID, a
        assert _st_call(lib, fwd, B=0) == E_INVALID and _st_call(lib, fwd, H=-1) == E_INVALID
        assert _st_call(lib, fwd, rs=65) == E_UNSUPPORTED
    assert _st_call(lib, True, ws=None) == E_WORKSPACE
    assert _st_call(lib, True, nbytes=16) == E_WORKSPACE
    assert _st_call(lib, True, taps=generic, nbytes=lib.srst_st_workspace_bytes(2, 20, 24)) == E_WORKSPACE
    assert _st_call(lib, False, taps=generic, ws=None) == E_WORKSPACE
    assert _st_call(lib, False, ws=None, nbytes=0) == 0   # compiled classes: the backward needs no workspace


def _patch_call(lib, name, **over):
    B, H, W = 2, 12, 14
    rng = np.random.default_rng(2)
    sr, gt = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    g, dg, k = _taps()
    geom = (4, 1, 2)
    n = max((H // 3) * (W // 3), lib.srst_bbg_num_patches(H, W, *geom))
    nb = max(lib.srst_bb_workspace_bytes(B, H, W), lib.srst_bbg_workspace_bytes(B, H, W, *geom))
    v = dict(mode=2, sr=sr, gt=gt, gt2=None, gt4=None, B=B, H=H, W=W, g=g, dg=dg, rs=len(g) // 2, k=k, rk=len(k) // 2,
             alpha=1.0, beta=0.5, criterion=1 | DIST_L1, idx=np.zeros((B, n), np.int64), loss=np.zeros(B, np.float32),
             grad_out=np.ones(B, np.float32), d_sr=np.zeros_like(sr), d_gt=np.zeros_like(sr),
             ws=np.zeros(nb // 4 + 8, np.float32), nbytes=nb, ksize=geom[0], pad=geom[1], stride=geom[2])
    v.update(over)
    a = {n_: (x.ctypes.data if isinstance(x, np.ndarray) else x) for n_, x in v.items()}
    for t in ("g", "dg", "k"):
        a[t] = _fp(v[t]) if v[t] is not None else None
    if name == "forward":
        return lib.srst_patch_forward_per_image(v["mode"], a["sr"], a["gt"], a["gt2"], a["gt4"], v["B"], v["H"], v["W"], a["g"],
                                                a["dg"], v["rs"], a["k"], v["rk"], v["alpha"], v["beta"], v["criterion"],
                                                a["idx"], a["loss"], a["ws"], v["nbytes"], None)
    if name == "backward":
        return lib.srst_patch_backward_per_image(v["mode"], a["sr"], a["gt"], a["gt2"], a["gt4"], a["idx"], a["grad_out"],
                                                 v["B"], v["H"], v["W"], a["g"], a["dg"], v["rs"], a["k"], v["rk"],
                                                 v["criterion"], a["d_sr"], a["d_gt"], a["ws"], v["nbytes"], None)
    if name == "bbg_forward":
        return lib.srst_bbg_forward_per_image(a["sr"], a["gt"], a["gt2"], a["gt4"], v["B"], v["H"], v["W"], v["ksize"],
                                              v["pad"], v["stride"], v["alpha"], v["beta"], v["criterion"], a["idx"],
                                              a["loss"], a["ws"], v["nbytes"], None)
    return lib.srst_bbg_backward_per_image(a["sr"], a["gt"], a["gt2"], a["gt4"], a["idx"], a["grad_out"], v["B"], v["H"],
                                           v["W"], v["ksize"], v["pad"], v["stride"], v["criterion"], a["d_sr"], a["d_gt"],
                                           a["ws"], v["nbytes"], None)


@pytest.mark.parametrize("name", ["forward", "backward", "bbg_forward", "bbg_backward"])
def test_patch_per_image_contract(lib, name):
    for mode in ((0, 1, 2) if not name.startswith("bbg") else (0,)):
        assert _patch_call(lib, name, mode=mode) == 0, mode
        assert _patch_call(lib, name, mode=mode, criterion=0) == 0, mode
    bad = [({"sr": None}, E_INVALID), ({"gt": None}, E_INVALID), ({"idx": None}, E_INVALID), ({"B": 0}, E_INVALID),
           ({"ws": None}, E_WORKSPACE), ({"nbytes": 256}, E_WORKSPACE), ({"gt2": np.zeros(4, np.float32)}, E_INVALID)]
    bad += [({"criterion": c}, E_INVALID) for c in (2, -1, 2 | DIST_L1, 0x200)]
    bad += [({"loss": None}, E_INVALID)] if "forward" in name else [({"grad_out": None}, E_INVALID),
                                                                     ({"d_sr": None, "d_gt": None}, E_INVALID)]
    if name.startswith("bbg"):
        bad += [({"H": 3}, E_SHAPE), ({"pad": -1}, E_UNSUPPORTED), ({"stride": 0}, E_UNSUPPORTED)]
    else:
        bad += [({"mode": -1}, E_INVALID), ({"mode": 3}, E_INVALID), ({"H": 11}, E_SHAPE), ({"B": 65536}, E_SHAPE),
                ({"g": None}, E_INVALID), ({"rk": 0}, E_INVALID)]
    wrong = [(o, rc, want) for o, want in bad if (rc := _patch_call(lib, name, **o)) != want]
    assert not wrong, f"(bad argument, returned, expected): {wrong}"
    # modes 0 and 1 take no taps
    if not name.startswith("bbg"):
        assert _patch_call(lib, name, mode=0, g=None, dg=None, k=None, rs=0, rk=0) == 0


def test_scalar_entry_points_still_reject_unknown_criterion_bits(lib):
    B, H, W = 1, 12, 12
    sr = np.zeros((B, 3, H, W), np.float32)
    nb = lib.srst_bb_workspace_bytes(B, H, W)
    ws, idx, loss = np.zeros(nb // 4 + 8, np.float32), np.zeros((B, 16), np.int64), np.zeros(1, np.float32)
    assert lib.srst_bb_forward(_p(sr), _p(sr), None, None, B, H, W, 1.0, 1.0, 0x200, _p(idx), _p(loss), _p(ws), nb,
                               None) == E_INVALID


# ---- poison ------------------------------------------------------------------------------------------------------
def _twice(lib, run):
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


def _same(clean, poisoned, keys):
    for key in keys:
        assert clean[key].tobytes() == poisoned[key].tobytes(), key
        assert not np.isnan(clean[key]).any(), key


@pytest.mark.parametrize("case", ["march-chunk", "tiled-ragged", "generic"])
def test_st_per_image_poison(lib, case):
    shape, taps = {"march-chunk": ((2, 40, 100), _taps()), "tiled-ragged": ((3, 21, 30), _taps()),
                   "generic": ((2, 20, 28), _taps(1.5, 3.5))}[case]
    rng = np.random.default_rng(3)
    sr, hr = (rng.random((shape[0], 3, shape[1], shape[2]), dtype=np.float32) for _ in range(2))
    go = rng.uniform(-2, 2, shape[0]).astype(np.float32)
    if case == "march-chunk":
        assert lib.srst_st_force_cfg(3, -1) == 0 and lib.srst_st_force_chunk_blocks(1) == 0
    try:
        clean, poisoned = _twice(lib, lambda: emu_st_per_image(lib, sr, hr, taps, go, want_hr=True))
    finally:
        lib.srst_st_force_cfg(-1, -1)
        lib.srst_st_force_chunk_blocks(0)
    _same(clean, poisoned, ("loss", "d_sr", "d_hr"))


@pytest.mark.parametrize("mode", ["patch", "gram", "pst"])
def test_patch_per_image_poison(lib, mode):
    rng = np.random.default_rng(4)
    sr, gt = (rng.random((2, 3, 24, 26), dtype=np.float32) for _ in range(2))
    go = rng.uniform(-2, 2, 2).astype(np.float32)
    taps = _taps() if mode == "pst" else None
    clean, poisoned = _twice(lib, lambda: emu_patch_per_image(lib, mode, sr, gt, 1 | DIST_L1, go, taps))
    _same(clean, poisoned, ("loss", "idx", "d_sr"))
    assert maxnorm_err(poisoned["d_gt"], clean["d_gt"]) < 1e-6


def test_bbg_per_image_poison(lib):
    rng = np.random.default_rng(5)
    B, H, W, geom = 2, 20, 22, (3, 1, 2)
    sr, gt = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    go = rng.uniform(-2, 2, B).astype(np.float32)
    n, nb = lib.srst_bbg_num_patches(H, W, *geom), lib.srst_bbg_workspace_bytes(B, H, W, *geom)

    def run():
        ws = helpers._workspace(nb)
        out = dict(idx=np.full((B, n), -1, np.int64), loss=np.full(B, np.nan, np.float32), d_sr=np.full_like(sr, np.nan),
                   d_gt=np.full_like(sr, np.nan))
        assert lib.srst_bbg_forward_per_image(_p(sr), _p(gt), None, None, B, H, W, *geom, 1.0, 0.5, 0, _p(out["idx"]),
                                              _p(out["loss"]), _p(ws), nb, None) == 0
        assert lib.srst_bbg_backward_per_image(_p(sr), _p(gt), None, None, _p(out["idx"]), _p(go), B, H, W, *geom, 0,
                                               _p(out["d_sr"]), _p(out["d_gt"]), _p(ws), nb, None) == 0
        return out

    clean, poisoned = _twice(lib, run)
    _same(clean, poisoned, ("loss", "idx", "d_sr"))
    assert maxnorm_err(poisoned["d_gt"], clean["d_gt"]) < 1e-6
