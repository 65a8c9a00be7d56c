"""CPU: the argument contract of the patch-loss entry points of include/srst.h (Best-Buddy, Gram, PatchwiseST, their
gradient w.r.t. gt and the arbitrary-geometry Best-Buddy), run on the emulation library.

Every argument that is bad on its own gets the code the entry point documents for it; which code wins when several
arguments are bad is not part of srst.h and is not tested.  The good call each case starts from succeeds, so a
rejection cannot come from another argument.  The backward entry points need no workspace when the caller passes
the pyramid levels."""
import ctypes

import numpy as np
import pytest

from oracle import st_oracle as O
from tests.helpers import emu_lib

E_INVALID, E_UNSUPPORTED, E_WORKSPACE, E_SHAPE = -1, -2, -3, -4
DIST_L1 = 0x100   # SRST_BB_DIST_L1
B, H, W = 2, 12, 14   # W % 3 != 0: the Gram and PatchwiseST backward zero-fill d_sr before their per-patch kernel
GEOM = dict(ksize=4, pad=1, stride=2)   # a non-default geometry for the srst_bbg_* entry points

# argument lists in the order of include/srst.h; "ws" is the workspace pointer, "nbytes" its size
SIG = {
    "srst_bb_forward": "sr gt gt2 gt4 B H W alpha beta criterion idx loss ws nbytes stream",
    "srst_gram_forward": "sr gt gt2 gt4 B H W alpha beta criterion idx loss ws nbytes stream",
    "srst_pst_forward": "sr gt gt2 gt4 B H W g dg rs k rk alpha beta criterion idx loss ws nbytes stream",
    "srst_bb_backward": "sr gt gt2 gt4 idx grad_out B H W criterion d_sr ws nbytes stream",
    "srst_gram_backward": "sr gt gt2 gt4 idx grad_out B H W criterion d_sr ws nbytes stream",
    "srst_pst_backward": "sr gt gt2 gt4 idx grad_out B H W g dg rs k rk criterion d_sr ws nbytes stream",
    "srst_patch_backward_gt": "mode sr gt gt2 gt4 idx grad_out B H W g dg rs k rk criterion d_gt ws nbytes stream",
    "srst_bbg_forward": "sr gt gt2 gt4 B H W ksize pad stride alpha beta criterion idx loss ws nbytes stream",
    "srst_bbg_backward": "sr gt gt2 gt4 idx grad_out B H W ksize pad stride criterion d_sr d_gt ws nbytes stream",
}
TAP_ARGS = ("g", "dg", "k")
NO_TAPS = dict(g=None, dg=None, rs=0, k=None, rk=0)
# entry point id -> (symbol, overrides of the good call)
ENTRIES = {
    "bb_forward": ("srst_bb_forward", {}),
    "gram_forward": ("srst_gram_forward", {}),
    "pst_forward": ("srst_pst_forward", {}),
    "bb_backward": ("srst_bb_backward", {}),
    "gram_backward": ("srst_gram_backward", {}),
    "pst_backward": ("srst_pst_backward", {}),
    "patch_backward_gt_0": ("srst_patch_backward_gt", dict(mode=0, **NO_TAPS)),
    "patch_backward_gt_1": ("srst_patch_backward_gt", dict(mode=1, **NO_TAPS)),
    "patch_backward_gt_2": ("srst_patch_backward_gt", dict(mode=2)),
    "bbg_forward": ("srst_bbg_forward", {}),
    "bbg_backward": ("srst_bbg_backward", {}),
}
DEFAULT_GEOMETRY = [e for e in ENTRIES if not e.startswith("bbg")]


@pytest.fixture(scope="module")
def env():
    lib = emu_lib()
    rng = np.random.default_rng(7)
    sr, gt = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    pyr2 = np.zeros((B, 3, H // 2, W // 2), np.float32)
    pyr4 = np.zeros((B, 3, H // 4, W // 4), np.float32)
    assert lib.srst_bb_pyramid(sr.ctypes.data, B, H, W, pyr2.ctypes.data, pyr4.ctypes.data, None) == 0
    g, dg = O.gaussian_taps(0.5, True)
    k = O.gaussian_taps(2.0)
    # ksize 1 at stride 1 has the most patches of any geometry at this shape: idx and the workspace fit every case
    nbytes = max(lib.srst_bb_workspace_bytes(B, H, W), lib.srst_bbg_workspace_bytes(B, H, W, 1, 0, 1))
    n = lib.srst_bbg_num_patches(H, W, 1, 0, 1)
    good = dict(sr=sr, gt=gt, gt2=None, gt4=None, B=B, H=H, W=W, alpha=1.0, beta=0.5, criterion=1 | DIST_L1,
                g=np.ascontiguousarray(g, np.float32), dg=np.ascontiguousarray(dg, np.float32), rs=len(g) // 2,
                k=np.ascontiguousarray(k, np.float32), rk=len(k) // 2, idx=np.zeros((B, n), np.int64),
                loss=np.zeros(1, np.float32), grad_out=np.ones(1, np.float32), d_sr=np.zeros_like(sr),
                d_gt=np.zeros_like(sr), ws=np.zeros(nbytes // 4 + 4, np.float32), nbytes=nbytes, stream=None, mode=0,
                **GEOM)
    return lib, good, pyr2, pyr4


def _call(env, entry, **over):
    lib, good, _, _ = env
    name, fixed = ENTRIES[entry]
    v = {**good, **fixed, **over}
    args = []
    for a in SIG[name].split():
        x = v[a]
        if isinstance(x, np.ndarray):
            x = x.ctypes.data_as(ctypes.POINTER(ctypes.c_float)) if a in TAP_ARGS else x.ctypes.data
        args.append(x)
    return getattr(lib, name)(*args)


def _bad_args(entry, pyr2, pyr4, misaligned):
    """(overrides, expected code) for every argument of `entry` that is bad on its own."""
    name = ENTRIES[entry][0]
    sig = SIG[name].split()
    out = [({a: None}, E_INVALID) for a in ("sr", "gt", "idx", "loss", "grad_out", "d_sr", "d_gt") if a in sig]
    out += [({"B": 0}, E_INVALID), ({"B": -1}, E_INVALID)]
    out += [({"criterion": c}, E_INVALID) for c in (2, -1, 2 | DIST_L1, 0x200)]
    out += [({"gt2": pyr2}, E_INVALID), ({"gt4": pyr4}, E_INVALID)]
    out += [({"ws": None}, E_WORKSPACE), ({"ws": misaligned}, E_WORKSPACE)]
    if name == "srst_bbg_backward":   # either gradient may be left out, not both
        out = [c for c in out if c[0] not in ({"d_sr": None}, {"d_gt": None})] + [({"d_sr": None, "d_gt": None}, E_INVALID)]
    if name.startswith("srst_bbg"):
        out += [({"B": 65536}, E_SHAPE), ({"H": 3}, E_SHAPE), ({"W": 3}, E_SHAPE),
                ({"ksize": 4, "pad": 0, "stride": 1}, E_SHAPE),   # the x1/4 level (3x3) holds no 4x4 patch
                ({"pad": -1}, E_UNSUPPORTED), ({"stride": 0}, E_UNSUPPORTED)]
        if name == "srst_bbg_backward":   # test_bb_geometry.py::test_entry_points_reject_unusable_geometry has these
            out += [({"ksize": 9}, E_UNSUPPORTED), ({"nbytes": 256}, E_WORKSPACE)]   # for the forward
        return out
    out += [({"B": 65536}, E_SHAPE), ({"H": 11}, E_SHAPE), ({"W": 11}, E_SHAPE), ({"nbytes": 256}, E_WORKSPACE)]
    if "g" in sig and entry != "patch_backward_gt_0" and entry != "patch_backward_gt_1":
        out += [({a: None}, E_INVALID) for a in TAP_ARGS]
        out += [({"rs": 0}, E_INVALID), ({"rk": 0}, E_INVALID), ({"rs": 4097}, E_INVALID), ({"rk": 4097}, E_INVALID)]
    if name == "srst_patch_backward_gt":
        out += [({"mode": -1}, E_INVALID), ({"mode": 3}, E_INVALID)]
    return out


@pytest.mark.parametrize("entry", list(ENTRIES))
def test_good_call_succeeds(env, entry):
    assert _call(env, entry) == 0
    _, _, pyr2, pyr4 = env
    assert _call(env, entry, gt2=pyr2, gt4=pyr4, criterion=0) == 0


@pytest.mark.parametrize("entry", list(ENTRIES))
def test_each_bad_argument_gets_its_code(env, entry):
    _, good, pyr2, pyr4 = env
    misaligned = good["ws"].ctypes.data + 4
    got = [(over, _call(env, entry, **over), want) for over, want in _bad_args(entry, pyr2, pyr4, misaligned)]
    wrong = [(over, rc, want) for over, rc, want in got if rc != want]
    assert not wrong, f"(bad argument, returned, expected): {wrong}"


@pytest.mark.parametrize("entry", ["bbg_forward", "bbg_backward"])
def test_bbg_accepts_images_down_to_4x4(env, entry):
    """Unlike the default-geometry entry points (H, W >= 12), any shape whose three pyramid levels hold a patch."""
    assert _call(env, entry, H=4, W=4, ksize=1, pad=0, stride=1) == 0
    assert _call(env, entry, H=4, W=5, ksize=1, pad=0, stride=1) == 0
    assert _call(env, entry, H=12, W=12, ksize=3, pad=0, stride=1) == 0


@pytest.mark.parametrize("entry", ["bb_backward", "gram_backward", "pst_backward"])
def test_backward_needs_no_workspace_when_given_the_pyramid(env, entry):
    """srst.h asks for the workspace to hold gt2 / gt4 only when the library builds them: with both given, a NULL
    workspace gives the same d_sr, bit for bit, as a call with one."""
    _, good, pyr2, pyr4 = env
    fwd = entry.replace("backward", "forward")
    idx = np.full_like(good["idx"], -1)
    assert _call(env, fwd, gt2=pyr2, gt4=pyr4, idx=idx) == 0
    d_ws, d_none = np.full_like(good["sr"], np.nan), np.full_like(good["sr"], np.nan)
    assert _call(env, entry, gt2=pyr2, gt4=pyr4, idx=idx, d_sr=d_ws) == 0
    assert _call(env, entry, gt2=pyr2, gt4=pyr4, idx=idx, d_sr=d_none, ws=None, nbytes=0) == 0
    assert not np.isnan(d_ws).any()
    assert d_ws.tobytes() == d_none.tobytes()
