"""CPU: the per-patch loss map entry points of include/srst.h (srst_patch_forward_map / srst_patch_backward_map and the
arbitrary-geometry srst_bbg_forward_map / srst_bbg_backward_map), run on the emulation library.

For the three patch losses with both search norms and both criteria, and for the Best-Buddy geometries of the golden
fixtures (k2p0s3, k3p1s1, k4p1s2, k5p0s5), on shapes with H % 3 != 0 and W % 3 != 0:
  * the map matches the float64 restatement built from the returned indices (max-norm 1e-5) and averages to loss_out;
  * idx and loss_out are bit-identical to the scalar forward;
  * d_sr and d_gt under a random signed grad_map match the float64 backward restatements with that per-patch weight
    (max-norm 1e-4);
  * a constant grad_map gives the scalar backward, and a per-image-constant one the per-image backward (1e-6).
Then the argument contract of the four entry points, and 0xFF-poisoned outputs, workspaces and shared memory."""
import numpy as np
import pytest

from oracle import st_oracle as O
from tests import patch_map_ref as R
from tests.helpers import _fp, _p, emu_bb, emu_bbg, emu_lib, emu_patch_gt, maxnorm_err, rel_err

E_INVALID, E_WORKSPACE = -1, -3
DIST_L1 = 0x100   # SRST_BB_DIST_L1
MODES = {"patch": 0, "gram": 1, "pst": 2}
POISON = 0xFF


@pytest.fixture(scope="module")
def lib():
    lib = emu_lib()
    assert lib.srst_emu_set_poison(0xCD) == 0xCD
    yield lib
    lib.srst_emu_set_poison(0xCD)


def _taps():
    return tuple(np.ascontiguousarray(t, np.float32) for t in (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0)))


def _tp(taps):
    return (_fp(taps[0]), _fp(taps[1]), len(taps[0]) // 2, _fp(taps[2]), len(taps[2]) // 2) if taps else (None, None, 0, None, 0)


def _ws(nbytes, fill=None):
    ws = np.zeros(nbytes // 4 + 4, np.float32)
    if fill is not None:
        ws.view(np.uint8)[16:] = fill   # all but the 16-byte ticket header, which srst.h requires to be zero
    return ws


def _out(shape, fill):
    a = np.empty(shape, np.float32)
    a.view(np.uint8)[...] = fill
    return a


class Patch:
    """srst_patch_*_map (geom None) or srst_bbg_*_map (geom = (ksize, pad, stride)) on host arrays."""

    def __init__(self, lib, mode, sr, gt, crit, taps=None, geom=None):
        self.lib, self.mode, self.sr, self.gt, self.crit, self.taps, self.geom = lib, mode, sr, gt, crit, taps, geom
        B, _, H, W = sr.shape
        self.shape = (B, H, W)
        if geom is None:
            self.N = (H // 3) * (W // 3)
            self.nbytes = lib.srst_bb_workspace_bytes(B, H, W)
        else:
            self.N = lib.srst_bbg_num_patches(H, W, *geom)
            self.nbytes = lib.srst_bbg_workspace_bytes(B, H, W, *geom)

    def forward(self, fill=0xCD, ws_fill=None, ws=None):
        B, H, W = self.shape
        ws = _ws(self.nbytes, ws_fill) if ws is None else ws
        idx = np.full((B, self.N), -1, np.int64)
        loss, m = _out(1, fill), _out((B, self.N), fill)
        if self.geom is None:
            rc = self.lib.srst_patch_forward_map(MODES[self.mode], _p(self.sr), _p(self.gt), None, None, B, H, W,
                                                 *_tp(self.taps), 1.0, 0.5, self.crit, _p(idx), _p(loss), _p(m), _p(ws),
                                                 self.nbytes, None)
        else:
            rc = self.lib.srst_bbg_forward_map(_p(self.sr), _p(self.gt), None, None, B, H, W, *self.geom, 1.0, 0.5,
                                               self.crit, _p(idx), _p(loss), _p(m), _p(ws), self.nbytes, None)
        assert rc == 0, rc
        assert np.all(ws[:4] == 0)   # the ticket is handed back zeroed
        return dict(idx=idx, loss=loss, map=m)

    def backward(self, idx, grad_map, fill=0xCD, ws_fill=None, per_image=False):
        B, H, W = self.shape
        ws = _ws(self.nbytes, ws_fill)
        go = np.ascontiguousarray(grad_map, np.float32)
        d_sr, d_gt = _out(self.sr.shape, fill), _out(self.sr.shape, fill)
        if self.geom is None:
            fn = self.lib.srst_patch_backward_per_image if per_image else self.lib.srst_patch_backward_map
            rc = fn(MODES[self.mode], _p(self.sr), _p(self.gt), None, None, _p(idx), _p(go), B, H, W, *_tp(self.taps),
                    self.crit, _p(d_sr), _p(d_gt), _p(ws), self.nbytes, None)
        else:
            fn = self.lib.srst_bbg_backward_per_image if per_image else self.lib.srst_bbg_backward_map
            rc = fn(_p(self.sr), _p(self.gt), None, None, _p(idx), _p(go), B, H, W, *self.geom, self.crit, _p(d_sr),
                    _p(d_gt), _p(ws), self.nbytes, None)
        assert rc == 0, rc
        return d_sr, d_gt


def _check(run, ref_map, ref_grads, scalar, scalar_gt):
    """The checks every case shares.  ref_map(idx), ref_grads(idx, w): float64 references; scalar(grad_out): the
    scalar entry points' (loss, idx, d_sr); scalar_gt(idx, grad_out): their d_gt."""
    B = run.shape[0]
    N = run.N
    f = run.forward()
    loss, idx, d_sr1 = scalar(1.0)
    assert f["idx"].tobytes() == idx.tobytes()
    assert f["loss"][0] == np.float32(loss)                       # bit-identical: same kernels, same reduction order
    assert maxnorm_err(f["map"], ref_map(f["idx"])) < 1e-5
    assert rel_err(float(np.mean(f["map"].astype(np.float64))), float(f["loss"][0])) < 1e-6
    rng = np.random.default_rng(B * N)
    w = rng.uniform(-2.0, 2.0, (B, N)).astype(np.float32)
    d_sr, d_gt = run.backward(f["idx"], w)
    r_sr, r_gt = ref_grads(f["idx"], w)
    assert maxnorm_err(d_sr, r_sr) < 1e-4
    assert maxnorm_err(d_gt, r_gt) < 1e-4
    # constant grad_map = 1/(B N): the gradient of map.mean(), i.e. of the scalar loss with grad_out = 1
    d_sr, d_gt = run.backward(f["idx"], np.full((B, N), 1.0 / (B * N), np.float32))
    assert maxnorm_err(d_sr, d_sr1) < 1e-6
    assert maxnorm_err(d_gt, scalar_gt(f["idx"], 1.0)) < 1e-6
    # per-image-constant grad_map g[b] / N: the per-image backward with grad_out = g
    g = rng.uniform(-2.0, 2.0, B).astype(np.float32)
    d_sr, d_gt = run.backward(f["idx"], np.repeat((g / np.float32(N))[:, None], N, 1))
    p_sr, p_gt = run.backward(f["idx"], g, per_image=True)
    assert maxnorm_err(d_sr, p_sr) < 1e-6
    assert maxnorm_err(d_gt, p_gt) < 1e-6


@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("dist_norm", ["l2", "l1"])
@pytest.mark.parametrize("criterion", ["l1", "l2"])
def test_patch_map(lib, mode, dist_norm, criterion):
    # W % 3 != 0 for criterion l1, H % 3 != 0 and W % 3 != 0 for l2
    B, H, W = (3, 24, 28) if criterion == "l1" else (2, 26, 25)
    rng = np.random.default_rng(len(mode) + 3 * len(dist_norm) + (criterion == "l2"))
    sr, gt = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    taps = _taps() if mode == "pst" else None
    crit = (0 if criterion == "l1" else 1) | (DIST_L1 if dist_norm == "l1" else 0)
    run = Patch(lib, mode, sr, gt, crit, taps)

    def scalar(grad_out):
        o = emu_bb(lib, sr, gt, alpha=1.0, beta=0.5, criterion=crit, grad_out=grad_out, mode=mode, taps=taps)
        return o["loss"], o["idx"], o["d_sr"]

    _check(run, lambda idx: R.patch_map(sr, gt, idx, mode, taps, criterion),
           lambda idx, w: R.patch_grads(sr, gt, idx, w, mode, taps, criterion), scalar,
           lambda idx, go: emu_patch_gt(lib, sr, gt, idx, criterion=crit, grad_out=go, mode=mode, taps=taps))


# the geometries of the golden fixtures tests/golden/bbg_*.npz
@pytest.mark.parametrize("geom,criterion,dist_norm", [((2, 0, 3), "l1", "l2"), ((3, 1, 1), "l2", "l2"),
                                                      ((4, 1, 2), "l1", "l1"), ((5, 0, 5), "l2", "l1")])
def test_bbg_map(lib, geom, criterion, dist_norm):
    B, H, W = 2, 22, 25   # H % 3 != 0, W % 3 != 0; the x1/4 level holds a 5x5 patch
    rng = np.random.default_rng(sum(geom))
    sr, gt = (rng.random((B, 3, H, W), dtype=np.float32) for _ in range(2))
    crit = (0 if criterion == "l1" else 1) | (DIST_L1 if dist_norm == "l1" else 0)
    run = Patch(lib, "patch", sr, gt, crit, geom=geom)
    gt2, gt4 = R.BO.pyramid_c(gt)

    def scalar(grad_out):
        o = emu_bbg(lib, sr, gt, *geom, alpha=1.0, beta=0.5, criterion=crit, grad_out=grad_out)
        return o["loss"], o["idx"], o["d_sr"]

    def scalar_gt(idx, grad_out):
        return emu_bbg(lib, sr, gt, *geom, alpha=1.0, beta=0.5, criterion=crit, grad_out=grad_out, want_gt=True)["d_gt"]

    _check(run, lambda idx: R.bbg_map(sr, gt, idx, *geom, criterion, gt2, gt4),
           lambda idx, w: R.bbg_grads(sr, gt, idx, *geom, criterion, w), scalar, scalar_gt)


# ---- argument contract -------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def small(lib):
    rng = np.random.default_rng(3)
    sr, gt = (rng.random((2, 3, 12, 14), dtype=np.float32) for _ in range(2))
    return sr, gt


@pytest.mark.parametrize("geom", [None, (4, 1, 2)])
def test_map_argument_contract(lib, small, geom):
    sr, gt = small
    taps = _taps()
    run = Patch(lib, "pst" if geom is None else "patch", sr, gt, 1, taps if geom is None else None, geom)
    B, H, W = run.shape
    f = run.forward()
    idx, go = f["idx"], np.ones((B, run.N), np.float32)
    ws = _ws(run.nbytes)
    loss, m, d_sr, d_gt = np.zeros(1, np.float32), np.zeros((B, run.N), np.float32), np.zeros_like(sr), np.zeros_like(sr)

    if geom is None:
        def fwd(m_, nbytes=run.nbytes, mode=2):
            return lib.srst_patch_forward_map(mode, _p(sr), _p(gt), None, None, B, H, W, *_tp(taps), 1.0, 0.5, 1, _p(idx),
                                              _p(loss), _p(m_), _p(ws), nbytes, None)

        def bwd(g_, a, b, nbytes=run.nbytes, mode=2):
            return lib.srst_patch_backward_map(mode, _p(sr), _p(gt), None, None, _p(idx), _p(g_), B, H, W, *_tp(taps), 1,
                                               _p(a), _p(b), _p(ws), nbytes, None)
    else:
        def fwd(m_, nbytes=run.nbytes, mode=None):
            return lib.srst_bbg_forward_map(_p(sr), _p(gt), None, None, B, H, W, *geom, 1.0, 0.5, 1, _p(idx), _p(loss),
                                            _p(m_), _p(ws), nbytes, None)

        def bwd(g_, a, b, nbytes=run.nbytes, mode=None):
            return lib.srst_bbg_backward_map(_p(sr), _p(gt), None, None, _p(idx), _p(g_), B, H, W, *geom, 1, _p(a), _p(b),
                                             _p(ws), nbytes, None)

    assert fwd(m) == 0 and bwd(go, d_sr, d_gt) == 0 and bwd(go, d_sr, None) == 0 and bwd(go, None, d_gt) == 0
    assert fwd(None) == E_INVALID                       # map_out is required
    assert bwd(None, d_sr, d_gt) == E_INVALID           # grad_map is required
    assert bwd(go, None, None) == E_INVALID             # at least one output
    assert fwd(m, nbytes=run.nbytes - 256) == E_WORKSPACE
    assert bwd(go, d_sr, d_gt, nbytes=run.nbytes - 256) == E_WORKSPACE
    if geom is None:
        assert fwd(m, mode=3) == E_INVALID and bwd(go, d_sr, d_gt, mode=-1) == E_INVALID
        assert lib.srst_patch_forward_map(0, _p(sr), _p(gt), None, None, B, H, W, None, None, 0, None, 0, 1.0, 0.5, 1,
                                          _p(idx), _p(loss), _p(m), _p(ws), run.nbytes, None) == 0   # taps: mode 2 only


# ---- poisoned memory -----------------------------------------------------------------------------------------------
@pytest.mark.parametrize("mode,geom", [("patch", None), ("gram", None), ("pst", None), ("patch", (3, 1, 1))])
def test_map_poisoned_memory(lib, mode, geom):
    """0xFF (NaN) in map_out, d_sr, d_gt, the workspace past its ticket header and shared memory: the same bits for the
    loss, the indices, the map and d_sr; d_gt (summed with atomics) without NaN and within 1e-6."""
    rng = np.random.default_rng(17)
    sr, gt = (rng.random((2, 3, 24, 28), dtype=np.float32) for _ in range(2))
    run = Patch(lib, mode, sr, gt, 0, _taps() if mode == "pst" else None, geom)
    w = rng.uniform(-1.0, 1.0, (2, run.N)).astype(np.float32)
    clean = run.forward(fill=0)
    c_sr, c_gt = run.backward(clean["idx"], w, fill=0)
    lib.srst_emu_set_poison(POISON)
    try:
        bad = run.forward(fill=POISON, ws_fill=POISON)
        b_sr, b_gt = run.backward(bad["idx"], w, fill=POISON, ws_fill=POISON)
    finally:
        lib.srst_emu_set_poison(0xCD)
    for k in ("idx", "loss", "map"):
        assert bad[k].tobytes() == clean[k].tobytes(), k
    assert b_sr.tobytes() == c_sr.tobytes()
    assert not np.isnan(b_gt).any() and maxnorm_err(b_gt, c_gt) < 1e-6
