"""Shared test helpers: golden fixtures, error metrics, the test-only host emulation library."""
import ctypes
import glob
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
EMU_DIR = os.path.join(ROOT, "tests", "emu")
EMU_LIB = os.path.join(EMU_DIR, "_build", "libsrst_emu.so")
CSRC = os.path.join(ROOT, "srgan_st_b200", "csrc")


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


def golden_names(prefix, suffix=""):
    """Fixture names starting with `prefix`; the `_dgt` companions (gradient w.r.t. gt only) are listed on request."""
    names = sorted(os.path.basename(p)[:-4] for p in glob.glob(os.path.join(GOLDEN, prefix + "*" + suffix + ".npz")))
    return [n for n in names if suffix or not n.endswith("_dgt")]


def rel_err(x, ref):
    """|x - ref| / |ref| for scalars."""
    return abs(float(x) - float(ref)) / max(abs(float(ref)), 1e-30)


def maxnorm_err(x, ref):
    """max|x - ref| / max|ref|: the gradient metric of SURVEY.md section 8(c)."""
    x = np.asarray(x, dtype=np.float64)
    ref = np.asarray(ref, dtype=np.float64)
    return float(np.abs(x - ref).max() / max(np.abs(ref).max(), 1e-30))


def emu_lib():
    """Build (if stale) and load the host emulation of the kernels.  TEST-ONLY: same sources as
    libsrst.so compiled with g++ -DSRST_EMULATE; it lets the CPU suite execute the kernels' index
    logic.  The product package never loads this."""
    from srgan_st_b200 import _cabi
    ld = os.path.join(EMU_DIR, "shared.ld")   # gathers the kernels' static __shared__ arrays for the poison fill
    srcs = [os.path.join(CSRC, f) for f in os.listdir(CSRC)] + [os.path.join(EMU_DIR, "cuda_emu.h"), ld,
                                                                os.path.join(ROOT, "include", "srst.h")]
    stale = (not os.path.exists(EMU_LIB)) or any(os.path.getmtime(s) > os.path.getmtime(EMU_LIB) for s in srcs)
    if stale:
        os.makedirs(os.path.dirname(EMU_LIB), exist_ok=True)
        cmd = ["g++", "-x", "c++", "-std=c++20", "-O2", "-DSRST_EMULATE", "-fdata-sections", "-I" + EMU_DIR, "-I" + CSRC,
               "-shared", "-fPIC", "-pthread", "-Wl,-T," + ld, "-o", EMU_LIB, os.path.join(CSRC, "srst_cabi.cu")]
        subprocess.run(cmd, check=True, capture_output=True)
    lib = _cabi.bind(EMU_LIB)
    lib.srst_emu_set_poison.restype = ctypes.c_int
    lib.srst_emu_set_poison.argtypes = [ctypes.c_int]
    return lib


# Fill of the workspaces the emu_* helpers below hand to the kernels: None = all zeros; a byte value = that byte
# everywhere but the 16-byte ticket header, which is all srst.h promises to be zero (tests/test_emu_poison.py).
WORKSPACE_FILL = None
FILLED_WORKSPACES = []   # every workspace filled that way, for checks that the ticket header came back zeroed


def _workspace(nbytes):
    ws = np.zeros(nbytes // 4 + 4, np.float32)
    if WORKSPACE_FILL is not None:
        ws.view(np.uint8)[16:] = WORKSPACE_FILL
        FILLED_WORKSPACES.append(ws)
    return ws


def _p(a):
    return ctypes.c_void_p(a.ctypes.data) if a is not None else None


def _fp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_float))


def emu_st(lib, sr, hr, taps, normalize=True, want_hr=False, grad_out=1.0):
    """Run srst_st_forward + srst_st_backward of `lib` on host arrays (emulation library only)."""
    sr = np.ascontiguousarray(sr, np.float32)
    hr = np.ascontiguousarray(hr, np.float32)
    B, _, H, W = sr.shape
    g, dg, k = [np.ascontiguousarray(t, np.float32) for t in taps]
    rs, rk = len(g) // 2, len(k) // 2
    generic = lib.srst_st_supported(rs, rk) == 2   # radii beyond the compiled classes: scratch planes in the workspace
    nb = lib.srst_st_workspace_bytes_r(B, H, W, rs, rk)
    assert nb >= lib.srst_st_workspace_bytes(B, H, W) and (generic or nb == lib.srst_st_workspace_bytes(B, H, W))
    ws = _workspace(nb)
    nbb = lib.srst_st_backward_workspace_bytes(B, H, W, rs, rk)
    assert (nbb > 0) == generic
    bws = np.full(nbb // 4 + 4, np.nan, np.float32)
    loss = np.zeros(1, np.float32)
    n_ixy = lib.srst_st_ixy_floats(B, H, W)
    ds_sr = np.full_like(sr, np.nan)
    ds_hr = np.full_like(sr, np.nan) if want_hr else None
    ixy_sr = np.full(n_ixy, np.nan, np.float32)
    ixy_hr = np.full(n_ixy, np.nan, np.float32) if want_hr else None
    rc = lib.srst_st_forward(_p(sr), _p(hr), B, H, W, _fp(g), _fp(dg), len(g) // 2, _fp(k), len(k) // 2,
                             int(normalize), 1e-12, _p(loss), _p(ds_sr), _p(ds_hr), _p(ixy_sr), _p(ixy_hr), _p(ws), nb,
                             None)
    assert rc == 0, rc
    go = np.full(1, grad_out, np.float32)
    # only the ticket header of the workspace is promised to come back zeroed (the generic path's planes are scratch)
    out = dict(loss=float(loss[0]), ds_sr=ds_sr, ws=ws[:lib.srst_st_workspace_bytes(B, H, W) // 4] if not generic else ws[:4],
               ixy_sr=ixy_sr.reshape(B, 2, (H + 1) // 2, W, 2))

    def backward(ixy, ds):
        d = np.full_like(sr, np.nan)
        if generic:
            assert lib.srst_st_backward(_p(ixy), _p(ds), _p(go), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, _p(d), None) == -3
            rc = lib.srst_st_backward_ws(_p(ixy), _p(ds), _p(go), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, _p(d), _p(bws),
                                         nbb, None)
        else:
            rc = lib.srst_st_backward(_p(ixy), _p(ds), _p(go), B, H, W, _fp(g), _fp(dg), rs, _fp(k), rk, _p(d), None)
        assert rc == 0, rc
        return d

    out["d_sr"] = backward(ixy_sr, ds_sr)
    if want_hr:
        out["d_hr"] = backward(ixy_hr, ds_hr)
    return out


def emu_bb(lib, sr, gt, gt2=None, gt4=None, alpha=1.0, beta=1.0, criterion=0, grad_out=1.0, mode="patch", taps=None):
    """Run srst_bb_forward + srst_bb_backward of `lib` on host arrays (emulation library only).
    mode: "patch" (BestBuddyLoss), "gram" (GramLoss) or "pst" (PatchwiseStructureTensorLoss, taps = (g, dg, k))."""
    sr = np.ascontiguousarray(sr, np.float32)
    gt = np.ascontiguousarray(gt, np.float32)
    gt2 = np.ascontiguousarray(gt2, np.float32) if gt2 is not None else None
    gt4 = np.ascontiguousarray(gt4, np.float32) if gt4 is not None else None
    B, _, H, W = sr.shape
    N = (H // 3) * (W // 3)
    nb = lib.srst_bb_workspace_bytes(B, H, W)
    ws = _workspace(nb)
    idx = np.full((B, N), -1, np.int64)
    loss = np.zeros(1, np.float32)
    go = np.full(1, grad_out, np.float32)
    d_sr = np.full_like(sr, np.nan)
    if mode == "pst":
        g, dg, k = [np.ascontiguousarray(t, np.float32) for t in taps]
        tp = (_fp(g), _fp(dg), len(g) // 2, _fp(k), len(k) // 2)
        rc = lib.srst_pst_forward(_p(sr), _p(gt), _p(gt2), _p(gt4), B, H, W, *tp, alpha, beta, criterion, _p(idx),
                                  _p(loss), _p(ws), nb, None)
        assert rc == 0, rc
        rc = lib.srst_pst_backward(_p(sr), _p(gt), _p(gt2), _p(gt4), _p(idx), _p(go), B, H, W, *tp, criterion, _p(d_sr),
                                   _p(ws), nb, None)
        assert rc == 0, rc
        return dict(loss=float(loss[0]), idx=idx, d_sr=d_sr)
    fwd = lib.srst_bb_forward if mode == "patch" else lib.srst_gram_forward
    bwd = lib.srst_bb_backward if mode == "patch" else lib.srst_gram_backward
    rc = fwd(_p(sr), _p(gt), _p(gt2), _p(gt4), B, H, W, alpha, beta, criterion, _p(idx), _p(loss), _p(ws), nb, None)
    assert rc == 0, rc
    rc = bwd(_p(sr), _p(gt), _p(gt2), _p(gt4), _p(idx), _p(go), B, H, W, criterion, _p(d_sr), _p(ws), nb, None)
    assert rc == 0, rc
    return dict(loss=float(loss[0]), idx=idx, d_sr=d_sr)


def emu_stpx(lib, sr, hr, taps, grad_st=1.0, grad_px=1.0):
    """Run srst_stpx_forward + srst_stpx_backward of `lib` on host arrays (emulation library only)."""
    sr = np.ascontiguousarray(sr, np.float32)
    hr = np.ascontiguousarray(hr, np.float32)
    B, _, H, W = sr.shape
    g, dg, k = [np.ascontiguousarray(t, np.float32) for t in taps]
    nb = lib.srst_st_workspace_bytes(B, H, W)
    ws = _workspace(nb)
    both = np.zeros(2, np.float32)
    ds_sr = np.full_like(sr, np.nan)
    ixy_sr = np.full(lib.srst_st_ixy_floats(B, H, W), np.nan, np.float32)
    rc = lib.srst_stpx_forward(_p(sr), _p(hr), B, H, W, _fp(g), _fp(dg), len(g) // 2, _fp(k), len(k) // 2, 1, 1e-12,
                               _p(both), _p(ds_sr), _p(ixy_sr), _p(ws), nb, None)
    assert rc == 0, rc
    gs, gp = np.full(1, grad_st, np.float32), np.full(1, grad_px, np.float32)
    d_sr = np.full_like(sr, np.nan)
    rc = lib.srst_stpx_backward(_p(sr), _p(hr), _p(ixy_sr), _p(ds_sr), _p(gs), _p(gp), B, H, W, _fp(g), _fp(dg),
                                len(g) // 2, _fp(k), len(k) // 2, _p(d_sr), None)
    assert rc == 0, rc
    return dict(st=float(both[0]), px=float(both[1]), d_sr=d_sr, ws=ws)


def emu_patch_gt(lib, sr, gt, idx, gt2=None, gt4=None, criterion=0, grad_out=1.0, mode="patch", taps=None):
    """Run srst_patch_backward_gt of `lib` on host arrays (emulation library only): d loss / d gt."""
    sr = np.ascontiguousarray(sr, np.float32)
    gt = np.ascontiguousarray(gt, np.float32)
    gt2 = np.ascontiguousarray(gt2, np.float32) if gt2 is not None else None
    gt4 = np.ascontiguousarray(gt4, np.float32) if gt4 is not None else None
    idx = np.ascontiguousarray(idx, np.int64)
    B, _, H, W = sr.shape
    nb = lib.srst_bb_workspace_bytes(B, H, W)
    ws = _workspace(nb)
    go = np.full(1, grad_out, np.float32)
    d_gt = np.full_like(gt, np.nan)
    if taps is not None:
        g, dg, k = [np.ascontiguousarray(t, np.float32) for t in taps]
        tp = (_fp(g), _fp(dg), len(g) // 2, _fp(k), len(k) // 2)
    else:
        tp = (None, None, 0, None, 0)
    rc = lib.srst_patch_backward_gt({"patch": 0, "gram": 1, "pst": 2}[mode], _p(sr), _p(gt), _p(gt2), _p(gt4), _p(idx), _p(go),
                                    B, H, W, *tp, criterion, _p(d_gt), _p(ws), nb, None)
    assert rc == 0, rc
    return d_gt


def emu_bbg(lib, sr, gt, ksize, pad, stride, gt2=None, gt4=None, alpha=1.0, beta=1.0, criterion=0, grad_out=1.0,
            want_gt=False):
    """Run srst_bbg_forward + srst_bbg_backward (arbitrary patch geometry) of `lib` on host arrays (emulation only)."""
    sr = np.ascontiguousarray(sr, np.float32)
    gt = np.ascontiguousarray(gt, np.float32)
    gt2 = np.ascontiguousarray(gt2, np.float32) if gt2 is not None else None
    gt4 = np.ascontiguousarray(gt4, np.float32) if gt4 is not None else None
    B, _, H, W = sr.shape
    N = lib.srst_bbg_num_patches(H, W, ksize, pad, stride)
    nb = lib.srst_bbg_workspace_bytes(B, H, W, ksize, pad, stride)
    assert N > 0 and nb > 0
    ws = _workspace(nb)
    idx = np.full((B, N), -1, np.int64)
    loss = np.zeros(1, np.float32)
    go = np.full(1, grad_out, np.float32)
    d_sr = np.full_like(sr, np.nan)
    d_gt = np.full_like(sr, np.nan) if want_gt else None
    rc = lib.srst_bbg_forward(_p(sr), _p(gt), _p(gt2), _p(gt4), B, H, W, ksize, pad, stride, alpha, beta, criterion,
                              _p(idx), _p(loss), _p(ws), nb, None)
    assert rc == 0, rc
    rc = lib.srst_bbg_backward(_p(sr), _p(gt), _p(gt2), _p(gt4), _p(idx), _p(go), B, H, W, ksize, pad, stride, criterion,
                               _p(d_sr), _p(d_gt), _p(ws), nb, None)
    assert rc == 0, rc
    return dict(loss=float(loss[0]), idx=idx, d_sr=d_sr, d_gt=d_gt)
