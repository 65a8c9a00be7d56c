"""BestBuddyLoss with a non-default patch geometry (reference loss.py:86, F.unfold(kernel_size=ksize, padding=pad,
stride=stride) at loss.py:116-129): overlapping patches, gaps, zero padding, 12..75-dimensional patches.

Fixtures ``tests/golden/bbg_*.npz`` are outputs of the reference itself (``make_golden.py geom``): loss, indices,
top-2 scores, d_sr and d_gt.  The C oracle (oracle/bbg_oracle.c) and the CUDA kernels (bb_generic.cuh; emulated on the
CPU, real on the GPU) accumulate patch elements in one fixed order: their indices are bit-exact against each other,
and against the reference rows may differ only inside fp32 noise of its own top-2 gap (near-tie protocol)."""
import numpy as np
import pytest

from oracle import bb_oracle as OB
from oracle import bbg_oracle as O
from tests.helpers import emu_bb, emu_bbg, emu_lib, golden, golden_names, maxnorm_err, rel_err

CASES = golden_names("bbg_")
DIST_L1 = 0x100   # SRST_BB_DIST_L1


def _args(z):
    return (int(z["ksize"]), int(z["pad"]), int(z["stride"]), float(z["alpha"]), float(z["beta"]), str(z["criterion"]),
            str(z["dist_norm"]))


def _crit(crit, dn):
    return (0 if crit == "l1" else 1) | (DIST_L1 if dn == "l1" else 0)


def _same_up_to_ties(idx, z):
    gap = z["top2"][..., 1] - z["top2"][..., 0]
    noise = 1e-5 * np.maximum(z["top2"][..., 1], 1e-6)
    differ = idx != z["ind"]
    assert not (differ & (gap > noise)).any()
    return not differ.any()


def test_fixture_inventory():
    assert len(CASES) >= 4


@pytest.mark.parametrize("name", CASES)
def test_oracle_matches_reference(name):
    z = golden(name)
    k, p, s, a, b, crit, dn = _args(z)
    r = O.bbg_forward_c(z["sr"], z["hr"], z["hr2"], z["hr4"], k, p, s, a, b, crit, dn)
    assert r["idx"].shape == z["ind"].shape
    if _same_up_to_ties(r["idx"], z):
        assert rel_err(r["loss"], z["loss"]) < 1e-5
        assert maxnorm_err(r["d_sr"], z["d_sr"]) < 1e-5
    s64, _, _ = O.bbg_scores_f64(z["sr"], z["hr"], z["hr2"], z["hr4"], k, p, s, a, b, dn)
    # xx + yy - 2xy in fp32 cancels against norms of ~10: the reference's own scores carry ~1e-6 absolute noise
    assert np.allclose(np.sort(s64, 2)[..., :2], z["top2"], rtol=2e-5, atol=1e-5)


def test_oracle_default_geometry_is_the_27_dim_oracle():
    z = golden("bb_srlike_2x48x48")
    r = O.bbg_forward_c(z["sr"], z["hr"], z["hr2"], z["hr4"], 3, 0, 3)
    q = OB.bb_forward_c(z["sr"], z["hr"], z["hr2"], z["hr4"])
    assert np.array_equal(r["idx"], q["idx"]) and r["loss"] == q["loss"]


@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("own_pyramid", [False, True])
def test_emulated_kernels_match_oracle_and_reference(name, own_pyramid):
    lib = emu_lib()
    z = golden(name)
    k, p, s, a, b, crit, dn = _args(z)
    gt2, gt4 = (None, None) if own_pyramid else (z["hr2"], z["hr4"])
    out = emu_bbg(lib, z["sr"], z["hr"], k, p, s, gt2, gt4, a, b, _crit(crit, dn), want_gt=True)
    orc = O.bbg_forward_c(z["sr"], z["hr"], gt2, gt4, k, p, s, a, b, crit, dn)
    assert np.array_equal(out["idx"], orc["idx"]), "indices must be bit-exact vs the C oracle"
    assert rel_err(out["loss"], orc["loss"]) < 1e-6
    assert maxnorm_err(out["d_sr"], orc["d_sr"]) < 1e-6
    if _same_up_to_ties(out["idx"], z):   # the reference's torch.min indices, its loss and both of its gradients
        assert rel_err(out["loss"], z["loss"]) < 1e-5
        assert maxnorm_err(out["d_sr"], z["d_sr"]) < 1e-5
        assert maxnorm_err(out["d_gt"], z["d_gt"]) < 1e-5


@pytest.mark.parametrize("dist_l1", [0, DIST_L1])
def test_emulated_default_geometry_equals_the_tuned_path(dist_l1):
    """(3, 0, 3) through the generic kernels = the filter + exact re-scoring search: same fixed-order scores."""
    lib = emu_lib()
    z = golden("bb_rand_1x48x36")
    a = emu_bbg(lib, z["sr"], z["hr"], 3, 0, 3, criterion=dist_l1, want_gt=True)
    b = emu_bb(lib, z["sr"], z["hr"], criterion=dist_l1)
    assert np.array_equal(a["idx"], b["idx"])
    assert rel_err(a["loss"], b["loss"]) < 1e-6 and maxnorm_err(a["d_sr"], b["d_sr"]) < 1e-6


def test_emulated_edge_cases():
    lib = emu_lib()
    # every score equal (no padding: all patches of a flat image are the same): index 0 (torch.min), zero loss / gradient
    flat = np.full((1, 3, 16, 20), 0.25, np.float32)
    out = emu_bbg(lib, flat, flat, 4, 0, 3)
    assert np.all(out["idx"] == 0) and out["loss"] == 0.0 and not out["d_sr"].any()
    # with padding the border patches see zeros: each query still takes the FIRST of its co-minimal candidates
    out = emu_bbg(lib, flat, flat, 4, 2, 3)
    orc = O.bbg_forward_c(flat, flat, None, None, 4, 2, 3)
    assert np.array_equal(out["idx"], orc["idx"]) and out["loss"] == 0.0
    # ksize 1 (3-dim patches), a stride larger than the image (one patch per level), the largest ksize
    rng = np.random.default_rng(3)
    sr = rng.random((2, 3, 33, 35), dtype=np.float32)
    gt = rng.random((2, 3, 33, 35), dtype=np.float32)
    for k, p, s in [(1, 0, 1), (3, 0, 100), (8, 3, 5), (2, 5, 2)]:
        out = emu_bbg(lib, sr, gt, k, p, s, want_gt=True)
        orc = O.bbg_forward_c(sr, gt, None, None, k, p, s)
        assert np.array_equal(out["idx"], orc["idx"]), (k, p, s)
        assert rel_err(out["loss"], orc["loss"]) < 1e-6 and maxnorm_err(out["d_sr"], orc["d_sr"]) < 1e-6
        assert np.isfinite(out["d_gt"]).all()
    # a NaN pixel: NaN loss like the reference, indices stay in range, nothing faults
    bad = sr.copy()
    bad[0, 1, 5, 7] = np.nan
    out = emu_bbg(lib, bad, gt, 4, 1, 2, want_gt=True)
    M = O.geometry(33, 35, 4, 1, 2)[1]
    assert np.isnan(out["loss"]) and out["idx"].min() >= 0 and out["idx"].max() < M


def test_entry_points_reject_unusable_geometry():
    lib = emu_lib()
    assert lib.srst_bbg_supported(3, 0, 3) == 1 and lib.srst_bbg_supported(9, 0, 1) == 0
    assert lib.srst_bbg_supported(3, -1, 1) == 0 and lib.srst_bbg_supported(3, 0, 0) == 0
    assert lib.srst_bbg_workspace_bytes(1, 16, 16, 5, 0, 1) == 0      # the x1/4 level (4x4) holds no 5x5 patch
    assert lib.srst_bbg_num_patches(16, 16, 5, 0, 1) == 0
    assert lib.srst_bbg_num_patches(24, 28, 4, 1, 2) == 12 * 14
    x = np.zeros((1, 3, 16, 16), np.float32)
    idx = np.zeros((1, 144), np.int64)
    loss = np.zeros(1, np.float32)
    ws = np.zeros(1 << 16, np.float32)
    vp = lambda a: a.ctypes.data
    rc = lib.srst_bbg_forward(vp(x), vp(x), None, None, 1, 16, 16, 5, 0, 1, 1.0, 1.0, 0, vp(idx), vp(loss), vp(ws), ws.nbytes, None)
    assert rc == -4   # SRST_E_SHAPE
    rc = lib.srst_bbg_forward(vp(x), vp(x), None, None, 1, 16, 16, 9, 0, 1, 1.0, 1.0, 0, vp(idx), vp(loss), vp(ws), ws.nbytes, None)
    assert rc == -2   # SRST_E_UNSUPPORTED
    rc = lib.srst_bbg_forward(vp(x), vp(x), None, None, 1, 16, 16, 3, 0, 1, 1.0, 1.0, 0, vp(idx), vp(loss), vp(ws), 64, None)
    assert rc == -3   # SRST_E_WORKSPACE


def test_module_constructor_contract():
    import srgan_st_b200 as pkg
    m = pkg.BestBuddyLoss(ksize=4, pad=1, stride=2)
    assert (m.ksize, m.pad, m.stride) == (4, 1, 2) and m._geom == (4, 1, 2)
    assert pkg.BestBuddyLoss()._geom is None
    with pytest.raises(NotImplementedError):
        pkg.BestBuddyLoss(ksize=9)
    with pytest.raises(NotImplementedError):
        pkg.BestBuddyLoss(ksize=3, stride=0)
    with pytest.raises(TypeError):
        pkg.BestBuddyLoss(ksize=3.0, stride=2)


# ---- GPU ---------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("name", CASES)
@pytest.mark.parametrize("pyramid", ["fused", "aten"])
def test_gpu_module_matches_reference(name, pyramid):
    import torch
    import srgan_st_b200 as pkg
    z = golden(name)
    k, p, s, a, b, crit, dn = _args(z)
    m = pkg.BestBuddyLoss(alpha=a, beta=b, ksize=k, pad=p, stride=s, dist_norm=dn, criterion=crit, pyramid=pyramid)
    x = torch.from_numpy(z["sr"]).cuda().requires_grad_(True)
    y = torch.from_numpy(z["hr"]).cuda().requires_grad_(True)
    loss = m(x, y)
    loss.backward()
    idx = m.last_indices.cpu().numpy()
    if pyramid == "fused":
        orc = O.bbg_forward_c(z["sr"], z["hr"], None, None, k, p, s, a, b, crit, dn)
        assert np.array_equal(idx, orc["idx"]), "indices must be bit-exact vs the C oracle"
        assert rel_err(loss.item(), orc["loss"]) < 1e-5
    if _same_up_to_ties(idx, z):
        assert rel_err(loss.item(), z["loss"]) < 1e-5
        assert maxnorm_err(x.grad.cpu().numpy(), z["d_sr"]) < 1e-5
        assert maxnorm_err(y.grad.cpu().numpy(), z["d_gt"]) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("k,p,s,dn", [(4, 1, 2, "l2"), (3, 1, 1, "l2"), (6, 0, 6, "l1"), (8, 4, 7, "l2")])
def test_gpu_matches_oracle_at_training_crop_size(k, p, s, dn):
    """2 x 96x96 (the warm-up crop of BASELINE configs[1]); overlapping 3x3/stride-1 patches give N = 9216, M = 12096."""
    import torch
    import srgan_st_b200 as pkg
    rng = np.random.default_rng(100 * k + s)
    sr = rng.random((2, 3, 96, 96), dtype=np.float32)
    gt = rng.random((2, 3, 96, 96), dtype=np.float32)
    m = pkg.BestBuddyLoss(ksize=k, pad=p, stride=s, dist_norm=dn, criterion="l2")
    x = torch.from_numpy(sr).cuda().requires_grad_(True)
    loss = m(x, torch.from_numpy(gt).cuda())
    loss.backward()
    orc = O.bbg_forward_c(sr, gt, None, None, k, p, s, 1.0, 1.0, "l2", dn)
    assert np.array_equal(m.last_indices.cpu().numpy(), orc["idx"])
    assert rel_err(loss.item(), orc["loss"]) < 1e-5
    assert maxnorm_err(x.grad.cpu().numpy(), orc["d_sr"]) < 1e-5


@pytest.mark.gpu
def test_gpu_default_geometry_through_both_paths():
    """(3, 0, 3) forced through the generic kernels picks the tuned search's indices bit for bit (4 x 192x192)."""
    import torch
    import srgan_st_b200 as pkg
    g = torch.Generator(device="cuda").manual_seed(5)
    sr = torch.rand(4, 3, 192, 192, device="cuda", generator=g)
    gt = torch.rand(4, 3, 192, 192, device="cuda", generator=g)
    fast = pkg.BestBuddyLoss()
    slow = pkg.BestBuddyLoss()
    slow._geom = (3, 0, 3)
    xa = sr.clone().requires_grad_(True)
    xb = sr.clone().requires_grad_(True)
    la, lb = fast(xa, gt), slow(xb, gt)
    la.backward()
    lb.backward()
    assert torch.equal(fast.last_indices, slow.last_indices)
    assert rel_err(lb.item(), la.item()) < 1e-6
    assert maxnorm_err(xb.grad.cpu().numpy(), xa.grad.cpu().numpy()) < 1e-6


@pytest.mark.gpu
def test_gpu_nan_input_gives_nan_loss_and_no_fault():
    import torch
    import srgan_st_b200 as pkg
    sr = torch.rand(1, 3, 40, 40, device="cuda")
    gt = torch.rand(1, 3, 40, 40, device="cuda")
    sr[0, 0, 3, 3] = float("nan")
    m = pkg.BestBuddyLoss(ksize=4, pad=1, stride=2)
    x = sr.clone().requires_grad_(True)
    loss = m(x, gt)
    loss.backward()
    torch.cuda.synchronize()
    assert torch.isnan(loss) and 0 <= int(m.last_indices.min()) and int(m.last_indices.max()) < O.geometry(40, 40, 4, 1, 2)[1]


def _f64_bb_reference(sr, hr, k, p, s):
    """BestBuddyLoss at its defaults (loss.py:116-139: l2 search, l1 criterion) restated in float64 with autograd, in
    the reference's place where it is not staged: scores, indices, the loss and its gradients in sr and gt."""
    import torch
    import torch.nn.functional as F
    x = sr.double().requires_grad_(True)
    y = hr.double().requires_grad_(True)
    unf = lambda t: F.unfold(t, kernel_size=k, padding=p, stride=s).permute(0, 2, 1)
    p1, p2 = unf(x), unf(y)
    cat = torch.cat([p2, unf(F.interpolate(y, scale_factor=0.5, mode="bicubic", align_corners=False)),
                     unf(F.interpolate(y, scale_factor=0.25, mode="bicubic", align_corners=False))], 1)
    with torch.no_grad():
        dist = lambda a, b: ((a * a).sum(2)[:, :, None] + (b * b).sum(2)[:, None, :]
                             - 2.0 * torch.bmm(a, b.transpose(1, 2))).clamp_min(0.0)
        score = dist(p1, cat) + dist(p2, cat)
    ind = score.argmin(2)
    loss = (p1 - torch.gather(cat, 1, ind.unsqueeze(-1).expand(-1, -1, cat.shape[2]))).abs().mean()
    loss.backward()
    return score, ind, loss.item(), x.grad, y.grad


@pytest.mark.gpu
@pytest.mark.parametrize("k,p,s", [(5, 2, 3), (2, 0, 2)])
def test_gpu_matches_the_live_reference(k, p, s):
    """The unmodified reference on the same B200 (oracle/_ref), 4 x 128x128, near-tie protocol on its own scores.
    Where the reference is not staged, its float64 restatement (_f64_bb_reference) takes its place."""
    import torch
    import torch.nn.functional as F
    import srgan_st_b200 as pkg
    from oracle import make_ref as R
    torch.backends.cuda.matmul.allow_tf32 = False
    ref = R.load() if R.available() else None
    g = torch.Generator(device="cuda").manual_seed(17 + k)
    hr = torch.rand(4, 3, 128, 128, device="cuda", generator=g)
    sr = (hr + 0.1 * torch.randn(4, 3, 128, 128, device="cuda", generator=g)).clamp(0, 1)
    ours_m = pkg.BestBuddyLoss(ksize=k, pad=p, stride=s)
    x = sr.clone().requires_grad_(True)
    y = hr.clone().requires_grad_(True)
    lo = ours_m(x, y)
    lo.backward()
    if ref is not None:
        ref_m = ref.loss.BestBuddyLoss(ksize=k, pad=p, stride=s)
        xr = sr.clone().requires_grad_(True)
        yr = hr.clone().requires_grad_(True)
        lr_ = ref_m(xr, yr)
        lr_.backward()
        ref_loss, ref_dx, ref_dy = lr_.item(), xr.grad, yr.grad
        with torch.no_grad():
            unf = lambda t: F.unfold(t, kernel_size=k, padding=p, stride=s).permute(0, 2, 1).contiguous()
            p1, p2 = unf(sr), unf(hr)
            cat = torch.cat([p2, unf(F.interpolate(hr, scale_factor=0.5, mode="bicubic", align_corners=False)),
                             unf(F.interpolate(hr, scale_factor=0.25, mode="bicubic", align_corners=False))], 1)
            score = ref.utils.batch_pairwise_distance(p1, cat, "l2") + ref.utils.batch_pairwise_distance(p2, cat, "l2")
            ind_ref = score.argmin(2)
    else:
        score, ind_ref, ref_loss, ref_dx, ref_dy = _f64_bb_reference(sr, hr, k, p, s)
    top2 = torch.topk(score, 2, dim=2, largest=False).values
    differ = ours_m.last_indices != ind_ref
    noise = 4e-6 * top2[..., 1].clamp_min(1e-6) + 1e-6
    assert not (differ & ((top2[..., 1] - top2[..., 0]) > noise)).any()
    if not differ.any():
        assert rel_err(lo.item(), ref_loss) < 1e-5
        assert maxnorm_err(x.grad.cpu().numpy(), ref_dx.cpu().numpy()) < 1e-5
        assert maxnorm_err(y.grad.cpu().numpy(), ref_dy.cpu().numpy()) < 1e-4   # atomicAdd order + bicubic adjoint
    else:
        assert rel_err(lo.item(), ref_loss) < 1e-4
