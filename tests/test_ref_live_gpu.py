"""GPU: the CUDA path against the UNMODIFIED reference modules running on the same B200 (oracle/_ref,
staged by oracle/make_ref.py) at the BASELINE.json sizes -- configs[1] (64 x 96x96), configs[4] (one
1356x2040 image), configs[3]-shaped patch losses (4 x 192x192: the reference needs ~1.4 GB of [B,N,M]
score matrices per image batch of 4; batch 64 does not fit its own memory appetite).

The reference on a GPU runs its ten 1-channel convolutions per image through cuDNN, which by default may
use TF32 (torch.backends.cudnn.allow_tf32 = True, ~1e-3 accuracy); BASELINE.json asks for fp32 parity,
so TF32 is switched off for the reference here -- that is the only setting touched.

The reference's sources are not part of this repository.  Where they are not staged, the ST and patch-loss tests
judge against the float64 restatements in oracle/ instead (held to the reference's own outputs by
tests/test_oracle_*.py): same assertions, the restatement in the reference's place.  The two training-loop tests
need the reference's model.py and config.py themselves and skip without them.

Tolerances (north_star): loss rel 1e-5, input gradients 1e-4 (max-norm relative).  Every measured error
is appended to gpurun_out/r02_parity.json (copied to profiles/ by hand after a run).
Gradient conditioning: where SR and HR tensors nearly coincide 1/(2 sqrt(disc)) amplifies fp32 rounding
and the reference's own gradient wanders from the fp64 truth (measured on the B200: up to 1.6e-3 max-norm on a
64 x 96x96 SR-like batch, 4e-4 on uniform noise); the assertion is therefore  |ours - ref| <= 1e-4 + |ref - fp64 oracle|  and,
independently,  |ours - fp64 oracle| <= 1e-4.
"""
import json
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from oracle import make_ref as R
from oracle import st_oracle as O
from tests.helpers import ROOT, maxnorm_err, rel_err

pytestmark = pytest.mark.gpu

PARITY_LOG = os.path.join(ROOT, "gpurun_out", "r02_parity.json")


def _record(key, **vals):
    os.makedirs(os.path.dirname(PARITY_LOG), exist_ok=True)
    try:
        data = json.load(open(PARITY_LOG))
    except Exception:
        data = {}
    data[key] = {k: (float(v) if not isinstance(v, (int, str)) else v) for k, v in vals.items()}
    json.dump(data, open(PARITY_LOG, "w"), indent=1, sort_keys=True)


@pytest.fixture(scope="module")
def staged_ref():
    """The reference modules when oracle/_ref is staged, else None."""
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return R.load() if R.available() else None


@pytest.fixture(scope="module")
def ref(staged_ref):
    if staged_ref is None:
        pytest.skip("oracle/_ref is not staged (SRST_REFERENCE=<SRGAN-ST checkout> python oracle/make_ref.py)")
    return staged_ref


def _pair(kind, B, H, W, seed):
    g = torch.Generator(device="cuda").manual_seed(seed)
    if kind == "rand":
        return (torch.rand(B, 3, H, W, device="cuda", generator=g), torch.rand(B, 3, H, W, device="cuda", generator=g))
    hr = torch.randint(0, 256, (B, 3, H, W), device="cuda", generator=g).float()
    hr = (F.avg_pool2d(hr, 3, 1, 1, count_include_pad=False).round() / 255).contiguous()
    lo = F.interpolate(hr, size=(max(H // 4, 1), max(W // 4, 1)), mode="bicubic", align_corners=False)
    sr = F.interpolate(lo, size=(H, W), mode="bicubic", align_corners=False)
    sr = (sr + 0.02 * torch.randn(B, 3, H, W, device="cuda", generator=g)).clamp_(0, 1).contiguous()
    return sr, hr


@pytest.mark.parametrize("kind,B,H,W", [("srlike", 64, 96, 96), ("rand", 64, 96, 96), ("srlike", 1, 1356, 2040),
                                         ("rand", 2, 333, 517)])
def test_st_loss_and_gradients_match_the_live_reference(staged_ref, kind, B, H, W):
    from srgan_st_b200 import StructureTensorLoss
    ref = staged_ref
    sr, hr = _pair(kind, B, H, W, 7 * B + H)
    x = sr.clone().requires_grad_(True)
    y = hr.clone().requires_grad_(True)
    ours = StructureTensorLoss()(x, y)
    ours.backward()
    if ref is not None:
        xr = sr.clone().requires_grad_(True)
        yr = hr.clone().requires_grad_(True)
        theirs = ref.loss.StructureTensorLoss()(xr, yr)          # reference loss.py:380-413, its own ATen path
        theirs.backward()
    torch.cuda.synchronize()
    o64 = O.st_loss(sr.cpu().numpy(), hr.cpu().numpy(), want_hr_grad=True)   # fp64 referee
    e = dict(loss_vs_fp64=rel_err(ours.item(), o64["loss"]))
    if ref is not None:
        e.update(loss_vs_ref=rel_err(ours.item(), theirs.item()), ref_loss_vs_fp64=rel_err(theirs.item(), o64["loss"]))
    ref_grads = {"dsr": xr.grad, "dhr": yr.grad} if ref is not None else {}
    for nm, g_ours, g64 in (("dsr", x.grad, o64["d_sr"]), ("dhr", y.grad, o64["d_hr"])):
        a = g_ours.cpu().numpy()
        e[nm + "_vs_fp64"] = maxnorm_err(a, g64)
        if nm in ref_grads:
            b = ref_grads[nm].cpu().numpy()
            e[nm + "_vs_ref"] = maxnorm_err(a, b)
            e[nm + "_ref_vs_fp64"] = maxnorm_err(b, g64)
    _record(f"st_{kind}_{B}x{H}x{W}" + ("" if ref is not None else "_without_reference"), **e)
    assert e["loss_vs_fp64"] < 1e-5
    for nm in ("dsr", "dhr"):
        assert e[nm + "_vs_fp64"] < 1e-4
    if ref is not None:
        assert e["loss_vs_ref"] < 1e-5
        for nm in ("dsr", "dhr"):
            assert e[nm + "_vs_ref"] < 1e-4 + e[nm + "_ref_vs_fp64"]
    # Measured on B200 (profiles/r02_parity.json): on SR-like batches the reference's own fp32 autograd sits ~1e-3 from the
    # fp64 truth (cancellation in utils.py:261 at pixels where both tensors nearly coincide) while this path stays at ~3e-6,
    # so a strict 1e-4 against the reference's gradient cannot hold for ANY accurate implementation; the two assertions
    # above (1e-4 to fp64, and 1e-4 + the reference's own error to the reference) are the meaningful ones.


def _ref_indices(ref, m_ref, sr, hr, alpha, beta, patches):
    """The reference's own argmin (loss.py:132-135) re-derived with its helpers, plus the top-2 gap."""
    with torch.no_grad():
        p1, p2 = patches(sr), patches(hr)
        hr2 = F.interpolate(hr, scale_factor=0.5, mode="bicubic", align_corners=False)
        hr4 = F.interpolate(hr, scale_factor=0.25, mode="bicubic", align_corners=False)
        cat = torch.cat([p2, patches(hr2), patches(hr4)], 1)
        score = alpha * ref.utils.batch_pairwise_distance(p1, cat, "l2") \
            + beta * ref.utils.batch_pairwise_distance(p2, cat, "l2")
        _, ind = torch.min(score, dim=2)
        top2 = torch.topk(score, 2, dim=2, largest=False).values
    return ind, top2, score


def _pst_taps64():
    from srgan_st_b200 import taps as T
    g_, dg_ = T.gaussian_taps(0.5)
    k_, _ = T.gaussian_taps(2.0)
    return np.asarray(g_, np.float64), np.asarray(dg_, np.float64), np.asarray(k_, np.float64)


def _f64_patch_referee(which, sr, hr):
    """The reference's patch losses at their defaults (alpha = beta = 1, l2 search, l1 criterion) restated in float64
    by oracle/bb_oracle.py: descriptors on the host, scores / argmin / top-2 on the GPU.  Returns what the test reads
    from the reference: indices, top-2, scores, the loss and d loss / d sr."""
    from oracle import bb_oracle as OB
    taps64 = _pst_taps64()
    desc = {"bb": lambda a: OB.unfold3(a.astype(np.float64)), "gram": OB.gram_descriptors,
            "pst": lambda a: OB.pst_descriptors(a, taps64)}[which]
    d64 = lambda t: torch.from_numpy(np.ascontiguousarray(desc(t.cpu().numpy()))).cuda()
    hr2 = F.interpolate(hr, scale_factor=0.5, mode="bicubic", align_corners=False)
    hr4 = F.interpolate(hr, scale_factor=0.25, mode="bicubic", align_corners=False)
    p1, p2 = d64(sr), d64(hr)
    cat = torch.cat([p2, d64(hr2), d64(hr4)], 1)

    def dist(a, b):   # utils.py batch_pairwise_distance, 'l2'
        return ((a * a).sum(2)[:, :, None] + (b * b).sum(2)[:, None, :] - 2.0 * torch.bmm(a, b.transpose(1, 2))).clamp_min(0.0)

    score = dist(p1, cat) + dist(p2, cat)
    ind = score.argmin(2)
    top2 = torch.topk(score, 2, dim=2, largest=False).values
    sel = torch.gather(cat, 1, ind.unsqueeze(-1).expand(-1, -1, cat.shape[2]))
    sr_np, sel_np = sr.cpu().numpy(), sel.cpu().numpy()
    d_sr = {"bb": lambda: OB.bb_backward(sr_np, sel_np), "gram": lambda: OB.gram_backward(sr_np, sel_np),
            "pst": lambda: OB.pst_backward(sr_np, sel_np, taps64)}[which]()
    return ind, top2, score, (p1 - sel).abs().mean().item(), torch.from_numpy(d_sr).cuda()


@pytest.mark.parametrize("which", ["bb", "gram", "pst"])
@pytest.mark.parametrize("kind", ["rand", "srlike"])
def test_patch_losses_match_the_live_reference(staged_ref, which, kind):
    import srgan_st_b200 as pkg
    ref = staged_ref
    B, H, W = 4, 192, 192
    sr, hr = _pair(kind, B, H, W, 11 + len(which))
    if kind == "srlike":
        sr = (hr + 0.1 * torch.randn_like(hr)).clamp(0, 1)   # noisier SR: real competition between candidates
    unf = lambda t: F.unfold(t, kernel_size=3, padding=0, stride=3).permute(0, 2, 1).contiguous()
    ours_m = {"bb": pkg.BestBuddyLoss, "gram": pkg.GramLoss, "pst": pkg.PatchwiseStructureTensorLoss}[which]()
    x = sr.clone().requires_grad_(True)
    lo = ours_m(x, hr)
    lo.backward()
    if ref is not None:
        if which == "bb":
            ref_m, patches = ref.loss.BestBuddyLoss(), unf
        elif which == "gram":
            ref_m = ref.loss.GramLoss()
            patches = ref_m.compute_patches
        else:
            ref_m = ref.loss.PatchwiseStructureTensorLoss()
            patches = ref_m.compute_patches
        xr = sr.clone().requires_grad_(True)
        lr_ = ref_m(xr, hr)
        lr_.backward()
        ref_loss, ref_grad = lr_.item(), xr.grad
        ind_ref, top2, score = _ref_indices(ref, ref_m, sr, hr, 1.0, 1.0, patches)
    else:
        ind_ref, top2, score, ref_loss, ref_grad = _f64_patch_referee(which, sr, hr)
    ours_idx = ours_m.last_indices
    gap = top2[..., 1] - top2[..., 0]
    # Rounding band of the reference's own scores.  Raw patches / Gram matrices: fp32 rounding of a ~|x|^2+|y|^2 sized sum
    # (torch.bmm's summation order is unspecified).  PatchwiseST: the descriptors are S / sqrt(det S + 1e-12) with
    # det = Jxx*Jyy - Jxy^2 computed in fp32 -- where the 3x3 patch is nearly one-dimensional that difference cancels
    # several digits, so two correct fp32 evaluations of the SAME descriptor (cuDNN on the GPU here, MKL-DNN in the
    # golden fixtures, our kernel) already differ by ~1e-4 relative; the band is widened accordingly and the measured
    # worst relative gap among differing rows is recorded.
    rel_band = 2e-4 if which == "pst" else 4e-6
    noise = rel_band * top2[..., 1].clamp_min(1e-6) + 1e-6
    differ = ours_idx != ind_ref
    clear = gap > noise
    n_diff = int(differ.sum().item())
    co_min, worst_gap = True, 0.0
    if n_diff:
        s_ours = torch.gather(score, 2, ours_idx.unsqueeze(-1)).squeeze(-1)
        co_min = bool(((s_ours - top2[..., 0])[differ] <= noise[differ]).all().item())
        worst_gap = float(((s_ours - top2[..., 0]) / top2[..., 1].clamp_min(1e-6))[differ].max().item())
    # Rows outside the band: judged by the float64 restatement of the reference's score (oracle/bb_oracle.py).  Both fp32
    # paths round ill-conditioned descriptors differently and neither is "the" fp32 answer (measured on B200: of the rows
    # outside the band the reference found the float64 argmin on 7, this path on 4): the float64 scores of the two picks
    # must agree to within the conditioning of the descriptor (5e-3 relative; worst measured 1.1e-3), and the counts of
    # rows where each path found the float64 argmin are recorded.
    better_or_equal, ours_hits64, ref_hits64, worst64 = True, 0, 0, 0.0
    if n_diff and not co_min and which == "pst":
        from oracle import bb_oracle as OB
        taps64 = _pst_taps64()
        hr_np, sr_np = hr.cpu().numpy(), sr.cpu().numpy()
        hr2_np = F.interpolate(hr, scale_factor=0.5, mode="bicubic", align_corners=False).cpu().numpy()
        hr4_np = F.interpolate(hr, scale_factor=0.25, mode="bicubic", align_corners=False).cpu().numpy()
        q1, q2 = OB.pst_descriptors(sr_np, taps64), OB.pst_descriptors(hr_np, taps64)
        cat64 = np.concatenate([q2, OB.pst_descriptors(hr2_np, taps64), OB.pst_descriptors(hr4_np, taps64)], 1)
        s_ours = torch.gather(score, 2, ours_idx.unsqueeze(-1)).squeeze(-1)
        outside = (differ & ((s_ours - top2[..., 0]) > noise)).cpu().numpy()
        oi, ri = ours_idx.cpu().numpy(), ind_ref.cpu().numpy()
        for bb_, i in zip(*np.nonzero(outside)):
            s64 = ((q1[bb_, i][None] - cat64[bb_]) ** 2).sum(1) + ((q2[bb_, i][None] - cat64[bb_]) ** 2).sum(1)
            j64 = int(np.argmin(s64))
            ours_hits64 += int(oi[bb_, i] == j64)
            ref_hits64 += int(ri[bb_, i] == j64)
            worst64 = max(worst64, abs(s64[oi[bb_, i]] - s64[ri[bb_, i]]) / max(s64[ri[bb_, i]], 1e-30))
            if worst64 > 5e-3:      # conditioning bound: det-cancellation costs up to ~3 digits of the descriptors
                better_or_equal = False
        co_min = better_or_equal
        clear = clear & torch.from_numpy(~outside).to(clear.device)   # those rows were judged in float64 instead
    # gradients: compared on the pixels of patches where both picked the same candidate
    agree = (~differ).view(B, H // 3, W // 3).repeat_interleave(3, 1).repeat_interleave(3, 2).unsqueeze(1).expand(-1, 3, -1, -1)
    ga, gb = x.grad[agree].cpu().numpy(), ref_grad[agree].cpu().numpy()
    e = dict(loss_vs_ref=rel_err(lo.item(), ref_loss), rows=int(differ.numel()), rows_differ=n_diff,
             rows_differ_clear=int((differ & clear).sum().item()), differ_are_cominimal=int(co_min),
             worst_relative_score_gap_of_differing_rows=worst_gap, dsr_vs_ref_on_agreeing_patches=maxnorm_err(ga, gb),
             worst_fp64_score_gap_between_the_two_picks=worst64,
             rows_outside_band_where_ours_is_the_fp64_argmin=ours_hits64,
             rows_outside_band_where_the_reference_is_the_fp64_argmin=ref_hits64)
    _record(f"{which}_{kind}_{B}x{H}x{W}" + ("" if ref is not None else "_without_reference"), **e)
    assert e["rows_differ_clear"] == 0, "a clearly separated row picked a different candidate than the reference"
    assert co_min, "a differing row is neither co-minimal in the reference's scores nor equivalent to its pick in float64"
    # Judged against the float64 restatement, every fp32 rounding of an ill-conditioned PatchwiseST descriptor shows up as
    # a differing row, not only those where two fp32 evaluations disagree: measured on the B200, pst/srlike differs on
    # 51 of 16384 rows against float64 (39 against the reference's fp32 scores), every one co-minimal or within the
    # float64 conditioning bound above.
    max_differ = 4e-3 if ref is None and which == "pst" else 3e-3
    assert n_diff <= max_differ * differ.numel()
    assert e["loss_vs_ref"] < 1e-4 if n_diff else e["loss_vs_ref"] < 1e-5
    assert e["dsr_vs_ref_on_agreeing_patches"] < (2e-3 if which == "pst" else 1e-4)


def test_reference_warmup_loop_with_our_criteria(ref):
    """The reference's OWN registry and loop body (config.py:122-125 add_g_criterion, warmup.py:86-96) driven on
    synthetic tensors with model.Generator: our modules register and train exactly where the reference's do, and
    one step gives the same loss values and the same generator gradients as the reference's criteria."""
    import copy
    import srgan_st_b200 as pkg
    torch.manual_seed(0)
    dev = torch.device("cuda:0")

    def make_config(st_module):
        cfg = ref.config.Config()
        cfg.DEVICE = "cuda:0"
        cfg.MODEL.G_LOSS.WARMUP_CRITERIONS = {"Pixel": torch.nn.MSELoss()}
        cfg.MODEL.G_LOSS.WARMUP_WEIGHTS = {"Pixel": 1.0}
        cfg.MODEL.G_LOSS.WARMUP_CRITERIONS["ST"] = st_module.to(dev)      # "ST + MSE" of BASELINE configs[1]
        cfg.MODEL.G_LOSS.WARMUP_WEIGHTS["ST"] = 1.0 / 3.0                 # config.py:80
        cfg.add_g_criterion("ST", st_module, 1.0 / 3.0)                   # config.py:122-125 (the GAN-phase registry)
        return cfg

    gen0 = ref.model.Generator(ref.config.Config()).to(dev)
    gt, _ = _pair("srlike", 16, 96, 96, 3)
    lr = F.interpolate(gt, scale_factor=0.25, mode="bicubic", align_corners=False).clamp(0, 1)
    results = []
    for st_module in (pkg.StructureTensorLoss(), ref.loss.StructureTensorLoss()):
        config = make_config(st_module)
        generator = copy.deepcopy(gen0)
        optimizer = torch.optim.Adam(generator.parameters(), lr=1e-4)
        # ---- warmup.py:83-96, verbatim control flow ----
        loss_values = {}
        generator.zero_grad()
        sr = generator(lr)
        loss = torch.tensor(0.0, device=config.DEVICE)
        for name, criterion in config.MODEL.G_LOSS.WARMUP_CRITERIONS.items():
            weight = config.MODEL.G_LOSS.WARMUP_WEIGHTS[name]
            l = criterion(sr, gt)
            loss = loss + (l * weight)
            loss_values[name] = (l * weight).item()
        loss.backward()
        grads = torch.cat([p.grad.flatten() for p in generator.parameters()])
        optimizer.step()
        results.append((loss_values, grads, loss.item()))
        assert "ST" in config.MODEL.G_LOSS.CRITERIONS and config.MODEL.G_LOSS.CRITERION_WEIGHTS["ST"] == 1.0 / 3.0
    (lv_o, g_o, l_o), (lv_r, g_r, l_r) = results
    assert rel_err(lv_o["ST"], lv_r["ST"]) < 1e-5 and rel_err(lv_o["Pixel"], lv_r["Pixel"]) < 1e-6
    gerr = maxnorm_err(g_o.cpu().numpy(), g_r.cpu().numpy())
    _record("warmup_step_16x96x96", st_loss_vs_ref=rel_err(lv_o["ST"], lv_r["ST"]), total_vs_ref=rel_err(l_o, l_r),
            generator_grad_vs_ref=gerr)
    assert gerr < 1e-3   # generator weights' gradients: the loss gradient (1e-4) pushed through 37 conv layers of cuDNN


def test_reference_train_loop_step_with_our_criteria(ref):
    """BASELINE configs[2] at its per-GPU batch (128 / 8 = 16): the reference's GAN-phase loop body (train.py:121-164:
    generator update over config.MODEL.G_LOSS.CRITERIONS with the 'Adversarial' special case, then the discriminator
    update) with model.Generator and model.Discriminator, once with our ST + BestBuddy criteria registered through
    config.add_g_criterion (config.py:122-125) and once with the reference's own.  Loss values, generator gradients and
    the discriminator step must agree.  The VGG content criterion needs downloaded weights (no network here) and is
    not registered -- it does not touch the loss path under test."""
    import copy
    import srgan_st_b200 as pkg
    torch.manual_seed(1)
    dev = torch.device("cuda:0")
    base = ref.config.Config()
    base.DEVICE = "cuda:0"
    gen0 = ref.model.Generator(base).to(dev)
    disc0 = ref.model.Discriminator(base).to(dev)
    B = 16
    gt, _ = _pair("srlike", B, 96, 96, 5)
    lr = F.interpolate(gt, scale_factor=0.25, mode="bicubic", align_corners=False).clamp(0, 1)
    results = []
    for ours in (True, False):
        config = ref.config.Config()
        config.DEVICE = "cuda:0"
        config.DATA.BATCH_SIZE = B
        config.MODEL.G_LOSS.CRITERIONS = {"Adversarial": torch.nn.BCEWithLogitsLoss()}
        config.add_g_criterion("Pixel", torch.nn.MSELoss(), 1.0)
        config.add_g_criterion("ST", pkg.StructureTensorLoss() if ours else ref.loss.StructureTensorLoss(), 1.0 / 3.0)
        config.add_g_criterion("BestBuddy", pkg.BestBuddyLoss() if ours else ref.loss.BestBuddyLoss(), 50.0)
        generator, discriminator = copy.deepcopy(gen0), copy.deepcopy(disc0)
        generator.train()
        discriminator.train()
        g_optimizer = torch.optim.Adam(generator.parameters(), lr=1e-4)
        d_optimizer = torch.optim.Adam(discriminator.parameters(), lr=1e-4)
        adversarial_criterion = torch.nn.BCEWithLogitsLoss().to(config.DEVICE)
        real_label = torch.full([config.DATA.BATCH_SIZE, 1], 1.0 - config.EXP.LABEL_SMOOTHING, dtype=torch.float, device=config.DEVICE)
        fake_label = torch.full([config.DATA.BATCH_SIZE, 1], 0.0, dtype=torch.float, device=config.DEVICE)
        loss_values = {}
        # ---- train.py:121-164, verbatim control flow ----
        for p in discriminator.parameters():
            p.requires_grad = False
        generator.zero_grad()
        sr = generator(lr)
        g_loss = torch.tensor(0.0, device=config.DEVICE)
        for name, criterion in config.MODEL.G_LOSS.CRITERIONS.items():
            weight = config.MODEL.G_LOSS.CRITERION_WEIGHTS[name]
            if name == 'Adversarial':
                loss = criterion(discriminator(sr), real_label)
            else:
                loss = criterion(sr, gt)
            g_loss = g_loss + (loss * weight)
            loss_values[name] = (loss * weight).item()
        g_loss.backward()
        g_grads = torch.cat([p.grad.flatten() for p in generator.parameters()])
        g_optimizer.step()
        for p in discriminator.parameters():
            p.requires_grad = True
        discriminator.zero_grad()
        pred_gt = discriminator(gt)
        loss_real = adversarial_criterion(pred_gt, real_label)
        pred_sr = discriminator(sr.detach().clone())
        loss_fake = adversarial_criterion(pred_sr, fake_label)
        d_loss = loss_real + loss_fake
        d_loss.backward()
        d_optimizer.step()
        results.append((loss_values, g_grads, g_loss.item(), d_loss.item()))
    (lv_o, g_o, gl_o, dl_o), (lv_r, g_r, gl_r, dl_r) = results
    e = dict(st_vs_ref=rel_err(lv_o["ST"], lv_r["ST"]), bb_vs_ref=rel_err(lv_o["BestBuddy"], lv_r["BestBuddy"]),
             g_loss_vs_ref=rel_err(gl_o, gl_r), d_loss_vs_ref=rel_err(dl_o, dl_r),
             generator_grad_vs_ref=maxnorm_err(g_o.cpu().numpy(), g_r.cpu().numpy()))
    _record("train_step_16x96x96", **e)
    assert e["st_vs_ref"] < 1e-5 and e["bb_vs_ref"] < 1e-4 and e["g_loss_vs_ref"] < 1e-4
    assert rel_err(lv_o["Pixel"], lv_r["Pixel"]) < 1e-6 and rel_err(lv_o["Adversarial"], lv_r["Adversarial"]) < 1e-5
    assert e["d_loss_vs_ref"] < 1e-5
    assert e["generator_grad_vs_ref"] < 1e-3   # the loss gradients (1e-4) pushed through the generator's cuDNN layers
