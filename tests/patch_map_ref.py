"""Float64 restatements of the per-patch loss map of the three patch losses (``loss_map``) and of its gradients under a
per-patch weight, for the tests.

Given the argmin indices under test, map entry [b, n] is the mean over the D criterion terms of query patch n of image
b against its selected candidate (reference loss.py:139, :222, :371 before the mean).  The weighted gradients reuse the
oracle's backward restatements: on the default 3x3 / stride-3 grid every pixel belongs to at most one query patch, so
the gradient of sum(w * map) is the batch-mean gradient with each query's block scaled by w[b, n] * B * N; the
arbitrary-geometry path goes through torch float64 autograd."""
import numpy as np

from oracle import bb_oracle as BO
from oracle import bbg_oracle as GO


def _crit(d, criterion):
    return np.abs(d) if criterion == "l1" else d * d


def _levels(gt, gt2, gt4):
    if gt2 is None:
        gt2, gt4 = BO.pyramid_c(gt)   # the library's own pyramid taps
    return gt2, gt4


def _desc(img, mode, taps):
    img = np.asarray(img, np.float64)
    if mode == "patch":
        return BO.unfold3(img)
    if mode == "gram":
        return BO.gram_descriptors(img)
    return BO.pst_descriptors(img, taps)


def _selected(gt, gt2, gt4, idx, mode, taps):
    cat = np.concatenate([_desc(t, mode, taps) for t in (gt, gt2, gt4)], 1)
    return np.take_along_axis(cat, np.asarray(idx, np.int64)[:, :, None], 1)


def patch_map(sr, gt, idx, mode="patch", taps=None, criterion="l1", gt2=None, gt4=None):
    """[B,N] map of the default 3x3 / stride-3 geometry (mode "patch", "gram" or "pst")."""
    gt2, gt4 = _levels(gt, gt2, gt4)
    return _crit(_desc(sr, mode, taps) - _selected(gt, gt2, gt4, idx, mode, taps), criterion).mean(-1)


def _backward(img, sel, mode, taps, criterion):
    """The oracle's batch-mean gradient of the criterion w.r.t. the patches of `img` against `sel` ([B,N,D])."""
    if mode == "patch":
        return BO.bb_backward(img, sel, criterion)
    if mode == "gram":
        return BO.gram_backward(img, sel, criterion)
    return BO.pst_backward(img, sel, taps, criterion)


def _weighted(g_img, weight):
    """Scale the batch-mean gradient image (1/(B N D) per term) patch by patch to weight[b, n] / D."""
    B, _, H, W = g_img.shape
    ny, nx = H // 3, W // 3
    w = np.asarray(weight, np.float64).reshape(B, ny, nx) * (B * ny * nx)
    out = np.zeros_like(g_img)
    out[:, :, :3 * ny, :3 * nx] = g_img[:, :, :3 * ny, :3 * nx] * np.repeat(np.repeat(w, 3, 1), 3, 2)[:, None]
    return out


def patch_grads(sr, gt, idx, weight, mode="patch", taps=None, criterion="l1", gt2=None, gt4=None):
    """(d_sr, d_gt) of sum(weight * map) for the default geometry; weight is [B,N].  d_gt follows
    oracle.bb_oracle.patch_backward_gt: the candidate-side gradient of every query, accumulated over the queries that
    selected a candidate and folded back through the bicubic pyramid."""
    gt2, gt4 = _levels(gt, gt2, gt4)
    sr, gt = np.asarray(sr, np.float64), np.asarray(gt, np.float64)
    gt2, gt4 = np.asarray(gt2, np.float64), np.asarray(gt4, np.float64)
    idx = np.asarray(idx, np.int64)
    d_sr = _weighted(_backward(sr, _selected(gt, gt2, gt4, idx, mode, taps), mode, taps, criterion), weight)
    B, _, H, W = sr.shape
    ny, nx = H // 3, W // 3
    cat = np.concatenate([BO.unfold3(t) for t in (gt, gt2, gt4)], 1)             # [B,M,27] candidate patches
    sel_img = BO._fold3(np.take_along_axis(cat, idx[:, :, None], 1), 3 * ny, 3 * nx)
    sr_c = sr[:, :, :3 * ny, :3 * nx]
    g_sel = BO.unfold3(_weighted(_backward(sel_img, _desc(sr_c, mode, taps), mode, taps, criterion), weight))
    g_cat = np.zeros_like(cat)
    for b in range(B):
        np.add.at(g_cat[b], idx[b], g_sel[b])
    N0, N2 = ny * nx, (gt2.shape[2] // 3) * (gt2.shape[3] // 3)
    return d_sr, (BO._fold3(g_cat[:, :N0], H, W)
                  + BO._bicubic_adjoint(BO._fold3(g_cat[:, N0:N0 + N2], gt2.shape[2], gt2.shape[3]), H, W, 2)
                  + BO._bicubic_adjoint(BO._fold3(g_cat[:, N0 + N2:], gt4.shape[2], gt4.shape[3]), H, W, 4))


def bbg_map(sr, gt, idx, ksize, pad, stride, criterion="l1", gt2=None, gt4=None):
    """[B,N] map of an arbitrary patch geometry (F.unfold(ksize, pad, stride), row-major patch order)."""
    gt2, gt4 = _levels(gt, gt2, gt4)
    u = lambda t: GO.unfold(np.asarray(t, np.float64), ksize, pad, stride)
    cat = np.concatenate([u(gt), u(gt2), u(gt4)], 1)
    sel = np.take_along_axis(cat, np.asarray(idx, np.int64)[:, :, None], 1)
    return _crit(u(sr) - sel, criterion).mean(-1)


def bbg_grads(sr, gt, idx, ksize, pad, stride, criterion="l1", weight=None):
    """(d_sr, d_gt) in float64 of sum(weight * map) for an arbitrary geometry (weight None: the batch mean), given the
    argmin indices [B,N]: torch autograd on the CPU through F.unfold, the gather of the selected candidates and
    F.interpolate(bicubic) of the pyramid (loss.py:116-139)."""
    import torch
    import torch.nn.functional as F

    x = torch.tensor(np.asarray(sr, np.float64), requires_grad=True)
    g = torch.tensor(np.asarray(gt, np.float64), requires_grad=True)
    u = lambda t: F.unfold(t, kernel_size=ksize, padding=pad, stride=stride).permute(0, 2, 1)
    levels = [g] + [F.interpolate(g, scale_factor=s, mode="bicubic", align_corners=False) for s in (0.5, 0.25)]
    cat = torch.cat([u(t) for t in levels], 1)                                      # [B,M,D]
    ind = torch.as_tensor(np.asarray(idx, np.int64))
    sel = torch.gather(cat, 1, ind[:, :, None].expand(-1, -1, cat.shape[2]))        # [B,N,D]
    d = u(x) - sel
    terms = (d.abs() if criterion == "l1" else d * d).mean(-1)
    if weight is None:
        loss = terms.mean()
    else:
        loss = (terms * torch.as_tensor(np.asarray(weight, np.float64).reshape(terms.shape))).sum()
    d_sr, d_gt = torch.autograd.grad(loss, (x, g))
    return d_sr.numpy(), d_gt.numpy()
