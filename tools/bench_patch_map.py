"""Time the per-patch loss map (loss_map) of the patch losses against their scalar forward on the B200.

    python tools/bench_patch_map.py [--rounds R] [--iters K]

One forward + backward step w.r.t. sr each, alternated round by round (CUDA events, median of R rounds of K steps):
  (a) module(sr, gt)                           -- reduction='mean'
  (b) (module.loss_map(sr, gt) * w).sum()      -- a fixed per-patch weight map w
  (c) BestBuddy only: the torch workaround -- the module's search under no_grad for last_indices, then F.unfold of sr
      and of the three HR levels, a gather on last_indices and the weighted mean of the L1 terms
for BestBuddyLoss, GramLoss and PatchwiseStructureTensorLoss at 64 x 192x192 and for BestBuddyLoss(ksize=4, stride=4)
on 64 x 96x96 crops.  The card's name, power limit and max SM clock are printed first: the numbers belong to them.
"""
import argparse
import os
import sys

import torch
import torch.nn.functional as F

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from bench_st_map import card, pair, report, time_alternating  # noqa: E402  (the same timing protocol)
from srgan_st_b200 import BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss  # noqa: E402


def workaround(module, ksize, stride):
    """The loss map without loss_map: the module's search for last_indices, then the reference's ATen chain."""
    def step(sr, gt, w):
        with torch.no_grad():
            module(sr, gt)
        idx = module.last_indices
        u = lambda t: F.unfold(t, kernel_size=ksize, stride=stride).permute(0, 2, 1)
        with torch.no_grad():
            cat = torch.cat([u(gt)] + [u(F.interpolate(gt, scale_factor=s, mode="bicubic", align_corners=False))
                                       for s in (0.5, 0.25)], 1)
            sel = torch.gather(cat, 1, idx[:, :, None].expand(-1, -1, cat.shape[2]))
        terms = (u(sr) - sel).abs().mean(-1)
        (terms * w.reshape(terms.shape)).sum().backward()
    return step


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=10)
    a = ap.parse_args()
    print("card:", card(), flush=True)
    print(f"rounds {a.rounds} x {a.iters} steps, median / min / max of the rounds; x = relative to the first row",
          flush=True)
    cases = [("BestBuddyLoss", BestBuddyLoss(), (64, 192, 192), (3, 3)),
             ("GramLoss", GramLoss(), (64, 192, 192), None),
             ("PatchwiseSTLoss", PatchwiseStructureTensorLoss(), (64, 192, 192), None),
             ("BestBuddyLoss k4s4", BestBuddyLoss(ksize=4, stride=4), (64, 96, 96), (4, 4))]
    for name, m, (B, H, W), geom in cases:
        sr, gt = pair(B, H, W)
        ny, nx = m.loss_map(sr, gt).shape[1:]
        w = torch.rand(B, ny, nx, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) / (B * ny * nx)
        fns = {"(a) forward mean": lambda: m(sr, gt).backward(),
               "(b) (map*w).sum": lambda: (m.loss_map(sr, gt) * w).sum().backward()}
        if geom is not None:
            wk = workaround(m, *geom)
            fns["(c) torch unfold"] = lambda: wk(sr, gt, w)
        report(f"{name} {B}x{H}x{W}", time_alternating(fns, a.rounds, a.iters))
        del sr, gt, w
        torch.cuda.synchronize()


if __name__ == "__main__":
    main()
