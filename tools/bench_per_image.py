"""Time reduction='none' against reduction='mean' on the B200, and one per-image call against B one-image calls.

    python tools/bench_per_image.py [--rounds R] [--iters K]

Every case is a forward + backward step.  The 'none' step backpropagates loss.mean() (the gradient of the 'mean'
step), so the two differ only by the per-image kernels and the tiny reduction torch adds.  Variants of one case are
timed alternately, R rounds of K steps each, with CUDA events; the median of the rounds is printed, with the spread.
The card's name and power limit are printed first: the numbers belong to them.

The fused ST + Pixel cases also time 'split': the per-image losses without the fused module,
st_weight * StructureTensorLoss(reduction='none') + pixel_weight * ((x - gt)**2).mean((1, 2, 3)), same backward.
"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from srgan_st_b200 import BestBuddyLoss, StructureTensorLoss, StructureTensorPixelLoss  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:   # the timing does not depend on it; say why it is missing
        q = f"nvidia-smi unavailable ({e})"
    return f"{torch.cuda.get_device_name(0)} | {q}"


def pair(B, H, W, seed=0):
    g = torch.Generator(device="cuda").manual_seed(seed)
    gt = torch.rand(B, 3, H, W, device="cuda", generator=g)
    sr = (gt + 0.05 * torch.randn(B, 3, H, W, device="cuda", generator=g)).clamp(0, 1).requires_grad_(True)
    return sr, gt


def step_fn(module, sr, gt, how):
    if how == "mean":
        return lambda: module(sr, gt).backward()
    if how in ("none", "split"):
        return lambda: module(sr, gt).mean().backward()
    B = sr.shape[0]   # "calls": B separate one-image calls, the workaround without reduction='none'

    def calls():
        for b in range(B):
            (module(sr[b:b + 1], gt[b:b + 1]) / B).backward()
    return calls


def time_alternating(fns, rounds, iters):
    """{name: [ms per step of each round]}, the variants interleaved round by round."""
    for f in fns.values():   # warm-up: modules, workspaces, tensor maps
        for _ in range(3):
            f()
    torch.cuda.synchronize()
    out = {k: [] for k in fns}
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    for _ in range(rounds):
        for k, f in fns.items():
            ev[0].record()
            for _ in range(iters):
                f()
            ev[1].record()
            torch.cuda.synchronize()
            out[k].append(ev[0].elapsed_time(ev[1]) / iters)
    return out


def report(case, res):
    base = statistics.median(res[next(iter(res))])
    for k, v in res.items():
        med = statistics.median(v)
        print(f"  {case:<44s} {k:<6s} {med:9.3f} ms/step  (min {min(v):.3f}, max {max(v):.3f})  x{med / base:.3f}",
              flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    print("card:", card(), flush=True)
    print(f"rounds {a.rounds} x {a.iters} steps, median / min / max of the rounds; x = relative to the first row", flush=True)
    st_mean, st_none = StructureTensorLoss(), StructureTensorLoss(reduction="none")
    for B, H, W, name in ((64, 96, 96, "ST configs[1] 64x96x96"), (1024, 96, 96, "ST 1024x96x96"),
                          (1, 1356, 2040, "ST 1x1356x2040")):
        sr, gt = pair(B, H, W)
        iters = a.iters if B * H * W < 50_000_000 else max(a.iters // 4, 3)
        report(name, time_alternating({"mean": step_fn(st_mean, sr, gt, "mean"),
                                       "none": step_fn(st_none, sr, gt, "none")}, a.rounds, iters))
        del sr, gt
    w_st, w_px = 0.5, 2.0
    px_mean = StructureTensorPixelLoss(st_weight=w_st, pixel_weight=w_px)
    px_none = StructureTensorPixelLoss(st_weight=w_st, pixel_weight=w_px, reduction="none")

    def split(x, y):
        return w_st * st_none(x, y) + w_px * ((x - y) ** 2).mean((1, 2, 3))

    for B, H, W, name in ((64, 96, 96, "ST+Pixel configs[1] 64x96x96"), (1, 1356, 2040, "ST+Pixel 1x1356x2040")):
        sr, gt = pair(B, H, W)
        report(name, time_alternating({"mean": step_fn(px_mean, sr, gt, "mean"), "none": step_fn(px_none, sr, gt, "none"),
                                       "split": step_fn(split, sr, gt, "split")}, a.rounds, a.iters))
        del sr, gt
    sr, gt = pair(64, 192, 192)
    report("BestBuddy configs[3] 64x192x192", time_alternating(
        {"mean": step_fn(BestBuddyLoss(), sr, gt, "mean"), "none": step_fn(BestBuddyLoss(reduction="none"), sr, gt, "none")},
        a.rounds, max(a.iters // 4, 3)))
    sr, gt = pair(64, 96, 96)
    report("ST configs[1]: one 'none' call vs 64 calls", time_alternating(
        {"none": step_fn(st_none, sr, gt, "none"), "calls": step_fn(st_mean, sr, gt, "calls")}, a.rounds,
        max(a.iters // 4, 3)))


if __name__ == "__main__":
    main()
