"""Time the per-pixel distance map (structure_tensor_distance) against the ST loss on the B200.

    python tools/bench_st_map.py [--rounds R] [--iters K]

Module level, one forward + backward step each, alternated round by round (CUDA events, median of R rounds of K steps):
  (a) StructureTensorLoss()(sr, gt)
  (b) structure_tensor_distance(sr, gt).mean()          -- the same gradient as (a)
  (c) (structure_tensor_distance(sr, gt) * w).sum()     -- a fixed per-pixel weight w
at 64 x 96x96, 1024 x 96x96 and 1 x 1356x2040.  Then at the C ABI, with CUDA events around the calls only:
srst_st_forward_map against srst_st_forward, and srst_st_backward_map (prepass + backward kernel) against
srst_st_backward, with ds_sr / ixy_sr saved (as a generator step does).  The card's name, power limit and max SM
clock are printed first: the numbers belong to them.
"""
import argparse
import os
import statistics
import subprocess
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from srgan_st_b200 import StructureTensorLoss, _cabi, structure_tensor_distance  # noqa: E402
from srgan_st_b200.loss import _st_taps  # noqa: E402


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


def time_alternating(fns, rounds, iters):
    """{name: [ms per call of each round]}, the variants interleaved round by round."""
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


def report(case, res, unit="ms/step"):
    base = statistics.median(res[next(iter(res))])
    for k, v in res.items():
        med = statistics.median(v)
        print(f"  {case:<24s} {k:<14s} {med:9.4f} {unit}  (min {min(v):.4f}, max {max(v):.4f})  x{med / base:.3f}",
              flush=True)


def abi_fns(B, H, W):
    """Forward / backward ABI calls of the plain loss and of the map on one problem (default radii)."""
    lib = _cabi.lib()
    tp = _st_taps(0.5, 2.0, "bench_st_map")[:5]   # ctypes tap pointers; the module cache keeps the arrays alive
    sr, gt = pair(B, H, W, seed=1)
    sr = sr.detach()
    ws = torch.zeros(lib.srst_st_workspace_bytes(B, H, W), dtype=torch.uint8, device="cuda")
    bws = torch.zeros(lib.srst_st_backward_map_workspace_bytes(B, H, W, tp[2], tp[4]), dtype=torch.uint8, device="cuda")
    loss = torch.empty((), device="cuda")
    dmap = torch.empty(B, H, W, device="cuda")
    ds = torch.empty(B, 3, H, W, device="cuda")
    ixy = torch.empty(lib.srst_st_ixy_floats(B, H, W), device="cuda")
    d_img = torch.empty(B, 3, H, W, device="cuda")
    one = torch.ones((), device="cuda")
    grad_map = torch.full((B, H, W), 1.0 / (B * H * W), device="cuda")
    s = torch.cuda.current_stream().cuda_stream
    common = (sr.data_ptr(), gt.data_ptr(), B, H, W, *tp, 1, 1e-12, loss.data_ptr())
    tail = (ds.data_ptr(), None, ixy.data_ptr(), None, ws.data_ptr(), ws.numel(), s)

    def check(rc):
        if rc:
            _cabi.check(rc, "bench_st_map")

    fwd = {"srst_st_forward": lambda: check(lib.srst_st_forward(*common, *tail)),
           "forward_map": lambda: check(lib.srst_st_forward_map(*common, dmap.data_ptr(), *tail))}
    bwd = {"srst_st_backward": lambda: check(lib.srst_st_backward(ixy.data_ptr(), ds.data_ptr(), one.data_ptr(), B, H, W,
                                                                   *tp, d_img.data_ptr(), s)),
           "backward_map": lambda: check(lib.srst_st_backward_map(ixy.data_ptr(), ds.data_ptr(), grad_map.data_ptr(), B,
                                                                   H, W, *tp, d_img.data_ptr(), bws.data_ptr(),
                                                                   bws.numel(), s))}
    return fwd, bwd


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--iters", type=int, default=20)
    a = ap.parse_args()
    print("card:", card(), flush=True)
    print(f"rounds {a.rounds} x {a.iters} calls, median / min / max of the rounds; x = relative to the first row",
          flush=True)
    st = StructureTensorLoss()
    shapes = ((64, 96, 96), (1024, 96, 96), (1, 1356, 2040))
    for B, H, W in shapes:
        sr, gt = pair(B, H, W)
        w = torch.rand(B, H, W, device="cuda", generator=torch.Generator(device="cuda").manual_seed(2)) / (B * H * W)
        report(f"step {B}x{H}x{W}", time_alternating({
            "(a) loss": lambda: st(sr, gt).backward(),
            "(b) map.mean": lambda: structure_tensor_distance(sr, gt).mean().backward(),
            "(c) (map*w).sum": lambda: (structure_tensor_distance(sr, gt) * w).sum().backward()}, a.rounds, a.iters))
        del sr, gt, w
    for B, H, W in shapes:
        fwd, bwd = abi_fns(B, H, W)
        report(f"abi fwd {B}x{H}x{W}", time_alternating(fwd, a.rounds, 5 * a.iters), "ms/call")
        report(f"abi bwd {B}x{H}x{W}", time_alternating(bwd, a.rounds, 5 * a.iters), "ms/call")
        torch.cuda.synchronize()


if __name__ == "__main__":
    main()
