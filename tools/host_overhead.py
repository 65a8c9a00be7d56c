"""Where the eager module path spends host time: host enqueue and wall time per fwd+bwd of every loss module, then a
cProfile of StructureTensorLoss fwd+bwd, at batch 64 x 96x96 with device-resident inputs (the ST kernels take ~31 us;
everything else is Python / torch / ctypes overhead).
    python tools/host_overhead.py > gpurun_out/host_overhead.log"""
import cProfile
import os
import pstats
import sys
import time

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from srgan_st_b200 import (BestBuddyLoss, GramLoss, PatchwiseStructureTensorLoss, StructureTensorLoss,  # noqa: E402
                           StructureTensorPixelLoss)

torch.manual_seed(0)
y = torch.rand(64, 3, 96, 96, device="cuda")
x = (y + 0.05 * torch.randn_like(y)).clamp(0, 1).requires_grad_(True)


def bench(m, n=300):
    for _ in range(20):
        x.grad = None
        m(x, y).backward()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(n):
        x.grad = None
        m(x, y).backward()
    t_enq = (time.perf_counter() - t0) / n
    torch.cuda.synchronize()
    t_all = (time.perf_counter() - t0) / n
    return t_enq * 1e6, t_all * 1e6


for name, m in (("StructureTensorLoss", StructureTensorLoss()), ("StructureTensorPixelLoss", StructureTensorPixelLoss()),
                ("BestBuddyLoss", BestBuddyLoss()), ("BestBuddyLoss(ksize=4, stride=4)", BestBuddyLoss(ksize=4, stride=4)),
                ("GramLoss", GramLoss()), ("PatchwiseStructureTensorLoss", PatchwiseStructureTensorLoss())):
    enq, tot = bench(m)
    print(f"{name}: host enqueue {enq:.1f} us per fwd+bwd, wall {tot:.1f} us per fwd+bwd (device-resident inputs, eager)")
m = StructureTensorLoss()
pr = cProfile.Profile()
pr.enable()
for _ in range(300):
    x.grad = None
    m(x, y).backward()
pr.disable()
torch.cuda.synchronize()
st = pstats.Stats(pr)
st.sort_stats("tottime").print_stats(22)
