#!/usr/bin/env python
"""bench.py -- structure-tensor loss fwd+bwd throughput on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload c2|c2x|c5|c1] [--impl reference]
                    [--dump-outputs DIR]

One "step" = one forward + backward pass of the fused ST loss over one batch of synthetic
SR/HR images (the hot path of SURVEY.md section 8).  Printed: ONE JSON line.

--dump-outputs DIR writes what the timed path returned in its last step -- the loss and d loss / d sr -- as
DIR/loss.npy and DIR/d_sr.npy (float32).  The inputs are seeded, so two builds run with the same arguments
can be compared output for output.  A gradient larger than 60 MB (--workload c2x) is written as
DIR/d_sr_sample.npy instead: the values at a fixed, seeded set of element indices.

  value      images/s with inputs resident in HBM: the two kernels (forward, backward) are enqueued
             through the C ABI on one stream, K steps captured in a CUDA graph, timed with CUDA
             events on that stream, max over ranks.  Every step reads a different batch from a pool
             larger than the 126 MB L2, so no step sees L2-warm inputs.
  e2e        the same metric through the public API (StructureTensorLoss()(sr, gt); backward();
             read the loss on the host) with each step's inputs copied host->device from pinned memory,
             as the reference's train.py:119-144 does.  At N > 1 the step also all-reduces a
             generator-sized gradient bucket (+ the loss in its tail).  `e2e.variants` separates the
             costs: strict (collective and .item() inside the step, round 1's definition), pipelined
             (collective on a side stream, the previous step's loss read while this step runs: the
             headline), h2d_only, collective_only (device-resident inputs).
  roofline   forward kernel (dominant) against the measured HBM copy bandwidth of
             MEASURED_PEAKS.json; algorithmic bytes = 24 B/pixel forward, 36 B/pixel backward
             (SURVEY.md section 8d).  The fwd+bwd pair is reported beside it.
  cpu_baseline  the reference's OWN modules (oracle/_ref, staged from /root/reference by
             oracle/make_ref.py: loss.py:380-413 on ATen/MKL-DNN, fp32) on the host cores, one process
             per core, on a bounded sample; `port` = the numpy restatement (oracle/st_oracle.py) beside it.

`--impl reference` times that CPU arm alone (and, when a GPU is visible, adds the reference modules'
own unfused ATen path on the B200 and the configs[1] warm-up step for context).
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.dont_write_bytecode = True   # the benchmark writes nothing into the tree it runs from (which may be read-only)

METRIC = "st_loss_fwd_bwd_images_per_sec"
UNIT = "images/s"

# per-rank workloads (weak scaling: every rank processes its own batch)
WORKLOADS = {
    # BASELINE.json configs[1]: warmup.py step's loss, batch 64 of 96x96 crops per GPU
    "c2": dict(B=64, H=96, W=96, desc="ST loss fwd+bwd, batch 64 x 3x96x96 per GPU (configs[1] loss path)"),
    # configs[4]: DIV2K-shaped validation image, one 1356x2040 image per GPU
    "c5": dict(B=1, H=1356, W=2040, desc="ST loss fwd+bwd, 1 x 3x1356x2040 per GPU (configs[4])"),
    # configs[0]/[2]: batch 16 of 96x96 per GPU
    "c1": dict(B=16, H=96, W=96, desc="ST loss fwd+bwd, batch 16 x 3x96x96 per GPU (configs[0]/[2])"),
    # steady state of the training shape (SURVEY 7.2-5): 1024 crops = 9.4 Mpx, 4096+ tiles, many waves
    "c2x": dict(B=1024, H=96, W=96, desc="ST loss fwd+bwd, batch 1024 x 3x96x96 per GPU (steady state of the configs[1] shape)"),
}
BYTES_FWD, BYTES_BWD = 24, 36  # algorithmic bytes per pixel (SURVEY.md 8d)


def _traffic(workload, kernel):
    """dram bytes per launch from the committed ncu --set full capture (profiles/r02_traffic.json)."""
    p = os.path.join(ROOT, "profiles", "r02_traffic.json")
    try:
        return int(json.load(open(p))[workload][kernel])
    except Exception:
        return None


FP32_FLOOR_LANE_OPS_PER_PX = {"fwd": 340, "bwd": 155}   # DESIGN.md section 3


def _fp32_context(torch, res, wl):
    props = torch.cuda.get_device_properties(0)
    mhz = (res.get("clocks") or {}).get("sm_mhz") or 1965.0
    peak = props.multi_processor_count * 128 * mhz * 1e6
    px = wl["B"] * wl["H"] * wl["W"]
    ops = px * (FP32_FLOOR_LANE_OPS_PER_PX["fwd"] + FP32_FLOOR_LANE_OPS_PER_PX["bwd"])
    ach = ops / (res["ms_step"] * 1e-3)
    return {"floor_lane_ops_per_px": FP32_FLOOR_LANE_OPS_PER_PX, "achieved_lane_ops_per_s": ach,
            "peak_lane_ops_per_s": peak, "frac": ach / peak,
            "hbm_frac_if_fp32_pipe_saturated": (BYTES_FWD + BYTES_BWD) * peak /
            (FP32_FLOOR_LANE_OPS_PER_PX["fwd"] + FP32_FLOOR_LANE_OPS_PER_PX["bwd"]) / 1e9 / _peaks()[0]}


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own modules (oracle/_ref) on the host cores, one process per core;
#          the numpy port (oracle/st_oracle.py) beside it
# ------------------------------------------------------------------------------------------------
def _avail_cores():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


def _cpu_worker(args):
    import numpy as np
    from oracle import st_oracle as O
    seed, n, H, W = args
    rng = np.random.default_rng(seed)
    taps = (*O.gaussian_taps(0.5, True), O.gaussian_taps(2.0))
    t = 0.0
    for _ in range(n):
        sr = rng.random((1, 3, H, W), dtype=np.float32)
        hr = rng.random((1, 3, H, W), dtype=np.float32)
        t0 = time.perf_counter()
        O.st_loss(sr, hr, taps=taps, dtype=np.float32)
        t += time.perf_counter() - t0
    return t


def cpu_port_images_per_sec(H, W, n_images, cores=None):
    """Times oracle/st_oracle.py (fp32 port of the reference's algorithm, fwd + bwd) on
    `n_images` synthetic images split over `cores` processes.  Returns (images/s, cores)."""
    import multiprocessing as mp
    cores = max(1, min(cores or _avail_cores(), n_images))
    per = [n_images // cores + (1 if i < n_images % cores else 0) for i in range(cores)]
    os.environ.setdefault("OMP_NUM_THREADS", "1")
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        pool.map(_cpu_worker, [(i, 1, min(H, 32), min(W, 32)) for i in range(cores)])  # spin-up
        t0 = time.perf_counter()
        pool.map(_cpu_worker, [(100 + i, per[i], H, W) for i in range(cores)])
        dt = time.perf_counter() - t0
    return n_images / dt, cores


_REF_CRIT = None


def _ref_worker(args):
    """One process = one host core running the UNMODIFIED reference StructureTensorLoss (loss.py:380-413) forward +
    backward on its share of the images, in sub-batches of `b` (the reference vmaps over the batch)."""
    global _REF_CRIT
    import torch
    seed, n, b, H, W = args
    torch.set_num_threads(1)
    from oracle import make_ref as R
    if _REF_CRIT is None:
        _REF_CRIT = R.load().loss.StructureTensorLoss()
    g = torch.Generator().manual_seed(seed)
    t = 0.0
    with R.on_cpu():  # utils.py:206,208 hard-code .cuda() on the taps
        done = 0
        while done < n:
            bb = min(b, n - done)
            x = torch.rand(bb, 3, H, W, generator=g).requires_grad_(True)
            y = torch.rand(bb, 3, H, W, generator=g)
            t0 = time.perf_counter()
            _REF_CRIT(x, y).backward()
            t += time.perf_counter() - t0
            done += bb
    return t


class RefCpuPool:
    """Spawned (not forked: the parent may hold a CUDA context and OpenMP threads) worker processes, kept alive across
    steps -- importing torch + torchvision + cv2 in a fresh interpreter costs seconds."""

    def __init__(self, cores=None):
        import multiprocessing as mp
        self.cores = max(1, cores or _avail_cores())
        os.environ.setdefault("OMP_NUM_THREADS", "1")
        os.environ.setdefault("MKL_NUM_THREADS", "1")
        self.pool = mp.get_context("spawn").Pool(self.cores)
        self.pool.map(_ref_worker, [(i, 1, 1, 16, 16) for i in range(self.cores)])  # imports + first-call set-up

    def images_per_sec(self, H, W, n_images, sub_batch):
        use = max(1, min(self.cores, n_images))
        per = [n_images // use + (1 if i < n_images % use else 0) for i in range(use)]
        t0 = time.perf_counter()
        self.pool.map(_ref_worker, [(1000 + i, per[i], sub_batch, H, W) for i in range(use)], chunksize=1)
        return n_images / (time.perf_counter() - t0), use

    def close(self):
        self.pool.terminate()
        self.pool.join()


def ref_available():
    from oracle import make_ref as R
    return R.available()


def ref_inproc_images_per_sec(B, H, W, reps=3):
    """The reference module as a user would call it on the host: one process, all intra-op threads."""
    import torch
    from oracle import make_ref as R
    crit = R.load().loss.StructureTensorLoss()
    torch.set_num_threads(_avail_cores())
    x = torch.rand(B, 3, H, W).requires_grad_(True)
    y = torch.rand(B, 3, H, W)
    with R.on_cpu():
        crit(x, y).backward()
        t0 = time.perf_counter()
        for _ in range(reps):
            crit(x, y).backward()
        dt = (time.perf_counter() - t0) / reps
    return B / dt, torch.get_num_threads()


def _ref_gpu_context(wl):
    """Reference-arm context on a visible GPU (no kernel of ours involved): the reference modules' own unfused ATen path
    on the B200 (BASELINE.md's "same hardware" figure), and the configs[1] warm-up step (warmup.py:83-96) with the
    reference's Generator, Adam and its two criteria (Pixel + ST)."""
    import torch
    from oracle import make_ref as R
    if not torch.cuda.is_available():
        return None
    ns = R.load()
    dev = torch.device("cuda:0")
    out = {}

    def timed(fn, n=10, warm=3):
        for _ in range(warm):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / n

    B, H, W = wl["B"], wl["H"], wl["W"]
    B = min(B, 64)
    g = torch.Generator(device=dev).manual_seed(5)
    y = torch.rand(B, 3, H, W, device=dev, generator=g)
    x = (y + 0.05 * torch.randn(B, 3, H, W, device=dev, generator=g)).clamp(0, 1).requires_grad_(True)
    crit = ns.loss.StructureTensorLoss()

    def st_step():
        x.grad = None
        crit(x, y).backward()

    for tf32 in (True, False):
        torch.backends.cudnn.allow_tf32 = tf32
        ms = timed(st_step)
        out["st_fwd_bwd_tf32_conv" if tf32 else "st_fwd_bwd_fp32"] = {"ms_per_step": ms, "images_per_s": B / (ms * 1e-3)}
    torch.backends.cudnn.allow_tf32 = True
    out["note"] = (f"reference loss.py:380-413 fwd+bwd on cuda:0, batch {B} x 3x{H}x{W}, eager ATen/cuDNN (about 100 launches "
                   "forward, 300 backward); cuDNN's default allows TF32 convolutions, the fp32 line switches that off")
    if H == 96 and W == 96:
        cfg = ns.config.Config()
        gen = ns.model.Generator(cfg).to(dev)
        opt = torch.optim.Adam(gen.parameters(), lr=1e-4)
        lr_in = torch.nn.functional.interpolate(y, scale_factor=0.25, mode="bicubic", align_corners=False).clamp(0, 1)
        crits = {"Pixel": (torch.nn.MSELoss(), 1.0), "ST": (ns.loss.StructureTensorLoss(), 1.0 / 3.0)}

        def warm_step():
            gen.zero_grad()
            sr = gen(lr_in)
            loss = torch.tensor(0.0, device=dev)
            vals = {}
            for name, (c, w) in crits.items():
                l = c(sr, y)
                loss = loss + l * w
                vals[name] = (l * w).item()          # the per-criterion sync of warmup.py:93
            loss.backward()
            opt.step()

        ms = timed(warm_step, n=10, warm=3)
        out["warmup_step_reference"] = {"ms_per_step": ms, "images_per_s": B / (ms * 1e-3),
                                        "what": f"warmup.py:83-96 loop body, reference Generator (1 547 350 params) + Adam + Pixel "
                                                f"+ reference ST criterion, batch {B} x 96x96 HR, eager, default cuDNN settings"}
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    wl = WORKLOADS[args.workload]
    H, W = wl["H"], wl["W"]
    big = H * W > 1e6
    sub = 1 if big else 4
    use_ref = ref_available()
    if use_ref:
        pool = RefCpuPool()
        measure = lambda n: pool.images_per_sec(H, W, n, sub)
        kind, how = "reference", "oracle/_ref loss.py StructureTensorLoss (unmodified reference, ATen/MKL-DNN fp32) fwd+bwd"
    else:  # not staged: the numpy port stands in (and says so)
        measure = lambda n: cpu_port_images_per_sec(H, W, n)
        kind, how = "port", "oracle/st_oracle.py fp32 fwd+bwd (oracle/_ref not staged on this box)"
    probe, cores = measure(max(2, _avail_cores()) if big else 4 * _avail_cores())
    budget_s = min(1.5, 150.0 / max(args.steps + args.warmup, 1))   # the whole run stays within a few minutes
    n_step = max(cores, int(probe * budget_s)) if not big else max(2, min(cores, 16))
    for _ in range(min(args.warmup, 3)):
        measure(max(1, n_step // 4))
    rates = []
    t0 = time.perf_counter()
    for _ in range(args.steps):
        r, cores = measure(n_step)
        rates.append(r)
    total = time.perf_counter() - t0
    value = statistics.median(rates)
    extra = {}
    if use_ref:
        pool.close()
        try:
            v, thr = ref_inproc_images_per_sec(min(wl["B"], 64), H, W)
            extra["inproc_all_threads"] = {"value": v, "unit": UNIT, "threads": thr,
                                           "what": "one process, torch intra-op threads = all cores (how a user would call it)"}
        except Exception as e:  # context only
            extra["inproc_all_threads"] = {"error": repr(e)}
        try:
            ctx = _ref_gpu_context(wl)
            if ctx:
                extra["reference_gpu_unfused"] = ctx
        except Exception as e:
            extra["reference_gpu_unfused"] = {"error": repr(e)}
    out = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": _config_dict(wl, args.gpus, extra={"sample_images_per_step": n_step}),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                         "sample": f"{n_step} images of 3x{H}x{W} per step, {how}, one process per core "
                                   f"(sub-batches of {sub})", **extra},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(out)
    return 0


def _config_dict(wl, world, extra=None):
    """The same keys on both arms (the driver compares the two `config` objects)."""
    c = {"workload": wl["desc"], "per_gpu_batch": wl["B"], "height": wl["H"], "width": wl["W"],
         "sigma": 0.5, "rho": 2.0, "parallelism": f"batch-sharded x{world}, no data-path collective"}
    if extra:
        c.update(extra)
    return c


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU in a background thread (NVML, ~2 ms period)
    while the timed regions run; falls back to `nvidia-smi -lms` when NVML is unavailable."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown"}

    def __init__(self, torch, local):
        self.samples, self.reason_bits, self.max_mhz = [], 0, None
        self._stop = False
        self._thread = None
        self._h = None
        self._nv = None
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                uuid = "GPU-" + str(torch.cuda.get_device_properties(local).uuid)
                self._h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(local)
            self._nv = pynvml
            self.max_mhz = float(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._nv = None

    def _loop(self):
        nv, h = self._nv, self._h
        while not self._stop:
            try:
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                self.reason_bits |= int(nv.nvmlDeviceGetCurrentClocksEventReasons(h))
            except Exception:
                pass
            time.sleep(0.002)

    def start(self):
        if self._nv is None:
            return
        import threading
        self._thread = threading.Thread(target=self._loop, daemon=True)
        self._thread.start()

    def stop(self):
        if self._thread is None:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["nvml unavailable"]}
        self._stop = True
        self._thread.join(timeout=2)
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["no samples"]}
        busy = [x for x in self.samples if x >= 0.5 * max(self.samples)]
        reasons = sorted(n for b, n in self.REASONS.items() if self.reason_bits & b)
        return {"sm_mhz": statistics.median(busy), "sm_min_mhz": min(busy), "sm_max_mhz": self.max_mhz,
                "reasons": reasons, "samples": len(self.samples)}


def make_pair(torch, B, H, W, gen, device):
    """Synthetic DIV2K-like pair (SURVEY.md 8d): HR = low-passed 8-bit noise, SR = 4x down/up
    sampled HR + noise, saturated to [0,1]."""
    import torch.nn.functional as F
    hr = torch.randint(0, 256, (B, 3, H, W), generator=gen, device=device).float()
    hr = (F.avg_pool2d(hr, 3, 1, 1, count_include_pad=False).round() / 255).contiguous()
    lo = F.interpolate(hr, size=(max(H // 4, 1), max(W // 4, 1)), mode="bicubic", align_corners=False)
    sr = F.interpolate(lo, size=(H, W), mode="bicubic", align_corners=False)
    sr = (sr + 0.02 * torch.randn(B, 3, H, W, generator=gen, device=device)).clamp_(0, 1).contiguous()
    return sr, hr


def run_gpu(args):
    import torch
    import torch.distributed as dist
    from srgan_st_b200 import StructureTensorLoss, _cabi, taps as T

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    torch.cuda.set_device(local)
    # Pin this process to the CPUs next to its GPU (NVML's ideal affinity): pinned host buffers are then
    # allocated on the GPU-local NUMA node, which is what the H2D copies of the e2e leg run at full rate
    # from.  The original affinity is restored before the CPU baseline leg uses every core.
    all_cpus = os.sched_getaffinity(0)
    numa_note = "unchanged"
    try:
        import pynvml
        pynvml.nvmlInit()
        h = pynvml.nvmlDeviceGetHandleByIndex(local)
        pynvml.nvmlDeviceSetCpuAffinity(h)
        numa_note = f"{len(os.sched_getaffinity(0))} GPU-local CPUs of {len(all_cpus)}"
    except Exception as e:  # NVML missing or no affinity information: run unpinned
        numa_note = f"unchanged ({type(e).__name__})"
    dev = torch.device("cuda", local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # stdout carries exactly one JSON line: NCCL's own banner / debug output goes to stderr
        os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    lib = _cabi.lib()
    g, dg = T.gaussian_taps(0.5)
    k, _ = T.gaussian_taps(2.0)
    hbm_peak, peak_src = _peaks()

    def measure(wl_name, K, Wm, with_e2e, keep_last=False):
        wl = WORKLOADS[wl_name]
        B, H, W = wl["B"], wl["H"], wl["W"]
        bytes_pair = 2 * B * 3 * H * W * 4
        pool_n = max(4, min(64, int(300e6 // bytes_pair) + 1))  # > 2x the 126 MB L2
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        pool = [make_pair(torch, B, H, W, gen, dev) for _ in range(pool_n)]
        ds = torch.empty(B, 3, H, W, device=dev)
        d_sr = torch.empty(B, 3, H, W, device=dev)
        ixy = torch.empty(lib.srst_st_ixy_floats(B, H, W), device=dev)
        loss = torch.zeros((), device=dev)
        go = torch.ones((), device=dev)
        nws = lib.srst_st_workspace_bytes(B, H, W)
        ws = torch.zeros(max(nws, 4096), dtype=torch.uint8, device=dev)
        vp = lambda t: ctypes.c_void_p(t.data_ptr())
        s = torch.cuda.Stream(device=dev)
        sp = ctypes.c_void_p(s.cuda_stream)

        def fwd(i):
            sr, hr = pool[i % pool_n]
            _cabi.check(lib.srst_st_forward(vp(sr), vp(hr), B, H, W, T.as_c(g), T.as_c(dg), 2, T.as_c(k), 8, 1,
                                            1e-12, vp(loss), vp(ds), None, vp(ixy), None, vp(ws), ws.numel(), sp), "fwd")

        def bwd(i):
            _cabi.check(lib.srst_st_backward(vp(ixy), vp(ds), vp(go), B, H, W, T.as_c(g), T.as_c(dg), 2,
                                             T.as_c(k), 8, vp(d_sr), sp), "bwd")

        def graph_of(fn_list, n):
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr, stream=s):
                for i in range(n):
                    for fn in fn_list:
                        fn(i)
            return gr

        def time_graph(gr):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with torch.cuda.stream(s):
                e0.record(s)
                gr.replay()
                e1.record(s)
            barrier()
            return max_over_ranks(e0.elapsed_time(e1))

        with torch.cuda.stream(s):
            for i in range(max(Wm, 3)):
                fwd(i); bwd(i)
        torch.cuda.synchronize()
        g_pair = graph_of([fwd, bwd], K)
        g_f = graph_of([fwd], K)
        g_b = graph_of([bwd], K)
        for gr in (g_pair, g_f, g_b):  # untimed replay: graph upload + instruction cache
            with torch.cuda.stream(s):
                gr.replay()
        torch.cuda.synchronize()
        sampler = ClockSampler(torch, local)
        if rank == 0:
            sampler.start()
        ms_pair = min(time_graph(g_pair) for _ in range(3))
        # what the caller of the timed path holds after its last step (step K-1, batch (K-1) % pool_n)
        last_step = {"loss": loss.cpu().numpy(), "d_sr": d_sr.cpu().numpy()} if keep_last else None
        ms_f = min(time_graph(g_f) for _ in range(3))
        ms_b = min(time_graph(g_b) for _ in range(3))
        loss_val = float(loss.item())
        res = dict(wl=wl, ms_step=ms_pair / K, ms_fwd=ms_f / K, ms_bwd=ms_b / K, clocks=None, pool_n=pool_n,
                   loss=loss_val, images_per_s=world * B * K / (ms_pair * 1e-3), last_step=last_step)
        px = B * H * W
        res["roofline_fwd"] = BYTES_FWD * px / (res["ms_fwd"] * 1e-3) / 1e9
        res["roofline_bwd"] = BYTES_BWD * px / (res["ms_bwd"] * 1e-3) / 1e9
        res["roofline_pair"] = (BYTES_FWD + BYTES_BWD) * px / (res["ms_step"] * 1e-3) / 1e9

        if with_e2e:
            crit = StructureTensorLoss()
            bucket = None
            if world > 1:
                # the step's only exchange (SURVEY 8e): one all-reduce of a generator-sized flat
                # gradient bucket (SRResNet: 1 547 350 fp32 params, model.py:193) with the loss in its tail
                from srgan_st_b200.dist import FlatGradBucket
                gen_like = torch.nn.Parameter(torch.zeros(1547350, device=dev))
                bucket = FlatGradBucket([gen_like])
            n_host = 4
            # one pinned [2,B,3,H,W] buffer per batch: SR and HR travel in a single copy
            host = [torch.stack([sr, hr]).cpu().pin_memory() for sr, hr in pool[:n_host]]
            # two device slots: the copy stream fills slot (i+1)%2 while step i computes on slot i%2
            # (the DataLoader pin_memory + non_blocking pattern of train.py:47,119-120); every step's
            # copy is issued and completed inside the timed region
            slots = [torch.empty(2, B, 3, H, W, device=dev) for _ in range(2)]
            copy_stream = torch.cuda.Stream(device=dev)

            def run_e2e(h2d, collective, pipelined, Ksteps):
                """K steps through the public module.  h2d: copy each step's inputs from pinned host memory (else the
                slots keep their contents); collective: all-reduce the gradient bucket every step (N > 1);
                pipelined: the host reads the PREVIOUS step's loss (one read per step, one step late) instead of
                stalling on its own loss, so enqueueing step i+1 overlaps the execution of step i."""
                copied = [torch.cuda.Event(), torch.cuda.Event()]
                consumed = [torch.cuda.Event(), torch.cuda.Event()]
                use_bucket = bucket is not None and collective
                loss_ring = [torch.zeros((), device=dev) for _ in range(2)]
                host_loss = [torch.zeros((), pin_memory=True) for _ in range(2)]
                read_done = [torch.cuda.Event(), torch.cuda.Event()]

                def issue_copy(i):
                    if not h2d:
                        return
                    with torch.cuda.stream(copy_stream):
                        copy_stream.wait_event(consumed[i % 2])     # slot free (previous user finished)
                        slots[i % 2].copy_(host[i % n_host], non_blocking=True)
                        copied[i % 2].record(copy_stream)

                def step(i, last):
                    sr_d, hr_d = slots[i % 2][0], slots[i % 2][1]
                    cur = torch.cuda.current_stream()
                    if h2d:
                        cur.wait_event(copied[i % 2])
                        if not last:
                            issue_copy(i + 1)
                    x = sr_d.detach().requires_grad_(True)
                    l = crit(x, hr_d)
                    l.backward()
                    consumed[i % 2].record(cur)
                    if not pipelined:
                        if use_bucket:
                            bucket.set_loss(l)
                            l = bucket.all_reduce_mean()
                        return l.item()  # device->host read of the step's result, as train.py:141
                    # pipelined: nothing blocks the host inside the step.  The collective stays on the compute stream (it
                    # overlaps the NEXT step's H2D copy, which runs on the copy stream; the kernels are ~30 us of a
                    # ~260 us step) and the host reads the PREVIOUS step's loss from a pinned slot.
                    if use_bucket:
                        bucket.set_loss(l)
                        src = bucket.all_reduce_mean()
                    else:
                        src = l.detach()
                    host_loss[i % 2].copy_(src, non_blocking=True)
                    read_done[i % 2].record(cur)
                    if i > 0:
                        read_done[(i - 1) % 2].synchronize()   # the host now holds step i-1's loss
                        return float(host_loss[(i - 1) % 2])
                    return None

                def drain(n):
                    if pipelined and n > 0:
                        read_done[(n - 1) % 2].synchronize()
                        _ = float(host_loss[(n - 1) % 2])

                for ev in consumed:
                    ev.record()
                nw = max(Wm, 3)
                issue_copy(0)
                for i in range(nw):
                    step(i, i == nw - 1)
                drain(nw)
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                issue_copy(0)
                for i in range(Ksteps):
                    step(i, i == Ksteps - 1)
                drain(Ksteps)
                e1.record()
                barrier()
                ms = max_over_ranks(e0.elapsed_time(e1))
                return {"value": world * B * Ksteps / (ms * 1e-3), "ms_per_step": ms / Ksteps}

            # PCIe links idle down between phases of this script (the CPU arm runs for seconds before this leg on a
            # fresh box): bring the H2D path to its steady state with an untimed burst of copies first, otherwise
            # the short timed region (K steps of ~0.3 ms) measures the link's ramp-up (observed: 28 vs 52 GB/s)
            t_burst = time.perf_counter()
            while time.perf_counter() - t_burst < 0.3:
                for j in range(8):
                    slots[j % 2].copy_(host[j % n_host], non_blocking=True)
                torch.cuda.synchronize()
            variants = {}
            variants["strict"] = run_e2e(True, True, False, K)
            variants["pipelined"] = run_e2e(True, True, True, K)
            if world > 1:
                variants["h2d_only"] = run_e2e(True, False, True, K)
                variants["collective_only"] = run_e2e(False, True, True, K)
            variants["device_resident_module"] = run_e2e(False, False, True, K)
            # headline: the faster of the two complete definitions (both copy every step's inputs H2D, both read one loss
            # per step on the host); at N = 1 the strict loop is PCIe-bound either way, at N > 1 the pipelined one wins
            # because the collective leaves the critical path
            head_name = "pipelined" if variants["pipelined"]["value"] >= variants["strict"]["value"] else "strict"
            head = variants[head_name]
            res["e2e"] = {"value": head["value"], "unit": UNIT, "headline_variant": head_name,
                          "h2d_bytes_per_step": bytes_pair, "d2h_bytes_per_step": 4,
                          "ms_per_step": head["ms_per_step"],
                          "h2d_gbs_per_gpu": bytes_pair / (head["ms_per_step"] * 1e-3) / 1e9,
                          "definition": "strict: every step copies its inputs H2D from pinned memory (next batch prefetched on a copy "
                                        "stream), runs fwd+bwd (+ the bucket all-reduce at N > 1) and reads its own loss with .item(); "
                                        "pipelined: same copies and collective, but the host reads the previous step's loss, so it never "
                                        "stalls inside a step",
                          "variants": variants,
                          "host_affinity": numa_note,
                          "collective": (f"one NCCL all-reduce of {bucket.nbytes} B (generator-grad bucket + loss) per step"
                                         if bucket is not None else "none (1 GPU)")}
        res["clocks"] = sampler.stop() if rank == 0 else None
        del pool
        torch.cuda.empty_cache()
        return res

    K, Wm = args.steps, args.warmup
    main = measure(args.workload, K, Wm, with_e2e=True, keep_last=args.dump_outputs is not None)
    if args.dump_outputs is not None and rank == 0:
        dump_outputs(args.dump_outputs, main["last_step"])
    others = {}
    if not args.no_extra:
        for name in WORKLOADS:
            if name != args.workload:
                r = measure(name, 40 if name == "c2x" else max(20, min(K, 200)), Wm, with_e2e=False)
                others[name] = {"workload": r["wl"]["desc"], "images_per_s": r["images_per_s"],
                                "ms_per_step": r["ms_step"], "ms_fwd": r["ms_fwd"], "ms_bwd": r["ms_bwd"],
                                "hbm_frac_fwd": r["roofline_fwd"] / hbm_peak, "hbm_frac_bwd": r["roofline_bwd"] / hbm_peak,
                                "hbm_frac_pair": r["roofline_pair"] / hbm_peak}

    if not args.no_extra:
        # BASELINE.json configs[3]: Best-Buddy patch search, batch 64 of 192x192 crops (per GPU), through the
        # public module (pyramid built by libsrst).  FP32-FMA bound, no HBM claim (SURVEY.md 8d).
        from srgan_st_b200 import BestBuddyLoss
        Bb, Hb, Wb = 64, 192, 192
        gen = torch.Generator(device=dev).manual_seed(99 + rank)
        gtb = torch.rand(Bb, 3, Hb, Wb, device=dev, generator=gen)
        xb = (gtb + 0.1 * torch.randn(Bb, 3, Hb, Wb, device=dev, generator=gen)).clamp(0, 1).requires_grad_(True)
        mb = BestBuddyLoss(pyramid="fused")
        for _ in range(3):
            mb(xb, gtb).backward()
        torch.cuda.synchronize()
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
        tf = tb = 0.0
        nb = 10
        for _ in range(nb):
            ev[0].record(); lb = mb(xb, gtb); ev[1].record(); lb.backward(); ev[2].record()
            torch.cuda.synchronize()
            tf += ev[0].elapsed_time(ev[1]) / nb; tb += ev[1].elapsed_time(ev[2]) / nb
        Nq = (Hb // 3) * (Wb // 3)
        Mc = Nq + ((Hb // 2) // 3) * ((Wb // 2) // 3) + ((Hb // 4) // 3) * ((Wb // 4) // 3)
        others["bb_c4"] = {"workload": "Best-Buddy loss fwd+bwd, batch 64 x 3x192x192 per GPU (configs[3]), "
                                       "pyramid+pack+search+loss kernels through the nn.Module",
                           "images_per_s_per_gpu": Bb / ((tf + tb) * 1e-3), "ms_fwd": tf, "ms_bwd": tb,
                           "reference_flop_per_step": 4.0 * Nq * Mc * 27 * Bb,
                           "reference_tflops_equiv": 4.0 * Nq * Mc * 27 * Bb / (tf * 1e-3) / 1e12,
                           "note": "reference work = two [N,M,27] SGEMMs (utils.py:183); the search kernel does ONE "
                                   "filtered dot product per pair and re-scores survivors exactly (bit-identical indices)"}
        # the same crops with a non-default patch geometry (BestBuddyLoss(ksize=4, stride=4), loss.py:86): the exact
        # all-pairs path (bb_generic.cuh) -- both dot products of every pair, no filter
        mg = BestBuddyLoss(ksize=4, pad=0, stride=4, pyramid="fused")
        for _ in range(2):
            mg(xb, gtb).backward()
        torch.cuda.synchronize()
        tfg = tbg = 0.0
        for _ in range(nb):
            ev[0].record(); lb = mg(xb, gtb); ev[1].record(); lb.backward(); ev[2].record()
            torch.cuda.synchronize()
            tfg += ev[0].elapsed_time(ev[1]) / nb; tbg += ev[1].elapsed_time(ev[2]) / nb
        Ng = (Hb // 4) * (Wb // 4)
        Mg = Ng + ((Hb // 2) // 4) * ((Wb // 2) // 4) + ((Hb // 4) // 4) * ((Wb // 4) // 4)
        others["bb_k4s4"] = {"workload": "Best-Buddy loss fwd+bwd with ksize=4, pad=0, stride=4 (48-dim patches), batch 64 x "
                                         "3x192x192 per GPU, exact all-pairs kernels through the nn.Module",
                             "images_per_s_per_gpu": Bb / ((tfg + tbg) * 1e-3), "ms_fwd": tfg, "ms_bwd": tbg,
                             "reference_tflops_equiv": 4.0 * Ng * Mg * 48 * Bb / (tfg * 1e-3) / 1e12}
        del gtb, xb

    if not args.no_extra:
        # BASELINE.json configs[1]: "SRResNet warmup.py step with ST + MSE loss, batch 64, 96x96 patches": the loop body of
        # warmup.py:83-96 (generator forward, the registered criteria with .item() after each, backward, Adam) on an
        # SRResNet-shaped generator built from stock torch layers (the generator is ballast here, not part of the hot
        # path: 16 residual blocks, 64 channels, two PixelShuffle stages -- 1 547 350 parameters like model.py:193).
        nn = torch.nn

        class _Res(nn.Module):
            def __init__(self, c):
                super().__init__()
                self.f = nn.Sequential(nn.Conv2d(c, c, 3, 1, 1, bias=False), nn.BatchNorm2d(c), nn.PReLU(),
                                       nn.Conv2d(c, c, 3, 1, 1, bias=False), nn.BatchNorm2d(c))

            def forward(self, x):
                return x + self.f(x)

        class _SRResNet(nn.Module):
            def __init__(self, c=64, nb=16):
                super().__init__()
                self.head = nn.Sequential(nn.Conv2d(3, c, 9, 1, 4), nn.PReLU())
                self.body = nn.Sequential(*[_Res(c) for _ in range(nb)])
                self.fuse = nn.Sequential(nn.Conv2d(c, c, 3, 1, 1, bias=False), nn.BatchNorm2d(c))
                self.up = nn.Sequential(*[nn.Sequential(nn.Conv2d(c, 4 * c, 3, 1, 1), nn.PixelShuffle(2), nn.PReLU())
                                          for _ in range(2)])
                self.tail = nn.Conv2d(c, 3, 9, 1, 4)

            def forward(self, x):
                h = self.head(x)
                return self.tail(self.up(h + self.fuse(self.body(h)))).clamp(0.0, 1.0)

        from srgan_st_b200 import StructureTensorPixelLoss
        torch.manual_seed(7 + rank)
        gen = _SRResNet().to(dev)
        n_par = sum(p.numel() for p in gen.parameters())
        Bw = 64
        gtw = torch.rand(Bw, 3, 96, 96, device=dev)
        lrw = torch.nn.functional.interpolate(gtw, scale_factor=0.25, mode="bicubic", align_corners=False).clamp(0, 1)
        opt = torch.optim.Adam(gen.parameters(), lr=1e-4)

        def loop_body(crits):
            gen.zero_grad()
            sr = gen(lrw)
            loss = torch.tensor(0.0, device=dev)
            vals = {}
            for name, (c, w) in crits.items():
                l = c(sr, gtw)
                loss = loss + l * w
                vals[name] = (l * w).item()            # warmup.py:93
            loss.backward()
            opt.step()

        def timed(fn, n=20, warm=5):
            for _ in range(warm):
                fn()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(n):
                fn()
            e1.record()
            torch.cuda.synchronize()
            return e0.elapsed_time(e1) / n

        two = {"Pixel": (nn.MSELoss(), 1.0), "ST": (StructureTensorLoss(), 1.0 / 3.0)}
        one = {"ST+Pixel": (StructureTensorPixelLoss(st_weight=1.0 / 3.0, pixel_weight=1.0), 1.0)}
        only_px = {"Pixel": (nn.MSELoss(), 1.0)}
        ms_two, ms_one, ms_px = timed(lambda: loop_body(two)), timed(lambda: loop_body(one)), timed(lambda: loop_body(only_px))
        others["warmup_step"] = {
            "workload": f"warmup.py:83-96 loop body, SRResNet-shaped generator ({n_par} params, stock torch/cuDNN eager) + Adam, "
                        f"batch {Bw} x 96x96 HR per GPU (BASELINE configs[1])",
            "ms_per_step_pixel_plus_st": ms_two, "ms_per_step_fused_st_pixel": ms_one, "ms_per_step_pixel_only": ms_px,
            "images_per_s_per_gpu": Bw / (ms_two * 1e-3),
            "st_criterion_cost_ms": ms_two - ms_px,
            "note": "the ST criterion's whole cost inside the step (module call, two kernels, .item()) is the difference to the "
                    "Pixel-only step; the reference's own criteria on the same step are timed by `--impl reference` "
                    "(reference_gpu_unfused.warmup_step_reference)"}
        del gen, opt, gtw, lrw
        torch.cuda.empty_cache()

    os.sched_setaffinity(0, all_cpus)
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu:
        wl = main["wl"]
        big = wl["H"] * wl["W"] > 1e6
        probe, cores = cpu_port_images_per_sec(wl["H"], wl["W"], 4 if big else 128)
        n = int(min(max(probe * 6, cores), 200000)) if not big else max(cores, 8)
        v, cores = cpu_port_images_per_sec(wl["H"], wl["W"], n)
        port = {"value": v, "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"{n} synthetic images of 3x{wl['H']}x{wl['W']}, oracle/st_oracle.py fp32 fwd+bwd, one process per core"}
        cpu = port
        if ref_available():
            try:
                rp = RefCpuPool()
                sub = 1 if big else 4
                probe, cores = rp.images_per_sec(wl["H"], wl["W"], max(2, cores) if big else 4 * cores, sub)
                n = int(min(max(probe * 12, cores), 50000)) if not big else max(cores, 8)
                v, cores = rp.images_per_sec(wl["H"], wl["W"], n, sub)
                rp.close()
                cpu = {"value": v, "unit": UNIT, "cores": cores, "kind": "reference",
                       "sample": f"{n} synthetic images of 3x{wl['H']}x{wl['W']}, oracle/_ref loss.py StructureTensorLoss (the unmodified "
                                 f"reference on ATen/MKL-DNN, fp32) fwd+bwd, one process per core, sub-batches of {sub}",
                       "port": port}
            except Exception as e:  # the reference could not run on this host: keep the port, say why
                port["reference_error"] = repr(e)

    if rank == 0:
        wl = main["wl"]
        out = {
            "metric": METRIC, "value": main["images_per_s"], "unit": UNIT, "n_gpus": world, "steps": K, "warmup": Wm,
            "ms_per_step": main["ms_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": _config_dict(wl, world, extra={
                "l2_policy": f"inputs cycle through a pool of {main['pool_n']} batches (> 2x L2) so every step is L2-cold",
                "timing": "CUDA graph of K (fwd,bwd) kernel pairs on one stream, CUDA events, max over ranks, best of 3"}),
            "clocks": main["clocks"],
            "e2e": main.get("e2e"),
            "gpu_launches": 2 * K,
            "roofline": {"bound": "hbm", "kernel": "st_forward_march_kernel", "achieved": main["roofline_fwd"], "peak": hbm_peak,
                         "unit": "GB/s", "frac": main["roofline_fwd"] / hbm_peak,
                         "traffic": _traffic(args.workload, "st_forward_march_kernel"),
                         "traffic_source": "profiles/r02_traffic.json (ncu --set full, dram__bytes_read+write per launch)",
                         "peak_source": peak_src, "bytes_per_pixel": BYTES_FWD,
                         "backward": {"kernel": "st_backward_kernel", "achieved": main["roofline_bwd"],
                                      "frac": main["roofline_bwd"] / hbm_peak, "bytes_per_pixel": BYTES_BWD},
                         "fwd_bwd_pair": {"achieved": main["roofline_pair"], "frac": main["roofline_pair"] / hbm_peak,
                                          "bytes_per_pixel": BYTES_FWD + BYTES_BWD},
                         "ms_fwd": main["ms_fwd"], "ms_bwd": main["ms_bwd"],
                         # context (DESIGN.md section 3): the kernels are bound on-chip, not by HBM.  Minimum fp32
                         # lane-operations of the algorithm (no halo recompute) against the FP32 pipe at the
                         # sampled SM clock (128 lanes/clk/SM, tools/ubench_fma.cu)
                         "fp32_pipe": _fp32_context(torch, main, wl)},
            "cpu_baseline": cpu,
            "loss_check": main["loss"],
            "other_workloads": others,
        }
        emit(out)
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="c2", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary workloads")
    ap.add_argument("--no-cpu", action="store_true", help="skip the cpu_baseline leg")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the loss and d_sr of the last timed step as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl == "reference":
        ap.error("--dump-outputs applies to the CUDA path (--impl ours)")
    if args.gpus > 1 and "RANK" not in os.environ and args.impl != "reference":
        # convenience: re-launch under torchrun on one node
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", "29533", os.path.abspath(__file__)] + sys.argv[1:]
        return subprocess.call(cmd)
    # stdout carries exactly ONE JSON line: everything else that writes to fd 1 (NCCL's version banner,
    # library chatter) is sent to stderr, and the line itself goes to the saved descriptor
    global _RESULT_FD
    sys.stdout.flush()
    _RESULT_FD = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference(args)
    return run_gpu(args)


_RESULT_FD = None
DUMP_ARRAY_BYTES = 60 << 20   # per array; loss + d_sr stay within 64 MB


def dump_outputs(path, arrays):
    """Write each array as path/<name>.npy (float32); one larger than DUMP_ARRAY_BYTES is written as
    path/<name>_sample.npy, its values at a fixed, seeded, sorted set of flat indices."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    for name, a in arrays.items():
        a = np.ascontiguousarray(a, dtype=np.float32)
        if a.nbytes > DUMP_ARRAY_BYTES:
            idx = np.sort(np.random.default_rng(0).choice(a.size, DUMP_ARRAY_BYTES // 4, replace=False))
            a, name = a.reshape(-1)[idx], name + "_sample"
        np.save(os.path.join(path, name + ".npy"), a)


def emit(obj):
    line = (json.dumps(obj) + "\n").encode()
    if _RESULT_FD is None:
        sys.stdout.write(line.decode()); sys.stdout.flush()
    else:
        os.write(_RESULT_FD, line)


if __name__ == "__main__":
    sys.exit(main())
