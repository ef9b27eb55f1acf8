#!/usr/bin/env python
"""bench.py -- CRF-loss fwd+bwd frames/s at 224^2 on N B200s (BASELINE.json's metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # our CUDA path
    python bench.py --impl reference [...]                         # the reference's CPU path
    python bench.py --dump-outputs DIR [...]                       # also write the last timed step's outputs

A step is one fwd+bwd of DenseCRFLoss over one batch of synthetic frames per GPU
(configs[1] of BASELINE.json: 32 frames x 10 classes x 224x224, sigma_rgb=15, sigma_xy=100):
lattice build + splat + blur + slice + loss reduction (forward) and the gradient kernel (backward).
For N > 1 the step goes through the product's sharding module (tcam_wsol_video_b200/dist.py, ShardedCRFLoss):
every rank runs its own --frames (weak scaling; 8 GPUs = configs[4]'s 256 frames), or --global-frames 256 shards a
fixed batch (strong scaling); the path's only exchange, a 4-byte all-reduce of the loss over NCCL, is issued every
step inside the timed region (on a side stream with the default --reduction global_async).

One JSON line is printed by rank 0; see DESIGN.md "Measurement" for every key.
"""
from __future__ import annotations

import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

METRIC = "crf_loss_fwd_bwd_frames_per_sec_224"
UNIT = "frames/s"
H = W = 224
SIGMA_RGB, SIGMA_XY = 15.0, 100.0
D = 5


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=600, help="timed steps (default: >= 0.5 s of timed region)")
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--frames", type=int, default=32, help="frames per GPU per step")
    ap.add_argument("--classes", type=int, default=10)
    ap.add_argument("--kind", choices=["noise", "natural"], default="noise")
    ap.add_argument("--rotate", type=int, default=4, help="distinct input batches cycled through (defeats L2 reuse)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the short runs on the other input regimes")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 -> min(steps, 50)")
    ap.add_argument("--global-frames", type=int, default=0,
                    help="strong scaling: a fixed global batch sharded over the ranks (BASELINE configs[4]: 256)")
    ap.add_argument("--reduction", choices=["global_async", "global", "local"], default="global_async",
                    help="N > 1: how dist.ShardedCRFLoss forms the loss (see tcam_wsol_video_b200/dist.py)")
    ap.add_argument("--no-train-step", dest="train_step", action="store_false",
                    help="skip the ResNet-50 train-step context run (other_inputs.train_step_resnet50)")
    ap.add_argument("--no-occupancy-sweep", dest="occupancy_sweep", action="store_false",
                    help="skip the 448x448 hash-load sweep (other_inputs.occupancy_sweep_448)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write what the last timed step returned (rank 0: loss, segmentation gradient) as DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


# ---------------------------------------------------------------------------
# algorithmic bytes (SURVEY.md §8d, restated in DESIGN.md "Roofline accounting")
# ---------------------------------------------------------------------------
def stage_bytes(P: int, d: int, K: int, M: float):
    """Algorithmic bytes per FRAME of each pipeline stage; they sum to SURVEY §8(d)'s B_frame."""
    dp1 = d + 1
    return {
        "build": 12 * P + 8 * dp1 * P,             # image in; offset + barycentric out
        "neighbour": 8 * dp1 * M,                  # neighbour table out
        "splat": 4 * K * P + 8 * dp1 * P + 4 * K * M,   # seg in; offset + bary in; value table out
        "blur": dp1 * (8 * M + 16 * K * M),        # per axis: neighbour ids in, 3 values in, 1 value out
        "slice": 8 * dp1 * P + 4 * K * M + 4 * K * P,   # offset + bary in; value table in; AS out
        "loss": 0,
        "backward": 4 * K * P,                     # gradient out
        "prepare": 0,                              # table clear: not algorithmic traffic
        "seed": 0,
    }


def frame_bytes(P, d, K, M):
    return float(sum(stage_bytes(P, d, K, M).values()))


# ---------------------------------------------------------------------------
# clocks
# ---------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock and throttle reasons of one GPU through NVML while the timed region runs."""

    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, device_index: int):
        self.samples = []
        self.reasons = set()
        self.max_mhz = None
        self._stop = threading.Event()
        self._thread = None
        self._h = None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            self._nvml = pynvml
            try:
                uuid = str(torch.cuda.get_device_properties(device_index).uuid)
                if not uuid.startswith("GPU-"):
                    uuid = "GPU-" + uuid
                self._h = pynvml.nvmlDeviceGetHandleByUUID(uuid)
            except Exception:
                self._h = pynvml.nvmlDeviceGetHandleByIndex(device_index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self._h, pynvml.NVML_CLOCK_SM))
        except Exception:
            self._h = None

    def _loop(self):
        nv = self._nvml
        while not self._stop.is_set():
            try:
                mhz = int(nv.nvmlDeviceGetClockInfo(self._h, nv.NVML_CLOCK_SM))
                try:
                    mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self._h))
                except Exception:
                    mask = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self._h))
                self.samples.append(mhz)
                for bit, name in self.REASONS.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def start(self):
        if os.environ.get("TCAMCRF_BENCH_NOCLOCK") == "1":
            return
        if self._h is not None:
            self._thread = threading.Thread(target=self._loop, daemon=True)
            self._thread.start()

    def stop(self):
        self._stop.set()
        if self._thread is not None:
            self._thread.join(timeout=2)

    def summary(self):
        if not self.samples:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.samples)), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(self.samples)}


# ---------------------------------------------------------------------------
# CPU reference timing (oracle/_ref when built, else the C port)
# ---------------------------------------------------------------------------
def cpu_fwd_bwd_frames_per_sec(frames: int, K: int, kind: str, reps: int, warmup: int = 1, keep_result: bool = False):
    """Times the reference's CPU implementation of the same fwd+bwd on `frames` frames of the workload."""
    import oracle
    from tcam_wsol_video_b200 import synth

    fn, which = oracle.best_filter(color=False)
    img = synth.make_images(frames, H, W, kind, seed=0)
    seg = synth.make_segs(frames, K, H, W, seed=0)
    cores = len(os.sched_getaffinity(0))
    if which == "reference":
        # torchrun exports OMP_NUM_THREADS=1; give the reference every host core it is allowed to use
        # (its own code then takes min(max_threads, N), bilateralfilter.cpp:45-47)
        oracle.ref_set_threads(cores)
        threads = min(oracle.load_ref()[0].ref_omp_max_threads(), frames)
    else:
        threads = 1
    times = []
    for i in range(warmup + reps):
        t0 = time.perf_counter()
        out = oracle.densecrf_loss_fwd_bwd(img, seg, SIGMA_RGB, SIGMA_XY, 1.0, fn)
        dt = time.perf_counter() - t0
        if i >= warmup:
            times.append(dt)
    res = (frames / min(times), frames / (sum(times) / len(times)), which, threads, cores, times)
    return res + ((out[0], out[1]),) if keep_result else res


def cpu_context_runs(K: int, kind: str):
    """SURVEY 8d's two other CPU arms, as context next to the all-cores number: (i) one thread, (iii) all cores with
    glibc malloc kept from returning the per-class buffers to the OS (the reference allocates and frees two
    [H*W] float arrays per class, bilateralfilter.cpp:31-37).  Small samples; (iii) needs the environment set
    before the process starts, so it runs in a child."""
    out = {}
    try:
        import oracle
        if not oracle.have_ref():
            return out
        cores = len(os.sched_getaffinity(0))
        fn, _ = oracle.best_filter(color=False)
        from tcam_wsol_video_b200 import synth
        img = synth.make_images(2, H, W, kind, seed=0)
        seg = synth.make_segs(2, K, H, W, seed=0)
        oracle.ref_set_threads(1)
        best = 1e30
        for _ in range(2):
            t0 = time.perf_counter()
            oracle.densecrf_loss_fwd_bwd(img, seg, SIGMA_RGB, SIGMA_XY, 1.0, fn)
            best = min(best, time.perf_counter() - t0)
        oracle.ref_set_threads(cores)
        out["one_thread"] = {"value": 2 / best, "unit": UNIT, "cores": 1, "sample": "2 frames, best of 2"}
        env = dict(os.environ, MALLOC_MMAP_THRESHOLD_="1073741824", MALLOC_TRIM_THRESHOLD_="1073741824",
                   MALLOC_TOP_PAD_="268435456", OMP_NUM_THREADS=str(cores))
        code = ("import sys, time; sys.path.insert(0, %r); import bench\n"
                "b, m, which, threads, cores, t = bench.cpu_fwd_bwd_frames_per_sec(%d, %d, %r, reps=2, warmup=1)\n"
                "print('MALLOC_TUNED', b, threads)" % (ROOT, min(32, max(cores, 2)), K, kind))
        res = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=120)
        for ln in res.stdout.splitlines():
            if ln.startswith("MALLOC_TUNED"):
                _, v, th = ln.split()
                out["malloc_tuned"] = {"value": float(v), "unit": UNIT, "cores": int(th),
                                       "sample": f"{min(32, max(cores, 2))} frames, best of 2 after 1 warm-up, "
                                                 "MALLOC_MMAP_THRESHOLD_/TRIM_THRESHOLD_=1 GiB, TOP_PAD_=256 MiB"}
    except Exception as exc:   # context only: never fail the bench line over it
        out["error"] = repr(exc)[:200]
    return out


def run_reference(args, rank: int, world: int):
    if rank != 0:
        return
    frames = args.frames
    t0 = time.perf_counter()
    # bounded sample: keep the whole run within ~150 s whatever --steps is (calibrate on a few frames)
    cal = min(frames, max(2, len(os.sched_getaffinity(0))))
    _, cal_fps, *_ = cpu_fwd_bwd_frames_per_sec(cal, args.classes, args.kind, reps=1, warmup=0)
    budget_frames = int(150.0 * cal_fps / max(args.steps + args.warmup, 1))
    frames = max(1, min(frames, budget_frames))
    best, mean, which, threads, cores, times = cpu_fwd_bwd_frames_per_sec(frames, args.classes, args.kind,
                                                                          reps=max(args.steps, 1),
                                                                          warmup=max(args.warmup, 0))
    value = frames * len(times) / sum(times)
    line = {
        "impl": "reference",
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(times),
        "warmup": args.warmup, "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, 1),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": which, "host_cores": cores,
                         "sample": f"{frames} frames x K={args.classes} x {H}x{W} ({args.kind}), fwd+bwd, "
                                   f"{len(times)} steps, OpenMP over frames as shipped"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
        "wall_s": time.perf_counter() - t0,
    }
    emit(line)


def workload_config(args, world, frames=None, n_global=None):
    frames = args.frames if frames is None else frames
    n_global = frames * world if n_global is None else n_global
    which = ("BASELINE configs[4]: batch-sharded CRF loss over %d frames" % n_global) if args.global_frames > 0 \
        else "BASELINE configs[1]: DenseCRFLoss fwd+bwd"
    return {
        "workload": f"{which}, {frames} frames/GPU x {args.classes} classes x "
                    f"{H}x{W} RGB, sigma_rgb={SIGMA_RGB:g}, sigma_xy={SIGMA_XY:g}, 5-D lattice, '{args.kind}' images",
        "frames_per_gpu": frames, "classes": args.classes, "height": H, "width": W,
        "image_kind": args.kind, "global_frames": n_global,
        "parallelism": (f"dp{world}: dist.ShardedCRFLoss(reduction='{args.reduction}'), frames sharded, one 4-byte "
                        f"all-reduce per step") if world > 1 else "single GPU",
        "l2": f"{args.rotate} distinct input batches rotated; per-step working set (segs+AS+grad+tables) > 126 MB L2",
    }


# ---------------------------------------------------------------------------
# our arm
# ---------------------------------------------------------------------------
def source_sha() -> str:
    """sha256 (first 16 hex digits) of the CUDA sources the timed kernels are built from: ties profiles/traffic.json
    (ncu captures) to the build that is being timed."""
    import hashlib
    h = hashlib.sha256()
    for name in ("tcamcrf.cu", "lattice.cuh"):
        with open(os.path.join(ROOT, "tcam_wsol_video_b200", "csrc", name), "rb") as f:
            h.update(f.read())
    return h.hexdigest()[:16]


def load_traffic(kind: str, K: int, N: int):
    """Per-stage ncu counters of one launch (profiles/traffic.json, written by tools/make_traffic.py from the
    `ncu --set full` raw pages); None when there is no capture of this workload or it is from another build."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        doc = json.load(open(path))
    except Exception:
        return None, "no profiles/traffic.json"
    if doc.get("_meta", {}).get("source_sha") != source_sha():
        return None, "profiles/traffic.json is from another build of csrc/ (stale): dropped"
    ent = doc.get("workloads", {}).get(f"{kind}:K{K}:N{N}")
    if not ent:
        return None, f"no ncu capture of {kind}:K{K}:N{N}"
    return ent, doc["_meta"].get("capture", "")


def timed_loop(torch, fn, steps, warmup=0):
    for i in range(warmup):
        fn(i)
        if i < 3:
            # let the library's density hint of this workspace land (it travels device -> pinned host word behind the
            # call): a burst of calls queued faster than the first one finishes would all be planned without it
            torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for i in range(steps):
        fn(i)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def link_probe(torch, h2d_bytes: int, d2h_bytes: int, reps: int = 10):
    """What the PCIe link alone takes for one step's traffic: the step's host->device bytes on one stream and its
    device->host bytes on another, concurrently, pinned memory both ways (best of `reps`, wall clock around a sync)."""
    dev = torch.device("cuda", torch.cuda.current_device())
    hin = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8).pin_memory()
    hout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8).pin_memory()
    din = torch.empty(max(h2d_bytes, 1), dtype=torch.uint8, device=dev)
    dout = torch.empty(max(d2h_bytes, 1), dtype=torch.uint8, device=dev)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    best = {"both": 1e30, "h2d": 1e30, "d2h": 1e30}
    for mode in ("both", "h2d", "d2h"):
        for _ in range(reps):
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            if mode in ("both", "h2d"):
                with torch.cuda.stream(s1):
                    din.copy_(hin, non_blocking=True)
            if mode in ("both", "d2h"):
                with torch.cuda.stream(s2):
                    hout.copy_(dout, non_blocking=True)
            torch.cuda.synchronize()
            best[mode] = min(best[mode], time.perf_counter() - t0)
    return {"link_bound_ms": 1e3 * best["both"], "h2d_alone_ms": 1e3 * best["h2d"], "d2h_alone_ms": 1e3 * best["d2h"],
            "h2d_gbs": h2d_bytes / best["h2d"] / 1e9, "d2h_gbs": d2h_bytes / best["d2h"] / 1e9}


def run_ours(args, rank: int, local_rank: int, world: int):
    import torch
    import torch.distributed as dist

    from tcam_wsol_video_b200 import _lib, ops, synth
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    from tcam_wsol_video_b200.dist import ShardedCRFLoss, shard_range

    assert torch.cuda.is_available(), "bench.py (impl=ours) needs a GPU; there is no CPU path"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    lib = _lib.load()
    assert lib.tcamcrf_device_count() >= 1

    K = args.classes
    if args.global_frames > 0:   # strong scaling (BASELINE configs[4]): a fixed batch sharded over the ranks
        lo, hi = shard_range(args.global_frames, rank, world)
        N, n_global = hi - lo, args.global_frames
    else:                        # weak scaling: every rank its own --frames
        N, n_global = args.frames, args.frames * world
    P = H * W
    sets = []
    for r in range(max(args.rotate, 1)):
        seed = 1000 * rank + r
        img = torch.from_numpy(synth.make_images(N, H, W, args.kind, seed=seed))
        seg = torch.from_numpy(synth.make_segs(N, K, H, W, seed=seed))
        sets.append((img.pin_memory(), seg.pin_memory(), img.to(dev), seg.to(dev).requires_grad_(True)))
    crf = DenseCRFLoss(weight=2e-9, sigma_rgb=SIGMA_RGB, sigma_xy=SIGMA_XY, scale_factor=1.0).to(dev)
    # N > 1: the product's sharding module (tcam_wsol_video_b200/dist.py).  "global_async": every rank's loss is its
    # share of the global mean (its gradient needs no exchange), the 4-byte all-reduce runs on a side stream behind
    # the forward kernels and the reduced value is read one step late -- nothing on the compute stream waits for NCCL.
    sharded = ShardedCRFLoss(crf, reduction=args.reduction) if world > 1 else None
    reduced = []

    def step(i):
        _, _, img_d, seg_d = sets[i % len(sets)]
        seg_d.grad = None
        if sharded is None:
            loss = crf(images=img_d, segmentations=seg_d)
        else:
            if args.reduction == "global_async":
                prev = sharded.global_loss()        # last step's reduced loss (its all-reduce finished long ago)
                if prev is not None:
                    reduced[:] = [prev]
            loss = sharded(img_d, seg_d, global_batch=n_global)
        loss.backward()
        return loss

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # lattice size of this input (for the algorithmic-bytes formula)
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, SIGMA_RGB, SIGMA_XY)
    _, _, ws = ops.crf_forward(sets[0][2], sets[0][3].detach(), cfg, check=True)
    _, m_total = ops.workspace_status(ws)
    M = m_total / N

    # ---- parity of what is being timed: rank 0's first batch through the module against the CPU reference
    # (filled in below, next to the cpu_baseline leg that produces the reference values)
    parity_gpu = None
    if rank == 0 and not args.no_cpu_baseline:
        crf1 = DenseCRFLoss(weight=1.0, sigma_rgb=SIGMA_RGB, sigma_xy=SIGMA_XY, scale_factor=1.0)
        nf = min(N, 32)
        seg_p = sets[0][3].detach()[:nf].clone().requires_grad_(True)
        loss_p = crf1(images=sets[0][2][:nf], segmentations=seg_p)
        loss_p.backward()
        parity_gpu = (float(loss_p.item()), seg_p.grad.cpu().numpy(), nf)
        del seg_p, loss_p

    sampler = ClockSampler(local_rank)
    sampler.start()   # warm-up, timed region and the per-stage pass: the same load throughout
    for i in range(args.warmup):
        step(i)
    barrier()

    launches0 = lib.tcamcrf_launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    barrier()
    ev0.record()
    for i in range(args.steps - 1):
        step(i)
    loss_last = step(args.steps - 1).detach()   # the graph (it holds the step's buffers) is freed as after any step
    ev1.record()
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = lib.tcamcrf_launch_count() - launches0
    # rank 0's outputs of the last timed step; every step returns fresh tensors, so these stay as that step left them
    dumped = (loss_last, sets[(args.steps - 1) % len(sets)][3].grad) if args.dump_outputs and rank == 0 else None
    del loss_last

    # per-stage times: the same steps again with CUDA events around every stage (tcamcrf_profile_*).  Kept out of
    # the timed region above because an event record between two kernels stops the next kernel's blocks from
    # becoming resident while the previous one drains (programmatic dependent launch).
    lib.tcamcrf_profile_enable(1)
    lib.tcamcrf_profile_read(None, None, 1)
    prof_steps = min(args.steps, 200)
    for i in range(prof_steps):
        step(i)
    barrier()
    lib.tcamcrf_profile_enable(0)
    st_ms = (ctypes.c_double * len(_lib.STAGES))()
    st_ln = (ctypes.c_longlong * len(_lib.STAGES))()
    lib.tcamcrf_profile_read(st_ms, st_ln, 1)

    t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total = float(t.item())
    ms_per_step = ms_total / args.steps
    value = n_global * args.steps / (ms_total / 1e3)

    # the collective on its own: latency of one 4-byte all-reduce on the compute stream (what "global" would add to
    # every step; "global_async" keeps it off the critical path)
    collective_us = None
    if world > 1:
        x = torch.zeros(1, device=dev)
        collective_us = 1e3 * timed_loop(torch, lambda i: dist.all_reduce(x), 200, warmup=20) / 200
        t = torch.tensor([collective_us], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        collective_us = float(t.item())

    def max_over_ranks(dt):
        t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def wall_loop(fn, steps):
        for i in range(3):
            fn(i)
        barrier()
        t0 = time.perf_counter()
        for i in range(steps):
            fn(i)
        torch.cuda.synchronize()
        return max_over_ranks(time.perf_counter() - t0)

    # ---- end to end through the host-pointer C ABI (pinned host buffers, copies inside the timed region)
    e2e = None
    e2e_trainer = None
    if not args.no_e2e:
        e2e_steps = args.e2e_steps or min(args.steps, 50)
        loss_h = torch.zeros(1).pin_memory()
        grad_h = torch.empty(N, K, H, W).pin_memory()
        cfg_h = _lib.make_config(_lib.FEAT_XY_RGB, 3, SIGMA_RGB, SIGMA_XY)

        def e2e_step(i):
            img_h, seg_h, _, _ = sets[i % len(sets)]
            rc = lib.tcamcrf_loss_fwd_bwd_host(ctypes.byref(cfg_h), img_h.data_ptr(), seg_h.data_ptr(),
                                               loss_h.data_ptr(), grad_h.data_ptr(), N, K, H, W, 2e-9)
            _lib.check(rc, "tcamcrf_loss_fwd_bwd_host")

        dt = wall_loop(e2e_step, e2e_steps)
        h2d = int(4 * N * 3 * P + 4 * N * K * P + 4)
        d2h = int(4 * N * K * P + 4 + 4)
        e2e = {"value": n_global * e2e_steps / dt, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
               "steps": e2e_steps, "ms_per_step": 1e3 * dt / e2e_steps,
               "api": "tcamcrf_loss_fwd_bwd_host (host pointers in, loss + gradient out)",
               "copies_declared": ["images float32 H2D", "segmentations float32 H2D", "gradient float32 D2H",
                                   "loss + status D2H"]}
        # the PCIe link alone, same bytes, same run: the bound of this call
        probe = link_probe(torch, h2d, d2h)
        probe["link_bound_ms"] = max_over_ranks(probe["link_bound_ms"] / 1e3) * 1e3
        e2e.update(probe)
        e2e["frac_of_link"] = e2e["link_bound_ms"] / e2e["ms_per_step"]

        # ---- the call the reference's trainer makes (dlib/losses/tcam.py:113-115): frames from pinned host memory
        # (train_wsol.py:1128 keeps raw_img on the CPU), segmentations where the network left them (device), loss read
        # back; the gradient stays on the device for the backbone's backward pass
        def module_step(i):
            img_h, _, _, seg_d = sets[i % len(sets)]
            seg_d.grad = None
            loss = crf(images=img_h, segmentations=seg_d)
            loss.backward()
            return loss.item()

        dtm = wall_loop(module_step, e2e_steps)
        # the same call with uint8 frames from the loader (SURVEY 8f.1): a quarter of the bytes on the wire
        img8_h = [(s[0].to(torch.uint8)).pin_memory() for s in sets]

        def module_step_u8(i):
            seg_d = sets[i % len(sets)][3]
            seg_d.grad = None
            loss = crf(images=img8_h[i % len(sets)], segmentations=seg_d)
            loss.backward()
            return loss.item()

        dtu = wall_loop(module_step_u8, e2e_steps)
        e2e_trainer = {
            "value": n_global * e2e_steps / dtu, "unit": UNIT, "ms_per_step": 1e3 * dtu / e2e_steps,
            "steps": e2e_steps, "h2d_bytes_per_step": int(N * 3 * P), "d2h_bytes_per_step": 4,
            "api": "DenseCRFLoss(images=pinned host uint8 [N,3,H,W], segmentations=device float32).backward(); "
                   "loss.item()  -- the reference's own call shape (train_wsol.py:1128, losses/tcam.py:113-115)",
            "copies_declared": ["images uint8 H2D (overlapped with the lattice build, section by section)",
                                "loss float32 D2H (.item())"],
            "segmentations": "device-resident, as the network leaves them (the reference copies them D2H and AS "
                             "H2D around its CPU filter, dense_crf_loss.py:44-61)",
            "float32_frames": {"value": n_global * e2e_steps / dtm, "ms_per_step": 1e3 * dtm / e2e_steps,
                               "h2d_bytes_per_step": int(4 * N * 3 * P), "d2h_bytes_per_step": 4},
        }
        # kept under the old keys too (round-1 readers)
        e2e["trainer_call"] = {"value": e2e_trainer["float32_frames"]["value"], "unit": UNIT,
                               "ms_per_step": e2e_trainer["float32_frames"]["ms_per_step"]}
        e2e["trainer_call_u8"] = {"value": e2e_trainer["value"], "unit": UNIT, "ms_per_step": e2e_trainer["ms_per_step"]}

    sampler.stop()   # the GPU has been under this benchmark's load since the warm-up: timed region, per-stage pass, e2e legs

    # ---- the same step on the other input regimes (short, device-resident; context for the headline number)
    extra = {}
    if world == 1 and not args.no_extra:
        extra = other_inputs(args, torch, dev, lib, N, K, local_rank)

    if rank != 0:
        return

    # ---- roofline: the whole step in SURVEY 8(d)'s algorithmic bytes (headline), every stage underneath
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback (of fallback)"
    sb = stage_bytes(P, D, K, M)
    counters, traffic_note = load_traffic(args.kind, K, N)
    stages = {}
    step_dram = 0.0
    for i, name in enumerate(_lib.STAGES):
        if st_ln[i] <= 0:
            continue
        per_launch_ms = st_ms[i] / st_ln[i]
        launches_per_step = st_ln[i] / prof_steps
        alg = sb[name] * N / launches_per_step
        ent = {"ms_per_step": st_ms[i] / prof_steps, "launches_per_step": launches_per_step,
               "ms_per_launch": per_launch_ms, "algorithmic_bytes_per_launch": alg,
               "algorithmic_gbs": alg / (per_launch_ms * 1e-3) / 1e9 if per_launch_ms > 0 else None}
        ent["gbs"] = ent["algorithmic_gbs"]
        c = (counters or {}).get(name)
        if c and per_launch_ms > 0:
            ent["dram_bytes_per_launch"] = c["dram_bytes"]
            ent["dram_gbs"] = c["dram_bytes"] / (per_launch_ms * 1e-3) / 1e9
            ent["frac_dram"] = ent["dram_gbs"] / peak
            ent["dram_over_algorithmic"] = c["dram_bytes"] / alg if alg > 0 else None
            for k2 in ("lts_sectors", "lts_requests", "lts_requests_atom", "lts_requests_red", "l1_sectors_atom",
                       "l1_sectors_red"):
                if k2 in c:
                    ent[k2] = c[k2]
            if c.get("lts_requests"):
                # the L2-side view: requests and 32-byte sectors per second of the live launch (the kernels that only
                # gather and stream -- blur, neighbour, slice -- all sit at ~190-220 G requests/s on B200) and ncu's
                # own percentage of the sustained sector peak (measured under ncu, cold cache)
                ent["lts_requests_per_s"] = c["lts_requests"] / (per_launch_ms * 1e-3)
                ent["lts_sectors_per_s"] = c["lts_sectors"] / (per_launch_ms * 1e-3)
                ent["lts_sectors_pct_of_peak_ncu"] = c.get("lts_sectors_pct_of_peak")
            step_dram += c["dram_bytes"] * launches_per_step
        stages[name] = ent
    dom = max(stages, key=lambda s_: stages[s_]["ms_per_step"]) if stages else None
    b_frame = frame_bytes(P, D, K, M)
    fps_per_gpu = value / world
    roofline = {
        "bound": "hbm", "scope": "whole step (all kernels of the fwd+bwd)",
        "achieved": b_frame * fps_per_gpu / 1e9, "peak": peak, "unit": "GB/s",
        "frac": b_frame * fps_per_gpu / 1e9 / peak,
        "traffic": step_dram if counters else None,
        "traffic_what": ("measured DRAM bytes of one step (sum over its kernels of ncu dram__bytes_read.sum + "
                         "dram__bytes_write.sum per launch); " + str(traffic_note)) if counters else traffic_note,
        "peak_source": peak_src, "bytes_per_frame": b_frame, "vertices_per_frame": M,
        "formula": "SURVEY 8(d): B_frame * frames/s per GPU / peak",
        "pipeline": {"bytes_per_frame": b_frame, "vertices_per_frame": M,
                     "achieved": b_frame * fps_per_gpu / 1e9, "frac": b_frame * fps_per_gpu / 1e9 / peak},
        "stages": stages,
    }
    if counters and ms_per_step > 0:
        roofline["dram"] = {"achieved": step_dram / (ms_per_step * 1e-3) / 1e9, "unit": "GB/s",
                            "frac": step_dram / (ms_per_step * 1e-3) / 1e9 / peak,
                            "what": "measured DRAM bytes of the step over the live step time"}
    if dom:
        d_ = stages[dom]
        roofline["dominant_kernel"] = {
            "kernel": dom, "ms_per_launch": d_["ms_per_launch"],
            "algorithmic_bytes_per_launch": d_["algorithmic_bytes_per_launch"],
            "algorithmic_gbs": d_["algorithmic_gbs"],
            "frac_algorithmic": d_["algorithmic_gbs"] / peak if d_["algorithmic_gbs"] else None,
            "traffic": d_.get("dram_bytes_per_launch"), "dram_gbs": d_.get("dram_gbs"), "frac_dram": d_.get("frac_dram"),
            "note": "SURVEY 8(d)'s bytes of the blur count two neighbour-row gathers per vertex which the L2 serves: "
                    "its algorithmic rate may exceed the HBM peak; frac_dram is what the HBM carried"}

    cpu = None
    parity = None
    if world == 1 and not args.no_cpu_baseline:
        frames = min(N, 32)
        best, mean, which, threads, cores, times, ref_out = cpu_fwd_bwd_frames_per_sec(
            frames, K, args.kind, reps=3, warmup=1, keep_result=True)
        cpu = {"value": best, "unit": UNIT, "cores": threads, "kind": which, "host_cores": cores,
               "sample": f"{frames} frames x K={K} x {H}x{W} ({args.kind}), fwd+bwd, best of 3 after 1 warm-up, "
                         f"OpenMP over frames as shipped", "mean_value": mean,
               "context": cpu_context_runs(K, args.kind)}
        if parity_gpu is not None and parity_gpu[2] == frames:
            ref_loss, ref_grad = float(ref_out[0]), ref_out[1]
            loss_rel = abs(parity_gpu[0] - ref_loss) / abs(ref_loss)
            grad_rel = float(np.abs(parity_gpu[1] - ref_grad).max() / np.abs(ref_grad).max())
            parity = {"loss_rel": loss_rel, "grad_rel": grad_rel, "tolerance": 1e-4,
                      "ok": bool(loss_rel < 1e-4 and grad_rel < 1e-4), "against": which,
                      "what": f"DenseCRFLoss(weight=1) fwd+bwd on the first {frames} frames of rank 0's first timed "
                              f"batch (seed 0) against the CPU {which}'s loss and gradient on the same inputs; "
                              f"grad_rel = max |diff| / max |grad|"}

    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True,
        "scaling": "strong" if args.global_frames > 0 else "weak", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic", "config": workload_config(args, world, N, n_global),
        "roofline": roofline, "cpu_baseline": cpu, "parity": parity, "e2e": e2e, "e2e_trainer": e2e_trainer,
        "gpu_launches": int(launches), "collective_us": collective_us,
        "clocks": dict(sampler.summary(), window="warm-up + timed region + per-stage pass + e2e legs"),
        "other_inputs": extra,
    }
    if dumped is not None:
        dump_outputs(args.dump_outputs, *dumped)
    emit(line)
    if parity is not None and not parity["ok"]:
        sys.stderr.write("bench.py: PARITY FAILED: %r\n" % (parity,))
        sys.exit(3)


def other_inputs(args, torch, dev, lib, N, K, local_rank):
    """Short device-resident runs on the other input regimes and the other BASELINE configs (context)."""
    from tcam_wsol_video_b200 import _lib, ops, synth
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    crf = DenseCRFLoss(weight=2e-9, sigma_rgb=SIGMA_RGB, sigma_xy=SIGMA_XY, scale_factor=1.0).to(dev)
    extra = {}
    for kind, k in (("natural", K), ("noise", 2), ("natural", 2)):
        if kind == args.kind and k == K:
            continue
        img = torch.from_numpy(synth.make_images(N, H, W, kind, seed=7)).to(dev)
        seg = torch.from_numpy(synth.make_segs(N, k, H, W, seed=7)).to(dev).requires_grad_(True)

        def fn(i):
            seg.grad = None
            crf(images=img, segmentations=seg).backward()

        ms = timed_loop(torch, fn, 100, warmup=10)
        extra[f"{kind}_k{k}"] = {"value": N * 100 / (ms / 1e3), "unit": UNIT, "steps": 100, "ms_per_step": ms / 100}
        del img, seg

    # BASELINE configs[2] without the backbone: per step, for 32 clips -- temporal max over the current + 4
    # previous frames' CAMs fused with fg/bg seeding, CRF loss from logits (K=2, uint8 frames resident on the
    # GPU, fused softmax) + cross-entropy on the seeds, backward to the logits.
    try:
        from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLossFromLogits
        from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder
        low = torch.from_numpy(synth.make_low_res_cams(N, 5, 28, 28, seed=3)).squeeze(2)
        cams = torch.nn.functional.interpolate(low, size=(H, W), mode="bilinear", align_corners=False).to(dev)
        roi = (cams.amax(dim=1, keepdim=True) >= 0.5).long()
        img8 = torch.from_numpy(synth.make_images(N, H, W, "natural", seed=3).astype(np.uint8)).to(dev)
        logits = torch.randn((N, 2, H, W), device=dev, requires_grad=True)
        seeder = TCAMSeeder(seed_tech="seed_weighted", min_=1, max_=1, max_p=0.6, min_p=0.1, fg_erode_k=11,
                            fg_erode_iter=0, ksz=3, support_background=True, multi_label_flag=False,
                            seg_ignore_idx=-255, cuda_id=local_rank, roi_method="roi_all", p_min_area_roi=0.05,
                            use_roi=True, rng_parity=False)
        crf2 = DenseCRFLossFromLogits(2e-9, SIGMA_RGB, SIGMA_XY, 1.0)

        def tcam_step(i):
            logits.grad = None
            seeds, _ = seeder.forward_stack(cams, roi)
            loss = crf2(images=img8, logits=logits) + torch.nn.functional.cross_entropy(logits, seeds,
                                                                                         ignore_index=-255)
            loss.backward()

        ms = timed_loop(torch, tcam_step, 100, warmup=10)
        extra["tcam_seed_crf_step_natural_k2"] = {
            "value": N * 100 / (ms / 1e3), "unit": UNIT, "steps": 100, "ms_per_step": ms / 100,
            "what": "temporal max (T=5) + seeding + CRF-from-logits + CE on seeds, fwd+bwd, no backbone"}
        ms = timed_loop(torch, lambda i: seeder.forward_stack(cams, roi), 100, warmup=10)
        extra["tcam_seeder_forward_stack"] = {"ms_per_call": ms / 100, "samples": N, "frames_per_sample": 5,
                                              "what": "TCAMSeeder.forward_stack alone (temporal max + fg/bg seeds)"}
        # the same step with the sparse seeds: FusedTcamLosses = CE on the labelled pixels + CRF as one autograd node
        from tcam_wsol_video_b200.losses import ConRanFieldTcams, FusedTcamLosses, SelfLearningTcams
        fused = FusedTcamLosses(SelfLearningTcams(cuda_id=local_rank, lambda_=1.0),
                                ConRanFieldTcams(cuda_id=local_rank, lambda_=2e-9, sigma_rgb=SIGMA_RGB,
                                                 sigma_xy=SIGMA_XY, scale_factor=1.0, fuse_softmax=True))

        def tcam_step_fused(i):
            logits.grad = None
            seeds, _ = seeder.forward_stack(cams, roi, sparse=True)
            fused(epoch=0, fcams=logits, raw_img=img8, seeds=seeds).backward()

        ms = timed_loop(torch, tcam_step_fused, 100, warmup=10)
        extra["tcam_seed_crf_step_natural_k2_fused"] = {
            "value": N * 100 / (ms / 1e3), "unit": UNIT, "steps": 100, "ms_per_step": ms / 100,
            "what": "the same step with TCAMSeeder(sparse=True) + FusedTcamLosses: no label map, the cross-entropy "
                    "computed on the labelled pixels and added in place to the CRF gradient"}
        # the same step captured once in a CUDA graph and replayed (what a trainer does with torch.cuda.graphs): the
        # ~25 launches of the step cost more on the CPU than on the GPU, the replay shows the GPU side alone
        try:
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for i in range(3):
                    tcam_step(i)
                    torch.cuda.synchronize()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            logits.grad = None
            with torch.cuda.graph(graph, stream=side):
                tcam_step(0)
            ms = timed_loop(torch, lambda i: graph.replay(), 100, warmup=10)
            extra["tcam_seed_crf_step_natural_k2_cuda_graph"] = {
                "value": N * 100 / (ms / 1e3), "unit": UNIT, "steps": 100, "ms_per_step": ms / 100,
                "what": "the (unfused) step captured with torch.cuda.graph and replayed"}
            del graph
            with torch.cuda.stream(side):
                for i in range(3):
                    tcam_step_fused(i)
                    torch.cuda.synchronize()
            torch.cuda.current_stream().wait_stream(side)
            graph = torch.cuda.CUDAGraph()
            logits.grad = None
            with torch.cuda.graph(graph, stream=side):
                tcam_step_fused(0)
            ms = timed_loop(torch, lambda i: graph.replay(), 100, warmup=10)
            extra["tcam_seed_crf_step_natural_k2_fused_cuda_graph"] = {
                "value": N * 100 / (ms / 1e3), "unit": UNIT, "steps": 100, "ms_per_step": ms / 100,
                "what": "the fused step captured with torch.cuda.graph and replayed"}
            del graph
        except Exception as exc:
            extra["tcam_seed_crf_step_natural_k2_cuda_graph"] = {"error": repr(exc)[:200]}
    except Exception as exc:  # context only; never fail the headline line
        extra["tcam_seed_crf_step_natural_k2"] = {"error": repr(exc)[:200]}

    # BASELINE configs[3]: lattice-size stress at 448x448 -- the 5-D colour lattice (x, y, r, g, b) and the 3-D
    # grayscale one (x, y, gray), 8 frames, K=2, noise frames (largest lattices), fwd+bwd like the headline; and
    # the hash-table occupancy sweep: the same step with the primary table tier sized for loads 0.125 .. 2.
    try:
        n4, k4, s4 = 8, 2, 448
        img4 = torch.from_numpy(synth.make_images(n4, s4, s4, "noise", seed=11)).to(dev)
        seg4 = torch.from_numpy(synth.make_segs(n4, k4, s4, s4, seed=11)).to(dev)
        g_one = torch.ones(1, device=dev)
        sweep = {}
        for name, feat_channels in (("xyrgb_5d", 3), ("xygray_3d", 1)):
            for load in (None, 0.125, 0.25, 0.5, 1.0, 2.0):
                if load is not None and not args.occupancy_sweep:
                    continue
                cfg4 = _lib.make_config(_lib.FEAT_XY_RGB, feat_channels, SIGMA_RGB, SIGMA_XY,
                                        **({} if load is None else {"hash_load": load}))

                def step4(i):
                    as4, _, _ = ops.crf_forward(img4, seg4, cfg4, want_loss=True, n_norm=float(n4))
                    ops.crf_backward(as4, g_one, float(n4))

                ms = timed_loop(torch, step4, 30, warmup=5)
                ws4 = ops.crf_forward(img4, seg4, cfg4, check=True)[2]
                _, m4 = ops.workspace_status(ws4)
                ent = {"value": n4 * 30 / (ms / 1e3), "unit": UNIT, "steps": 30, "frames": n4, "ms_per_step": ms / 30,
                       "vertices_per_frame": m4 / n4}
                if load is None:
                    extra[f"noise_448_{name}_k2"] = ent
                else:
                    sweep[f"{name}:load{load:g}"] = ent
        if sweep:
            extra["occupancy_sweep_448"] = dict(sweep, what="primary table tier sized for `hash_load` = vertices (at 1.2 "
                                                "per pixel) / slots; above ~1 most vertices live in the overflow tier")
        del img4, seg4
    except Exception as exc:
        extra["noise_448"] = {"error": repr(exc)[:200]}

    if args.train_step:
        try:
            extra["train_step_resnet50"] = train_step_context(args, torch, dev, local_rank)
        except Exception as exc:
            extra["train_step_resnet50"] = {"error": repr(exc)[:300]}
    return extra


def train_step_context(args, torch, dev, local_rank):
    """BASELINE configs[2] as written: a ResNet-50 train step on 32 clips of 224x224 with the TCAM losses around
    it -- what share of the step this op is.  torchvision ResNet-50 at stride 8 (dlib/encoders/resnet.py:78-79 keeps
    layer3/4 at stride 1 with dilation) + a 1x1 two-class head + bilinear upsampling, AMP (fp16 autocast like
    `--amp True`), SGD; losses as in the README recipe: SelfLearningTcams (CE on TCAMSeeder's seeds) +
    ConRanFieldTcams (CRF, lambda 2e-9).  Random weights, synthetic frames; the backbone is PyTorch's, not ours."""
    import torchvision
    from tcam_wsol_video_b200 import synth
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLossFromLogits
    from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder
    B = 32
    net = torchvision.models.resnet50(weights=None, replace_stride_with_dilation=[False, True, True])
    net.fc = torch.nn.Identity()
    net.avgpool = torch.nn.Identity()

    class Model(torch.nn.Module):
        def __init__(self):
            super().__init__()
            self.body = torch.nn.Sequential(net.conv1, net.bn1, net.relu, net.maxpool, net.layer1, net.layer2,
                                            net.layer3, net.layer4)
            self.head = torch.nn.Conv2d(2048, 2, 1)

        def forward(self, x):
            y = self.head(self.body(x))
            return torch.nn.functional.interpolate(y, size=x.shape[2:], mode="bilinear", align_corners=False)

    model = Model().to(dev).to(memory_format=torch.channels_last)
    opt = torch.optim.SGD(model.parameters(), lr=1e-3, momentum=0.9)
    scaler = torch.amp.GradScaler("cuda")
    img_np = synth.make_images(B, H, W, "natural", seed=5)
    raw8_h = torch.from_numpy(img_np.astype(np.uint8)).pin_memory()          # raw_img stays on the CPU (train_wsol.py:1128)
    raw32_h = torch.from_numpy(img_np).pin_memory()
    x = ((torch.from_numpy(img_np) / 255.0 - 0.45) / 0.225).to(dev).contiguous(memory_format=torch.channels_last)
    low = torch.from_numpy(synth.make_low_res_cams(B, 5, 28, 28, seed=3)).squeeze(2)
    cams = torch.nn.functional.interpolate(low, size=(H, W), mode="bilinear", align_corners=False).to(dev)
    roi = (cams.amax(dim=1, keepdim=True) >= 0.5).long()
    fixed_seeds = torch.randint(0, 2, (B, H, W), device=dev)
    seeder = TCAMSeeder(seed_tech="seed_weighted", min_=1, max_=1, max_p=0.6, min_p=0.1, fg_erode_k=11,
                        fg_erode_iter=0, ksz=3, support_background=True, multi_label_flag=False, seg_ignore_idx=-255,
                        cuda_id=local_rank, roi_method="roi_all", p_min_area_roi=0.05, use_roi=True, rng_parity=False)
    crf = DenseCRFLossFromLogits(2e-9, SIGMA_RGB, SIGMA_XY, 1.0)

    def make_step(mode):
        def fn(i):
            opt.zero_grad(set_to_none=True)
            with torch.autocast("cuda", dtype=torch.float16):
                logits = model(x)
            lf = logits.float()
            if mode == "ours":
                seeds, _ = seeder.forward_stack(cams, roi)
                loss = torch.nn.functional.cross_entropy(lf, seeds, ignore_index=-255) + crf(images=raw8_h, logits=lf)
            elif mode == "reference_cpu_op":
                seeds, _ = seeder.forward_stack(cams, roi)
                loss = torch.nn.functional.cross_entropy(lf, seeds, ignore_index=-255) + \
                    2e-9 * reference_cpu_crf(torch).apply(raw32_h, torch.softmax(lf, dim=1))
            else:
                loss = torch.nn.functional.cross_entropy(lf, fixed_seeds)
            scaler.scale(loss).backward()
            scaler.step(opt)
            scaler.update()
        return fn

    out = {"what": "torchvision ResNet-50 (stride 8) + 1x1 head + bilinear upsampling, batch 32 x 224x224, fp16 "
                   "autocast, SGD step; 'natural' frames, K=2; ms per train step", "batch": B}
    ms_without = timed_loop(torch, make_step("none"), 10, warmup=3) / 10
    ms_ours = timed_loop(torch, make_step("ours"), 10, warmup=3) / 10
    out["without_op_ms"] = ms_without
    out["with_our_op_ms"] = ms_ours
    out["op_share_of_step"] = (ms_ours - ms_without) / ms_ours
    if not args.no_cpu_baseline:
        try:
            ms_ref = timed_loop(torch, make_step("reference_cpu_op"), 2, warmup=1) / 2
            out["with_reference_cpu_op_ms"] = ms_ref
            out["reference_op_share_of_step"] = (ms_ref - ms_without) / ms_ref
            out["reference_cpu_op"] = ("the reference's DenseCRFLossFunction restated around its own C++ filter "
                                       "(oracle/_ref when built): synchronize, segmentations D2H, CPU filter on all "
                                       "host cores, AS H2D (dense_crf_loss.py:36-74); cpu_baseline leg only")
        except Exception as exc:
            out["with_reference_cpu_op_ms"] = {"error": repr(exc)[:200]}
    return out


_REF_CPU_CRF = None


def reference_cpu_crf(torch):
    """The reference's DenseCRFLossFunction (dlib/crf/dense_crf_loss.py:36-74) around the reference's own C++ filter, as an
    autograd Function (torch is imported lazily in this file, hence the factory).  cpu_baseline leg only -- never on the
    product path."""
    global _REF_CPU_CRF
    if _REF_CPU_CRF is None:
        class Fn(torch.autograd.Function):
            @staticmethod
            def forward(ctx, images, segmentations):
                import oracle
                fn, _ = oracle.best_filter(color=False)
                if oracle.have_ref():
                    oracle.ref_set_threads(len(os.sched_getaffinity(0)))
                torch.cuda.synchronize()
                n, k, h, w = segmentations.shape
                seg = segmentations.detach().float().cpu().numpy()
                AS = fn(images.numpy(), seg, n, k, h, w, SIGMA_RGB, SIGMA_XY).reshape(seg.shape)
                loss = -float((seg.ravel() * AS.ravel()).sum(dtype=np.float32)) / n
                ctx.AS = torch.from_numpy(AS).to(segmentations.device)
                ctx.N = n
                return torch.tensor([loss], device=segmentations.device)

            @staticmethod
            def backward(ctx, g):
                return None, -2 * g * ctx.AS / ctx.N

        _REF_CPU_CRF = Fn
    return _REF_CPU_CRF


DUMP_MAX_VALUES = 1 << 23   # 32 MiB of float32


def dump_outputs(out_dir: str, loss, grad) -> None:
    """Writes the loss (loss.npy) and the gradient of the segmentations (segmentations_grad.npy) in float32.  A
    gradient of more than DUMP_MAX_VALUES values is written as its values at a fixed set of flat positions
    (numpy default_rng(0), ascending), the same for every build of the project, so that two builds can be compared
    output for output."""
    import torch
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "loss.npy"), loss.detach().float().cpu().numpy())
    grad = grad.detach()
    if grad.numel() > DUMP_MAX_VALUES:
        idx = np.sort(np.random.default_rng(0).choice(grad.numel(), DUMP_MAX_VALUES, replace=False))
        grad = grad.reshape(-1)[torch.from_numpy(idx).to(grad.device)]
    np.save(os.path.join(out_dir, "segmentations_grad.npy"), grad.float().cpu().numpy())


_REAL_STDOUT = None


def emit(line: dict) -> None:
    """The one JSON line goes to the real stdout; everything else (NCCL banners, warnings) to stderr."""
    text = json.dumps(line) + "\n"
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, text.encode())
    else:
        sys.stdout.write(text)
        sys.stdout.flush()


def main():
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)   # libraries that print to fd 1 (e.g. "NCCL version ...") must not pollute the JSON line
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(args, rank, local_rank, world)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
