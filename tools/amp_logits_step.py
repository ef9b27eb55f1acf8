#!/usr/bin/env python
"""Times the TCAM loss step with fp16 / bf16 logits: read natively by the logits kernels, against the same logits cast
to float32 first (`.float()` before the loss; autograd casts the gradient back), which is what the loss did before
it read 2-byte logits.

    python tools/amp_logits_step.py [--steps 250] [--rounds 4] [--out DIR]

Step = seeder forward_stack (temporal max + seeding, in-kernel draws) + FusedTcamLosses forward and backward, on 32
clips of 224 x 224, K = 2, natural frames as pinned uint8 on the host (the trainer's call shape).  Timed with CUDA
events, eagerly and as CUDA-graph replays, the two variants alternating in the same process (`rounds` x `steps` each).
A separate run under torch.profiler lists the time per kernel.  Writes amp_logits_step.json under --out."""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from tcam_wsol_video_b200 import synth  # noqa: E402
from tcam_wsol_video_b200.losses import ConRanFieldTcams, FusedTcamLosses, SelfLearningTcams  # noqa: E402
from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder  # noqa: E402

B, T, K, H, W = 32, 3, 2, 224, 224


def card():
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        limit = "unknown"
    return name, limit


class Step:
    """One variant of the step on its own static inputs (same values for both variants)."""

    def __init__(self, dtype, native):
        self.native = native
        g = torch.Generator().manual_seed(0)
        self.cams = torch.rand((B, T, H, W), generator=g).cuda()
        self.roi = torch.ones((B, 1, H, W), dtype=torch.long, device="cuda")
        self.frames = torch.from_numpy(synth.make_images(B, H, W, "natural", seed=1).astype(np.uint8)).pin_memory()
        self.logits = (3 * torch.randn((B, K, H, W), generator=g)).to(dtype).cuda().requires_grad_(True)
        self.seeder = TCAMSeeder(seed_tech="seed_weighted", min_=1, max_=1, max_p=0.6, min_p=0.1, fg_erode_k=11,
                                 fg_erode_iter=0, ksz=3, support_background=True, multi_label_flag=False,
                                 seg_ignore_idx=-255, cuda_id=0, roi_method="roi_all", p_min_area_roi=0.05,
                                 use_roi=True, rng_parity=False)
        self.loss = FusedTcamLosses(
            SelfLearningTcams(cuda_id=0, lambda_=1.0, seg_ignore_idx=-255),
            ConRanFieldTcams(cuda_id=0, lambda_=2e-9, sigma_rgb=15., sigma_xy=100., scale_factor=1.0,
                             fuse_softmax=True, seg_ignore_idx=-255))
        self.graph = None

    def __call__(self):
        seeds, _ = self.seeder.forward_stack(self.cams, self.roi, sparse=True)
        fcams = self.logits if self.native else self.logits.float()
        total = self.loss(epoch=0, fcams=fcams, raw_img=self.frames, seeds=seeds)
        total.backward()
        return total

    def eager(self, n):
        for _ in range(n):
            self.logits.grad = None
            self()

    def capture(self):
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            self.eager(3)
            self.logits.grad = None
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=s):
                self()
        torch.cuda.current_stream().wait_stream(s)

    def replay(self, n):
        for _ in range(n):
            self.graph.replay()


def timed(fn, n):
    start, end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    start.record()
    fn(n)
    end.record()
    end.synchronize()
    return start.elapsed_time(end) / n


def kernel_times(step, n):
    from torch.profiler import ProfilerActivity, profile
    step.eager(3)
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        step.eager(n)
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        t = getattr(e, "device_time_total", None) or getattr(e, "cuda_time_total", 0)
        if t > 0 and e.count >= n:
            out[e.key] = (round(t / n, 2), e.count // n)
    return dict(sorted(out.items(), key=lambda kv: -kv[1][0]))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=250)
    ap.add_argument("--rounds", type=int, default=4)
    ap.add_argument("--profile-steps", type=int, default=20)
    ap.add_argument("--out", default=".", help="directory for amp_logits_step.json (default: the current one)")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a GPU"
    name, limit = card()
    result = {"card": name, "power_limit": limit, "shape": [B, K, H, W], "steps": a.steps, "rounds": a.rounds,
              "ms_per_step": {}, "kernels_us_per_step": {}}
    print(f"{name}, power limit {limit}; {B} x {K} x {H} x {W} logits, {a.rounds} rounds x {a.steps} steps per cell")
    for dt_name, dtype in (("float16", torch.float16), ("bfloat16", torch.bfloat16)):
        native, cast = Step(dtype, True), Step(dtype, False)
        for s in (native, cast):
            s.eager(5)
            s.capture()
        torch.cuda.synchronize()
        # same gradient from both paths (up to the CRF term's splat-atomic order and the rounding to `dtype`): the
        # seeder draws from torch's generator, so both steps start from the same generator state
        for s in (native, cast):
            torch.manual_seed(7)
            s.eager(1)
        gn, gc = native.logits.grad.float(), cast.logits.grad.float()
        agree = float((gn - gc).abs().max() / gc.abs().max())
        for mode in ("eager", "graph"):
            times = {"native": [], "cast": []}
            for _ in range(a.rounds):
                for label, s in (("native", native), ("cast", cast)):
                    times[label].append(timed(s.eager if mode == "eager" else s.replay, a.steps))
            cell = {k: {"median": float(np.median(v)), "min": float(np.min(v)), "all": [round(x, 4) for x in v]}
                    for k, v in times.items()}
            cell["gain_us"] = round(1000 * (cell["cast"]["median"] - cell["native"]["median"]), 2)
            result["ms_per_step"][f"{dt_name}/{mode}"] = cell
            print(f"{dt_name:9s} {mode:5s}: native {cell['native']['median']:.4f} ms, cast {cell['cast']['median']:.4f}"
                  f" ms per step (median of {a.rounds}); gain {cell['gain_us']:+.2f} us")
        result[f"{dt_name}/grad_rel_diff"] = agree
        print(f"{dt_name:9s} gradient, native against cast: max |diff| / max |cast| = {agree:.2e}")
        for label, s in (("native", native), ("cast", cast)):
            result["kernels_us_per_step"][f"{dt_name}/{label}"] = kernel_times(s, a.profile_steps)
        del native, cast
        torch.cuda.synchronize()
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "amp_logits_step.json"), "w") as f:
        json.dump(result, f, indent=1)
    for key, ks in result["kernels_us_per_step"].items():
        print(key)
        for kname, (us, cnt) in list(ks.items())[:14]:
            print(f"  {us:9.2f} us  x{cnt}  {kname[:110]}")


if __name__ == "__main__":
    main()
