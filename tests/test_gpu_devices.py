"""GPU suite, several devices in ONE process: the library keeps its limits, kernel attributes, streams, events and
buffers per device.  Which device a process touches first decides what a process-wide cache would hold, so each
scenario runs in a fresh interpreter (tests/devices_worker.py) that uses cuda:0 first, then cuda:1.  Needs >= 2 GPUs;
skipped otherwise."""
import json
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("scenario", [
    "fused_seeding",        # tcam_seed_fused at 224x224 needs the shared-memory opt-in on each device
    "two_kernel_seeding",   # so does seed_select_smem_kernel
    "crf_paths",            # density hints, the host-frames copy lane, the host-pointer buffers and graphs
    "stage_timing",         # the profiler's events belong to the device whose stream records them
])
def test_second_device_in_one_process(scenario):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs at least two GPUs")
    res = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "devices_worker.py"), scenario],
                         capture_output=True, text=True, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    line = [ln for ln in res.stdout.splitlines() if ln.startswith("DEVICES_WORKER ")][-1]
    assert json.loads(line[len("DEVICES_WORKER "):])["scenario"] == scenario
