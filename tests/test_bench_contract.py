"""bench.py: the reference arm's JSON line, the algorithmic-bytes formula of SURVEY.md 8(d) and the
outputs --dump-outputs writes (CPU), and the dump of a real run being its last timed step (GPU)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _bench():
    sys.path.insert(0, ROOT)
    import bench
    return bench


def test_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` times the reference's own CPU path (oracle/_ref, or the port when the reference
    was not built) and prints one JSON line with the arm's keys."""
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "0", "--frames", "2", "--classes", "2"],
                         capture_output=True, text=True, timeout=300, cwd=ROOT)
    assert res.returncode == 0, res.stderr[-2000:]
    lines = [ln for ln in res.stdout.splitlines() if ln.startswith("{")]
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference"
    assert d["metric"] == _bench().METRIC and d["unit"] == "frames/s" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["steps"] == 1 and d["vs_baseline"] is None and d["data"] == "synthetic"
    assert d["config"]["frames_per_gpu"] == 2 and d["config"]["classes"] == 2
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0


def test_stage_bytes_sum_to_the_survey_formula():
    """bench.stage_bytes splits SURVEY 8(d)'s B_frame = 12P + 12KP + 24(d+1)P + 8(d+1)M + (d+1)(8M + 16KM) + 8KM."""
    bench = _bench()
    for P, d, K, M in ((224 * 224, 5, 2, 56141.0), (224 * 224, 5, 10, 3070.0), (448 * 448, 3, 2, 735.6), (1, 1, 1, 2.0)):
        want = 12 * P + 12 * K * P + 24 * (d + 1) * P + 8 * (d + 1) * M + (d + 1) * (8 * M + 16 * K * M) + 8 * K * M
        assert abs(bench.frame_bytes(P, d, K, M) - want) < 1e-6 * want
    # the worked example of the survey: 224^2, d = 5, K = 2, noise (M = 56 141) -> 26.1 MB per frame
    assert abs(bench.frame_bytes(224 * 224, 5, 2, 56141.0) / 1e6 - 26.1) < 0.1


def test_dump_outputs_writes_the_whole_gradient_or_a_fixed_sample(tmp_path, monkeypatch):
    import torch
    bench = _bench()
    loss = torch.tensor([-1.5])
    grad = torch.arange(2 * 3 * 4 * 5, dtype=torch.float32).reshape(2, 3, 4, 5)
    bench.dump_outputs(str(tmp_path / "whole"), loss, grad)
    assert np.load(tmp_path / "whole" / "loss.npy").tolist() == [-1.5]
    got = np.load(tmp_path / "whole" / "segmentations_grad.npy")
    assert got.dtype == np.float32 and np.array_equal(got, grad.numpy())
    # above the cap: the values at the same ascending positions on every call
    monkeypatch.setattr(bench, "DUMP_MAX_VALUES", 16)
    bench.dump_outputs(str(tmp_path / "a"), loss, grad)
    bench.dump_outputs(str(tmp_path / "b"), loss, grad)
    a = np.load(tmp_path / "a" / "segmentations_grad.npy")
    assert a.shape == (16,) and np.all(np.diff(a) > 0) and np.array_equal(a, np.load(tmp_path / "b" / "segmentations_grad.npy"))


@pytest.mark.parametrize("extra", [["--steps", "0"], ["--impl", "reference", "--dump-outputs", "out"]])
def test_bench_refuses_arguments_it_cannot_honour(extra):
    res = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py")] + extra, capture_output=True, text=True,
                         timeout=120, cwd=ROOT)
    assert res.returncode == 2 and "error" in res.stderr and not res.stdout.strip()


@pytest.mark.gpu
def test_dumped_outputs_are_those_of_the_last_timed_step(tmp_path):
    """--steps 202 over 4 rotated input batches: the last timed step is the one on batch 1 (seed 1), while the
    per-stage pass after it (min(steps, 200) steps) ends on batch 3.  Only rank 0 writes: the same run as rank 1
    (RANK, as torchrun sets it) leaves DIR alone."""
    import torch
    from tcam_wsol_video_b200 import synth
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    n, k = 2, 2

    def run(steps, out_dir, rank):
        env = dict(os.environ, RANK=str(rank), LOCAL_RANK="0", WORLD_SIZE="1")
        return subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", str(steps),
                               "--warmup", "1", "--rotate", "4", "--frames", str(n), "--classes", str(k),
                               "--no-cpu-baseline", "--no-e2e", "--no-extra", "--dump-outputs", str(out_dir)],
                              capture_output=True, text=True, timeout=600, cwd=ROOT, env=env)

    res = run(202, tmp_path / "rank0", 0)
    assert res.returncode == 0, res.stderr[-2000:]
    assert json.loads(res.stdout.strip().splitlines()[-1])["steps"] == 202
    b = _bench()
    img = torch.from_numpy(synth.make_images(n, b.H, b.W, "noise", seed=1)).cuda()
    seg = torch.from_numpy(synth.make_segs(n, k, b.H, b.W, seed=1)).cuda().requires_grad_(True)
    loss = DenseCRFLoss(weight=2e-9, sigma_rgb=b.SIGMA_RGB, sigma_xy=b.SIGMA_XY, scale_factor=1.0)(
        images=img, segmentations=seg)
    loss.backward()
    got_loss = np.load(tmp_path / "rank0" / "loss.npy")
    got_grad = np.load(tmp_path / "rank0" / "segmentations_grad.npy")
    assert got_loss.dtype == np.float32 and got_grad.shape == (n, k, b.H, b.W)
    assert abs(float(got_loss[0]) - loss.item()) <= 1e-5 * abs(loss.item())
    want = seg.grad.cpu().numpy()
    assert np.abs(got_grad - want).max() <= 1e-5 * np.abs(want).max()
    res = run(2, tmp_path / "rank1", 1)
    assert res.returncode == 0, res.stderr[-2000:]
    assert not (tmp_path / "rank1").exists() and not res.stdout.strip()
