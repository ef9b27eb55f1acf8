"""Randomised parity run: random shapes, class counts, lattice dimensions, bandwidths, image kinds, frame dtypes and
forced kernel variants, each filtered on the GPU and compared with the oracle's C restatement (rel 1e-4, the north
star's tolerance).  python tools/r2_fuzz.py [seconds] [seed]    (a stand-in for the sanitizer runs this pool refuses:
hundreds of odd shapes through every variant, on one workspace that keeps being resized)"""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
import oracle
from tcam_wsol_video_b200 import _lib, ops, synth

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 90.0
rng = np.random.default_rng(int(sys.argv[2]) if len(sys.argv) > 2 else 1)
t0 = time.time()
cases = fails = 0
worst = 0.0
kinds = {}
while time.time() - t0 < budget:
    n = int(rng.integers(1, 6)); k = int(rng.integers(1, 13))
    h = int(rng.integers(1, 72)); w = int(rng.integers(1, 72))
    kind = "noise" if rng.random() < 0.5 else "natural"
    colour = rng.random() < 0.3
    srgb = float(rng.choice([3.0, 8.0, 15.0, 40.0, 120.0])); sxy = float(rng.choice([5.0, 30.0, 100.0, 400.0]))
    u8 = rng.random() < 0.4
    for name in ("BUILD_DEDUP", "DENSE"):
        _lib.set_tuning(name, int(rng.integers(-1, 2)))
    chunk = int(rng.choice([0, 0, 1, 2, 3]))   # frames per pass (0: the library's default)
    seg = synth.make_segs(n, k, h, w, seed=int(rng.integers(1 << 30)))
    if colour:
        dim = int(rng.integers(1, 7))
        planes = rng.integers(0, 256, size=(1, dim, h, w)).astype(np.float32)      # one frame: the batch loop strides by 3
        n = 1; seg = seg[:1]
        want = oracle.port_colorbilateralfilter_batch(planes, seg, 1, k, h, w, srgb, dim).reshape(seg.shape)
        cfg = _lib.make_config(_lib.FEAT_COLOR, dim, srgb, chunk_frames=chunk)
        img = planes
        tag = f"colour{dim}"
    else:
        ch = int(rng.choice([1, 2, 3, 3, 3, 4]))
        img = synth.make_images(n, h, w, kind, seed=int(rng.integers(1 << 30)), channels=ch)
        want = np.stack([oracle.port_filter_features(oracle.xy_features(h, w, sxy, img[i], srgb), seg[i])
                         for i in range(n)]).reshape(seg.shape)
        cfg = _lib.make_config(_lib.FEAT_XY_RGB, ch, srgb, sxy, chunk_frames=chunk)
        tag = f"xy+{ch}"
    if not _lib.load().tcamcrf_key_range_ok(cfg, h, w, 255.0):
        continue
    timg = torch.from_numpy(img.astype(np.uint8) if u8 else img).cuda()
    got, loss, _ = ops.crf_forward(timg, torch.from_numpy(seg).cuda(), cfg, check=True)
    got = got.cpu().numpy()
    den = np.linalg.norm(want.ravel()) or 1.0
    err = float(np.linalg.norm((got - want).ravel()) / den)
    worst = max(worst, err)
    cases += 1
    kinds[tag] = kinds.get(tag, 0) + 1
    if not (err < 1e-4) or not np.isfinite(loss.item()):
        fails += 1
        print("FAIL", dict(n=n, k=k, h=h, w=w, kind=kind, tag=tag, srgb=srgb, sxy=sxy, u8=u8, err=err), flush=True)
for name in ("BUILD_DEDUP", "DENSE"):
    _lib.set_tuning(name, -1)
print(f"fuzz: {cases} cases in {time.time() - t0:.0f} s, {fails} failures, worst normwise rel err {worst:.2e}; lattices {kinds}")
sys.exit(1 if fails else 0)
