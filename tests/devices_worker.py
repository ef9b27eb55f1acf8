"""Worker of tests/test_gpu_devices.py: one scenario in a fresh interpreter that drives two devices.

Which device the library meets first is part of what is tested, so every scenario starts in a new process, uses the
first device, then the second (ordinals from argv[2], default "0,1").  Prints one JSON line and exits non-zero when a
check fails.

    python tests/devices_worker.py fused_seeding|two_kernel_seeding|crf_paths|stage_timing [first,second]
"""
import ctypes
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

from tcam_wsol_video_b200 import _lib, synth  # noqa: E402

REL_TOL = 1e-4   # splat atomics: two runs differ in the last bits (tests/test_gpu_parity.py)


def _rel(got, want):
    got, want = np.asarray(got, np.float64), np.asarray(want, np.float64)
    return float(np.abs(got - want).max() / max(np.abs(want).max(), 1e-30))


def _stack_cams(b, t, h, w, seed):
    """CAMs of the current + (t-1) neighbour frames [B,T,H,W] (CPU) and a roi on their temporal max [B,1,H,W]."""
    low = torch.from_numpy(synth.make_low_res_cams(b, t, 28, 28, seed=seed)).squeeze(2)
    cams = torch.nn.functional.interpolate(low, size=(h, w), mode="bilinear", align_corners=False)
    return cams, (cams.amax(dim=1, keepdim=True) >= 0.5).long()


def fused_seeding(devices):
    """TCAMSeeder.forward_stack (one tcam_seed_fused launch) bit-exact against oracle/seeding.py on each device."""
    from oracle import seeding as ref
    from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder
    lib = _lib.load()
    b, t, h, w, ksz = 4, 5, 224, 224, 3
    cams_cpu, roi_cpu = _stack_cams(b, t, h, w, seed=0)
    out = {}
    for d in devices:
        dev = torch.device("cuda", d)
        with torch.cuda.device(dev):
            assert lib.tcam_seed_fused_supported(h * w, 1) == 1, d
        seeder = TCAMSeeder(seed_tech="seed_weighted", min_=1, max_=1, max_p=0.6, min_p=0.1, fg_erode_k=11,
                            fg_erode_iter=0, ksz=ksz, support_background=True, multi_label_flag=False,
                            seg_ignore_idx=-255, cuda_id=d, roi_method="roi_all", p_min_area_roi=0.05, use_roi=True,
                            rng_parity=True)
        cams, roi = cams_cpu.to(dev), roi_cpu.to(dev)
        torch.manual_seed(99)
        labels, cam_max = seeder.forward_stack(cams, roi)
        sel = seeder._last_sel
        want_max = ref.temporal_max(cams)
        kw = dict(seed_tech="seed_weighted", min_=1, max_=1, min_p=0.1, max_p=0.6, use_roi=True)
        torch.manual_seed(99)
        want = ref.tcam_seeder_forward(want_max.unsqueeze(1), roi, ksz=ksz, ignore_idx=-255, **kw)
        assert torch.equal(cam_max, want_max), d
        assert torch.equal(labels, want), d
        torch.manual_seed(99)   # the same stream again, for the seeds before their dilation
        for i in range(b):
            fg, bg = ref.one_sample(want_max[i], roi[i, 0], **kw)
            for side, m in ((0, fg), (1, bg)):
                got = sorted(v for v in sel[i, side].tolist() if v >= 0)
                assert got == m.flatten().nonzero().flatten().tolist(), (d, i, side)
        out[d] = {"fg": int((labels == 1).sum()), "bg": int((labels == 0).sum())}
    return out


def two_kernel_seeding(devices):
    """tcam_seed_select + tcam_seed_labels at 224x224 (the shared-memory select kernel) on each device, with the same
    draws made on the CPU: identical results."""
    lib = _lib.load()
    b, t, h, w, k, ksz = 4, 5, 224, 224, 3, 3
    hw = h * w
    cams_cpu, roi_cpu = _stack_cams(b, t, h, w, seed=1)
    n_fg = [int(np.float32(0.6) * np.float32(int(roi_cpu[i].sum()))) for i in range(b)]   # tcam_seeding.py:510,519
    counts = np.array([[f, int(0.1 * hw)] for f in n_fg], np.int32)                        # :567
    offsets = (np.cumsum(counts.reshape(-1)) - counts.reshape(-1)).astype(np.int32)
    q_cpu = torch.empty(int(counts.sum()), dtype=torch.float32).exponential_(1, generator=torch.Generator().manual_seed(5))
    results = []
    for d in devices:
        dev = torch.device("cuda", d)
        cams, roi, q = cams_cpu.to(dev), roi_cpu.to(dev), q_cpu.to(dev)
        q_off, n_cand = torch.from_numpy(offsets).to(dev), torch.from_numpy(counts.reshape(-1)).to(dev)
        cam_max = torch.empty((b, hw), dtype=torch.float32, device=dev)
        scratch = torch.empty((b, 2, hw), dtype=torch.float32, device=dev)
        sel = torch.empty((b, 2, k), dtype=torch.int32, device=dev)
        labels = torch.empty((b, h, w), dtype=torch.long, device=dev)
        with torch.cuda.device(dev):
            stream = torch.cuda.current_stream(dev).cuda_stream
            _lib.check(lib.tcam_seed_select(cams.data_ptr(), t, roi.data_ptr(), q.data_ptr(), q_off.data_ptr(),
                                            n_cand.data_ptr(), k, k, 1, b, hw, cam_max.data_ptr(), scratch.data_ptr(),
                                            sel.data_ptr(), k, stream), "tcam_seed_select")
            _lib.check(lib.tcam_seed_labels(sel.data_ptr(), k, b, h, w, ksz, -255, labels.data_ptr(), stream),
                       "tcam_seed_labels")
        assert torch.equal(cam_max, cams.amax(dim=1).reshape(b, hw)), d
        assert bool((sel >= 0).all()), d   # k seeds on each side: there are more candidates than that
        results.append((sel.cpu(), cam_max.cpu(), labels.cpu()))
    for a, b_ in zip(results[0], results[1]):
        assert torch.equal(a, b_)
    return {"fg": int((results[0][2] == 1).sum()), "bg": int((results[0][2] == 0).sum())}


def crf_paths(devices):
    """The CRF loss alternating first -> second -> first device: device frames, the trainer-shaped call with pinned
    uint8 host frames (the library's copy stream), and the host-pointer entry point (cached buffers, graph replay)."""
    import oracle
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    lib = _lib.load()
    n, k, h, w = 4, 3, 48, 56
    img = synth.make_images(n, h, w, "natural", seed=3)
    seg = synth.make_segs(n, k, h, w, seed=3)
    want_loss, want_grad, _ = oracle.densecrf_loss_fwd_bwd(img, seg, 15.0, 100.0, 1.0, oracle.port_bilateralfilter_batch)
    img8 = torch.from_numpy(img.astype(np.uint8)).pin_memory()
    img_h, seg_h = torch.from_numpy(img).pin_memory(), torch.from_numpy(seg).pin_memory()
    loss_h, grad_h = torch.zeros(1).pin_memory(), torch.zeros(n, k, h, w).pin_memory()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    errs = []
    for d in (devices[0], devices[1], devices[0]):
        dev = torch.device("cuda", d)
        for what, images in (("device frames", torch.from_numpy(img).to(dev)), ("pinned uint8 host frames", img8)):
            s = torch.from_numpy(seg).to(dev).requires_grad_(True)
            loss = DenseCRFLoss(1.0, 15.0, 100.0, 1.0)(images=images, segmentations=s)
            loss.backward()
            errs.append((d, what, _rel(loss.item(), want_loss), _rel(s.grad.cpu().numpy(), want_grad)))
        torch.cuda.set_device(d)
        for _ in range(2):   # eager + captured, then a replay of the captured schedule
            _lib.check(lib.tcamcrf_loss_fwd_bwd_host(ctypes.byref(cfg), img_h.data_ptr(), seg_h.data_ptr(),
                                                     loss_h.data_ptr(), grad_h.data_ptr(), n, k, h, w, 1.0),
                       "tcamcrf_loss_fwd_bwd_host")
            errs.append((d, "host pointers", _rel(loss_h.numpy(), want_loss), _rel(grad_h.numpy(), want_grad)))
    for e in errs:
        assert e[2] < REL_TOL and e[3] < REL_TOL, e
    return {"max_rel": max(max(e[2], e[3]) for e in errs), "calls": len(errs)}


def stage_timing(devices):
    """Per-stage timing on: one step on the first device, read, one step on the second, read again."""
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    lib = _lib.load()
    n, k, h, w = 2, 2, 32, 40
    img = torch.from_numpy(synth.make_images(n, h, w, "natural", seed=4))
    seg = torch.from_numpy(synth.make_segs(n, k, h, w, seed=4))
    ms = (ctypes.c_double * len(_lib.STAGES))()
    launches = (ctypes.c_longlong * len(_lib.STAGES))()
    lib.tcamcrf_profile_enable(1)
    try:
        reads = []
        for d in devices:
            dev = torch.device("cuda", d)
            s = seg.to(dev).requires_grad_(True)
            DenseCRFLoss(1.0, 15.0, 100.0, 1.0)(images=img.to(dev), segmentations=s).backward()
            torch.cuda.synchronize(dev)
            _lib.check(lib.tcamcrf_profile_read(ms, launches, 1), "tcamcrf_profile_read")
            reads.append(dict(zip(_lib.STAGES, launches)))
    finally:
        lib.tcamcrf_profile_enable(0)
    for d, r in zip(devices, reads):
        assert r["build"] >= 1 and r["splat"] >= 1 and r["slice"] >= 1, (d, r)
    return reads


if __name__ == "__main__":
    scenario = sys.argv[1]
    devices = [int(x) for x in (sys.argv[2] if len(sys.argv) > 2 else "0,1").split(",")]
    result = globals()[scenario](devices)
    print("DEVICES_WORKER " + json.dumps({"scenario": scenario, "devices": devices, "result": result}), flush=True)
