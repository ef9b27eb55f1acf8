"""GPU suite (-m gpu): temporal-CAM max and fg/bg seeding, bit-exact against the torch restatement of the
reference (oracle/seeding.py) when both consume the same random stream."""
import numpy as np
import pytest

from tcam_wsol_video_b200 import synth

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def _make(torch, b, h, w, seed, low_res=28):
    """CAMs like the trainer sees them: low-res maps upsampled bilinearly to the image size
    (train_wsol.py:417-432), plus an Otsu-like roi."""
    g = torch.Generator().manual_seed(seed)
    low = torch.rand((b, 1, low_res, low_res), generator=g)
    cam = torch.nn.functional.interpolate(low, size=(h, w), mode="bilinear", align_corners=False)
    roi = (cam >= cam.flatten(1).median(dim=1).values.view(b, 1, 1, 1)).long()
    return cam.cuda(), roi.cuda()


def _seeder(**kw):
    from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder
    base = dict(seed_tech="seed_weighted", min_=1, max_=1, max_p=0.6, min_p=0.1, fg_erode_k=11, fg_erode_iter=0,
                ksz=3, support_background=True, multi_label_flag=False, seg_ignore_idx=-255, cuda_id=0,
                roi_method="roi_all", p_min_area_roi=0.05, use_roi=True)
    base.update(kw)
    return TCAMSeeder(**base)


CONFIGS = [
    dict(),                                                       # README recipe (SURVEY F5)
    dict(seed_tech="seed_uniform"),
    dict(min_=10, max_=10, ksz=1, min_p=0.2, max_p=0.2, use_roi=False),   # config.py defaults
    dict(min_=3, max_=5, ksz=5),
    dict(min_=0, max_=2, ksz=4),
    dict(min_=2, max_=0),
]


@pytest.mark.parametrize("cfg", CONFIGS, ids=[str(i) for i in range(len(CONFIGS))])
@pytest.mark.parametrize("shape", [(4, 224, 224), (3, 37, 53)])
def test_seeds_bit_exact_vs_reference_restatement(torch_cuda, cfg, shape):
    torch = torch_cuda
    from oracle import seeding as ref
    b, h, w = shape
    cam, roi = _make(torch, b, h, w, seed=5)
    cam[1] = 0.25                      # a flat CAM: the reference emits no seed for it and draws nothing
    mod = _seeder(**cfg)
    torch.manual_seed(1234)
    got = mod(x=cam, roi=roi)
    torch.manual_seed(1234)
    want = ref.tcam_seeder_forward(cam, roi, seed_tech=mod.seed_tech, min_=mod.min_, max_=mod.max_, min_p=mod.min_p,
                                   max_p=mod.max_p, ksz=mod.ksz, ignore_idx=-255, use_roi=mod.use_roi)
    assert got.dtype == torch.long and got.shape == (b, h, w)
    assert torch.equal(got, want)
    assert (got[1] == -255).all()
    # and the two random streams are at the same position afterwards
    assert torch.equal(torch.rand(4, device="cuda"), torch.rand(4, device="cuda")) is False
    torch.manual_seed(1234)
    mod(x=cam, roi=roi)
    a = torch.rand(4, device="cuda")
    torch.manual_seed(1234)
    ref.tcam_seeder_forward(cam, roi, seed_tech=mod.seed_tech, min_=mod.min_, max_=mod.max_, min_p=mod.min_p,
                            max_p=mod.max_p, ksz=mod.ksz, ignore_idx=-255, use_roi=mod.use_roi)
    assert torch.equal(a, torch.rand(4, device="cuda"))


def test_ties_follow_stable_sort_order(torch_cuda):
    """Heavily quantised CAMs: most of the n-th values tie, and a stable sort keeps the lower pixel index."""
    torch = torch_cuda
    from oracle import seeding as ref
    b, h, w = 3, 64, 48
    g = torch.Generator().manual_seed(3)
    cam = (torch.randint(0, 4, (b, 1, h, w), generator=g).float() / 4).cuda()
    roi = (torch.rand((b, 1, h, w), generator=g) > 0.3).long().cuda()
    for tech in ("seed_weighted", "seed_uniform"):
        mod = _seeder(seed_tech=tech, min_=4, max_=4, ksz=1)
        torch.manual_seed(7)
        got = mod(x=cam, roi=roi)
        torch.manual_seed(7)
        want = ref.tcam_seeder_forward(cam, roi, seed_tech=tech, min_=4, max_=4, min_p=0.1, max_p=0.6, ksz=1,
                                       ignore_idx=-255, use_roi=True)
        assert torch.equal(got, want)


def test_fused_temporal_max_and_seeding(torch_cuda):
    """BASELINE configs[2]: max over the current + 4 previous frames' CAMs fused with seeding == max chain
    followed by the reference seeder."""
    torch = torch_cuda
    from oracle import seeding as ref
    b, t, h, w = 32, 5, 224, 224
    low = torch.from_numpy(synth.make_low_res_cams(b, t, 28, 28, seed=0)).squeeze(2)       # [B,T,28,28]
    cams = torch.nn.functional.interpolate(low, size=(h, w), mode="bilinear", align_corners=False).cuda()
    cam_max_want = ref.temporal_max(cams)
    roi = (cam_max_want >= 0.5).long().unsqueeze(1)
    mod = _seeder()
    torch.manual_seed(99)
    got, cam_max = mod.forward_stack(cams, roi)
    torch.manual_seed(99)
    want = ref.tcam_seeder_forward(cam_max_want.unsqueeze(1), roi, seed_tech=mod.seed_tech, min_=1, max_=1,
                                   min_p=0.1, max_p=0.6, ksz=3, ignore_idx=-255, use_roi=True)
    assert torch.equal(cam_max, cam_max_want)
    assert torch.equal(got, want)
    assert int((got == 1).sum()) > 0 and int((got == 0).sum()) > 0


def test_seeder_api_surface(torch_cuda):
    torch = torch_cuda
    mod = _seeder()
    assert "min_=1, max_=1, min_p=0.1,max_p=0.6, ksz=3, fg_erode_k: 11, fg_erode_iter: 0" in mod.extra_repr()
    mod.set_seed_tech("seed_uniform")
    assert mod.seed_tech == "seed_uniform"
    cam, roi = _make(torch, 2, 32, 32, seed=1)
    out = mod.use_all_roi(cam, roi)
    assert torch.equal(out == 1, roi.squeeze(1) == 1) and ((out == 1) | (out == -255)).all()
    assert _seeder(roi_method="largest")(x=cam, roi=None).shape == (2, 32, 32)   # component roi computed on the GPU
    # erosion of the roi before sampling (fg_erode_iter > 0) keeps seeds inside the eroded region
    mod = _seeder(fg_erode_k=5, fg_erode_iter=1, ksz=1, max_=8)
    seeds = mod(x=cam, roi=roi)
    eroded = mod._erode(roi).squeeze(1)
    assert ((seeds == 1) <= (eroded == 1)).all()


OTSU_CASES = [pytest.param(kind, (224, 224), id=kind) for kind in ("bilinear", "uniform", "quantised", "flat")]
OTSU_CASES += [pytest.param(kind, shape, id=f"{kind}-{shape[0]}x{shape[1]}")
               for shape in ((1, 1), (1, 2), (2, 1), (1, 300)) for kind in ("bilinear", "uniform", "two_valued")]
OTSU_CASES += [pytest.param(kind, shape, id=f"{kind}-{shape[0]}x{shape[1]}")
               for shape in ((224, 224), (1, 300)) for kind in ("two_valued", "outlier", "unnormalised")]


@pytest.mark.parametrize("kind,shape", OTSU_CASES)
def test_otsu_roi_matches_numpy_restatement(torch_cuda, kind, shape):
    """tcam_otsu_roi vs the reference's CPU recipe (np.histogram + scikit-image's Otsu restated): same
    threshold bit for bit and the same mask, on CAM-like, uniform, heavily tied and flat inputs, two-valued maps, a
    flat map with one outlier and an unnormalised map in [-3, 40], at 224x224 and on 1x1, 1x2, 2x1 and 1x300 frames."""
    torch = torch_cuda
    from oracle import seeding as ref
    from tcam_wsol_video_b200 import ops
    b, (h, w) = 6, shape
    g = torch.Generator().manual_seed(17)
    if kind == "bilinear":
        cam = torch.nn.functional.interpolate(torch.rand((b, 1, 28, 28), generator=g), size=(h, w), mode="bilinear",
                                              align_corners=False)
    elif kind == "uniform":
        cam = torch.rand((b, 1, h, w), generator=g)
    elif kind == "quantised":
        cam = torch.randint(0, 7, (b, 1, h, w), generator=g).float() / 9 + 0.01
    elif kind == "two_valued":
        cam = torch.where(torch.rand((b, 1, h, w), generator=g) < 0.3, 0.8, 0.15)
    elif kind == "outlier":
        cam = torch.full((b, 1, h, w), 0.4)
        cam.view(b, -1)[torch.arange(b), torch.randint(0, h * w, (b,), generator=g)] = 0.9
    elif kind == "unnormalised":
        cam = torch.rand((b, 1, h, w), generator=g) * 43 - 3
    else:
        cam = torch.full((b, 1, h, w), 0.3)
        cam[1] = torch.rand((1, h, w), generator=g) * 0.5       # one non-flat sample among flat ones
    roi, th = ops.otsu_roi(cam.cuda())
    assert roi.shape == cam.shape and roi.dtype == torch.long
    for i in range(b):
        want_roi, want_th = ref.roi_all_single_cam(cam[i, 0].numpy())
        assert th[i].item() == np.float32(want_th), (i, th[i].item(), want_th)
        assert np.array_equal(roi[i, 0].cpu().numpy(), want_roi)


def test_seeder_computes_roi_when_none_is_given(torch_cuda):
    """use_roi=True, roi=None: the reference calls GetRoiSingleCam per sample on the CPU; here one kernel."""
    torch = torch_cuda
    from oracle import seeding as ref
    cam, _ = _make(torch, 4, 96, 80, seed=9)
    mod = _seeder()
    torch.manual_seed(5)
    got = mod(x=cam, roi=None)
    roi = torch.stack([torch.from_numpy(ref.roi_all_single_cam(cam[i, 0].cpu().numpy())[0]) for i in range(4)])
    torch.manual_seed(5)
    want = ref.tcam_seeder_forward(cam, roi.unsqueeze(1).cuda(), seed_tech=mod.seed_tech, min_=1, max_=1, min_p=0.1,
                                   max_p=0.6, ksz=3, ignore_idx=-255, use_roi=True)
    assert torch.equal(got, want)


@pytest.mark.parametrize("h_t", [0.0, 10.0, 50.0])
def test_temporal_aggregation_with_renormalisation(torch_cuda, h_t):
    """aggregate_temporal_cams = the loader's loop (wsol_loader.py:591-600) with re_normalize_cam (:630-635).
    Plain max: bit-exact.  With the exp re-normalisation the reference runs torch's CPU exp (SLEEF), the kernel
    CUDA's expf: equal within 2 ulp of exp -> rel 1e-6 in the ratio (tolerance stated here)."""
    torch = torch_cuda
    from oracle import seeding as oseed
    from tcam_wsol_video_b200 import temporal
    low = torch.from_numpy(synth.make_low_res_cams(6, 5, 28, 28, seed=11))        # [B,T,1,h,w]
    low[1, 2, 0, 3, 4] = float("nan")
    low[2, 0, 0, 0, 0] = float("inf")
    low[3, 1, 0, 5, 5] = float("-inf")
    want = oseed.temporal_max_renorm(low, h_t)                                     # CPU, [B,1,h,w]
    got = temporal.aggregate_temporal_cams(low.cuda(), knn_t=h_t).cpu()
    assert got.shape == want.shape == (6, 1, 28, 28)
    assert torch.equal(torch.isnan(got), torch.isnan(want))
    if h_t == 0.0:
        assert torch.equal(torch.nan_to_num(got, nan=-7.0), torch.nan_to_num(want, nan=-7.0))
    else:
        g, w = torch.nan_to_num(got, nan=-7.0), torch.nan_to_num(want, nan=-7.0)
        assert (g - w).abs().max().item() <= 1e-6 * max(w.abs().max().item(), 1.0)
    # single-frame form used by the loader
    one = temporal.re_normalize_cam(low[0, 0].cuda(), 10.0).cpu()
    assert (one - oseed.re_normalize_cam(low[0, 0], 10.0)).abs().max().item() <= 1e-6


@pytest.mark.parametrize("size", [(224, 224), (160, 288), (28, 28)])
def test_prepare_std_cams_disq(torch_cuda, size):
    """Fused nan_to_num -> bilinear(align_corners=False) -> nan_to_num against the trainer's three torch calls
    (train_wsol.py:417-432).  Same source-index / weight arithmetic as ATen; tolerance 1e-6 absolute on [0,1] maps
    (FMA contraction may differ between the two compilations)."""
    torch = torch_cuda
    from oracle import seeding as oseed
    from tcam_wsol_video_b200 import temporal
    low = torch.from_numpy(synth.make_low_res_cams(5, 1, 28, 28, seed=4))[:, 0]    # [B,1,h,w]
    low[0, 0, 2, 3] = float("nan")
    low[1, 0, 0, 0] = float("inf")
    low[2, 0, 27, 27] = float("-inf")
    want_cpu = oseed.prepare_std_cams_disq(low, size)
    want_gpu = oseed.prepare_std_cams_disq(low.cuda(), size).cpu()
    got = temporal.prepare_std_cams_disq(low.cuda(), size).cpu()
    assert got.shape == want_cpu.shape
    assert torch.isfinite(got).all()
    assert (got - want_gpu).abs().max().item() <= 1e-6
    assert (got - want_cpu).abs().max().item() <= 1e-6


@pytest.mark.parametrize("method", ["roi_high_density", "largest"])
@pytest.mark.parametrize("shape", [(224, 224), (37, 61), (8, 5)])
def test_roi_connected_components(torch_cuda, method, shape):
    """GetRoiSingleCam 'roi_high_density' / 'largest' on the GPU (union-find components, per-component density and
    area, bounding box) against the line-by-line restatement (oracle/seeding.py; scipy.ndimage.label for
    skimage.measure.label, bounding rectangle for the cv2 contour).  Masks, boxes and box masks must be identical."""
    torch = torch_cuda
    from oracle import seeding as oseed
    from tcam_wsol_video_b200 import ops
    from tcam_wsol_video_b200.tcam_seeding import GetRoiSingleCam
    h, w = shape
    g = torch.Generator().manual_seed(h * 1000 + w)
    low = torch.rand((6, 1, 7, 7), generator=g)
    cams = torch.nn.functional.interpolate(low, size=(h, w), mode="bilinear", align_corners=False)[:, 0]
    cams = cams + 0.05 * torch.rand((6, h, w), generator=g)                     # several blobs per map
    cams[4] = 0.3                                                                # flat: threshold 0, everything in
    cams[5] = torch.rand((h, w), generator=g)                                    # salt and pepper: many components
    for p_min in (0.05, 0.6):
        roi, mask, bbox = ops.roi_components(cams.cuda(), method == "largest", p_min)
        for i in range(cams.shape[0]):
            want_roi, want_mask, want_bbox = oseed.roi_components_single_cam(cams[i].numpy(), method, p_min)
            assert np.array_equal(roi[i].cpu().numpy(), want_roi), (i, p_min)
            assert np.array_equal(bbox[i].cpu().numpy().reshape(1, 4), want_bbox), (i, p_min)
            assert np.array_equal(mask[i].cpu().numpy(), want_mask), (i, p_min)
    # fixed threshold (the loader passes roi_thresholds when it has them) and the single-cam class
    getter = GetRoiSingleCam(roi_method=method, p_min_area_roi=0.05)
    r1, m1, b1 = getter(cams[1].cuda(), thresh=0.5)
    w1 = oseed.roi_components_single_cam(cams[1].numpy(), method, 0.05, thresh=0.5)
    assert np.array_equal(r1.cpu().numpy(), w1[0]) and np.array_equal(m1.cpu().numpy(), w1[1])
    assert np.array_equal(b1.cpu().numpy(), w1[2]) and r1.dtype == torch.long
    # nothing above the threshold: empty roi, box [0,0,0,0]
    r0, m0, b0 = getter(torch.zeros(h, w).cuda(), thresh=0.5)
    assert r0.sum().item() == 0 and m0.sum().item() == 0 and b0.abs().sum().item() == 0


def test_seeder_computes_component_roi_when_none_is_given(torch_cuda):
    """TCAMSeeder(roi_method='largest') with roi=None: the reference calls GetRoiSingleCam on the CPU per sample
    (tcam_seeding.py:476-479); here the batched kernel.  Same seeds as passing that roi explicitly."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    cam, _ = _make(torch, 4, 64, 64, seed=21)
    seeder = _seeder(roi_method="largest")
    roi, _, _ = ops.roi_components(cam, True, 0.05)
    torch.manual_seed(5)
    a = seeder(cam, None)
    torch.manual_seed(5)
    b = seeder(cam, roi)
    assert torch.equal(a, b)


def test_seeder_without_host_round_trip(torch_cuda):
    """rng_parity=False: candidate counts stay on the GPU (no host sync, fixed draw slots).  The counts must equal the
    host-computed ones -- flat CAMs, empty rois and float32 truncation of max_p * roi.sum() included -- and every
    foreground seed must be one of the n best roi pixels, every background seed one of the n lowest pixels."""
    torch = torch_cuda
    cam, roi = _make(torch, 6, 64, 80, seed=33)
    cam[2] = 0.25                       # flat: no seeds at all (tcam_seeding.py:465)
    roi[3] = 0                          # empty roi: no foreground candidates
    seeder = _seeder(rng_parity=False, ksz=1, max_=3, min_=2)
    x, r = seeder._prep(cam, roi)
    host_counts, _ = seeder._candidate_counts(x, r)
    dev_counts = seeder._candidate_counts_device(x, r)
    assert dev_counts.dtype == torch.int32 and np.array_equal(dev_counts.cpu().numpy(), host_counts)
    out = seeder(cam, roi)
    assert set(torch.unique(out).tolist()) <= {-255, 0, 1}
    assert (out[2] == -255).all()
    assert (out[3] != 1).all()
    flat = cam.reshape(6, -1)
    for i in (0, 1, 4, 5):
        n_fg, n_bg = int(host_counts[i, 0]), int(host_counts[i, 1])
        fg_vals = (flat[i] * roi[i].reshape(-1) + 1e-8)
        thr_fg = torch.sort(fg_vals, descending=True).values[n_fg - 1]
        thr_bg = torch.sort(flat[i] + 1e-8).values[n_bg - 1]
        seeds_fg = (out[i].reshape(-1) == 1).nonzero().flatten()
        seeds_bg = (out[i].reshape(-1) == 0).nonzero().flatten()
        assert 1 <= seeds_fg.numel() <= 3 and 1 <= seeds_bg.numel() <= 2
        assert (fg_vals[seeds_fg] >= thr_fg).all()
        assert ((flat[i] + 1e-8)[seeds_bg] <= thr_bg).all()


def test_temporal_kernels_match_the_reference_python(torch_cuda):
    """The temporal-aggregation and CAM-resize kernels against fixtures produced by EXECUTING the reference's own
    re_normalize_cam / torch.maximum loop / prepare_std_cams_disq on the CPU (tests/golden/make_golden_py.py).
    Plain max: bit-exact.  exp-based re-normalisation and the bilinear resize: 1e-6 (CUDA expf / FMA contraction
    against torch's CPU kernels)."""
    import os
    torch = torch_cuda
    from conftest import GOLDEN
    from tcam_wsol_video_b200 import temporal
    g = np.load(os.path.join(GOLDEN, "py", "py_temporal_agg.npz"))
    cams = torch.from_numpy(g["cams"]).cuda()
    for h_t in (0.0, 10.0, 50.0):
        got = temporal.aggregate_temporal_cams(cams, knn_t=h_t).cpu().numpy()
        want = g[f"agg_h{int(h_t)}"]
        assert np.array_equal(np.isnan(got), np.isnan(want))
        a, b = np.nan_to_num(got, nan=-7.0), np.nan_to_num(want, nan=-7.0)
        if h_t == 0.0:
            assert np.array_equal(a, b)
        else:
            assert np.abs(a - b).max() <= 1e-6
    g = np.load(os.path.join(GOLDEN, "py", "py_prepare_std_cams.npz"))
    std = torch.from_numpy(g["std_cams"]).cuda()
    for key in [k for k in g.files if k.startswith("out_")]:
        size = tuple(int(v) for v in key[4:].split("x"))
        got = temporal.prepare_std_cams_disq(std, size).cpu().numpy()
        assert np.abs(got - g[key]).max() <= 1e-6, key


def test_fused_and_two_kernel_paths(torch_cuda):
    """Frames whose slice does not fit an SM's shared memory (tcam_seed_fused_supported == 0) and k > 32 take
    tcam_seed_select + tcam_seed_labels; both paths are bit-exact against the reference restatement given its draws."""
    torch = torch_cuda
    import oracle.seeding as ref
    from tcam_wsol_video_b200 import _lib
    lib = _lib.load()
    assert lib.tcam_seed_fused_supported(224 * 224, 1) == 1
    assert lib.tcam_seed_fused_supported(224 * 224, 33) == 0
    assert lib.tcam_seed_fused_supported(640 * 640, 1) == 0
    for (b, h, w), kw in (((2, 640, 640), dict()), ((3, 48, 56), dict(min_=40, max_=35, ksz=1))):
        cam, roi = _make(torch, b, h, w, seed=5)
        mod = _seeder(**kw)
        torch.manual_seed(11)
        got = mod(cam, roi)
        torch.manual_seed(11)
        want = ref.tcam_seeder_forward(cam, roi, seed_tech=mod.seed_tech, min_=mod.min_, max_=mod.max_,
                                       min_p=mod.min_p, max_p=mod.max_p, ksz=mod.ksz, ignore_idx=-255,
                                       use_roi=mod.use_roi)
        assert torch.equal(got, want)


def test_in_kernel_draws(torch_cuda):
    """rng_parity=False: the Exp(1) draws are made in the kernel (Philox keyed from torch's CUDA generator).  Same
    torch seed -> same seeds; different seeds -> different picks; uniform sampling spreads over the candidates; weighted
    sampling prefers high CAM values."""
    torch = torch_cuda
    cam, roi = _make(torch, 8, 96, 96, seed=9)
    seeder = _seeder(rng_parity=False, ksz=1, seed_tech="seed_uniform")
    torch.manual_seed(3)
    a = seeder(cam, roi)
    torch.manual_seed(3)
    b = seeder(cam, roi)
    assert torch.equal(a, b)
    picks = []
    for _ in range(40):
        out = seeder(cam, roi)
        assert ((out == 1).flatten(1).sum(1) == 1).all() and ((out == 0).flatten(1).sum(1) == 1).all()
        picks.append((out[0] == 1).flatten().nonzero().item())
    assert len(set(picks)) >= 30                                  # ~14 k candidates: repeats are unlikely
    # weighted: the mean CAM value at the picks lies above the candidates' mean
    flat = cam[0].flatten()
    n_fg = int(np.float32(0.6) * np.float32(roi[0].sum().item()))
    cand = torch.sort(flat * roi[0].flatten() + 1e-8, descending=True).values[:n_fg]
    seeder_w = _seeder(rng_parity=False, ksz=1, seed_tech="seed_weighted")
    vals = []
    for _ in range(200):
        out = seeder_w(cam, roi)
        vals.append(flat[(out[0] == 1).flatten().nonzero().item()].item())
    se = cand.std().item() / np.sqrt(200)
    assert np.mean(vals) > cand.mean().item() + 1.0 * se
    # every pick is a candidate
    assert min(vals) + 1e-8 >= cand[-1].item() - 1e-12


def test_roi_components_match_the_reference_class_run_with_opencv(torch_cuda):
    """The GPU ROI kernels against the reference's own GetRoiSingleCam executed with real OpenCV (fixture made by
    tests/golden/make_golden_py.py): masks, boxes and box masks identical in all 48 cases."""
    import os
    torch = torch_cuda
    from tcam_wsol_video_b200.tcam_seeding import GetRoiSingleCam
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "py", "py_get_roi_single_cam.npz"))
    for ci in range(int(g["n_cases"])):
        method, thresh, cj = [str(v) for v in g[f"c{ci}_cfg"]]
        cam = torch.from_numpy(g[f"cam{cj}"]).cuda()
        roi, mask, bbox = GetRoiSingleCam(roi_method=method, p_min_area_roi=0.05)(cam, thresh=float(thresh) if thresh else None)
        assert np.array_equal(roi.cpu().numpy(), g[f"c{ci}_roi"]), ci
        assert np.array_equal(bbox.cpu().numpy(), g[f"c{ci}_bbox"]), ci
        assert np.array_equal(mask.cpu().numpy(), g[f"c{ci}_mask"]), ci


def _dyadic_cam(mask, seed):
    """mask [h,w] bool -> cam: foreground pixels take dyadic values in [0.5, 1) (exact float32 and float64 sums in
    any order), background 0."""
    rng = np.random.default_rng(seed)
    return np.where(mask, 0.5 + rng.integers(0, 32, mask.shape) / 64.0, 0.0).astype(np.float32)


def _roi_shapes():
    """(name, cam [h,w] float32, p_min_area) drawn to stress the union-find, the tie-breaking and the selection."""
    shapes = []

    def serpentine(h, w):
        y, x = np.mgrid[0:h, 0:w]
        return (y % 2 == 0) | ((y % 4 == 1) & (x == w - 1)) | ((y % 4 == 3) & (x == 0))

    for h, w in ((640, 640), (37, 61)):
        shapes.append((f"serpentine{h}x{w}", _dyadic_cam(serpentine(h, w), h), 0.05))
    h, w = 96, 96
    y, x = np.mgrid[0:h, 0:w] - (h - 1) / 2.0
    phase = np.mod(np.hypot(y, x) - 12.0 * np.arctan2(y, x) / (2 * np.pi), 12.0)
    shapes.append(("spirals", np.where(phase < 4, 0.75, np.where((phase >= 6) & (phase < 10), 0.625, 0.0))
                   .astype(np.float32), 0.05))
    comb = np.zeros((50, 40), bool)
    comb[:, ::2] = True
    comb[-1] = True                                              # the teeth join only in the last row
    shapes.append(("comb", _dyadic_cam(comb, 3), 0.05))
    stairs = np.zeros((40, 50), bool)
    for i in range(0, 38, 2):
        stairs[i:i + 2, i:i + 2] = True                          # 2x2 blocks touching only at corners
    for i in range(40):
        stairs[i, min(49, 45 - i)] = True                        # an anti-diagonal line: single pixels
    shapes.append(("diagonal", _dyadic_cam(stairs, 4), 0.05))
    y, x = np.mgrid[0:37, 0:53]
    shapes.append(("checkerboard", np.where((x + y) % 2 == 0, 0.75, 0.0).astype(np.float32), 0.0005))
    ties = np.zeros((40, 50), np.float32)
    block = np.array([[0.5, 0.75, 0.875], [0.625, 0.9375, 0.5], [0.75, 0.5, 0.5625]], np.float32)
    for k, (y0, x0) in enumerate([(30, 5), (3, 40), (3, 10), (20, 25)]):
        ties[y0:y0 + 3, x0:x0 + 3] = np.rot90(block, k)          # same values, another order: same sum exactly
    shapes.append(("equal_density", ties, 0.004))   # min area 8: the densest is kept
    # the p_min_area boundary: the densest component's area is exactly H*W*p (kept) or one less (the largest wins)
    for (h, w, p, dense_hw, big_hw) in ((40, 50, 0.05, (10, 10), (15, 20)), (100, 100, 0.05, (20, 25), (30, 30)),
                                        (10, 10, 0.6, (6, 10), (3, 10))):
        for drop in (0, 1):
            cam = np.zeros((h, w), np.float32)
            cam[:dense_hw[0], :dense_hw[1]] = 0.9375
            if drop:
                cam[0, 0] = 0.0
            cam[h - big_hw[0]:, w - big_hw[1]:] = 0.5
            assert (cam == 0.9375).sum() == h * w * p - drop
            shapes.append((f"min_area{h}x{w}_p{p}_minus{drop}", cam, p))
    border = np.zeros((30, 45), bool)
    border[10:20, 40:] = True                                    # touches the right border
    border[25:, 5:15] = True                                     # touches the bottom border
    border[26:, 30:] = True                                      # the bottom-right corner
    shapes.append(("borders", _dyadic_cam(border, 5), 0.05))
    rng = np.random.default_rng(6)
    for h, w in ((1, 64), (64, 1), (1, 1)):
        shapes.append((f"line{h}x{w}", _dyadic_cam(rng.random((h, w)) < 0.5, h + w), 0.05))
        shapes.append((f"full{h}x{w}", _dyadic_cam(np.ones((h, w), bool), 7), 0.05))
    shapes.append(("full", _dyadic_cam(np.ones((33, 47), bool), 8), 0.05))
    shapes.append(("empty", np.zeros((33, 47), np.float32), 0.05))
    return shapes


@pytest.mark.parametrize("method", ["roi_high_density", "largest"])
@pytest.mark.parametrize("thresh", [0.5, None], ids=["fixed", "otsu"])
def test_roi_components_on_drawn_shapes(torch_cuda, method, thresh):
    """roi_components_kernel on masks drawn to break it: a serpentine and two interleaved spirals (long union chains),
    a comb joined in its last row, corner-touching blocks (4-connectivity), a checkerboard and equal-density
    components (exact ties: the first component in raster order wins), the p_min_area boundary (area exactly H*W*p
    is kept), border-touching components, 1xW / Hx1 / 1x1 frames, full and empty frames.  Every shape runs alone and
    batched with the other shapes of its frame size; roi, bbox and bbox mask must equal the restatement's exactly."""
    torch = torch_cuda
    from oracle import seeding as oseed
    from tcam_wsol_video_b200 import ops
    groups = {}
    for name, cam, p in _roi_shapes():
        groups.setdefault((cam.shape, p), []).append((name, cam))
    for (_, p), items in groups.items():
        batch = torch.from_numpy(np.stack([cam for _, cam in items])).cuda()
        batched = ops.roi_components(batch, method == "largest", p, thresh)
        for i, (name, cam) in enumerate(items):
            want = oseed.roi_components_single_cam(cam, method, p, thresh=thresh)
            alone = ops.roi_components(batch[i:i + 1], method == "largest", p, thresh)
            for got in ((batched[0][i], batched[1][i], batched[2][i]), (alone[0][0], alone[1][0], alone[2][0])):
                assert np.array_equal(got[0].cpu().numpy(), want[0]), name
                assert np.array_equal(got[2].cpu().numpy().reshape(1, 4), want[2]), name
                assert np.array_equal(got[1].cpu().numpy(), want[1]), name
