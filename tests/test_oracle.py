"""CPU suite, part 1: pins the oracle.

* the C restatement (oracle/permuto_oracle.c) reproduces, bit for bit, every committed golden
  fixture -- those were produced by the reference's own C++ (tests/golden/make_golden.py);
* for six more cases the filtered tensors and the lattice internals (offset_, barycentric_, neighbours, M)
  match, bit for bit, digests stored from the reference build in tests/golden/lattice/, and the reference
  build itself wherever it is present (oracle/_ref).
"""
import hashlib
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_golden
from tcam_wsol_video_b200 import synth


def _run_port(oracle_mod, g, image=None):
    img = g["image_u8"].astype(np.float32) if image is None else image
    seg = g["seg"]
    dim = int(g["dim"])
    if dim:
        return oracle_mod.color_densecrf_loss_fwd_bwd(img, seg, float(g["sigma_rgb"]), 1.0,
                                                      oracle_mod.port_colorbilateralfilter_batch)
    return oracle_mod.densecrf_loss_fwd_bwd(img, seg, float(g["sigma_rgb"]), float(g["sigma_xy"]), 1.0,
                                            oracle_mod.port_bilateralfilter_batch)


@pytest.mark.parametrize("path", golden_cases(), ids=os.path.basename)
def test_port_matches_golden_bit_exact(oracle_mod, path):
    g = load_golden(path)
    loss, grad, AS = _run_port(oracle_mod, g)
    assert np.array_equal(AS, g["AS"])
    assert np.array_equal(grad, g["grad"])
    assert np.float32(loss) == g["loss"]


def test_port_matches_golden_224(oracle_mod):
    g = load_golden(os.path.join(GOLDEN, "bf5_noise_n1_k2_224x224.npz"))
    n, k, h, w = (int(v) for v in g["shape"])
    img = synth.make_images(n, h, w, str(g["kind"]), seed=int(g["seed"]))
    seg = synth.make_segs(n, k, h, w, seed=int(g["seed"]))
    # the seeded generator must reproduce the inputs the fixture was made from
    assert img.sum(dtype=np.float64) == g["image_sum"]
    assert abs(seg.sum(dtype=np.float64) - g["seg_sum"]) < 1e-6
    loss, grad, AS = oracle_mod.densecrf_loss_fwd_bwd(img, seg, float(g["sigma_rgb"]), float(g["sigma_xy"]), 1.0,
                                                      oracle_mod.port_bilateralfilter_batch)
    assert np.array_equal(AS.ravel()[:: int(g["stride"])], g["AS_sample"])
    assert AS.astype(np.float64).sum() == g["AS_sum"]
    assert np.float32(loss) == g["loss"]
    assert oracle_mod.port_lattice_bilateral(img[0], h, w, float(g["sigma_rgb"]), float(g["sigma_xy"])).m == int(g["M0"])


@pytest.mark.parametrize("path", golden_cases(), ids=os.path.basename)
def test_port_lattice_size_matches_golden(oracle_mod, path):
    g = load_golden(path)
    img = g["image_u8"].astype(np.float32)
    h, w = img.shape[2:]
    dim = int(g["dim"])
    if dim:
        L = oracle_mod.port_lattice_color(img[0], h, w, float(g["sigma_rgb"]), dim)
    else:
        L = oracle_mod.port_lattice_bilateral(img[0], h, w, float(g["sigma_rgb"]), float(g["sigma_xy"]))
    assert L.m == int(g["M0"])
    # structural invariants of a permutohedral lattice
    assert np.all(L.offset >= 0) and np.all(L.offset < L.m)
    assert np.allclose(L.bary.sum(axis=1), 1.0, atol=1e-5)
    assert L.bary.min() > -1e-5
    assert L.nbr.min() >= -1 and L.nbr.max() < L.m


LATTICE_KINDS = ("noise", "natural")
LATTICE_SHAPES = ((2, 2, 32, 40), (1, 3, 31, 37), (1, 1, 7, 5))


def lattice_case_name(kind, shape):
    return "%s_n%d_k%d_%dx%d" % ((kind,) + tuple(shape))


def lattice_case_arrays(oracle_mod, kind, shape, ref):
    """Filtered tensors of both wrappers and the first frame's two lattices (offset_, barycentric_, neighbour table,
    M) for one case, from the reference build (ref=True) or the C restatement."""
    n, k, h, w = shape
    img = synth.make_images(n, h, w, kind, seed=7)
    seg = synth.make_segs(n, k, h, w, seed=7)
    o = oracle_mod
    bf = o.ref_bilateralfilter_batch if ref else o.port_bilateralfilter_batch
    cbf = o.ref_colorbilateralfilter_batch if ref else o.port_colorbilateralfilter_batch
    out = {"bf_AS": bf(img, seg, n, k, h, w, 15.0, 100.0), "cbf_AS": cbf(img, seg, n, k, h, w, 15.0, 3)}
    for tag, L in (("bf", (o.ref_lattice_bilateral if ref else o.port_lattice_bilateral)(img[0], h, w, 15.0, 100.0)),
                   ("cbf", (o.ref_lattice_color if ref else o.port_lattice_color)(img[0], h, w, 15.0, 3))):
        out[tag + "_M"] = np.int32(L.m)
        out[tag + "_offset"] = np.ascontiguousarray(L.offset, dtype=np.int32)
        out[tag + "_bary"] = np.ascontiguousarray(L.bary, dtype=np.float32)
        out[tag + "_nbr"] = np.ascontiguousarray(L.nbr, dtype=np.int32)
    return out


def sha256_of(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


@pytest.mark.parametrize("kind", LATTICE_KINDS)
@pytest.mark.parametrize("shape", LATTICE_SHAPES)
def test_port_vs_reference_build(oracle_mod, kind, shape):
    """Bit for bit: against the digests stored in tests/golden/lattice/ (tests/golden/make_golden_lattice.py) and,
    where oracle/_ref is built, against the live reference build too."""
    port = lattice_case_arrays(oracle_mod, kind, shape, ref=False)
    g = load_golden(os.path.join(GOLDEN, "lattice", lattice_case_name(kind, shape) + ".npz"))
    for key, a in port.items():
        assert a.dtype == np.dtype(str(g[key + "_dtype"])) and a.shape == tuple(g[key + "_shape"]), key
        assert sha256_of(a) == str(g[key + "_sha256"]), (key, a.sum(dtype=np.float64), float(g[key + "_sum"]))
    if oracle_mod.have_ref():
        ref = lattice_case_arrays(oracle_mod, kind, shape, ref=True)
        for key, a in port.items():
            assert np.array_equal(a, ref[key]), key


def test_filter_is_linear_and_symmetric_enough(oracle_mod):
    """Properties the loss relies on: linearity in the segmentation, positivity for positive input."""
    n, k, h, w = 1, 2, 20, 24
    img = synth.make_images(n, h, w, "noise", seed=3)
    s1 = synth.make_segs(n, k, h, w, seed=3)
    s2 = synth.make_segs(n, k, h, w, seed=4)
    f = lambda s: oracle_mod.port_bilateralfilter_batch(img, s, n, k, h, w, 15.0, 100.0).astype(np.float64)
    lhs = f((2.0 * s1 + 0.5 * s2).astype(np.float32))
    rhs = 2.0 * f(s1) + 0.5 * f(s2)
    assert np.abs(lhs - rhs).max() / np.abs(rhs).max() < 1e-5
    assert f(s1).min() > 0.0


def test_loss_wrapper_restates_reference_lines(oracle_mod):
    """loss = -sum(S*AS)/N and grad = -2*g*AS/N (dense_crf_loss.py:63-74)."""
    n, k, h, w = 3, 2, 12, 10
    img = synth.make_images(n, h, w, "natural", seed=5)
    seg = synth.make_segs(n, k, h, w, seed=5)
    loss, grad, AS = oracle_mod.densecrf_loss_fwd_bwd(img, seg, 15.0, 100.0, grad_output=0.25,
                                                      filter_fn=oracle_mod.port_bilateralfilter_batch)
    assert AS.shape == seg.shape and grad.shape == seg.shape
    assert abs(float(loss) + float((seg.astype(np.float64) * AS).sum() / n)) < 1e-3 * abs(float(loss))
    assert np.allclose(grad, -2.0 * 0.25 * AS / n, rtol=1e-6)


# ---------------------------------------------------------------------------
# fixtures made by EXECUTING the reference's own Python (tests/golden/make_golden_py.py)
# ---------------------------------------------------------------------------
def _py_golden(name):
    import os
    from conftest import GOLDEN
    z = np.load(os.path.join(GOLDEN, "py", name), allow_pickle=False)
    return {k: z[k] for k in z.files}


def test_restatements_match_the_reference_python():
    """oracle/seeding.py's re_normalize_cam / temporal max / prepare_std_cams_disq and the package's frame pickers
    against outputs of the reference's own functions (cut out of wsol_loader.py / train_wsol.py and executed)."""
    import torch
    from oracle import seeding as oseed
    from tcam_wsol_video_b200 import temporal as tp
    g = _py_golden("py_temporal_agg.npz")
    cams = torch.from_numpy(g["cams"])
    for h_t in (0.0, 10.0, 50.0):
        got = oseed.temporal_max_renorm(cams, h_t).numpy()
        want = g[f"agg_h{int(h_t)}"]
        assert np.array_equal(np.isnan(got), np.isnan(want))
        assert np.array_equal(np.nan_to_num(got, nan=-7.0), np.nan_to_num(want, nan=-7.0)), h_t   # same torch, same bits
    assert np.array_equal(oseed.re_normalize_cam(cams[0, 0], 10.0).numpy(), g["renorm_single_h10"])
    g = _py_golden("py_prepare_std_cams.npz")
    std = torch.from_numpy(g["std_cams"])
    for key in [k for k in g if k.startswith("out_")]:
        size = tuple(int(v) for v in key[4:].split("x"))
        assert np.array_equal(oseed.prepare_std_cams_disq(std, size).numpy(), g[key]), key
    g = _py_golden("py_frame_pickers.npz")
    frames = [str(f) for f in g["frames"]]
    for key in [k for k in g if k.startswith(("left_", "right_"))]:
        side, k, f = key.split("_")
        fn = tp.get_left_knn if side == "left" else tp.get_right_knn
        assert fn(frames, frames[int(f[1:])], int(k[1:])) == [str(v) for v in g[key]], key


def test_seed_sampling_restatement_matches_the_reference_modules():
    """oracle/seeding.py's sample_fg / sample_bg against the reference's own _SFG / _SBG modules executed on the CPU
    generator with the same seed (tests/golden/make_golden_py.py): same stable sort, same candidate order, same
    multinomial draws -> identical seed maps."""
    import torch
    from oracle import seeding as oseed
    g = _py_golden("py_seed_sampling.npz")
    cam, roi = torch.from_numpy(g["cam"]), torch.from_numpy(g["roi"])
    ci = 0
    while f"case{ci}_cfg" in g:
        tech, max_, min_, max_p, min_p, use_roi = [str(v) for v in g[f"case{ci}_cfg"]]
        torch.manual_seed(1000 + ci)
        for i in range(cam.shape[0]):
            fg = oseed.sample_fg(cam[i], roi[i] if use_roi == "1" else None, torch.zeros((48, 56), dtype=torch.long),
                                 float(max_p), int(max_), tech)
            bg = oseed.sample_bg(cam[i], torch.zeros((48, 56), dtype=torch.long), float(min_p), int(min_))
            assert np.array_equal(fg.numpy(), g[f"case{ci}_fg"][i]), (ci, i)
            assert np.array_equal(bg.numpy(), g[f"case{ci}_bg"][i]), (ci, i)
        ci += 1
    assert ci == 4


def test_loss_restatement_matches_the_reference_autograd_function(oracle_mod):
    """oracle.densecrf_loss_fwd_bwd (the 15 restated lines) against the reference's own DenseCRFLossFunction executed
    on CPU tensors with the reference's C++ behind it (tests/golden/make_golden_py.py).  The filter is bit-identical;
    the loss sums 2*3*31*37 float32 products in torch's order there and numpy's here: rel 1e-6."""
    g = _py_golden("py_dense_crf_loss.npz")
    w = float(g["weight"])
    loss, grad, _ = oracle_mod.densecrf_loss_fwd_bwd(g["image"], g["seg"], 15.0, 100.0, w,
                                                    oracle_mod.port_bilateralfilter_batch)
    assert abs(w * float(loss) - float(g["loss"][0])) <= 1e-6 * abs(float(g["loss"][0]))
    assert np.abs(grad - g["grad"]).max() <= 1e-6 * np.abs(g["grad"]).max()


def test_clip_grouping_matches_the_reference_functions():
    """losses.group_ordered_frames / RgbJointConRanFieldTcams.pair_samples against the reference's own functions
    (dlib/losses/tcam.py:32-45, 207-232) executed by tests/golden/make_golden_py.py."""
    import torch
    from tcam_wsol_video_b200.losses import RgbJointConRanFieldTcams, group_ordered_frames
    g = _py_golden("py_clip_grouping.npz")
    groups = group_ordered_frames(torch.from_numpy(g["seq_iter"]), torch.from_numpy(g["frm_iter"]))
    assert len(groups) == int(g["n_groups"])
    imgs, probs = torch.from_numpy(g["imgs"]), torch.from_numpy(g["probs"])
    for gi, grp in enumerate(groups):
        assert list(grp) == g[f"group{gi}"].tolist()
        if len(grp) > 1:
            pi, pc = RgbJointConRanFieldTcams.pair_samples(o_idx=grp, imgs=imgs, prob_cams=probs)
            assert np.array_equal(pi.numpy(), g[f"pair{gi}_img"]) and np.array_equal(pc.numpy(), g[f"pair{gi}_cam"])


def test_colour_loss_restatement_matches_the_reference_autograd_function(oracle_mod):
    g = _py_golden("py_color_dense_crf_loss.npz")
    w = float(g["weight"])
    loss, grad, _ = oracle_mod.color_densecrf_loss_fwd_bwd(g["image"], g["seg"], 15.0, w,
                                                          oracle_mod.port_colorbilateralfilter_batch)
    assert abs(w * float(loss) - float(g["loss"][0])) <= 1e-6 * abs(float(g["loss"][0]))
    assert np.abs(grad - g["grad"]).max() <= 1e-6 * np.abs(g["grad"]).max()


def test_seeder_forward_restatement_matches_the_reference_module():
    """oracle/seeding.py's tcam_seeder_forward against the reference's own TCAMSeeder.forward executed on the CPU
    generator (kornia's dilation replaced by the flat max-pool, torch.device(cuda_id) by the CPU device)."""
    import torch
    from oracle import seeding as oseed
    g = _py_golden("py_tcam_seeder.npz")
    cam, roi = torch.from_numpy(g["cam"]).unsqueeze(1), torch.from_numpy(g["roi"]).unsqueeze(1)
    ci = 0
    while f"case{ci}_cfg" in g:
        kw = {}
        for item in g[f"case{ci}_cfg"]:
            key, val = str(item).split("=")
            kw[key] = val if key == "seed_tech" else (val == "True" if key == "use_roi" else
                                                       (float(val) if key in ("min_p", "max_p") else int(val)))
        torch.manual_seed(2000 + ci)
        got = oseed.tcam_seeder_forward(cam, roi, ignore_idx=-255, **kw)
        assert np.array_equal(got.numpy(), g[f"case{ci}_out"]), ci
        ci += 1
    assert ci == 3


def test_roi_restatement_matches_the_reference_class_run_with_opencv():
    """oracle/seeding.py's GetRoiSingleCam restatement against the reference's own class (dlib/cams/tcam_seeding.py:
    316-430) executed with REAL OpenCV 4.13 for the contour / bounding-rectangle part (tests/golden/make_golden_py.py;
    skimage's label and Otsu stood in for, see there): 48 cases, both component modes, Otsu and fixed thresholds."""
    from oracle import seeding as oseed
    g = _py_golden("py_get_roi_single_cam.npz")
    for ci in range(int(g["n_cases"])):
        method, thresh, cj = [str(v) for v in g[f"c{ci}_cfg"]]
        cam = g[f"cam{cj}"]
        roi, mask, bbox = oseed.roi_components_single_cam(cam, method, 0.05, thresh=float(thresh) if thresh else None)
        assert np.array_equal(roi, g[f"c{ci}_roi"]), ci
        assert np.array_equal(bbox, g[f"c{ci}_bbox"]), ci
        assert np.array_equal(mask, g[f"c{ci}_mask"]), ci


def test_flat_dilation_agrees_with_opencv():
    """kornia 0.6.4 (not installable here) documents its flat-kernel dilation as the max over the ksz x ksz window
    anchored at ksz // 2 with the border ignored; OpenCV's cv2.dilate is an independent implementation of that same
    operator (default anchor = kernel centre = ksz // 2, default border = ignored).  The restatement every seeding
    test relies on (oracle/seeding.py flat_dilation) must agree with it, even kernel sizes included."""
    cv2 = pytest.importorskip("cv2")
    import torch
    from oracle import seeding as oseed
    rng = np.random.default_rng(3)
    for k in (1, 2, 3, 4, 5, 7):
        x = (rng.random((2, 1, 23, 31)) > 0.9).astype(np.float32)
        got = oseed.flat_dilation(torch.from_numpy(x), k).numpy()
        for b in range(2):
            want = cv2.dilate(x[b, 0], np.ones((k, k), np.uint8))
            assert np.array_equal(got[b, 0], want), k


@pytest.mark.parametrize("ksz", [1, 2, 3, 4, 5])
def test_seed_labels_from_sel_repaints_the_seeder(ksz):
    """seed_labels_from_sel (the label map of a [B,2,kmax] selection, which the sparse cross-entropy tests compare the
    kernels with) must repaint tcam_seeder_forward's map from the seeds the restated seeder picked: odd and even
    windows, windows that overlap on one side, fg/bg conflicts, a sample without seeds."""
    import torch
    from oracle import seeding as oseed
    b, h, w, k = 4, 13, 17, 12
    cam = torch.rand((b, 1, h, w), generator=torch.Generator().manual_seed(ksz))
    cam[2] = 0.5                                                 # flat: no seeds
    kw = dict(seed_tech="seed_uniform", min_=k, max_=k, min_p=0.5, max_p=0.5, use_roi=False)
    torch.manual_seed(11)
    want = oseed.tcam_seeder_forward(cam, None, ksz=ksz, ignore_idx=-255, **kw)
    torch.manual_seed(11)                                        # the same draws, sample by sample
    sel = torch.full((b, 2, k), -1, dtype=torch.int32)
    fg, bg = torch.zeros((b, h, w), dtype=torch.long), torch.zeros((b, h, w), dtype=torch.long)
    for i in range(b):
        fg[i], bg[i] = oseed.one_sample(cam[i, 0], None, **{n: kw[n] for n in ("min_p", "max_p", "min_", "max_",
                                                                              "seed_tech", "use_roi")})
        for side, m in enumerate((fg[i], bg[i])):
            idx = torch.nonzero(m.reshape(-1)).flatten()
            sel[i, side, :idx.numel()] = idx.int()
    got = oseed.seed_labels_from_sel(sel, ksz, h, w, -255)
    assert torch.equal(got, want)
    assert (sel[2] == -1).all() and (got[2] == -255).all()
    if ksz > 1:
        dil_fg = oseed.flat_dilation(fg.unsqueeze(1), ksz).squeeze(1)
        dil_bg = oseed.flat_dilation(bg.unsqueeze(1), ksz).squeeze(1)
        assert ((dil_fg == 1) & (dil_bg == 1)).any()             # conflicts: ignored
        win = torch.nn.functional.conv2d(fg.unsqueeze(1).float(), torch.ones(1, 1, ksz, ksz), padding=ksz - 1)
        assert (win > 1).any()                                   # windows overlapping on one side
