"""GPU suite (-m gpu): parity of the CUDA path against the oracle, through the C ABI.

Tolerances (BASELINE.json north_star): filtered tensors, loss and gradient within rel 1e-4 in
fp32; lattice structure (which vertices each pixel touches, barycentric weights) bit-exact.
The only non-bit-exact step is the splat's atomic summation order, so the errors seen are ~1e-6.

Nothing here reads /root/reference: the checker is the C restatement (oracle/permuto_oracle.c)
and the committed golden fixtures (made from the reference build by tests/golden/make_golden.py).
"""
import ctypes
import os

import numpy as np
import pytest

from conftest import GOLDEN, golden_cases, load_golden, pointwise_rel_err, rel_err
from tcam_wsol_video_b200 import _lib, synth

pytestmark = pytest.mark.gpu

REL_TOL = 1e-4  # north_star: "within rel 1e-4 on filtered tensors, CRF loss value and CRF gradient in fp32"


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU suite needs a B200"
    assert _lib.load().tcamcrf_device_count() >= 1
    return torch


@pytest.fixture
def tuning():
    """Sets library tuning knobs for one test (tcamcrf_set_tuning) and restores the defaults afterwards."""
    touched = []

    def set_(name, value):
        touched.append(name)
        _lib.set_tuning(name, -1 if value is None else int(value))

    yield set_
    for name in touched:
        _lib.set_tuning(name, -1)


def _gpu_filter_host(img, seg, srgb, sxy, dim=0):
    """AS through the drop-in host API (reference names, numpy 1-D contract)."""
    from tcam_wsol_video_b200 import bilateralfilter as bf
    from tcam_wsol_video_b200 import colorbilateralfilter as cbf
    n, k, h, w = seg.shape
    out = np.zeros(seg.size, np.float32)
    if dim:
        cbf.colorbilateralfilter_batch(np.ascontiguousarray(img.ravel()), np.ascontiguousarray(seg.ravel()), out,
                                       n, k, h, w, srgb, dim)
    else:
        bf.bilateralfilter_batch(np.ascontiguousarray(img.ravel()), np.ascontiguousarray(seg.ravel()), out,
                                 n, k, h, w, srgb, sxy)
    return out.reshape(seg.shape)


def _assert_close(got, want, what):
    e = rel_err(got, want)
    assert e < REL_TOL, f"{what}: normwise rel err {e:.3e}"
    # pointwise, with a floor at 1e-3 of the largest magnitude (outputs are positive and of similar scale)
    pe = pointwise_rel_err(got, want, floor=1e-3 * float(np.abs(want).max()))
    assert pe < REL_TOL, f"{what}: pointwise rel err {pe:.3e}"


# ---------------------------------------------------------------------------
# golden fixtures (reference-made)
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("path", golden_cases(), ids=os.path.basename)
def test_host_api_matches_golden(torch_cuda, path):
    g = load_golden(path)
    img = g["image_u8"].astype(np.float32)
    got = _gpu_filter_host(img, g["seg"], float(g["sigma_rgb"]), float(g["sigma_xy"]), int(g["dim"]))
    _assert_close(got, g["AS"], "AS")


@pytest.mark.parametrize("path", golden_cases(), ids=os.path.basename)
def test_module_loss_and_grad_match_golden(torch_cuda, path):
    torch = torch_cuda
    from tcam_wsol_video_b200.color_dense_crf_loss import ColorDenseCRFLoss
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    g = load_golden(path)
    images = torch.from_numpy(g["image_u8"].astype(np.float32))          # CPU, like the trainer passes it
    seg = torch.from_numpy(g["seg"]).cuda().requires_grad_(True)
    weight = 1.0
    if int(g["dim"]):
        mod = ColorDenseCRFLoss(weight=weight, sigma_rgb=float(g["sigma_rgb"]), scale_factor=1.0)
    else:
        mod = DenseCRFLoss(weight=weight, sigma_rgb=float(g["sigma_rgb"]), sigma_xy=float(g["sigma_xy"]),
                           scale_factor=1.0)
    loss = mod(images=images, segmentations=seg)
    assert loss.shape == (1,) and loss.device == seg.device and loss.dtype == torch.float32
    loss.backward()
    assert abs(loss.item() - float(g["loss"])) < REL_TOL * abs(float(g["loss"]))
    _assert_close(seg.grad.cpu().numpy(), g["grad"], "grad")


def test_golden_224_noise(torch_cuda):
    g = load_golden(os.path.join(GOLDEN, "bf5_noise_n1_k2_224x224.npz"))
    n, k, h, w = (int(v) for v in g["shape"])
    img = synth.make_images(n, h, w, str(g["kind"]), seed=int(g["seed"]))
    seg = synth.make_segs(n, k, h, w, seed=int(g["seed"]))
    got = _gpu_filter_host(img, seg, float(g["sigma_rgb"]), float(g["sigma_xy"]))
    _assert_close(got.ravel()[:: int(g["stride"])], g["AS_sample"], "AS sample")
    assert abs(got.astype(np.float64).sum() - float(g["AS_sum"])) < 1e-5 * float(g["AS_sum"])
    loss = -float((seg.astype(np.float64) * got).sum()) / n
    assert abs(loss - float(g["loss"])) < REL_TOL * abs(float(g["loss"]))


# ---------------------------------------------------------------------------
# lattice structure: bit-exact
# ---------------------------------------------------------------------------
def _debug_lattice(cfg, img, h, w):
    lib = _lib.load()
    d = (2 + cfg.channels) if cfg.feat == _lib.FEAT_XY_RGB else cfg.channels
    p = h * w
    off = np.zeros(p * (d + 1), np.int32)
    bary = np.zeros(p * (d + 1), np.float32)
    m = ctypes.c_int(0)
    img = np.ascontiguousarray(img, dtype=np.float32)
    nbr = np.zeros((d + 1) * p * (d + 1) * 2, np.int32)
    _lib.check(lib.tcamcrf_debug_lattice(ctypes.byref(cfg), img.ctypes.data, h, w, off.ctypes.data, bary.ctypes.data,
                                         ctypes.byref(m), nbr.ctypes.data, nbr.size), "tcamcrf_debug_lattice")
    M = m.value
    return off.reshape(p, d + 1), bary.reshape(p, d + 1), M, nbr[: (d + 1) * M * 2].reshape(d + 1, M, 2)


@pytest.mark.parametrize("build", ["0", "1"], ids=["build_kernel", "build_dedup_kernel"])
@pytest.mark.parametrize("kind", ["noise", "natural"])
@pytest.mark.parametrize("dim", [0, 3, 1])
@pytest.mark.parametrize("hw", [(32, 40), (31, 37), (224, 224)])
def test_lattice_structure_bit_exact(torch_cuda, oracle_mod, tuning, kind, dim, hw, build):
    """Both build kernels (lock-step probes per pixel / the block's distinct keys deduplicated in shared memory
    first), forced through TCAMCRF_BUILD_DEDUP; the library picks between them from the density hint."""
    tuning("BUILD_DEDUP", build)
    h, w = hw
    img = synth.make_images(1, h, w, kind, seed=21)[0]
    if dim:
        cfg = _lib.make_config(_lib.FEAT_COLOR, dim, 15.0)
        L = oracle_mod.port_lattice_color(img, h, w, 15.0, dim)
        img_in = img[:dim]
    else:
        cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
        L = oracle_mod.port_lattice_bilateral(img, h, w, 15.0, 100.0)
        img_in = img
    off, bary, M, nbr = _debug_lattice(cfg, img_in, h, w)
    p = h * w
    d = L.d
    # both sides also hold the vertices of the reference's zero-feature padding pixels when P % 4 != 0
    # (permutohedral.cpp:173,238-251); no real pixel points at those that are padding-only
    assert M == L.m
    used = np.unique(L.offset[:p])
    assert np.array_equal(bary, L.bary[:p])                     # bit-exact weights
    # ids are a relabelling: the map oracle id -> gpu id must be a bijection on the vertices pixels touch
    fwd = np.full(L.m, -1, np.int64)
    fwd[L.offset[:p].ravel()] = off.ravel()
    assert np.array_equal(fwd[L.offset[:p].ravel()], off.ravel())   # consistent
    assert len(np.unique(fwd[used])) == len(used)                   # injective
    gpu_used = set(fwd[used].tolist())
    # neighbour tables agree under the relabelling; missing stays missing; a padding-only neighbour (whose
    # relabelling is unknown) must at least exist on the gpu side and not be one of the pixel-touched vertices
    ext = np.concatenate([fwd, [-1]])
    for j in range(d + 1):
        want_ref = L.nbr[j][used]                                   # [len(used), 2] in oracle ids
        want = ext[want_ref]
        got = nbr[j][fwd[used]]
        known = (want_ref < 0) | (want >= 0)
        assert np.array_equal(want[known], got[known]), f"axis {j}"
        for g in got[~known].ravel().tolist():
            assert g >= 0 and g not in gpu_used, f"axis {j}: padding-only neighbour"


# ---------------------------------------------------------------------------
# oracle comparisons on seeded inputs
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["noise", "natural"])
@pytest.mark.parametrize("shape", [(1, 2, 224, 224), (3, 10, 64, 48), (2, 1, 33, 35), (2, 3, 17, 129), (1, 4, 1, 1),
                                   (2, 2, 1, 50), (1, 5, 3, 2), (1, 2, 448, 448)])
def test_filter_vs_oracle(torch_cuda, oracle_mod, kind, shape):
    n, k, h, w = shape
    img = synth.make_images(n, h, w, kind, seed=31)
    seg = synth.make_segs(n, k, h, w, seed=31)
    want = oracle_mod.port_bilateralfilter_batch(img, seg, n, k, h, w, 15.0, 100.0).reshape(seg.shape)
    got = _gpu_filter_host(img, seg, 15.0, 100.0)
    _assert_close(got, want, "5-D AS")
    want = oracle_mod.port_colorbilateralfilter_batch(img, seg, n, k, h, w, 15.0, 3).reshape(seg.shape)
    got = _gpu_filter_host(img, seg, 15.0, 0.0, dim=3)
    _assert_close(got, want, "3-D colour AS")


@pytest.mark.parametrize("sig", [(1.0, 1.0), (3.0, 10.0), (80.0, 300.0), (255.0, 1000.0)])
def test_sigma_extremes(torch_cuda, oracle_mod, sig):
    srgb, sxy = sig
    n, k, h, w = 1, 2, 40, 40
    img = synth.make_images(n, h, w, "noise", seed=41)
    seg = synth.make_segs(n, k, h, w, seed=41)
    want = oracle_mod.port_bilateralfilter_batch(img, seg, n, k, h, w, srgb, sxy).reshape(seg.shape)
    _assert_close(_gpu_filter_host(img, seg, srgb, sxy), want, f"sigma {sig}")


def test_constant_image_and_signed_input(torch_cuda, oracle_mod):
    """One colour everywhere (heavy key duplication: every warp inserts the same vertices) and a
    segmentation with negative entries (the filter is linear, not restricted to probabilities)."""
    n, k, h, w = 2, 2, 48, 64
    img = np.full((n, 3, h, w), 128.0, np.float32)
    rng = np.random.default_rng(5)
    seg = rng.standard_normal((n, k, h, w)).astype(np.float32)
    want = oracle_mod.port_bilateralfilter_batch(img, seg, n, k, h, w, 15.0, 100.0).reshape(seg.shape)
    got = _gpu_filter_host(img, seg, 15.0, 100.0)
    assert rel_err(got, want) < REL_TOL
    want = oracle_mod.port_colorbilateralfilter_batch(img, seg, n, k, h, w, 15.0, 3).reshape(seg.shape)
    got = _gpu_filter_host(img, seg, 15.0, 0.0, dim=3)
    assert rel_err(got, want) < REL_TOL


def test_single_image_entry_points(torch_cuda, oracle_mod):
    from tcam_wsol_video_b200 import bilateralfilter as bf
    from tcam_wsol_video_b200 import colorbilateralfilter as cbf
    k, h, w = 3, 30, 26
    img = synth.make_images(1, h, w, "natural", seed=51)
    seg = synth.make_segs(1, k, h, w, seed=51)
    out = np.zeros(seg.size, np.float32)
    bf.bilateralfilter(img.ravel(), seg.ravel(), out, h, w, 15.0, 100.0)     # K inferred from len(in)
    want = oracle_mod.port_bilateralfilter_batch(img, seg, 1, k, h, w, 15.0, 100.0)
    _assert_close(out, want, "bilateralfilter")
    out = np.zeros(seg.size, np.float32)
    cbf.colorbilateralfilter(img.ravel(), seg.ravel(), out, h, w, 15.0, 3)
    want = oracle_mod.port_colorbilateralfilter_batch(img, seg, 1, k, h, w, 15.0, 3)
    _assert_close(out, want, "colorbilateralfilter")
    # empty batch: the reference's loop runs zero times and leaves `outs` untouched
    out = np.full(4, 7.0, np.float32)
    bf.bilateralfilter_batch(np.zeros(0, np.float32), np.zeros(0, np.float32), out, 0, 2, 4, 4, 15.0, 100.0)
    assert np.all(out == 7.0)


@pytest.mark.parametrize("n,groups", [(70, None), (7, "3"), (5, "16"), (33, "1")])
def test_host_path_groups_and_chunks(torch_cuda, oracle_mod, tuning, n, groups):
    """Host-pointer path: the lattice of a whole chunk (<= 64 frames) is built at once, the value stages run group
    by group with a frame offset; more than 64 frames take several chunks.  Ragged group / chunk sizes included.
    Also the fused loss + gradient entry point (tcamcrf_loss_fwd_bwd_host)."""
    import ctypes
    from tcam_wsol_video_b200 import _lib
    tuning("HOST_GROUPS", groups)
    k, h, w = 3, 13, 18
    img = synth.make_images(n, h, w, "noise", seed=n)
    seg = synth.make_segs(n, k, h, w, seed=n)
    want = oracle_mod.port_bilateralfilter_batch(img, seg, n, k, h, w, 15.0, 100.0).reshape(seg.shape)
    got = _gpu_filter_host(img, seg, 15.0, 100.0, dim=0)
    _assert_close(got, want, "AS (host path)")
    lib = _lib.load()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    loss = np.zeros(1, np.float32)
    grad = np.zeros_like(seg)
    img_c, seg_c = np.ascontiguousarray(img), np.ascontiguousarray(seg)
    _lib.check(lib.tcamcrf_loss_fwd_bwd_host(ctypes.byref(cfg), img_c.ctypes.data, seg_c.ctypes.data,
                                             loss.ctypes.data, grad.ctypes.data, n, k, h, w, 0.5), "fwd_bwd_host")
    want_loss, want_grad, _ = oracle_mod.densecrf_loss_fwd_bwd(img, seg, 15.0, 100.0, 0.5,
                                                               oracle_mod.port_bilateralfilter_batch)
    assert abs(float(loss[0]) - float(want_loss)) < REL_TOL * abs(float(want_loss))
    assert rel_err(grad, want_grad) < REL_TOL


@pytest.mark.parametrize("n,k", [(32, 10), (32, 2), (21, 7), (70, 6), (5, 2), (1, 10)])
def test_host_path_graph_replay(torch_cuda, oracle_mod, n, k):
    """Host-pointer path with PINNED buffers: the first call runs the three-stream schedule eagerly and captures it,
    later calls replay the CUDA graph (one launch per call).  Eager call, two replays with new data in the same
    buffers, new buffers (a new schedule) and pageable buffers (eager, while the cache holds the pinned buffers'
    schedules) must all match the oracle.  The shapes cover one and several chunks, wide (K >= 6) and narrow value
    rows, and ragged sections and groups."""
    import ctypes
    torch = torch_cuda
    from tcam_wsol_video_b200 import _lib
    lib = _lib.load()
    h, w = 20, 24
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    bufs = [(torch.empty(n, 3, h, w).pin_memory(), torch.empty(n, k, h, w).pin_memory(),
             torch.empty(1).pin_memory(), torch.empty(n, k, h, w).pin_memory()) for _ in range(2)]
    launches = []
    for call in range(5):
        img = synth.make_images(n, h, w, "noise" if call % 2 == 0 else "natural", seed=50 + call)
        seg = synth.make_segs(n, k, h, w, seed=50 + call)
        if call == 4:
            img_h, seg_h = np.ascontiguousarray(img, np.float32), np.ascontiguousarray(seg, np.float32)
            loss_h, grad_h = np.zeros(1, np.float32), np.zeros_like(seg_h)
            ptrs = [a.ctypes.data for a in (img_h, seg_h, loss_h, grad_h)]
        else:
            img_h, seg_h, loss_h, grad_h = bufs[0] if call != 3 else bufs[1]
            img_h.copy_(torch.from_numpy(img))
            seg_h.copy_(torch.from_numpy(seg))
            grad_h.zero_()
            ptrs = [t.data_ptr() for t in (img_h, seg_h, loss_h, grad_h)]
        l0 = lib.tcamcrf_launch_count()
        _lib.check(lib.tcamcrf_loss_fwd_bwd_host(ctypes.byref(cfg), *ptrs, n, k, h, w, 0.25), "fwd_bwd_host")
        launches.append(lib.tcamcrf_launch_count() - l0)
        want_loss, want_grad, _ = oracle_mod.densecrf_loss_fwd_bwd(img, seg, 15.0, 100.0, 0.25,
                                                                   oracle_mod.port_bilateralfilter_batch)
        assert abs(float(loss_h[0]) - float(want_loss)) < REL_TOL * abs(float(want_loss)), f"call {call}"
        assert rel_err(np.asarray(grad_h), want_grad) < REL_TOL, f"call {call}"
    # a replay accounts for as many kernels as the eager call it was captured from
    assert launches[1] == launches[0] and launches[2] == launches[0] and launches[0] > 0, launches


@pytest.mark.parametrize("n,sections", [(32, None), (5, None), (70, None), (9, "1"), (13, "64"), (1, None)])
def test_host_frames_path(torch_cuda, oracle_mod, tuning, n, sections):
    """Frames left on the CPU in pinned memory (what the reference's trainer passes) take
    tcamcrf_loss_forward_host_frames: copied section by section on the library's copy stream while the lattice of
    the sections already in is built.  Same AS / loss as the oracle, for one and several chunks, ragged sections,
    the filter-only and the fused-softmax variants; pageable frames take the plain copy."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    tuning("HIMG_SECTIONS", sections)
    k, h, w = 3, 24, 20
    img = synth.make_images(n, h, w, "noise" if n % 2 else "natural", seed=90 + n)
    seg_np = synth.make_segs(n, k, h, w, seed=90 + n)
    seg = torch.from_numpy(seg_np).cuda()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    want_loss, _, want_as = oracle_mod.densecrf_loss_fwd_bwd(img, seg_np, 15.0, 100.0, 1.0,
                                                             oracle_mod.port_bilateralfilter_batch)
    pinned = torch.from_numpy(img).pin_memory()
    assert ops._host_frames(pinned, seg.device) and not ops._host_frames(torch.from_numpy(img), seg.device)
    lib = _lib.load()
    for rep in range(3):     # the staging buffer and the copy lane are reused from call to call
        l0 = lib.tcamcrf_launch_count()
        got, loss, _ = ops.crf_forward(pinned, seg, cfg, check=True)
        launches = lib.tcamcrf_launch_count() - l0
        _assert_close(got.cpu().numpy(), want_as, f"AS, host frames, call {rep}")
        assert abs(loss.item() - float(want_loss)) < REL_TOL * abs(float(want_loss))
    l0 = lib.tcamcrf_launch_count()
    got_dev, _, _ = ops.crf_forward(torch.from_numpy(img), seg, cfg, check=True)     # pageable: plain copy, one section
    torch.cuda.synchronize()
    if n > 4 and sections != "1":
        assert launches > lib.tcamcrf_launch_count() - l0      # the lattice stages really ran section by section
    assert rel_err(got.cpu().numpy(), got_dev.cpu().numpy()) < 1e-5
    # uint8 frames from the loader (a quarter of the bytes on the wire): identical features
    pinned8 = torch.from_numpy(img.astype(np.uint8)).pin_memory()
    assert ops._host_frames(pinned8, seg.device)
    got8, loss8, _ = ops.crf_forward(pinned8, seg, cfg, check=True)
    _assert_close(got8.cpu().numpy(), want_as, "AS, uint8 host frames")
    assert abs(loss8.item() - float(want_loss)) < REL_TOL * abs(float(want_loss))
    got, loss = ops.crf_forward(pinned, seg, cfg, want_loss=False, check=True)[:2]
    assert loss is None
    _assert_close(got.cpu().numpy(), want_as, "AS, host frames, filter only")
    logits = torch.from_numpy(np.log(seg_np)).cuda()       # softmax(log p) = p
    got, loss, _ = ops.crf_forward_logits(pinned, logits, cfg, check=True)
    _assert_close(got.cpu().numpy(), want_as, "AS, host frames, fused softmax")
    assert abs(loss.item() - float(want_loss)) < REL_TOL * abs(float(want_loss))


def test_u8_images_and_chunking_give_identical_results(torch_cuda):
    """uint8 images produce the same features as float images holding the same integers, and processing the
    batch in chunks of frames does not change anything but the summation order inside the loss."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    n, k, h, w = 5, 2, 40, 56
    img = synth.make_images(n, h, w, "natural", seed=61)
    seg = torch.from_numpy(synth.make_segs(n, k, h, w, seed=61)).cuda()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    as_f, loss_f, _ = ops.crf_forward(torch.from_numpy(img).cuda(), seg, cfg, check=True)
    as_u, loss_u, _ = ops.crf_forward(torch.from_numpy(img.astype(np.uint8)).cuda(), seg, cfg, check=True)
    cfg2 = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0, chunk_frames=2)
    as_c, loss_c, _ = ops.crf_forward(torch.from_numpy(img), seg, cfg2, check=True)
    assert rel_err(as_u.cpu().numpy(), as_f.cpu().numpy()) < 1e-5
    assert rel_err(as_c.cpu().numpy(), as_f.cpu().numpy()) < 1e-5
    assert abs(loss_u.item() - loss_f.item()) < 1e-5 * abs(loss_f.item())
    assert abs(loss_c.item() - loss_f.item()) < 1e-5 * abs(loss_f.item())


def test_backward_is_bit_exact_given_AS(torch_cuda):
    """grad = ((-2*g)*AS)/N with the reference's rounding order: identical bits to the torch expression."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    torch.manual_seed(0)
    as_t = torch.rand(3, 2, 31, 17, device="cuda") * 50
    g = torch.tensor([1e-7 * 3.3], device="cuda")
    got = ops.crf_backward(as_t, g, 3.0)
    want = -2 * g * as_t / torch.tensor([3.0], device="cuda")
    assert torch.equal(got, want)


def test_module_scale_factor_and_amp(torch_cuda, oracle_mod):
    """scale_factor != 1 (nearest / bilinear rescale first, sigma_xy scaled; dense_crf_loss.py:105-121) and
    a call under autocast (custom_fwd keeps the op in fp32)."""
    torch = torch_cuda
    import torch.nn.functional as F
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    n, k, h, w = 2, 2, 48, 64
    img = torch.from_numpy(synth.make_images(n, h, w, "natural", seed=71))
    seg = torch.from_numpy(synth.make_segs(n, k, h, w, seed=71)).cuda().requires_grad_(True)
    mod = DenseCRFLoss(weight=1e-3, sigma_rgb=15.0, sigma_xy=100.0, scale_factor=0.5).cuda()
    with torch.autocast("cuda", dtype=torch.float16):
        loss = mod(images=img, segmentations=seg)
    loss.backward()
    # oracle on the rescaled inputs
    simg = F.interpolate(img, scale_factor=0.5, mode="nearest", recompute_scale_factor=False).numpy()
    sseg = F.interpolate(seg.detach().cpu(), scale_factor=0.5, mode="bilinear", recompute_scale_factor=False,
                         align_corners=False)
    want_loss, want_grad, _ = oracle_mod.densecrf_loss_fwd_bwd(simg, sseg.numpy(), 15.0, 50.0, 1.0,
                                                               oracle_mod.port_bilateralfilter_batch)
    assert abs(loss.item() - 1e-3 * float(want_loss)) < REL_TOL * abs(1e-3 * float(want_loss))
    # gradient w.r.t. the full-resolution segmentation = bilinear-adjoint of the oracle's gradient
    sseg_t = F.interpolate(seg.detach().cpu().requires_grad_(True), scale_factor=0.5, mode="bilinear",
                           recompute_scale_factor=False, align_corners=False)
    ref_in = seg.detach().cpu().requires_grad_(True)
    F.interpolate(ref_in, scale_factor=0.5, mode="bilinear", recompute_scale_factor=False,
                  align_corners=False).backward(torch.from_numpy(want_grad) * 1e-3)
    assert rel_err(seg.grad.cpu().numpy(), ref_in.grad.numpy()) < REL_TOL


def test_device_status_poisons_outputs(torch_cuda):
    """A vertex pool that is too small must yield NaN outputs and a readable status, never wrong numbers."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    n, k, h, w = 1, 2, 64, 64
    img = torch.from_numpy(synth.make_images(n, h, w, "noise", seed=81))
    seg = torch.from_numpy(synth.make_segs(n, k, h, w, seed=81)).cuda()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0, pool_factor=0.01)
    as_t, loss, ws = ops.crf_forward(img, seg, cfg, check=False)
    st, _ = ops.workspace_status(ws)
    assert st & _lib.DEV_POOL_FULL
    assert torch.isnan(loss).all() and torch.isnan(as_t).all()
    with pytest.raises(_lib.TcamCrfError):
        ops.crf_forward(img, seg, cfg, check=True)
    # key range: sigma so small that lattice coordinates leave the packed fields
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 1e-3, 100.0)
    as_t, loss, ws = ops.crf_forward(img, seg, cfg, check=False)
    st, _ = ops.workspace_status(ws)
    assert st & _lib.DEV_KEY_RANGE and torch.isnan(loss).all()


@pytest.mark.parametrize("build", ["0", "1"], ids=["build_kernel", "build_dedup_kernel"])
@pytest.mark.parametrize("load", [0.25, 0.5, 0.9, 4.0, 64.0])
def test_hash_load_factor_sweep(torch_cuda, oracle_mod, tuning, load, build):
    """BASELINE config 4 (occupancy sweep): results do not depend on the table size.  Loads above ~1 make the
    primary tier smaller than the lattice, so most vertices live in the overflow tier."""
    torch = torch_cuda
    tuning("BUILD_DEDUP", build)
    from tcam_wsol_video_b200 import ops
    n, k, h, w = 1, 2, 96, 96
    img = synth.make_images(n, h, w, "noise", seed=91)
    seg = synth.make_segs(n, k, h, w, seed=91)
    want = oracle_mod.port_bilateralfilter_batch(img, seg, n, k, h, w, 15.0, 100.0).reshape(seg.shape)
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0, hash_load=load)
    as_t, _, _ = ops.crf_forward(torch.from_numpy(img), torch.from_numpy(seg).cuda(), cfg, check=True)
    _assert_close(as_t.cpu().numpy(), want, f"load {load}")


@pytest.mark.parametrize("build", ["0", "1"], ids=["build_kernel", "build_dedup_kernel"])
def test_overflow_tier_is_cleared_between_calls(torch_cuda, oracle_mod, tuning, build):
    """A call that spills into the overflow tier leaves keys there; the next call on the same workspace (same
    plan) must not see them.  Three different images back to back through a deliberately tiny primary tier."""
    torch = torch_cuda
    tuning("BUILD_DEDUP", build)
    from tcam_wsol_video_b200 import ops
    n, k, h, w = 2, 2, 64, 80
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0, hash_load=64.0)
    for seed in (101, 102, 103):
        img = synth.make_images(n, h, w, "noise", seed=seed)
        seg = synth.make_segs(n, k, h, w, seed=seed)
        want = oracle_mod.port_bilateralfilter_batch(img, seg, n, k, h, w, 15.0, 100.0).reshape(seg.shape)
        as_t, _, ws = ops.crf_forward(torch.from_numpy(img), torch.from_numpy(seg).cuda(), cfg, check=True)
        _assert_close(as_t.cpu().numpy(), want, f"seed {seed}")
        # vertex count equals the oracle's (stale keys would inflate it)
        _, m_total = ops.workspace_status(ws)
        m_want = sum(oracle_mod.port_lattice_bilateral(img[i], h, w, 15.0, 100.0).m for i in range(n))
        assert m_total == m_want


@pytest.mark.parametrize("k", [2, 10, 7])
def test_adaptive_table_size_follows_the_frames(torch_cuda, oracle_mod, k):
    """The primary table tier a call uses is sized from the previous call's vertex counts (effective_geom).  Alternate
    natural frames (few vertices) and iid-noise frames (the worst case) on ONE workspace, both ways round: a guess
    that is too small must only cost speed (overflow tier), never correctness."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import _lib, ops
    n, h, w = 3, 96, 112
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    seg_np = synth.make_segs(n, k, h, w, seed=3)
    seg = torch.from_numpy(seg_np).cuda()
    sizes = []
    for step, kind in enumerate(["natural", "natural", "noise", "noise", "natural", "noise", "natural"]):
        img = synth.make_images(n, h, w, kind, seed=40 + step)
        got, _, ws = ops.crf_forward(torch.from_numpy(img), seg, cfg, want_loss=False, check=True)
        want = oracle_mod.port_bilateralfilter_batch(img, seg_np, n, k, h, w, 15.0, 100.0).reshape(seg_np.shape)
        _assert_close(got.cpu().numpy(), want, f"AS, call {step} ({kind})")
        sizes.append(int(ws.view(torch.int32)[(ws.data_ptr() + 255) // 256 * 256 - ws.data_ptr():][18].item())
                     if ws.data_ptr() % 256 == 0 else None)
    # the size in use shrinks after a natural call and grows back after a noise call (word 18 of the ctrl block)
    if all(s is not None for s in sizes):
        assert sizes[1] < sizes[3], sizes
        assert sizes[4] == sizes[3] and sizes[5] < sizes[3], sizes     # call 4 still sized by the noise call 3


@pytest.mark.parametrize("kind", ["noise", "natural"])
@pytest.mark.parametrize("k,dim,hw", [(10, 0, (40, 52)), (5, 0, (33, 35)), (7, 0, (24, 130)), (12, 0, (31, 37)),
                                      (16, 0, (40, 40)), (13, 3, (40, 44)), (9, 0, (1, 50))])
def test_row_cooperative_kernels(torch_cuda, oracle_mod, tuning, kind, k, dim, hw):
    """splat_rows_kernel / slice_rows_kernel (the kernels the density hint selects for dense lattices, K = 5..16:
    neighbouring lanes share a vertex row) forced on with TCAMCRF_DENSE=1, against the oracle and against the
    per-pixel kernels (TCAMCRF_DENSE=0): every row width (2, 3, 4 float4s), ragged frames (pixel counts that are
    not multiples of 32), 5-D and colour lattices, probabilities and the fused softmax."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    h, w = hw
    n = 3
    img = synth.make_images(n, h, w, kind, seed=k)
    seg_np = synth.make_segs(n, k, h, w, seed=k)
    seg = torch.from_numpy(seg_np).cuda()
    logits = torch.from_numpy(np.log(seg_np)).cuda()       # softmax(log p) = p
    if dim:
        cfg = _lib.make_config(_lib.FEAT_COLOR, dim, 15.0)
        want = oracle_mod.port_colorbilateralfilter_batch(img, seg_np, n, k, h, w, 15.0, dim).reshape(seg_np.shape)
    else:
        cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
        want = oracle_mod.port_bilateralfilter_batch(img, seg_np, n, k, h, w, 15.0, 100.0).reshape(seg_np.shape)
    want_loss = -(seg_np.astype(np.float64) * want.astype(np.float64)).sum() / n
    out = {}
    for mode in ("0", "1"):
        tuning("DENSE", mode)
        got, loss, _ = ops.crf_forward(torch.from_numpy(img), seg, cfg, check=True)
        _assert_close(got.cpu().numpy(), want, f"AS, TCAMCRF_DENSE={mode}")
        assert abs(loss.item() - want_loss) < REL_TOL * abs(want_loss)
        out[mode] = got
        got, loss, _ = ops.crf_forward_logits(torch.from_numpy(img), logits, cfg, check=True)
        _assert_close(got.cpu().numpy(), want, f"AS from logits, TCAMCRF_DENSE={mode}")
        assert abs(loss.item() - want_loss) < REL_TOL * abs(want_loss)
    assert rel_err(out["1"].cpu().numpy(), out["0"].cpu().numpy()) < 1e-5


def test_large_frames_take_smaller_chunks(torch_cuda, oracle_mod):
    """1024x1024 frames: the default chunk drops below 64 (tcamcrf_chunk_frames) and a batch larger than it goes
    through several passes over one workspace; frames are independent, so the result equals the same frames
    filtered two at a time, and frame 0 equals the oracle."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    k, h, w = 2, 1024, 1024
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    cap = ops.lattice_capacity(cfg, k, h, w)
    assert 1 <= cap < 64
    n = cap + 3
    img_np = synth.make_images(n, h, w, "natural", seed=11)
    seg_np = synth.make_segs(n, k, h, w, seed=11)
    img = torch.from_numpy(img_np).cuda()
    seg = torch.from_numpy(seg_np).cuda()
    got, loss, _ = ops.crf_forward(img, seg, cfg, check=True)
    for n0 in (0, cap - 1, n - 2):          # first chunk, across the chunk boundary, last chunk
        part, _, _ = ops.crf_forward(img[n0:n0 + 2].contiguous(), seg[n0:n0 + 2].contiguous(), cfg, check=True)
        assert rel_err(part.cpu().numpy(), got[n0:n0 + 2].cpu().numpy()) < 1e-5
    want0 = oracle_mod.port_bilateralfilter_batch(img_np[:1], seg_np[:1], 1, k, h, w, 15.0, 100.0).reshape(1, k, h, w)
    _assert_close(got[:1].cpu().numpy(), want0, "AS, 1024x1024 frame 0")
    want_loss = -(seg.double() * got.double()).sum() / n
    assert abs(loss.item() - want_loss.item()) < 1e-5 * abs(want_loss.item())
    del got, img, seg, part
    ops.release_workspaces()       # ~19 GiB: do not keep it for the rest of the session
    torch.cuda.empty_cache()


def test_full_size_properties_config2(torch_cuda):
    """BASELINE configs[1] at full size (32 x 10 classes x 224^2): too slow for the scalar oracle in a unit
    test, so check size-independent properties: linearity, channel independence (K=10 in one pass equals
    ten K=1 passes), determinism of the lattice, and frame independence."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    n, k, h, w = 32, 10, 224, 224
    img = torch.from_numpy(synth.make_images(n, h, w, "noise", seed=0)).cuda()
    seg = torch.from_numpy(synth.make_segs(n, k, h, w, seed=0)).cuda()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    as1, loss1, _ = ops.crf_forward(img, seg, cfg, check=True)
    assert torch.isfinite(as1).all() and as1.min() > 0
    # loss definition
    want = -(seg.double() * as1.double()).sum() / n
    assert abs(loss1.item() - want.item()) < 1e-5 * abs(want.item())
    # linearity
    as2, _, _ = ops.crf_forward(img, (seg * 3.0).contiguous(), cfg, check=True)
    assert rel_err(as2.cpu().numpy(), (as1 * 3.0).cpu().numpy()) < 1e-5
    # channel independence: class 7 alone
    as7, _, _ = ops.crf_forward(img, seg[:, 7:8].contiguous(), cfg, check=True)
    assert rel_err(as7.cpu().numpy(), as1[:, 7:8].cpu().numpy()) < 1e-5
    # frame independence: frames 5..8 alone
    as_sub, _, _ = ops.crf_forward(img[5:9].contiguous(), seg[5:9].contiguous(), cfg, check=True)
    assert rel_err(as_sub.cpu().numpy(), as1[5:9].cpu().numpy()) < 1e-5


def test_cuda_graph_capture_and_replay(torch_cuda, oracle_mod):
    """The device API never synchronises or allocates, so a whole fwd+bwd can be captured in a CUDA graph and
    replayed on new data (table clearing, vertex counts and the loss ticket are all device-side)."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    n, k, h, w = 4, 2, 64, 72
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    img = torch.zeros((n, 3, h, w), device="cuda")
    seg = torch.zeros((n, k, h, w), device="cuda")
    g_out = torch.tensor([0.5], device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        img.copy_(torch.from_numpy(synth.make_images(n, h, w, "noise", seed=1)))
        seg.copy_(torch.from_numpy(synth.make_segs(n, k, h, w, seed=1)))
        for _ in range(2):                              # warm-up on the capture stream (allocates the workspace)
            as_t, loss, _ = ops.crf_forward(img, seg, cfg)
            grad = ops.crf_backward(as_t, g_out, float(n))
    torch.cuda.current_stream().wait_stream(side)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        as_t, loss, _ = ops.crf_forward(img, seg, cfg)
        grad = ops.crf_backward(as_t, g_out, float(n))
    for seed, kind in ((2, "natural"), (3, "noise")):
        img_np = synth.make_images(n, h, w, kind, seed=seed)
        seg_np = synth.make_segs(n, k, h, w, seed=seed)
        img.copy_(torch.from_numpy(img_np))
        seg.copy_(torch.from_numpy(seg_np))
        graph.replay()
        torch.cuda.synchronize()
        want_loss, want_grad, want_as = oracle_mod.densecrf_loss_fwd_bwd(img_np, seg_np, 15.0, 100.0, 0.5,
                                                                         oracle_mod.port_bilateralfilter_batch)
        _assert_close(as_t.cpu().numpy(), want_as, f"graph AS {kind}")
        _assert_close(grad.cpu().numpy(), want_grad, f"graph grad {kind}")
        assert abs(loss.item() - float(want_loss)) < REL_TOL * abs(float(want_loss))


def test_cuda_graph_capture_with_host_frames(torch_cuda, oracle_mod):
    """The host-frames forward only forks to the library's copy stream and joins back with events, so it can be
    captured too: the graph then re-reads the pinned frames on every replay."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    n, k, h, w = 6, 2, 40, 36
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    frames = torch.zeros((n, 3, h, w)).pin_memory()
    seg = torch.zeros((n, k, h, w), device="cuda")
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        frames.copy_(torch.from_numpy(synth.make_images(n, h, w, "natural", seed=5)))
        seg.copy_(torch.from_numpy(synth.make_segs(n, k, h, w, seed=5)))
        for _ in range(2):                              # warm-up on the capture stream (workspace, copy lane)
            as_t, loss, _ = ops.crf_forward(frames, seg, cfg)
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=side):
        as_t, loss, _ = ops.crf_forward(frames, seg, cfg)
    for seed, kind in ((6, "noise"), (7, "natural")):
        img_np = synth.make_images(n, h, w, kind, seed=seed)
        seg_np = synth.make_segs(n, k, h, w, seed=seed)
        frames.copy_(torch.from_numpy(img_np))          # host-side write: the replay below picks it up
        seg.copy_(torch.from_numpy(seg_np))
        torch.cuda.synchronize()
        graph.replay()
        torch.cuda.synchronize()
        want_loss, _, want_as = oracle_mod.densecrf_loss_fwd_bwd(img_np, seg_np, 15.0, 100.0, 1.0,
                                                                 oracle_mod.port_bilateralfilter_batch)
        _assert_close(as_t.cpu().numpy(), want_as, f"graph AS, host frames, {kind}")
        assert abs(loss.item() - float(want_loss)) < REL_TOL * abs(float(want_loss))


def test_temporal_max_bit_exact(torch_cuda):
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    cams = torch.from_numpy(synth.make_low_res_cams(32, 5, 28, 28, seed=0)).cuda()
    cams[3, 2, 0, 5, 5] = float("nan")
    cams[4, 0, 0, 1, 1] = float("nan")
    cams[6, 4, 0, 0, 0] = float("inf")
    got = ops.temporal_cam_max(cams)
    want = cams[:, 0]
    for t in range(1, cams.shape[1]):
        want = torch.maximum(want, cams[:, t])          # the chain in wsol_loader.py:591-600
    assert got.shape == want.shape
    assert torch.equal(torch.nan_to_num(got, nan=-7.0), torch.nan_to_num(want, nan=-7.0))
    assert torch.equal(torch.isnan(got), torch.isnan(want))


@pytest.mark.parametrize("case", ["k21_voc", "wide_clip_colour", "tall_512", "k1", "k33"])
def test_unusual_shapes(torch_cuda, oracle_mod, case):
    """Shapes away from the benchmark: 21 classes (run-time columns-per-row in the blur), a width-concatenated clip
    through the colour lattice (RgbJointConRanFieldTcams' [H, T*W] layout), a 512 x 384 frame, one class, 33 classes
    (nine float4 columns)."""
    from tcam_wsol_video_b200 import _lib, ops
    torch = torch_cuda
    n, k, h, w, color = {"k21_voc": (2, 21, 60, 70, False), "wide_clip_colour": (2, 2, 56, 5 * 56, True),
                         "tall_512": (1, 2, 512, 384, False), "k1": (3, 1, 33, 47, False),
                         "k33": (1, 33, 24, 31, False)}[case]
    img = synth.make_images(n, h, w, "natural" if case != "k33" else "noise", seed=len(case))
    seg = synth.make_segs(n, k, h, w, seed=len(case))
    if color:
        cfg = _lib.make_config(_lib.FEAT_COLOR, 3, 15.0)
        want = oracle_mod.port_colorbilateralfilter_batch(img, seg, n, k, h, w, 15.0, 3)
    else:
        cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
        want = oracle_mod.port_bilateralfilter_batch(img, seg, n, k, h, w, 15.0, 100.0)
    got, _, _ = ops.crf_forward(torch.from_numpy(img), torch.from_numpy(seg).cuda(), cfg, want_loss=False, check=True)
    _assert_close(got.cpu().numpy(), want.reshape(seg.shape), case)


# ---------------------------------------------------------------------------
# BASELINE configs at FULL size against the oracle (VERDICT r1, item 1)
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("kind", ["noise", "natural"])
def test_full_size_config2_vs_reference(torch_cuda, oracle_mod, kind):
    """BASELINE configs[1] as benchmarked -- 32 frames x 10 classes x 224^2 -- against the reference's own C++
    (oracle/_ref, bilateralfilter.cpp:42-55, when it travelled to this box; else the C restatement): AS, loss
    (dense_crf_loss.py:63-64) and gradient (:73) within rel 1e-4.  Three calls on one workspace: from the second
    on the density hint is in, so noise frames take the row-cooperative splat."""
    torch = torch_cuda
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    n, k, h, w = 32, 10, 224, 224
    img = synth.make_images(n, h, w, kind, seed=0)
    seg_np = synth.make_segs(n, k, h, w, seed=0)
    fn, _ = oracle_mod.best_filter(color=False)
    want_loss, want_grad, want_as = oracle_mod.densecrf_loss_fwd_bwd(img, seg_np, 15.0, 100.0, 1.0, fn)
    images = torch.from_numpy(img).cuda()
    mod = DenseCRFLoss(weight=1.0, sigma_rgb=15.0, sigma_xy=100.0, scale_factor=1.0)
    from tcam_wsol_video_b200 import ops
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    for call in range(3):
        seg = torch.from_numpy(seg_np).cuda().requires_grad_(True)
        loss = mod(images=images, segmentations=seg)
        loss.backward()
        torch.cuda.synchronize()
        assert abs(loss.item() - float(want_loss)) < REL_TOL * abs(float(want_loss)), f"loss, call {call}"
        _assert_close(seg.grad.cpu().numpy(), want_grad, f"grad, call {call} ({kind})")
        got_as, _, _ = ops.crf_forward(images, seg.detach(), cfg, want_loss=False, check=True)
        _assert_close(got_as.cpu().numpy(), want_as, f"AS, call {call} ({kind})")


@pytest.mark.parametrize("kind", ["noise", "natural"])
@pytest.mark.parametrize("channels,hw", [(1, (64, 64)), (1, (448, 448)), (2, (64, 64)), (2, (448, 448)),
                                         (4, (64, 64)), (1, (37, 53))])
@pytest.mark.parametrize("build", ["0", "1"], ids=["build_kernel", "build_dedup_kernel"])
def test_xy_lattices_of_other_dimensions(torch_cuda, oracle_mod, tuning, kind, channels, hw, build):
    """BASELINE configs[3]'s "grayscale 3-D bilateralfilter" (features x, y, gray: TCAMCRF_FEAT_XY_RGB with one
    image plane) and the 4-D / 6-D siblings, at 64^2 and 448^2, against Permutohedral::init / compute
    (permutohedral.cpp:115-297, 507-572) on explicit features built with initializePermutohedral's arithmetic
    (bilateralfilter.cpp:4-19).  Both build kernels."""
    torch = torch_cuda
    tuning("BUILD_DEDUP", build)
    from tcam_wsol_video_b200 import ops
    h, w = hw
    n, k = 2, 2
    rgb = synth.make_images(n, h, w, kind, seed=13 + channels)
    planes = rgb if channels <= 3 else np.concatenate([rgb, rgb[:, ::-1][:, :1] * 0.5 + 3.0], axis=1)
    planes = np.ascontiguousarray(planes[:, :channels])
    seg = synth.make_segs(n, k, h, w, seed=17)
    want = np.stack([oracle_mod.port_filter_features(oracle_mod.xy_features(h, w, 100.0, planes[i], 15.0), seg[i])
                     for i in range(n)]).reshape(seg.shape)
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, channels, 15.0, 100.0)
    got, _, _ = ops.crf_forward(torch.from_numpy(planes).cuda(), torch.from_numpy(seg).cuda(), cfg,
                                want_loss=False, check=True)
    _assert_close(got.cpu().numpy(), want, f"xy + {channels} planes, {h}x{w}, {kind}")


@pytest.mark.parametrize("build", ["0", "1"], ids=["build_kernel", "build_dedup_kernel"])
@pytest.mark.parametrize("dim", [4, 6])
def test_colour_lattices_of_other_dimensions(torch_cuda, oracle_mod, tuning, dim, build):
    """colorbilateralfilter with DIM = 4 and 6 image planes (one image: the batch function's 3-plane stride makes
    N > 1 read overlapping windows, colorbilateralfilter.cpp:50)."""
    tuning("BUILD_DEDUP", build)
    k, h, w = 2, 40, 44
    rng = np.random.default_rng(dim)
    img = rng.integers(0, 256, size=(1, dim, h, w)).astype(np.float32)
    seg = synth.make_segs(1, k, h, w, seed=dim)
    want = oracle_mod.port_colorbilateralfilter_batch(img, seg, 1, k, h, w, 15.0, dim).reshape(seg.shape)
    got = _gpu_filter_host(img, seg, 15.0, 0.0, dim=dim)
    _assert_close(got, want, f"colour lattice, DIM={dim}")


@pytest.mark.parametrize("dim,n", [(4, 3), (6, 2), (5, 9), (2, 4), (1, 2)])
def test_colour_batch_keeps_the_reference_three_plane_stride(torch_cuda, oracle_mod, dim, n):
    """colorbilateralfilter_batch strides the image buffer by THREE planes whatever DIM is (colorbilateralfilter.cpp:50):
    with DIM > 3 consecutive frames read overlapping windows [3n, 3n + DIM) of it, with DIM < 3 they skip planes.
    Same here, through the drop-in host API, against the reference's own loop (oracle)."""
    k, h, w = 2, 30, 34
    rng = np.random.default_rng(dim * 10 + n)
    planes = (n - 1) * 3 + max(dim, 3)
    img = rng.integers(0, 256, size=(planes, h, w)).astype(np.float32)
    seg = synth.make_segs(n, k, h, w, seed=dim)
    want = oracle_mod.port_colorbilateralfilter_batch(img, seg, n, k, h, w, 15.0, dim).reshape(seg.shape)
    got = _gpu_filter_host(img, seg, 15.0, 0.0, dim=dim)
    _assert_close(got, want, f"colour batch, DIM={dim}, N={n}")


def test_soak_alternating_inputs_on_one_workspace(torch_cuda, oracle_mod):
    """150 calls back to back on one workspace with the input regime changing under the library's feet: noise and
    natural frames (the density hint flips the build / splat variants two calls late), class counts 1..12, a tiny
    primary table tier every now and then (overflow tier in use, then clean again).  Every call must report status 0
    and a finite loss; every 10th is compared with the oracle."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    rng = np.random.default_rng(2024)
    n, h, w = 4, 40, 56
    checked = 0
    for call in range(150):
        kind = "noise" if (call // 7) % 2 == 0 else "natural"
        k = int(rng.integers(1, 13))
        load = 64.0 if call % 23 == 5 else 0.0
        img = synth.make_images(n, h, w, kind, seed=1000 + call)
        seg_np = synth.make_segs(n, k, h, w, seed=1000 + call)
        cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0, hash_load=load)
        got, loss, ws = ops.crf_forward(torch.from_numpy(img).cuda(), torch.from_numpy(seg_np).cuda(), cfg, check=True)
        assert torch.isfinite(loss).all(), call
        if call % 10 == 0:
            want = oracle_mod.port_bilateralfilter_batch(img, seg_np, n, k, h, w, 15.0, 100.0).reshape(seg_np.shape)
            _assert_close(got.cpu().numpy(), want, f"call {call} ({kind}, K={k}, load {load})")
            checked += 1
    assert checked == 15
