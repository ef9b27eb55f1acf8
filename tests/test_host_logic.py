"""CPU suite, part 2: host logic and the drop-in boundary (no GPU, no compute calls).

* the product's device header (lattice.cuh), compiled for the host, embeds pixels and steps to
  neighbours exactly like the oracle (keys, barycentric weights bit for bit);
* libtcamcrf.so loads here and exports every symbol include/tcamcrf.h declares;
* argument validation of the C ABI and of the python drop-in modules.
"""
import ctypes
import os
import re

import numpy as np
import pytest

from conftest import ROOT
from tcam_wsol_video_b200 import _lib, synth


def _features(img, h, w, srgb, sxy, color_dim=0):
    p = h * w
    if color_dim:
        return np.ascontiguousarray((img.reshape(img.shape[0], -1)[:color_dim].T / np.float32(srgb)).astype(np.float32))
    f = np.zeros((p, 5), np.float32)
    rows, cols = np.divmod(np.arange(p), w)
    f[:, 0] = cols.astype(np.float32) / np.float32(sxy)
    f[:, 1] = rows.astype(np.float32) / np.float32(sxy)
    for c in range(3):
        f[:, 2 + c] = img[c].reshape(-1) / np.float32(srgb)
    return f


def _embed(harness, feats, d, scale):
    n = feats.shape[0]
    coords = np.zeros((n, d + 1, d), np.int16)
    bary = np.zeros((n, d + 1), np.float32)
    packed = np.zeros((n, d + 1), np.uint64)
    fp = ctypes.POINTER(ctypes.c_float)
    bad = harness.harness_embed(d, feats.ctypes.data_as(fp), n, scale.ctypes.data_as(fp),
                                coords.ctypes.data_as(ctypes.c_void_p), bary.ctypes.data_as(fp),
                                packed.ctypes.data_as(ctypes.c_void_p))
    return bad, coords, bary, packed


@pytest.mark.parametrize("kind", ["noise", "natural"])
@pytest.mark.parametrize("d,sig", [(5, (15.0, 100.0)), (5, (3.0, 8.0)), (3, (15.0, 0.0)), (1, (15.0, 0.0))])
def test_device_embedding_matches_oracle(harness, oracle_mod, kind, d, sig):
    h, w = 36, 44
    srgb, sxy = sig
    img = synth.make_images(1, h, w, kind, seed=11)[0]
    if d == 5:
        feats = _features(img, h, w, srgb, sxy)
        L = oracle_mod.port_lattice_bilateral(img, h, w, srgb, sxy)
    else:
        feats = _features(img, h, w, srgb, sxy, color_dim=d)
        L = oracle_mod.port_lattice_color(img, h, w, srgb, d)
    scale = oracle_mod.port_scale_factors(d)
    bad, coords, bary, packed = _embed(harness, feats, d, scale)
    assert bad == 0
    n = h * w
    assert np.array_equal(L.keys[L.offset[:n]], coords)      # same lattice vertices, coordinate by coordinate
    assert np.array_equal(L.bary[:n], bary)                    # bit-exact barycentric weights
    uniq, first = np.unique(packed.reshape(-1), return_index=True)
    assert len(uniq) == L.m                                    # packing is injective on the vertices
    # neighbour stepping on packed keys == +-1 / -+d on the coordinates (permutohedral.cpp:285-290)
    kc = coords.reshape(-1, d)[first]
    m = len(uniq)
    n1 = np.zeros((d + 1, m, d), np.int16)
    n2 = np.zeros_like(n1)
    assert harness.harness_neighbours(d, uniq.ctypes.data_as(ctypes.c_void_p), m,
                                      n1.ctypes.data_as(ctypes.c_void_p), n2.ctypes.data_as(ctypes.c_void_p)) == 0
    for j in range(d + 1):
        e1, e2 = kc - 1, kc + 1
        if j < d:
            e1[:, j] = kc[:, j] + d
            e2[:, j] = kc[:, j] - d
        assert np.array_equal(e1, n1[j]) and np.array_equal(e2, n2[j])


def test_key_range_is_reported(harness, oracle_mod):
    """Features far outside the packed-key range must be flagged, never wrapped silently."""
    d = 5
    bits = harness.harness_field_bits(d)
    assert bits == 12
    scale = oracle_mod.port_scale_factors(d)
    feats = np.zeros((2, d), np.float32)
    feats[1, 4] = 1e6
    bad, _, _, _ = _embed(harness, feats, d, scale)
    assert bad == 1
    for dd, expect in ((1, 20), (2, 20), (3, 20), (4, 15), (6, 10)):
        assert harness.harness_field_bits(dd) == expect


def test_library_exports_every_declared_symbol():
    lib = _lib.load()
    header = open(os.path.join(ROOT, "include", "tcamcrf.h")).read()
    header = re.sub(r"/\*.*?\*/", "", header, flags=re.S)
    declared = set(re.findall(r"\b(\w+)\s*\([^;{]*\)\s*;", header))
    declared = {d for d in declared if not d.isupper()}
    assert declared, "no prototypes parsed"
    assert declared == set(_lib.SIGNATURES), declared ^ set(_lib.SIGNATURES)
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/tcamcrf.h but not exported"
    assert lib.tcamcrf_version() == 104


def test_workspace_sizing_and_argument_validation():
    lib = _lib.load()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    small = lib.tcamcrf_workspace_bytes(ctypes.byref(cfg), 1, 2, 224, 224)
    big = lib.tcamcrf_workspace_bytes(ctypes.byref(cfg), 32, 2, 224, 224)
    assert 0 < small < big
    # chunking bounds the workspace: 256 frames need no more than the default chunk of 64
    assert lib.tcamcrf_workspace_bytes(ctypes.byref(cfg), 256, 2, 224, 224) == \
        lib.tcamcrf_workspace_bytes(ctypes.byref(cfg), 64, 2, 224, 224)
    assert lib.tcamcrf_workspace_bytes(ctypes.byref(cfg), 0, 2, 224, 224) == 0
    assert b"positive" in lib.tcamcrf_last_error()
    bad = _lib.make_config(_lib.FEAT_XY_RGB, 5, 15.0, 100.0)   # d = 7 > 6
    assert lib.tcamcrf_workspace_bytes(ctypes.byref(bad), 1, 2, 8, 8) == 0
    assert b"dimension" in lib.tcamcrf_last_error()
    bad = _lib.make_config(_lib.FEAT_COLOR, 3, 0.0)
    assert lib.tcamcrf_workspace_bytes(ctypes.byref(bad), 1, 2, 8, 8) == 0
    # null pointers are rejected before anything touches the device
    assert lib.tcamcrf_filter(ctypes.byref(cfg), None, None, None, 1, 2, 8, 8, None, 0, None) == 1
    assert lib.tcamcrf_loss_backward(None, None, None, 16, 1.0, None) == 1
    assert lib.tcam_temporal_max(None, None, 1, 1, 1, None) == 1
    assert lib.tcam_temporal_max_renorm(None, None, 1, 1, 1, 10.0, None) == 1
    assert lib.tcam_prepare_std_cams(None, None, 1, 28, 28, 224, 224, None) == 1
    # lattice re-use API: one lattice holds at most chunk_frames (64) frames; pointers and workspace are checked
    assert lib.tcamcrf_lattice_build(ctypes.byref(cfg), None, 0, 1, 2, 8, 8, None, 0, None) == 1
    assert lib.tcamcrf_lattice_apply(ctypes.byref(cfg), None, None, None, 1, 2, 8, 8, 1.0, 0, None, 0, None) == 1
    fake = ctypes.c_void_p(256)   # never dereferenced: the frame-count check comes first
    assert lib.tcamcrf_lattice_build(ctypes.byref(cfg), fake, 0, 65, 2, 8, 8, fake, 1 << 40, None) == 1
    assert b"at most" in lib.tcamcrf_last_error()
    assert lib.tcamcrf_lattice_build(ctypes.byref(cfg), fake, 0, 2, 2, 8, 8, fake, 16, None) == 2   # workspace too small


def test_chunk_shrinks_for_large_frames():
    """Frames per pass: 64 by default, capped by N; large frames get a smaller chunk instead of an error (32-bit
    vertex / entry indices, ~16 GiB default workspace) -- the reference takes any image size."""
    lib = _lib.load()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    chunk = lambda c, n, k, h, w: lib.tcamcrf_chunk_frames(ctypes.byref(c), n, k, h, w)
    assert chunk(cfg, 32, 10, 224, 224) == 32
    assert chunk(cfg, 256, 2, 224, 224) == 64
    assert chunk(cfg, 256, 2, 448, 448) == 64
    big = chunk(cfg, 64, 2, 1024, 1024)
    assert 1 <= big < 64
    assert lib.tcamcrf_workspace_bytes(ctypes.byref(cfg), 64, 2, 1024, 1024) <= 17 * 2 ** 30
    assert chunk(cfg, 4, 2, 4096, 4096) == 1
    # an explicit chunk is only lowered when the 32-bit indices need it
    explicit = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0, chunk_frames=64)
    assert chunk(explicit, 64, 2, 1024, 1024) > big
    assert chunk(explicit, 64, 2, 4096, 4096) == 3
    assert lib.tcamcrf_workspace_bytes(ctypes.byref(explicit), 64, 2, 4096, 4096) > 0
    # beyond any chunk size
    assert chunk(cfg, 1, 2, 8192, 8192) == 0 and "too large" in _lib.last_error()
    assert chunk(cfg, 0, 2, 8, 8) == 0
    from tcam_wsol_video_b200 import ops
    assert ops.lattice_capacity(cfg, 2, 224, 224) == 64
    assert ops.lattice_capacity(cfg, 2, 1024, 1024) == big


def test_dropin_modules_validate_like_the_swig_typemaps():
    from tcam_wsol_video_b200 import bilateralfilter as bf
    from tcam_wsol_video_b200 import colorbilateralfilter as cbf
    img = np.zeros(3 * 4 * 4, np.float32)
    seg = np.zeros(2 * 4 * 4, np.float32)
    out = np.zeros_like(seg)
    with pytest.raises(TypeError):
        bf.bilateralfilter_batch(img.astype(np.float64), seg, out, 1, 2, 4, 4, 15.0, 100.0)
    with pytest.raises(TypeError):
        bf.bilateralfilter_batch(img.reshape(3, 16), seg, out, 1, 2, 4, 4, 15.0, 100.0)
    with pytest.raises(TypeError):
        cbf.colorbilateralfilter_batch(img, seg[::2], out, 1, 1, 4, 4, 15.0, 3)
    with pytest.raises(ValueError):
        bf.bilateralfilter_batch(img, seg, out, 2, 2, 4, 4, 15.0, 100.0)


def test_no_cpu_fallback_without_gpu():
    """On a box without a B200 every compute entry point must fail loudly."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    from tcam_wsol_video_b200 import bilateralfilter as bf
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
    img = np.zeros(3 * 4 * 4, np.float32)
    seg = np.zeros(2 * 4 * 4, np.float32)
    out = np.zeros_like(seg)
    with pytest.raises(_lib.TcamCrfError):
        bf.bilateralfilter_batch(img, seg, out, 1, 2, 4, 4, 15.0, 100.0)
    loss = DenseCRFLoss(weight=1e-7, sigma_rgb=15.0, sigma_xy=100.0, scale_factor=1.0)
    with pytest.raises(_lib.TcamCrfError):
        loss(images=torch.zeros(1, 3, 4, 4), segmentations=torch.zeros(1, 2, 4, 4))
    assert "sigma_rgb=15.0, sigma_xy=100.0, weight=1e-07, scale_factor=1.0" == loss.extra_repr()
    # the mean-field filter and the reusable lattice refuse a CPU-only box too; itera=0 is pure torch
    from tcam_wsol_video_b200 import ops
    from tcam_wsol_video_b200.crf_post_processing import DenseCRFFilter
    segs = torch.softmax(torch.randn(1, 2, 4, 4), dim=1)
    with pytest.raises(_lib.TcamCrfError):
        DenseCRFFilter(15, 100, 1.0, 2)(torch.zeros(1, 3, 4, 4), segs)
    assert torch.equal(DenseCRFFilter(15, 100, 1.0, 0)(torch.zeros(1, 3, 4, 4), segs), segs)
    with pytest.raises(_lib.TcamCrfError):
        ops.Lattice(torch.zeros(1, 3, 4, 4), _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0), 2)


def test_mean_field_oracle_restatement(oracle_mod):
    """oracle/crf_post_processing.py on its own: probabilities stay normalised, zero iterations = softmax(-U) = seg,
    and the image pydensecrf sees is the mirrored one for square frames (crf_post_processing.py:116-118)."""
    from oracle import crf_post_processing as ocp
    from tcam_wsol_video_b200 import synth
    rng = np.random.default_rng(0)
    img = synth.make_images(1, 12, 12, "natural", seed=1)[0]
    seen = ocp.quirk_image(img)
    assert np.array_equal(seen, img.astype(np.uint8).transpose(0, 2, 1))
    logits = rng.standard_normal((3, 12, 12)).astype(np.float32)
    seg = np.exp(logits) / np.exp(logits).sum(0, keepdims=True)
    q0 = ocp.mean_field(img, seg, 15, 100, 0, oracle_mod.port_bilateralfilter_batch)
    assert np.abs(q0 - seg).max() < 1e-6
    q2 = ocp.mean_field(img, seg, 15, 100, 2, oracle_mod.port_bilateralfilter_batch)
    assert np.abs(q2.sum(0) - 1).max() < 1e-5 and np.abs(q2 - seg).max() > 1e-3


def test_product_never_imports_the_oracle():
    pkg = os.path.join(ROOT, "tcam_wsol_video_b200")
    for dirpath, _, files in os.walk(pkg):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h", ".cpp")):
                text = open(os.path.join(dirpath, f)).read()
                assert "import oracle" not in text and "from oracle" not in text, f
                assert "liboracle" not in text and "_ref/" not in text, f


def test_temporal_frame_pickers():
    """left / right k-nearest frames of a shot, and the neighbourhood by mode (wsol_loader.py:448-459, 544-557)."""
    from tcam_wsol_video_b200 import temporal as tp
    frames = [f"f{i}" for i in range(6)]
    assert tp.get_left_knn(frames, "f3", 2) == ["f1", "f2"]
    assert tp.get_left_knn(frames, "f1", 4) == ["f0"]
    assert tp.get_left_knn(frames, "f0", 4) == []
    assert tp.get_right_knn(frames, "f3", 2) == ["f4", "f5"]
    assert tp.get_right_knn(frames, "f4", 4) == ["f5"]
    # reference quirk: for the last frame of a shot the slice is lframes[n-1:n] = the frame itself
    assert tp.get_right_knn(frames, "f5", 4) == ["f5"]
    assert tp.temporal_frames(frames, "f5", 2, tp.TIME_BEFORE_AFTER) == ["f3", "f4", "f5", "f5"]
    assert tp.temporal_frames(frames, "f2", 4, tp.TIME_BEFORE) == ["f0", "f1", "f2"]
    assert tp.temporal_frames(frames, "f2", 1, tp.TIME_BEFORE_AFTER) == ["f1", "f2", "f3"]
    assert tp.temporal_frames(frames, "f2", 1, tp.TIME_AFTER) == ["f2", "f3"]
    assert tp.temporal_frames(frames, "f2", 3, tp.TIME_INSTANT) == ["f2"]


def test_key_range_is_refused_on_the_host():
    """A sigma too small for the lattice dimension (or more than 6 feature dimensions) is refused up front with a
    clear message instead of coming back as a NaN loss (ADVICE r1); pure host arithmetic, no device needed."""
    ok = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    _lib.require_key_range(ok, 224, 224)
    _lib.require_key_range(_lib.make_config(_lib.FEAT_COLOR, 6, 1.0), 224, 224)
    for bad in (_lib.make_config(_lib.FEAT_XY_RGB, 3, 0.05, 100.0),      # 12-bit fields of the 5-D lattice
                _lib.make_config(_lib.FEAT_COLOR, 6, 0.5),               # 10-bit fields at d = 6
                _lib.make_config(_lib.FEAT_COLOR, 7, 15.0),              # d > 6 does not fit one 64-bit key
                _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 1e-4)):      # position term out of range
        with pytest.raises(_lib.TcamCrfError, match="out of range"):
            _lib.require_key_range(bad, 224, 224)


def test_tuning_knobs_are_set_at_run_time():
    """The TCAMCRF_* environment variables are read once; tests and sweeps change knobs through the C ABI.  Knobs
    whose experiments are decided (CHUNK, HOST_TAPER, HOST_GRAPH) are gone and are refused like any unknown name."""
    for name in ("DENSE", "BUILD_DEDUP", "HIMG_SECTIONS", "HOST_GROUPS", "HOST_SECTION0", "HOST_GROW", "HOST_TRACE"):
        _lib.set_tuning(name, 1)
        _lib.set_tuning(name, -1)
        _lib.set_tuning("TCAMCRF_" + name, 1)
        _lib.set_tuning("TCAMCRF_" + name, -1)
    for name in ("NO_SUCH_KNOB", "CHUNK", "HOST_TAPER", "HOST_GRAPH"):
        with pytest.raises(_lib.TcamCrfError, match="unknown tuning knob"):
            _lib.set_tuning(name, 1)


def test_release_workspaces_clears_every_cached_buffer():
    """Both caches keyed by (device, stream, ...) are dropped: a trainer that changes streams or batch sizes can
    release what it no longer uses."""
    from tcam_wsol_video_b200 import ops
    ops._workspaces[(0, 1)] = object()
    ops._seed_ce_scratch[(0, 1, 4)] = object()
    ops.release_workspaces()
    assert not ops._workspaces and not ops._seed_ce_scratch


def test_weight_is_folded_only_when_it_is_a_plain_number():
    import torch
    from tcam_wsol_video_b200.dense_crf_loss import _folded_weight
    assert _folded_weight(2e-9) == 2e-9 and _folded_weight(3) == 3.0
    assert _folded_weight(torch.tensor(2e-9)) is None and _folded_weight(0.0) is None
    assert _folded_weight(True) is None and _folded_weight(float("nan")) is None
