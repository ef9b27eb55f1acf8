"""GPU suite (-m gpu): fp16 and bf16 logits read natively by the logits paths (the *_lowp kernels of csrc/tcamcrf.cu
and csrc/seed.cuh, the *_typed entry points, ops and the loss modules).

Widening a 2-byte logit to float32 is exact and the kernels compute in float32 exactly as the float32 kernels do, so
the oracle is the float32 path itself: given the same AS, every gradient must have the bits of the float32 gradient
on the widened logits cast to the logits' dtype (NaN matching NaN), and the seed cross-entropy's loss and count must
equal the float32 kernels' exactly.  The forward (AS, loss) has splat atomics, so it is held to the bar of
tests/test_gpu_kernel_matrix.py instead: the float64 matrix form of the filter on softmax64 of the widened logits,
within 2x the float32 oracle's own error + 1e-7.  Every case runs for fp16 and for bf16; kernel tracing proves which
instantiation ran, and the last test fails on any compiled *_lowp instantiation that no case launched.
"""
import re
import shutil
import subprocess

import numpy as np
import pytest

from conftest import rel_err
from oracle import lattice_matrix as lm
from tcam_wsol_video_b200 import _lib, synth
from test_gpu_kernel_matrix import Reference, assert_bar, assert_loss, config, errs, make_planes, softmax32
from test_gpu_seed_ce import _hand_sel, _seeder_sel

pytestmark = pytest.mark.gpu

DTYPES = ["float16", "bfloat16"]
IGNORE = -255
UNIT_ROUNDOFF = {"float16": 2.0 ** -11, "bfloat16": 2.0 ** -8}

_launched = set()      # every *_lowp kernel the profiler saw in this module
_forward_cases_run = set()


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available(), "GPU suite needs a B200"
    assert _lib.load().tcamcrf_device_count() >= 1
    return torch


@pytest.fixture
def tuning():
    """Sets library tuning knobs for one test and restores the defaults afterwards."""
    touched = []

    def set_(name, value):
        touched.append(name)
        _lib.set_tuning(name, -1 if value is None else int(value))

    yield set_
    for name in touched:
        _lib.set_tuning(name, -1)


# ---------------------------------------------------------------------------
# kernel names
# ---------------------------------------------------------------------------
def _normalise(name):
    """Profiler name -> 'splat_lowp_kernel<5, 2>' / 'seed_ce_forward_lowp_kernel'; None for other kernels."""
    m = re.search(r"tcamcrf::(\w+_lowp_kernel)(?:<([^>]*)>)?", name)
    if not m:
        return None
    if m.group(2) is None:
        return m.group(1)
    return f"{m.group(1)}<{', '.join(a.strip() for a in m.group(2).split(','))}>"


def _demangle(mangled):
    """_ZN7tcamcrf22splat_rows_lowp_kernelILi4ELi3EEEvNS_11PixelParamsE -> splat_rows_lowp_kernel<4, 3>."""
    m = re.match(r"_ZN7tcamcrf(\d+)", mangled)
    if not m:
        return None
    name = mangled[m.end():m.end() + int(m.group(1))]
    if not name.endswith("_lowp_kernel"):
        return None
    rest = mangled[m.end() + int(m.group(1)):]
    if not rest.startswith("I"):
        return name
    args = re.match(r"I((?:Li\d+E)+)E", rest)
    assert args, f"cannot read the template arguments of {mangled}"
    return f"{name}<{', '.join(re.findall(r'Li(\d+)E', args.group(1)))}>"


def compiled_lowp_kernels():
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    text = subprocess.run([tool, "-sass", _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = {_demangle(n) for n in re.findall(r"Function : (\S+)", text)}
    names.discard(None)
    return names


class Traced:
    """torch.profiler with CUDA activities around library calls; records the *_lowp kernels that ran."""

    def __init__(self, torch):
        self.torch = torch
        self.kernels = set()

    def __enter__(self):
        from torch.profiler import ProfilerActivity, profile
        self.prof = profile(activities=[ProfilerActivity.CUDA])
        self.prof.__enter__()
        return self

    def __exit__(self, *exc):
        self.torch.cuda.synchronize()
        self.prof.__exit__(*exc)
        if exc[0] is None:
            names = {e.name for e in self.prof.events()}
            assert names, "torch.profiler recorded no CUDA kernel: kernel tracing is unavailable"
            self.kernels = {n for n in map(_normalise, names) if n}
            _launched.update(self.kernels)
        return False


# ---------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------
def tdtype(torch, name):
    return getattr(torch, name)


def same_bits(torch, got, want):
    """Identical bits, NaN matching NaN (the NaN payload of a cast is not specified)."""
    assert got.dtype == want.dtype and got.shape == want.shape
    nan_g, nan_w = torch.isnan(got), torch.isnan(want)
    if not torch.equal(nan_g, nan_w):
        return False
    bits = torch.int16 if got.element_size() == 2 else torch.int32
    return torch.equal(got.view(bits)[~nan_g], want.view(bits)[~nan_w])


def assert_same_bits(torch, got, want, what):
    if same_bits(torch, got, want):
        return
    diff = (got.view(torch.int16) != want.view(torch.int16)) & ~(torch.isnan(got) & torch.isnan(want))
    idx = diff.nonzero()[:4].tolist()
    pairs = [(got[tuple(i)].item(), want[tuple(i)].item()) for i in idx]
    raise AssertionError(f"{what}: {int(diff.sum())} elements differ, e.g. {pairs}")


def make_logits(torch, dtype, mode, n, k, h, w, seed):
    """[n,k,h,w] CUDA logits in `dtype`: confident (+-6e4 in fp16, +-1e30 in bf16), tied, subnormal, -inf (some
    pixels entirely -inf: NaN probabilities), or 3 * randn."""
    rng = np.random.default_rng(seed)
    z = 3.0 * rng.standard_normal((n, k, h, w))
    big = 6e4 if dtype == "float16" else 1e30
    tiny = 2.0 ** -20 if dtype == "float16" else 1e-39
    if mode == "confident":
        z = np.where(rng.random(z.shape) < 0.5, big, -big) + z
    elif mode == "tied":
        z[:] = z[:, :1]
    elif mode == "subnormal":
        z = z * tiny
    elif mode == "neginf":
        z[:, k - 1][rng.random((n, h, w)) < 0.5] = -np.inf
        z[:, :, 0, :3] = -np.inf                       # every class: 0 / 0 in the softmax
    t = torch.from_numpy(z).to(tdtype(torch, dtype))
    assert not mode == "subnormal" or bool(((t != 0) & (t.abs() < torch.finfo(t.dtype).tiny)).any())
    return t.cuda()


# ---------------------------------------------------------------------------
# 1. the logits backward, bit for bit given AS
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("mode", ["randn", "confident", "tied", "subnormal", "neginf"])
@pytest.mark.parametrize("k", [2, 3, 7])
@pytest.mark.parametrize("dtype", DTYPES)
def test_backward_bit_exact(torch_cuda, dtype, k, mode):
    """tcamcrf_loss_backward_logits_typed on 2-byte logits = the float32 backward on the widened logits, then a cast;
    K = 2 takes the Prob2 register path.  g = 65536 (a GradScaler-sized scale) overflows some elements to +-inf."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    n, h, w = 2, 19, 37
    z = make_logits(torch, dtype, mode, n, k, h, w, seed=k)
    zw = z.float()
    AS = torch.from_numpy(40.0 * np.random.default_rng(k + 1).standard_normal((n, k, h, w)).astype(np.float32)).cuda()
    for g in (1.0, 65536.0):
        for weight in (1.0, 0.37):
            gt = torch.tensor([g], device="cuda")
            with Traced(torch) as tr:
                got = ops.crf_backward_logits(AS, z, gt, float(n), weight)
            assert tr.kernels == {"loss_backward_logits_lowp_kernel"}, tr.kernels
            assert got.dtype == z.dtype
            want = ops.crf_backward_logits(AS, zw, gt, float(n), weight).to(z.dtype)
            assert_same_bits(torch, got, want, f"g={g}, weight={weight}")
            if g == 65536.0 and mode == "randn":
                assert bool(torch.isinf(got).any()) or dtype == "bfloat16"


# ---------------------------------------------------------------------------
# 2. the seed cross-entropy, bit for bit
# ---------------------------------------------------------------------------
# (id, B, K, H, W, ksz, kmax, placement)
SEED_CASES = [
    ("corners", 5, 2, 37, 53, 4, 3, "corners"),
    ("overlap", 1, 4, 37, 53, 5, 40, "overlap"),
    ("conflict", 5, 3, 37, 53, 3, 3, "conflict"),
    ("empty-sample", 5, 2, 37, 53, 3, 32, "empty_sample"),
    ("seeder-fused", 5, 2, 64, 64, 3, 3, "seeder"),
    ("seeder-two-kernel", 5, 3, 37, 53, 2, 40, "seeder"),
]


@pytest.mark.parametrize("logits_mode", ["randn", "confident"])
@pytest.mark.parametrize("case", SEED_CASES, ids=[c[0] for c in SEED_CASES])
@pytest.mark.parametrize("dtype", DTYPES)
def test_seed_ce_bit_exact(torch_cuda, dtype, case, logits_mode):
    """Forward loss and count equal the float32 kernels' on the widened logits; the unfused backward
    (SeedCrossEntropyFunction) and the fused CRF + CE backward (same AS) equal the float32 sequence cast once."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    from tcam_wsol_video_b200.dense_crf_loss import SeedCrossEntropyFunction
    from tcam_wsol_video_b200.tcam_seeding import SparseSeeds
    name, b, k, h, w, ksz, kmax, placement = case
    seed = sum(map(ord, name))
    if placement == "seeder":
        seeds = _seeder_sel(torch, b, h, w, ksz, kmax, seed)
    else:
        seeds = SparseSeeds(torch.from_numpy(_hand_sel(placement, b, h, w, ksz, kmax, seed)).cuda(), ksz, IGNORE, h, w)
    z = make_logits(torch, dtype, logits_mode, b, k, h, w, seed)
    zw = z.float()
    sel = seeds.sel

    with Traced(torch) as tr:
        loss, count, _ = ops.seed_ce_forward(z, sel, ksz)
    assert "seed_ce_forward_lowp_kernel" in tr.kernels
    loss32, count32, _ = ops.seed_ce_forward(zw, sel, ksz)
    assert count.item() == count32.item()
    assert same_bits(torch, loss, loss32), (loss.item(), loss32.item())

    # unfused: SeedCrossEntropyFunction starts from a zero gradient
    g = 0.625
    zz = z.clone().requires_grad_(True)
    with Traced(torch) as tr:
        SeedCrossEntropyFunction.apply(zz, sel, ksz).backward(torch.full((1,), g, device="cuda"))
    assert "seed_ce_backward_lowp_kernel" in tr.kernels
    z32 = zw.clone().requires_grad_(True)
    SeedCrossEntropyFunction.apply(z32, sel, ksz).backward(torch.full((1,), g, device="cuda"))
    assert zz.grad.dtype == z.dtype
    assert_same_bits(torch, zz.grad, z32.grad.to(z.dtype), "unfused backward")

    # fused: the CRF gradient, then the cross-entropy's added in place, rounded once -- given the same AS
    raw = torch.from_numpy(synth.make_images(b, h, w, "natural", seed=seed).astype(np.uint8)).cuda()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    as_t, _, _ = ops.crf_forward_logits(raw, zw, cfg)
    gt = torch.full((1,), 1.25, device="cuda")
    crf_w, ce_w = 3e-3, 0.75
    with Traced(torch) as tr:
        got = ops.crf_seed_ce_backward(as_t, z, sel, ksz, count, gt, float(b), crf_w, ce_w)
    assert {"loss_backward_logits_lowp_kernel", "seed_ce_backward_lowp_kernel"} <= tr.kernels
    want = ops.crf_backward_logits(as_t, zw, gt, float(b), crf_w)
    ops.seed_ce_backward_(want, zw, sel, ksz, count32, gt, ce_w)
    assert got.dtype == z.dtype
    assert_same_bits(torch, got, want.to(z.dtype), "fused backward")


# ---------------------------------------------------------------------------
# 3. the forward from 2-byte logits against the float64 matrix form of the filter
# ---------------------------------------------------------------------------
# one lattice per dimension 1..6 (xy + rgb is D = 5, colour rgb D = 3); (K, DENSE) covers splat / slice at V = 2
# (K = 2) and V = 4 (K = 3, 4), and the row splat at KV = 2 / 3 / 4 (K = 5..8 / 9..12 / 13..16, forced with DENSE)
FWD_LATTICES = [("colour", 1), ("colour", 2), ("colour", 3), ("xy", 2), ("xy", 3), ("colour", 6)]
FWD_VARIANTS = [(2, 0), (3, 0), (4, 1), (5, 1), (8, 1), (11, 1), (16, 1)]


def _fwd_cases():
    out = []
    for li, spec in enumerate(FWD_LATTICES):
        for vi, (k, dense) in enumerate(FWD_VARIANTS):
            i = li + vi
            out.append(dict(spec=spec, k=k, dense=dense, u8=i % 2 == 0, kind=("natural", "noise")[(i // 2) % 2],
                            host=(li + 2 * vi) % 3 == 0, chunk=2 if i % 3 == 1 else 0))
    return out


FWD_CASES = _fwd_cases()


def _fwd_id(c):
    s = c["spec"]
    return (f"{s[0]}{s[1]}-K{c['k']}-dense{c['dense']}-{'u8' if c['u8'] else 'f32'}-{c['kind']}"
            f"-{'host' if c['host'] else 'device'}{'-chunk2' if c['chunk'] else ''}")


def expected_lowp(c):
    d = c["spec"][1] + (2 if c["spec"][0] == "xy" else 0)
    k = c["k"]
    kp = k if k <= 2 else (k + 3) // 4 * 4
    v = 4 if kp % 4 == 0 else 2
    out = {f"slice_lowp_kernel<{d}, {v}>"}
    if c["dense"] and v == 4 and 2 <= kp // 4 <= 4:
        out.add(f"splat_rows_lowp_kernel<{d}, {kp // 4}>")
    else:
        out.add(f"splat_lowp_kernel<{d}, {v}>")
    return out


@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("c", FWD_CASES, ids=_fwd_id)
def test_forward_against_float64(torch_cuda, oracle_mod, tuning, c, dtype):
    """AS and the loss from 2-byte logits, through the device-frames and the pinned host-frames paths, against the
    float64 filter of softmax64(widened logits); then the backward on that AS, bit for bit."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    tuning("DENSE", c["dense"])
    n, k, (h, w) = 3, c["k"], (19, 37)
    seed = FWD_CASES.index(c) + 1
    planes = make_planes(n, h, w, c["kind"], seed)
    images = torch.from_numpy(planes.astype(np.uint8) if c["u8"] else planes)
    images = images.pin_memory() if c["host"] else images.cuda()
    z = make_logits(torch, dtype, "randn", n, k, h, w, seed)
    zw64 = z.double().cpu().numpy()
    ref = Reference(oracle_mod, c["spec"], planes)
    s64 = lm.softmax64(zw64)
    want = ref.apply(s64)
    bar = errs(ref.apply32(softmax32(zw64.astype(np.float32))), want)
    cfg = config(c["spec"], c["chunk"])
    with Traced(torch) as tr:
        as_t, loss_t, _ = ops.crf_forward_logits(images, z, cfg, check=True)
    assert expected_lowp(c) <= tr.kernels, f"launched {sorted(tr.kernels)}"
    assert as_t.dtype == torch.float32
    got = as_t.cpu().numpy()
    assert_bar(got, want, bar, "AS from 2-byte logits")
    assert_loss(loss_t.item(), lm.crf_loss64(s64, want, n), bar)
    g = torch.tensor([0.75], device="cuda")
    assert_same_bits(torch, ops.crf_backward_logits(as_t, z, g, float(n), 0.5),
                     ops.crf_backward_logits(as_t, z.float(), g, float(n), 0.5).to(z.dtype), "backward on this AS")
    _forward_cases_run.add((_fwd_id(c), dtype))


# ---------------------------------------------------------------------------
# 5. the loss modules under autocast
# ---------------------------------------------------------------------------
def _tcam_modules(fused):
    from tcam_wsol_video_b200.losses import ConRanFieldTcams, FusedTcamLosses, SelfLearningTcams
    sl = SelfLearningTcams(cuda_id=0, lambda_=0.75, seg_ignore_idx=IGNORE)
    crf = ConRanFieldTcams(cuda_id=0, lambda_=2e-3, sigma_rgb=15., sigma_xy=100., scale_factor=1.0,
                           fuse_softmax=True, seg_ignore_idx=IGNORE)
    if fused:
        f = FusedTcamLosses(sl, crf)
        return lambda fcams, raw, seeds: f(epoch=0, fcams=fcams, raw_img=raw, seeds=seeds)
    return lambda fcams, raw, seeds: sl(epoch=0, fcams=fcams, seeds=seeds) + crf(epoch=0, fcams=fcams, raw_img=raw)


def _step_inputs(torch, b, k, h, w, seed):
    raw = torch.from_numpy(synth.make_images(b, h, w, "natural", seed=seed).astype(np.uint8)).cuda()
    seeds = _seeder_sel(torch, b, h, w, 3, 3, seed)
    return raw, seeds


def _grad_tol(dtype, fused):
    """Normwise gradient tolerance against the float32 modules: the forward's 1e-5, plus one rounding to the logits'
    dtype for the fused node, three for two separate terms (each rounded, then their sum)."""
    return (1 if fused else 3) * UNIT_ROUNDOFF.get(dtype, 0.0) + 1e-5


def _copies_of(prof, numel):
    """aten::_to_copy / aten::copy_ calls on a tensor of `numel` elements."""
    out = []
    for e in prof.events():
        if e.name in ("aten::_to_copy", "aten::copy_"):
            for shape in e.input_shapes or []:
                if isinstance(shape, (list, tuple)) and shape and all(isinstance(s, int) for s in shape) \
                        and int(np.prod(shape)) == numel:
                    out.append((e.name, shape))
    return out


@pytest.mark.parametrize("fused", [True, False], ids=["FusedTcamLosses", "SelfLearning+ConRanField"])
@pytest.mark.parametrize("dtype", DTYPES)
def test_modules_under_autocast(torch_cuda, dtype, fused):
    """Inside torch.autocast: the gradient has the logits' dtype, loss and gradient agree with the same modules on
    fcams.float(), and nothing copies or casts a logits-sized tensor between the loss call and the end of backward."""
    torch = torch_cuda
    from torch.profiler import ProfilerActivity, profile
    b, k, h, w = 4, 2, 48, 56
    raw, seeds = _step_inputs(torch, b, k, h, w, seed=5)
    step = _tcam_modules(fused)
    z = make_logits(torch, dtype, "randn", b, k, h, w, seed=6)
    fcams = z.clone().requires_grad_(True)
    step(fcams.detach().clone().requires_grad_(True), raw, seeds).backward()     # warm-up: library, workspaces
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU], record_shapes=True) as prof:
        with torch.autocast("cuda", dtype=tdtype(torch, dtype)):
            loss = step(fcams, raw, seeds)
        loss.backward()
        torch.cuda.synchronize()
    assert fcams.grad.dtype == fcams.dtype
    assert not _copies_of(prof, z.numel()), _copies_of(prof, z.numel())
    f32 = z.float().requires_grad_(True)
    loss32 = step(f32, raw, seeds)
    loss32.backward()
    assert abs(loss.item() - loss32.item()) <= 1e-5 * abs(loss32.item())
    assert rel_err(fcams.grad.float().cpu().numpy(), f32.grad.cpu().numpy()) <= _grad_tol(dtype, fused)


# ---------------------------------------------------------------------------
# 6. the seeder + FusedTcamLosses step with fp16 logits in a CUDA graph
# ---------------------------------------------------------------------------
def test_fp16_step_in_a_cuda_graph(torch_cuda):
    """Captured once, replayed 3x on new inputs: the cross-entropy equals an eager call's bit for bit on the seeds the
    replay picked; the CRF term and the gradient agree with an eager step within the forward tolerance."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    from tcam_wsol_video_b200.losses import ConRanFieldTcams, FusedTcamLosses, SelfLearningTcams
    from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder
    b, t, k, h, w = 4, 3, 2, 64, 72
    seeder = TCAMSeeder(seed_tech="seed_weighted", min_=2, max_=2, max_p=0.6, min_p=0.1, fg_erode_k=11,
                        fg_erode_iter=0, ksz=3, support_background=True, multi_label_flag=False,
                        seg_ignore_idx=IGNORE, cuda_id=0, roi_method="roi_all", p_min_area_roi=0.05, use_roi=True,
                        rng_parity=False)
    fused = FusedTcamLosses(SelfLearningTcams(cuda_id=0, lambda_=0.75, seg_ignore_idx=IGNORE),
                            ConRanFieldTcams(cuda_id=0, lambda_=2e-3, sigma_rgb=15., sigma_xy=100., scale_factor=1.0,
                                             fuse_softmax=True, seg_ignore_idx=IGNORE))
    cams = torch.zeros((b, t, h, w), device="cuda")
    roi = torch.ones((b, 1, h, w), dtype=torch.long, device="cuda")
    img8 = torch.zeros((b, 3, h, w), dtype=torch.uint8, device="cuda")
    logits = torch.zeros((b, k, h, w), dtype=torch.float16, device="cuda", requires_grad=True)

    def load(seed):
        g = torch.Generator().manual_seed(seed)
        cams.copy_(torch.rand((b, t, h, w), generator=g))
        img8.copy_(torch.from_numpy(synth.make_images(b, h, w, "natural", seed=seed).astype(np.uint8)))
        with torch.no_grad():
            logits.copy_(3 * torch.randn((b, k, h, w), generator=g))

    stream = torch.cuda.Stream()
    stream.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(stream):
        load(1)
        graph = torch.cuda.CUDAGraph()
        logits.grad = None
        with torch.cuda.graph(graph, stream=stream):
            seeds, _ = seeder.forward_stack(cams, roi, sparse=True)
            total = fused(epoch=0, fcams=logits, raw_img=img8, seeds=seeds)
            total.backward()
        g_ce, g_crf = fused.last_ce, fused.last_crf
        for seed in (2, 3, 4):
            load(seed)
            logits.grad.zero_()
            graph.replay()
            stream.synchronize()
            assert logits.grad.dtype == torch.float16
            got_grad = logits.grad.float().cpu().numpy()
            got_ce, got_crf = g_ce.clone(), g_crf.item()
            z = logits.detach().clone()
            eager_ce, _, _ = ops.seed_ce_forward(z, seeds.sel, seeds.ksz)
            assert same_bits(torch, got_ce, eager_ce) and np.isfinite(eager_ce.item()), seed
            zz = z.clone().requires_grad_(True)
            fused(epoch=0, fcams=zz, raw_img=img8, seeds=seeds).backward()
            assert same_bits(torch, fused.last_ce, eager_ce), seed
            assert abs(got_crf - fused.last_crf.item()) <= 1e-5 * abs(fused.last_crf.item()), seed
            # both gradients are rounded to fp16: AS's atomic-order noise can move one by an ulp (2 unit roundoffs)
            assert rel_err(got_grad, zz.grad.float().cpu().numpy()) <= 2 * UNIT_ROUNDOFF["float16"] + 1e-5, seed
            fused.last_ce, fused.last_crf = g_ce, g_crf
    torch.cuda.synchronize()


# ---------------------------------------------------------------------------
# 7. outside autocast, and refusals
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("fused", [True, False], ids=["FusedTcamLosses", "SelfLearning+ConRanField"])
@pytest.mark.parametrize("dtype", DTYPES + ["float64"])
def test_modules_outside_autocast(torch_cuda, dtype, fused):
    """fp16, bf16 and float64 logits handed to the modules with no autocast region: the loss and gradient equal torch's
    F.cross_entropy on the seeds' label map plus the fused CRF, both on the logits widened (or, for float64, cast) to
    float32; the gradient has the logits' dtype."""
    torch = torch_cuda
    import torch.nn.functional as F
    from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLossFromLogits
    b, k, h, w = 4, 3, 48, 56
    raw, seeds = _step_inputs(torch, b, k, h, w, seed=7)
    step = _tcam_modules(fused)
    z = make_logits(torch, "float16", "randn", b, k, h, w, seed=8).to(tdtype(torch, dtype))
    fcams = z.clone().requires_grad_(True)
    loss = step(fcams, raw, seeds)
    loss.backward()
    assert fcams.grad.dtype == fcams.dtype
    z32 = z.float().requires_grad_(True)
    want = 0.75 * F.cross_entropy(z32, seeds.dense(), ignore_index=IGNORE) + \
        DenseCRFLossFromLogits(2e-3, 15., 100.)(images=raw, logits=z32)
    want.backward()
    assert abs(loss.item() - want.item()) <= 1e-5 * abs(want.item())
    assert rel_err(fcams.grad.double().cpu().numpy(), z32.grad.cpu().numpy()) <= _grad_tol(dtype, fused)


@pytest.mark.parametrize("fused", [True, False], ids=["FusedTcamLosses", "SelfLearningTcams"])
def test_seeds_of_other_frames_are_refused(torch_cuda, fused):
    torch = torch_cuda
    from tcam_wsol_video_b200.losses import SelfLearningTcams
    from tcam_wsol_video_b200.tcam_seeding import SparseSeeds
    b, k, h, w = 4, 2, 48, 56
    raw, seeds = _step_inputs(torch, b, k, h, w, seed=9)
    if fused:
        step = _tcam_modules(True)
    else:
        sl = SelfLearningTcams(cuda_id=0, lambda_=0.75, seg_ignore_idx=IGNORE)
        step = lambda fcams, raw, seeds: sl(epoch=0, fcams=fcams, seeds=seeds)   # noqa: E731
    z = make_logits(torch, "float16", "randn", b, k, h, w, seed=10)
    step(z, raw, seeds)   # the matching seeds are accepted
    with pytest.raises(ValueError):
        step(z, raw, SparseSeeds(seeds.sel, seeds.ksz, seeds.ignore_idx, h, w + 1))   # another resolution
    with pytest.raises(ValueError):
        step(z[:3], raw[:3], seeds)                                                     # another batch size


def test_ops_refuse_malformed_seeds_and_logits(torch_cuda):
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    b, k, h, w = 2, 2, 19, 37
    z = make_logits(torch, "bfloat16", "randn", b, k, h, w, seed=11)
    sel = torch.full((b, 2, 3), -1, dtype=torch.int32, device="cuda")
    sel[:, :, 0] = torch.tensor([5, 300], dtype=torch.int32)
    count = ops.seed_ce_forward(z, sel, 3)[1]
    for bad in (sel.long(), sel[:, :1].contiguous(), sel[:1].contiguous(), sel.cpu(), sel.transpose(1, 2)):
        with pytest.raises(_lib.TcamCrfError):
            ops.seed_ce_forward(z, bad, 3)
        with pytest.raises(_lib.TcamCrfError):
            ops.seed_ce_backward_(torch.zeros_like(z), z, bad, 3, count, torch.ones(1, device="cuda"))
    for bad_grad in (torch.zeros_like(z, dtype=torch.float32), torch.zeros_like(z)[:1],
                     torch.zeros((b, h, w, k), dtype=z.dtype, device="cuda").permute(0, 3, 1, 2)):
        with pytest.raises(_lib.TcamCrfError):
            ops.seed_ce_backward_(bad_grad, z, sel, 3, count, torch.ones(1, device="cuda"))
    with pytest.raises(_lib.TcamCrfError):
        ops.seed_ce_forward(z[:, :, :, :1].expand(b, k, h, w), sel, 3)   # not contiguous
    with pytest.raises(_lib.TcamCrfError):
        ops.seed_ce_forward(z[0], sel, 3)                                # not 4-D
    # K < 2 is still refused, by the softmax forward and by the cross-entropy
    z1 = z[:, :1].contiguous()
    images = torch.zeros((b, 3, h, w), dtype=torch.uint8, device="cuda")
    with pytest.raises(_lib.TcamCrfError):
        ops.crf_forward_logits(images, z1, _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0))
    with pytest.raises(_lib.TcamCrfError):
        ops.seed_ce_forward(z1, sel, 3)


def test_unknown_dtype_code_is_refused(torch_cuda):
    """Every typed entry point returns TCAMCRF_ERR_INVALID for a dtype code it does not know, before touching any
    pointer."""
    from ctypes import byref
    lib = _lib.load()
    cfg = _lib.make_config(_lib.FEAT_XY_RGB, 3, 15.0, 100.0)
    for code in (3, -1, 7):
        calls = {
            "tcamcrf_loss_forward_logits_typed": lambda: lib.tcamcrf_loss_forward_logits_typed(
                byref(cfg), None, 0, None, code, None, None, 1, 2, 4, 4, 1.0, None, 0, None),
            "tcamcrf_loss_forward_host_frames_typed": lambda: lib.tcamcrf_loss_forward_host_frames_typed(
                byref(cfg), None, None, 0, None, code, None, None, 1, 2, 4, 4, 1.0, None, 0, None),
            "tcamcrf_loss_backward_logits_typed": lambda: lib.tcamcrf_loss_backward_logits_typed(
                None, None, code, None, None, 1, 2, 4, 4, 1.0, 1.0, None),
            "tcam_seed_ce_forward_typed": lambda: lib.tcam_seed_ce_forward_typed(
                None, code, None, 1, 1, 2, 4, 4, 3, None, None, None, None, 1.0, None, None),
            "tcam_seed_ce_backward_typed": lambda: lib.tcam_seed_ce_backward_typed(
                None, code, None, 1, 1, 2, 4, 4, 3, None, None, 1.0, None, None),
            "tcam_crf_seed_ce_backward_typed": lambda: lib.tcam_crf_seed_ce_backward_typed(
                None, None, code, None, 1, 3, None, None, 1, 2, 4, 4, 1.0, 1.0, 1.0, None, None),
        }
        for name, call in calls.items():
            assert call() == 1, name                        # TCAMCRF_ERR_INVALID
            assert "dtype" in _lib.last_error(), (name, _lib.last_error())


# ---------------------------------------------------------------------------
# 4. coverage: must stay the last test of the module
# ---------------------------------------------------------------------------
def test_every_compiled_lowp_kernel_was_launched(torch_cuda):
    """Every *_lowp instantiation compiled into libtcamcrf.so ran in some case of this module."""
    want_cases = {(_fwd_id(c), d) for c in FWD_CASES for d in DTYPES}
    if not want_cases <= _forward_cases_run:
        pytest.skip(f"only {len(_forward_cases_run)} of {len(want_cases)} forward cases ran: run the whole module")
    compiled = compiled_lowp_kernels()
    assert len(compiled) >= 45, f"cuobjdump listed only {len(compiled)} *_lowp kernels: {sorted(compiled)}"
    missing = sorted(compiled - _launched)
    print(f"\n*_lowp kernels: {len(compiled)} compiled, {len(compiled & _launched)} launched")
    assert not missing, "compiled but never launched: " + ", ".join(missing)
