"""GPU suite (-m gpu): every compiled lattice-kernel instantiation against the float64 matrix form of the filter.

The reference is oracle/lattice_matrix.py: A = alpha * W * B_d ... B_0 * W^T built from the oracle's lattice of each
frame (bit-exact to the library's, tests/test_gpu_parity.py), evaluated in float64.  It gives A S, A^T S, the loss,
both gradients and the logits chain rule without any float32 rounding of its own.

The case table is a covering design: lattice (colour D = 1..6, xy + 1..4 planes = D 3..6) x images (float32, uint8)
x build (BUILD_DEDUP 0 / 1) x splat (DENSE 0 / 1) x K (1, 2, 3-4, 5-8, 9-12, 13-16, 17-20, 21-24) x input
(probabilities, logits) on ragged frames (P not a multiple of 4, 32, 256 or the 32 x 8 dedup tile, H = 1, W = 1),
one tile-exact 8 x 32 frame, iid noise (about one vertex per pixel), natural frames (long runs of pixels on one
vertex) and constant images (every pixel of a warp on the same d + 1 vertices).  Every call runs under
torch.profiler with CUPTI kernel tracing: each case asserts that the instantiations it aims at really ran, and the
last test fails on any instantiation compiled into the library that no case launched.

Tolerance: a kernel must be at least as accurate as the float32 code it replaces.  Normwise and pointwise error
(floor 1e-3 * max|want|) against float64 <= 2 x the float32 oracle's own error on the same case + 1e-7 (the oracle's
error is measured per case; tests/test_lattice_matrix.py records it at 1.4e-7 to 4.0e-7), and rel 1e-4 against the
float32 oracle like the rest of the suite.  The transposed filter has no float32 oracle: it is held to the forward
filter's bar on the same case.  The logits backward is held normwise to 2 x the error of the same chain rule evaluated
in float32 (what F.softmax + autograd compute), + 1e-7, and per element to the rounding-error bound of its expression
(assert_logits_grad): its pointwise relative error is not a measure where G - sum p G cancels.  Measured on a B200,
the fused backward reached 4x the float32 restatement's pointwise error at one element (K = 11) for that reason.
"""
import itertools
import re
import subprocess

import numpy as np
import pytest

from conftest import pointwise_rel_err, rel_err
from oracle import lattice_matrix as lm
from tcam_wsol_video_b200 import _lib, synth

pytestmark = pytest.mark.gpu

SIGMA_RGB, SIGMA_XY = 15.0, 10.0
SHAPES = [(19, 37), (1, 50), (50, 1), (7, 300), (8, 32)]
KINDS = ["noise", "natural", "constant"]
LATTICES = [("colour", d) for d in range(1, 7)] + [("xy", c) for c in range(1, 5)]
# (K, logits, dense): one entry per value-stage variant; K = 6 / 10 / 14 are the row kernels' KV = 2 / 3 / 4
VALUE_VARIANTS = [(1, False, 0), (2, False, 0), (2, True, 1), (3, False, 0), (4, True, 0),
                  (6, False, 1), (10, False, 1), (14, False, 1), (7, True, 1), (11, True, 1), (16, True, 1),
                  (13, False, 0), (19, True, 1), (22, False, 1)]
# the softmax needs two classes, so V = 1 (K = 1) has no logits variant that any entry point can launch
UNREACHABLE = {f"{k}<{d}, 1, true>" for k in ("splat_kernel", "slice_kernel") for d in range(1, 7)}

_launched = set()      # every lattice-kernel instantiation the profiler saw in this module
_cases_run = set()


def _dim(spec):
    return spec[1] + (2 if spec[0] == "xy" else 0)


def _cases():
    """Each lattice gets every value variant once; builds (float / uint8 x plain / dedup), shapes and frame kinds
    rotate through them, so every (D, image type, build kernel) meets several value variants."""
    out = []
    builds = list(itertools.product([False, True], [0, 1]))
    for li, spec in enumerate(LATTICES):
        for vi, (k, logits, dense) in enumerate(VALUE_VARIANTS):
            if spec[0] == "xy" and vi % 2:
                continue   # the xy lattices share D with the colour ones: half of the value variants suffice
            u8, dedup = builds[(vi + li) % 4]
            hw = SHAPES[(vi + li) % len(SHAPES)]
            kind = KINDS[(vi + 2 * li) % len(KINDS)]
            n, chunk = (5, 2) if (vi + li) % 3 == 0 else (2, 0)
            out.append(dict(spec=spec, u8=u8, dedup=dedup, dense=dense, k=k, logits=logits, hw=hw, kind=kind,
                            n=n, chunk=chunk))
    return out


CASES = _cases()


def _case_id(c):
    s = c["spec"]
    return (f"{s[0]}{s[1]}-{'u8' if c['u8'] else 'f32'}-dedup{c['dedup']}-dense{c['dense']}-K{c['k']}"
            f"{'-logits' if c['logits'] else ''}-{c['kind']}-{c['hw'][0]}x{c['hw'][1]}-n{c['n']}")


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


# ---------------------------------------------------------------------------
# kernel names: the profiler's (demangled by CUPTI) and the library's (mangled, from cuobjdump)
# ---------------------------------------------------------------------------
_LATTICE_KERNELS = ("build_kernel", "build_dedup_kernel", "neighbour_kernel", "splat_kernel", "splat_rows_kernel",
                    "slice_kernel", "blur_kernel")


def _normalise(name):
    if name.startswith("_ZN7tcamcrf"):
        return _demangle(name)
    m = re.search(r"tcamcrf::(\w+)<([^>]*)>", name)
    if not m or m.group(1) not in _LATTICE_KERNELS:
        return None
    return f"{m.group(1)}<{m.group(2).strip()}>"


def _demangle(mangled):
    """_ZN7tcamcrf17splat_rows_kernelILi4ELi3ELb1EEEvNS_11PixelParamsE -> splat_rows_kernel<4, 3, true>."""
    m = re.match(r"_ZN7tcamcrf(\d+)", mangled)
    if not m:
        return None
    pos = m.end()
    name = mangled[pos:pos + int(m.group(1))]
    rest = mangled[pos + int(m.group(1)):]
    if name not in _LATTICE_KERNELS or not rest.startswith("I"):
        return None
    args, rest = [], rest[1:]
    while not rest.startswith("E"):
        t = re.match(r"Li(n?\d+)E|Lb([01])E|(f)|(h)", rest)
        assert t, f"cannot read the template arguments of {mangled}"
        if t.group(1) is not None:
            args.append(t.group(1).replace("n", "-"))
        elif t.group(2) is not None:
            args.append("true" if t.group(2) == "1" else "false")
        else:
            args.append("float" if t.group(3) else "unsigned char")
        rest = rest[t.end():]
    return f"{name}<{', '.join(args)}>"


def compiled_lattice_kernels():
    """Every lattice-kernel instantiation in the built library, read like tools/dump_sass.py does."""
    import shutil
    tool = shutil.which("cuobjdump") or "/usr/local/cuda/bin/cuobjdump"
    text = subprocess.run([tool, "-sass", _lib.LIB_PATH], check=True, capture_output=True, text=True).stdout
    names = {_demangle(n) for n in re.findall(r"Function : (\S+)", text)}
    names.discard(None)
    return names


class Traced:
    """torch.profiler with CUDA activities (CUPTI kernel tracing, no counters) around library calls."""

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
# inputs and the float64 side
# ---------------------------------------------------------------------------
def make_planes(n, h, w, kind, seed):
    """float32 [n, 6, h, w] of integer values 0..255 (so a uint8 copy holds the same features)."""
    if kind == "constant":
        return np.full((n, 6, h, w), 128.0, np.float32)
    img = synth.make_images(n, h, w, kind, seed=seed)
    return np.ascontiguousarray(np.concatenate([img, np.floor(img[:, ::-1] * 0.5) + 3.0], axis=1))


def config(spec, chunk=0):
    if spec[0] == "colour":
        return _lib.make_config(_lib.FEAT_COLOR, spec[1], SIGMA_RGB, chunk_frames=chunk)
    return _lib.make_config(_lib.FEAT_XY_RGB, spec[1], SIGMA_RGB, SIGMA_XY, chunk_frames=chunk)


def features(oracle_mod, spec, frame, h, w):
    kind, c = spec
    if kind == "colour":
        return np.ascontiguousarray((frame[:c].reshape(c, -1).T / np.float32(SIGMA_RGB)).astype(np.float32))
    return oracle_mod.xy_features(h, w, SIGMA_XY, frame[:c], SIGMA_RGB)


class Reference:
    """Per frame: the oracle lattice as a float64 operator, and the float32 oracle filter on the same features."""

    def __init__(self, oracle_mod, spec, planes):
        n, _, h, w = planes.shape
        self.oracle = oracle_mod
        self.feats = [features(oracle_mod, spec, planes[i], h, w) for i in range(n)]
        self.ops = [lm.LatticeOperator(oracle_mod.port_lattice_features(f)) for f in self.feats]

    def apply(self, s, transposed=False):
        n, k = s.shape[:2]
        return np.stack([self.ops[i].apply(s[i].reshape(k, -1), transposed) for i in range(n)]).reshape(s.shape)

    def apply32(self, s):
        n, k = s.shape[:2]
        return np.stack([self.oracle.port_filter_features(self.feats[i], s[i].reshape(k, -1))
                         for i in range(n)]).reshape(s.shape)


def errs(got, want):
    want = np.asarray(want, np.float64)
    return rel_err(got, want), pointwise_rel_err(got, want, floor=1e-3 * max(float(np.abs(want).max()), 1e-30))


def assert_bar(got, want, bar, what):
    """Normwise and pointwise error against float64 within 2 x the float32 reference's (bar) + 1e-7."""
    e, pe = errs(got, want)
    assert e <= 2 * bar[0] + 1e-7, f"{what}: normwise {e:.3e} > 2 x {bar[0]:.3e} + 1e-7"
    assert pe <= 2 * bar[1] + 1e-7, f"{what}: pointwise {pe:.3e} > 2 x {bar[1]:.3e} + 1e-7"


def assert_loss(got, want, bar):
    """-sum(S * AS) / N: every term has one sign, so its relative error is at most AS's largest pointwise one."""
    assert abs(got - want) <= (2 * max(bar) + 1e-7) * abs(want), f"loss {got!r} against {want!r}"


def softmax32(z):
    z = np.asarray(z, np.float32)
    e = np.exp(z - z.max(axis=1, keepdims=True))
    return e / e.sum(axis=1, keepdims=True, dtype=np.float32)


def logits_grad32(z, AS, n_norm, g, weight):
    """The chain rule as float32 autograd would evaluate it: G = ((-2 g w) AS) / N, dz = p (G - sum p G)."""
    p = softmax32(z)
    G = (np.float32(-2.0) * np.float32(g * weight) * AS.astype(np.float32)) / np.float32(n_norm)
    return p * (G - (p * G).sum(axis=1, keepdims=True, dtype=np.float32))


def assert_logits_grad(dz, z, AS, n_norm, g, weight, what):
    """dz = p (G - sum_j p_j G_j) cancels where one class dominates, so a pointwise relative error says nothing there.
    Normwise: within 2 x the float32 chain rule's error + 1e-7.  Per element: within the rounding-error bound of the
    expression in ulps: K + 8 of p_k (|G_k| + sum_j p_j |G_j|) (a few for p and G, K for the inner sum, two for the
    difference and the product), plus what the rounding of z_j - max z costs expf: |z_j - max z| ulps of p_j, and one
    smallest normal float times max |G| for probabilities that flush to zero."""
    K = z.shape[1]
    p = lm.softmax64(z)
    G = lm.crf_grad_reference64(AS, n_norm, g, weight)
    want = lm.logits_grad64(p, G)
    e, e32 = rel_err(dz, want), rel_err(logits_grad32(z, AS, n_norm, g, weight), want)
    assert e <= 2 * e32 + 1e-7, f"{what}: normwise {e:.3e} > 2 x {e32:.3e} + 1e-7"
    dzmax = np.abs(z.astype(np.float64) - z.max(axis=1, keepdims=True))
    inner = (p * G).sum(axis=1, keepdims=True)
    with np.errstate(invalid="ignore"):
        pdz = np.nan_to_num(p * dzmax)    # 0 * 1e30 where a class sits at -1e30
    scale = p * ((K + 8) * (np.abs(G) + (p * np.abs(G)).sum(axis=1, keepdims=True)) + (pdz * np.abs(G)).sum(
        axis=1, keepdims=True)) + pdz * np.abs(G - inner)
    floor = (K + 8) * float(np.finfo(np.float32).tiny) * float(np.abs(G).max())
    excess = np.abs(dz - want) - (2.0 ** -23 * scale + floor)
    assert excess.max() <= 0, f"{what}: {int((excess > 0).sum())} elements beyond their rounding-error bound"


def expected_kernels(c):
    """The instantiations a forward call of case c must launch."""
    d, k = _dim(c["spec"]), c["k"]
    img = "unsigned char" if c["u8"] else "float"
    kp = k if k <= 2 else (k + 3) // 4 * 4
    v = 4 if kp % 4 == 0 else 2 if kp % 2 == 0 else 1
    lg = "true" if c["logits"] else "false"
    out = {f"{'build_dedup_kernel' if c['dedup'] else 'build_kernel'}<{d}, {img}>", f"neighbour_kernel<{d}>",
           f"slice_kernel<{d}, {v}, {lg}>"}
    kv = kp // 4
    if c["dense"] and v == 4 and 2 <= kv <= 4:
        out.add(f"splat_rows_kernel<{d}, {kv}, {lg}>")
    else:
        out.add(f"splat_kernel<{d}, {v}, {lg}>")
    if v < 4:
        out.add(f"blur_kernel<{v}, 1>")
    else:
        out.add(f"blur_kernel<4, {kv if kv in (1, 2, 3, 4, 6) else 0}>")
    return out


def _inputs(torch, c, seed):
    n, k, (h, w) = c["n"], c["k"], c["hw"]
    planes = make_planes(n, h, w, c["kind"], seed)
    images = torch.from_numpy(planes.astype(np.uint8) if c["u8"] else planes).cuda()
    gen = np.random.default_rng(seed)
    z = (3.0 * gen.standard_normal((n, k, h, w))).astype(np.float32)
    s = softmax32(z) if k > 1 else gen.random((n, k, h, w), dtype=np.float32)
    return planes, images, z, s


# ---------------------------------------------------------------------------
# the case table
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("c", CASES, ids=_case_id)
def test_lattice_kernels_against_float64(torch_cuda, oracle_mod, tuning, c):
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    tuning("DENSE", c["dense"])
    tuning("BUILD_DEDUP", c["dedup"])
    n, k = c["n"], c["k"]
    planes, images, z, s = _inputs(torch, c, seed=CASES.index(c) + 1)
    ref = Reference(oracle_mod, c["spec"], planes)
    cfg = config(c["spec"], c["chunk"])
    weight = 0.5
    if c["logits"]:
        s64 = lm.softmax64(z)
        want = ref.apply(s64)
        as32 = ref.apply32(s)                       # the unfused reference: float32 softmax, float32 filter
        bar = errs(as32, want)
        zt = torch.from_numpy(z).cuda()
        with Traced(torch) as tr:
            as_t, loss_t, _ = ops.crf_forward_logits(images, zt, cfg, check=True)
        assert expected_kernels(c) <= tr.kernels, f"launched {sorted(tr.kernels)}"
        got = as_t.cpu().numpy()
        assert_bar(got, want, bar, "AS from logits")
        assert rel_err(got, as32) < 1e-4
        assert_loss(loss_t.item(), lm.crf_loss64(s64, want, n), bar)
        g = torch.tensor([0.75], device="cuda")
        dz = ops.crf_backward_logits(as_t, zt, g, float(n), weight).cpu().numpy()
        assert_logits_grad(dz, z, got, n, 0.75, weight, "logits gradient")
        lib = _lib.load()
        out = torch.empty_like(as_t)
        _lib.check(lib.tcamcrf_loss_backward_logits(as_t.data_ptr(), zt.data_ptr(), g.data_ptr(), out.data_ptr(),
                                                    n, k, *c["hw"], float(n), ops._stream_ptr(as_t.device)),
                   "tcamcrf_loss_backward_logits")
        assert_logits_grad(out.cpu().numpy(), z, got, n, 0.75, 1.0, "logits gradient (unweighted)")
        _cases_run.add(_case_id(c))
        return

    want = ref.apply(s)
    want_t = ref.apply(s, transposed=True)
    as32 = ref.apply32(s)
    bar = errs(as32, want)
    st = torch.from_numpy(s).cuda()
    with Traced(torch) as tr:
        as_f, _, _ = ops.crf_forward(images, st, cfg, want_loss=False, check=True)       # tcamcrf_filter[_u8]
        as_l, loss_t, _ = ops.crf_forward(images, st, cfg, want_loss=True, check=True)   # tcamcrf_loss_forward[_u8]
        at_f = ops.crf_filter_transposed(images, st, cfg)                                # tcamcrf_filter_transposed
    assert expected_kernels(c) <= tr.kernels, f"launched {sorted(tr.kernels)}"
    for name, t in (("tcamcrf_filter", as_f), ("tcamcrf_loss_forward", as_l)):
        got = t.cpu().numpy()
        assert_bar(got, want, bar, name)
        assert rel_err(got, as32) < 1e-4, name
    assert_loss(loss_t.item(), lm.crf_loss64(s, want, n), bar)
    assert_bar(at_f.cpu().numpy(), want_t, bar, "tcamcrf_filter_transposed")

    # one lattice, four applications: the first splat turns entry indices into tagged vertex ids in place, the
    # others read tagged ids, in both splat kernels and in both blur orders
    if c["n"] <= cfg_capacity(cfg, k, c["hw"]):
        lat = ops.Lattice(images, cfg, k)
        with Traced(torch) as tr:
            outs = []
            for dense, transposed in ((1, False), (0, False), (1, True), (1, False)):
                tuning("DENSE", dense)
                outs.append((transposed, lat.apply(st, transposed=transposed).cpu().numpy()))
        for i, (transposed, got) in enumerate(outs):
            assert_bar(got, want_t if transposed else want, bar, f"lattice reuse, application {i}")
            fresh = at_f.cpu().numpy() if transposed else as_f.cpu().numpy()
            assert rel_err(got, fresh) < 1e-5
        assert lat.status()[0] == 0

    # backward: the reference's -2 g w AS / N is one rounding per element of the GPU's AS
    g = torch.tensor([0.75], device="cuda")
    grad = ops.crf_backward(as_l, g, float(n), weight).cpu().numpy()
    assert rel_err(grad, lm.crf_grad_reference64(as_l.cpu().numpy(), n, 0.75, weight)) < 3e-7
    if c["spec"] == ("xy", 3) and not c["u8"]:
        from tcam_wsol_video_b200.dense_crf_loss import DenseCRFLoss
        s1 = st.clone().requires_grad_(True)
        DenseCRFLoss(weight, SIGMA_RGB, SIGMA_XY, 1.0, exact_gradient=True)(
            images=images[:, :3].contiguous(), segmentations=s1).backward()
        want_g = lm.crf_grad_exact64(want, want_t, n, 1.0, weight)
        assert_bar(s1.grad.cpu().numpy(), want_g, bar, "exact gradient")
    _cases_run.add(_case_id(c))


def cfg_capacity(cfg, k, hw):
    from tcam_wsol_video_b200 import ops
    return ops.lattice_capacity(cfg, k, *hw)


# ---------------------------------------------------------------------------
# confident and degenerate logits; the K = 2 register path
# ---------------------------------------------------------------------------
def degenerate_logits(mode, n, k, h, w, seed):
    rng = np.random.default_rng(seed)
    z = rng.standard_normal((n, k, h, w))
    if mode in ("scale30", "scale80"):
        z = z * float(mode[5:])
    elif mode == "minus1e30":
        z[:, -1] = -1e30
    elif mode == "ties":
        z[:, 1] = z[:, 0] = np.maximum(z[:, 0], z[:, 1:].max(axis=1))
    elif mode == "equal":
        z[:] = 0.25
    elif mode == "denormal":
        z[:, -1] = z[:, :-1].max(axis=1) - 95.0     # p ~ e^-95 ~ 5e-42: a float32 denormal
    return z.astype(np.float32)


@pytest.mark.parametrize("mode", ["scale30", "scale80", "minus1e30", "ties", "equal", "denormal"])
@pytest.mark.parametrize("k,dense", [(2, 0), (4, 0), (10, 1), (21, 1)])
def test_degenerate_logits(torch_cuda, oracle_mod, tuning, mode, k, dense):
    """Probabilities at 1 and 0, a class at -1e30, ties in the maximum, p = 1/K, and a class whose probability is
    a float32 denormal.  The splat's reductions flush denormals to zero, so for that class AS is 0 where float64
    gives ~1e-41: harmless normwise and, with the floor at 1e-3 of the largest output, pointwise over the tensor."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    tuning("DENSE", dense)
    n, h, w = 2, 19, 37
    spec = ("xy", 3)
    planes = make_planes(n, h, w, "natural", seed=k)
    ref = Reference(oracle_mod, spec, planes)
    z = degenerate_logits(mode, n, k, h, w, seed=k)
    s64 = lm.softmax64(z)
    want = ref.apply(s64)
    bar = errs(ref.apply32(softmax32(z)), want)
    zt = torch.from_numpy(z).cuda()
    as_t, loss_t, _ = ops.crf_forward_logits(torch.from_numpy(planes).cuda(), zt, config(spec), check=True)
    got = as_t.cpu().numpy()
    assert np.isfinite(got).all()
    assert_bar(got, want, bar, f"AS, {mode}")
    assert_loss(loss_t.item(), lm.crf_loss64(s64, want, n), bar)
    dz = ops.crf_backward_logits(as_t, zt, torch.tensor([1.0], device="cuda"), float(n)).cpu().numpy()
    assert np.isfinite(dz).all()
    assert_logits_grad(dz, z, got, n, 1.0, 1.0, f"logits gradient, {mode}")


@pytest.mark.parametrize("mode", ["randn3", "scale30", "ties", "equal"])
@pytest.mark.parametrize("spec", [("colour", 1), ("colour", 4), ("xy", 3)], ids=lambda s: f"{s[0]}{s[1]}")
def test_two_class_register_path_equals_three_classes(torch_cuda, tuning, spec, mode):
    """K = 2 reads its probabilities through the two-class register path (Prob2); a K = 3 call whose third class is
    at -inf has the same probabilities bit for bit through the general softmax.  The two must agree within the
    atomic-order noise, and the extra class gets no gradient.  The gradients are compared given the same AS: the
    chain rule amplifies the atomic-order noise of AS by the cancellation in G - sum p G (3e-6 normwise was seen),
    and without that noise the two paths must give the same bits."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    tuning("DENSE", 0)
    n, h, w = 2, 19, 37
    planes = torch.from_numpy(make_planes(n, h, w, "noise", seed=3)).cuda()
    z2 = (3.0 * np.random.default_rng(4).standard_normal((n, 2, h, w))).astype(np.float32) if mode == "randn3" \
        else degenerate_logits(mode, n, 2, h, w, seed=4)
    z3 = np.concatenate([z2, np.full((n, 1, h, w), -np.inf, np.float32)], axis=1)
    g = torch.tensor([1.0], device="cuda")
    out = {}
    for name, z in (("2", z2), ("3", z3)):
        zt = torch.from_numpy(z).cuda()
        as_t, loss_t, _ = ops.crf_forward_logits(planes, zt, config(spec), check=True)
        out[name] = (as_t.cpu().numpy(), loss_t.item(), ops.crf_backward_logits(as_t, zt, g, float(n)).cpu().numpy())
    as2, l2, d2 = out["2"]
    as3, l3, d3 = out["3"]
    assert rel_err(as3[:, :2], as2) < 1e-6 and np.all(as3[:, 2] == 0)
    assert abs(l3 - l2) <= 1e-6 * abs(l2)
    assert np.all(d3[:, 2] == 0)
    # given the same AS, the backward has no atomics: the register path and the general softmax give the same bits
    as3_same = torch.from_numpy(np.concatenate([as2, np.zeros_like(as2[:, :1])], axis=1)).cuda()
    d3_same = ops.crf_backward_logits(as3_same, torch.from_numpy(z3).cuda(), g, float(n)).cpu().numpy()
    assert np.array_equal(d3_same[:, :2], d2) and np.all(d3_same[:, 2] == 0)


# ---------------------------------------------------------------------------
# value and build kernels at frame0 > 0 (only the host paths start a launch at a later frame of the workspace)
# ---------------------------------------------------------------------------
@pytest.mark.parametrize("spec,k", [(("colour", 2), 6), (("colour", 3), 10), (("xy", 3), 14), (("colour", 1), 3)],
                         ids=lambda v: f"{v[0]}{v[1]}" if isinstance(v, tuple) else f"K{v}")
def test_value_stages_at_later_frames(torch_cuda, oracle_mod, tuning, spec, k):
    """The host-pointer path runs the value stages group by group (two frames per group for K >= 6), so the splat,
    blur and slice of the later groups start at frame0 = 2 and 4 of the workspace.  DENSE = 1 forces the row splat."""
    torch = torch_cuda
    tuning("DENSE", 1)
    tuning("HOST_GROUPS", 3)
    n, h, w = 5, 19, 37
    planes = make_planes(n, h, w, "noise", seed=k)
    ref = Reference(oracle_mod, spec, planes)
    s = synth.make_segs(n, k, h, w, seed=k)
    want = ref.apply(s)
    bar = errs(ref.apply32(s), want)
    lib = _lib.load()
    got = np.zeros(s.size, np.float32)
    img = np.ascontiguousarray(planes[:, :3])
    if spec[0] == "xy":
        rc = lib.bilateralfilter_batch(img.ctypes.data, img.size, s.ctypes.data, s.size, got.ctypes.data, got.size,
                                       n, k, h, w, SIGMA_RGB, SIGMA_XY)
    else:
        # the drop-in batch strides frames by three planes (colorbilateralfilter.cpp:50): DIM <= 3 keeps them apart
        rc = lib.colorbilateralfilter_batch(img.ctypes.data, img.size, s.ctypes.data, s.size, got.ctypes.data,
                                            got.size, n, k, h, w, SIGMA_RGB, spec[1])
    _lib.check(rc, "host-pointer filter")
    for i in range(n):
        assert_bar(got.reshape(s.shape)[i], want[i], errs(ref.apply32(s[i:i + 1])[0], want[i]), f"frame {i}")
    assert_bar(got.reshape(s.shape), want, bar, "all frames")


@pytest.mark.parametrize("u8", [False, True], ids=["f32", "u8"])
@pytest.mark.parametrize("dedup", [0, 1])
@pytest.mark.parametrize("spec", [("colour", 2), ("xy", 1), ("colour", 6)], ids=lambda s: f"{s[0]}{s[1]}")
def test_build_at_later_frames(torch_cuda, oracle_mod, tuning, spec, dedup, u8):
    """Pinned host frames are copied and built section by section (four frames per section here), so the build
    kernels of the later sections start at frame0 = 4 and 8 of the workspace."""
    torch = torch_cuda
    from tcam_wsol_video_b200 import ops
    tuning("BUILD_DEDUP", dedup)
    tuning("HIMG_SECTIONS", 3)
    n, k, h, w = 9, 3, 7, 30
    planes = make_planes(n, h, w, "natural", seed=n)
    ref = Reference(oracle_mod, spec, planes)
    s = synth.make_segs(n, k, h, w, seed=2)
    want = ref.apply(s)
    host = torch.from_numpy(planes.astype(np.uint8) if u8 else planes).pin_memory()
    as_t, loss_t, _ = ops.crf_forward(host, torch.from_numpy(s).cuda(), config(spec), check=True)
    torch.cuda.synchronize()
    got = as_t.cpu().numpy()
    for i in range(n):
        assert_bar(got[i], want[i], errs(ref.apply32(s[i:i + 1])[0], want[i]), f"frame {i}")
    assert_loss(loss_t.item(), lm.crf_loss64(s, want, n), errs(ref.apply32(s), want))


# ---------------------------------------------------------------------------
# coverage: must stay the last test of the module
# ---------------------------------------------------------------------------
def test_every_compiled_lattice_kernel_was_launched(torch_cuda):
    """The union of the instantiations the cases launched must cover everything compiled into libtcamcrf.so, except
    the splat / slice of V = 1 with logits: V = 1 means K = 1, and every logits entry point refuses K < 2."""
    if len(_cases_run) < len(CASES):
        pytest.skip(f"only {len(_cases_run)} of {len(CASES)} cases ran: run the whole module for the coverage check")
    compiled = compiled_lattice_kernels()
    assert len(compiled) > 100, f"cuobjdump listed only {len(compiled)} lattice kernels"
    assert UNREACHABLE <= compiled
    missing = sorted(compiled - UNREACHABLE - _launched)
    print(f"\nlattice kernels: {len(compiled)} compiled, {len(compiled & _launched)} launched, "
          f"{len(UNREACHABLE)} unreachable through the C ABI")
    assert not missing, "compiled but never launched: " + ", ".join(missing)
