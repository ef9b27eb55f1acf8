"""The float64 matrix form of the filter (oracle/lattice_matrix.py), pinned before the GPU suite relies on it.

A = alpha * W * B_d ... B_0 * W^T is built from the oracle's own lattice, so the float32 C restatement
(permuto_oracle.c) and the reference build's fixtures must agree with it up to float32 rounding -- and how far they
are from it is the yardstick for the kernels (tests/test_gpu_kernel_matrix.py): a kernel must be at least as accurate
as the float32 code it replaces.

The float32 oracle's own error against float64, measured here (normwise ||a-b||_inf / ||b||_inf and pointwise with
a floor of 1e-3 * max|b|), worst case over the shapes 19x37, 1x50, 50x1, 7x300, 8x32, 1x1 and three classes:

    lattice            noise: norm / point      natural: norm / point
    colour D = 1       3.5e-7 / 3.5e-7          3.2e-7 / 4.0e-7
    colour D = 2       1.9e-7 / 2.2e-7          2.2e-7 / 3.3e-7
    colour D = 3       1.5e-7 / 2.1e-7          2.9e-7 / 3.6e-7
    colour D = 4       1.7e-7 / 2.5e-7          2.1e-7 / 2.5e-7
    colour D = 5       1.5e-7 / 2.7e-7          2.4e-7 / 3.1e-7
    colour D = 6       1.4e-7 / 2.3e-7          2.4e-7 / 2.8e-7
    xy + 1 (D = 3)     2.3e-7 / 2.8e-7          2.8e-7 / 3.4e-7
    xy + 2 (D = 4)     1.9e-7 / 2.1e-7          2.8e-7 / 3.0e-7
    xy + 4 (D = 6)     1.7e-7 / 2.6e-7          2.5e-7 / 2.9e-7

The reference build's own outputs (the fixtures in tests/golden/, 5-D and colour D = 1, 3) are within 1.4e-7 to
2.9e-7 normwise and 2.0e-7 to 3.2e-7 pointwise.  So float32 costs the reference a few ulps, never 1e-6.  The bar
below (ORACLE_BAR) holds every figure with a margin of 2x or more.
"""
import numpy as np
import pytest

from conftest import golden_cases, load_golden, pointwise_rel_err, rel_err
from oracle import lattice_matrix as lm
from tcam_wsol_video_b200 import synth

ORACLE_BAR = 1e-6        # the float32 oracle / reference build against float64, normwise and pointwise
SHAPES = [(19, 37), (1, 50), (50, 1), (7, 300), (8, 32), (1, 1)]


def _errs(got, want):
    want = np.asarray(want, np.float64)
    return rel_err(got, want), pointwise_rel_err(got, want, floor=1e-3 * max(float(np.abs(want).max()), 1e-30))


def _planes(h, w, kind, seed):
    """Six image planes: the three of synth.make_images and a second, scaled copy (for D = 4..6)."""
    img = synth.make_images(1, h, w, kind, seed=seed)[0]
    return np.ascontiguousarray(np.concatenate([img, img[::-1] * 0.5 + 3.0], axis=0))


def lattice_and_filter(oracle_mod, spec, planes, h, w):
    """(oracle lattice, float32 filter function) of one frame for spec ("colour", DIM) or ("xy", planes)."""
    kind, c = spec
    if kind == "colour":
        feats = (planes[:c].reshape(c, -1).T / np.float32(15.0)).astype(np.float32)
    else:
        feats = oracle_mod.xy_features(h, w, 100.0, planes[:c], 15.0)
    L = oracle_mod.port_lattice_features(feats)
    return L, (lambda s: oracle_mod.port_filter_features(feats, s))


@pytest.mark.parametrize("path", golden_cases(), ids=lambda p: p.rsplit("/", 1)[-1])
def test_matrix_matches_reference_fixtures(oracle_mod, path):
    """Every AS fixture the reference build made (tests/golden/*.npz; tests/golden/lattice/ stores digests only, and
    the port is bit-exact to those, tests/test_oracle.py)."""
    g = load_golden(path)
    img = g["image_u8"].astype(np.float32)
    n, k, h, w = g["seg"].shape
    dim = int(g["dim"])
    for i in range(n):
        if dim:
            L = oracle_mod.port_lattice_color(img[i], h, w, float(g["sigma_rgb"]), dim)
        else:
            L = oracle_mod.port_lattice_bilateral(img[i], h, w, float(g["sigma_rgb"]), float(g["sigma_xy"]))
        want = lm.apply(L, g["seg"][i].reshape(k, -1))
        e, pe = _errs(g["AS"][i].reshape(k, -1), want)
        assert e < ORACLE_BAR and pe < ORACLE_BAR, f"frame {i}: norm {e:.2e} point {pe:.2e}"
        # the port on the same lattice agrees too
        got = oracle_mod.port_bilateralfilter_batch(img[i], g["seg"][i], 1, k, h, w, float(g["sigma_rgb"]),
                                                    float(g["sigma_xy"])) if not dim else \
            oracle_mod.port_colorbilateralfilter_batch(img[i], g["seg"][i], 1, k, h, w, float(g["sigma_rgb"]), dim)
        assert max(_errs(got.reshape(k, -1), want)) < ORACLE_BAR


@pytest.mark.parametrize("kind", ["noise", "natural"])
@pytest.mark.parametrize("spec", [("colour", d) for d in range(1, 7)] + [("xy", c) for c in (1, 2, 4)],
                         ids=lambda s: f"{s[0]}{s[1]}")
def test_matrix_matches_port_on_random_frames(oracle_mod, spec, kind):
    """D = 1..6 colour lattices and the xy + 1/2/4-plane lattices (D = 3, 4, 6), with P % 4 != 0 (the reference's
    zero-feature ghost pixels put vertices in the lattice that only the blur reaches), H = 1, W = 1 and one pixel."""
    for h, w in SHAPES:
        planes = _planes(h, w, kind, seed=spec[1] + 7 * h)
        L, filt = lattice_and_filter(oracle_mod, spec, planes, h, w)
        seg = synth.make_segs(1, 3, h, w, seed=h + w)[0].reshape(3, -1)
        want = lm.apply(L, seg)
        e, pe = _errs(filt(seg), want)
        assert e < ORACLE_BAR and pe < ORACLE_BAR, f"{h}x{w}: norm {e:.2e} point {pe:.2e}"
        # signed input and the transpose: <V, A S> == <A^T V, S> in float64
        v = np.random.default_rng(h * w).standard_normal(seg.shape)
        lhs = (v * want).sum()
        rhs = (lm.apply(L, v, transposed=True) * seg).sum()
        assert abs(lhs - rhs) <= 1e-12 * max(abs(lhs), 1.0)


@pytest.mark.parametrize("spec", [("colour", 1), ("colour", 3), ("colour", 6), ("xy", 1), ("xy", 3), ("xy", 4)],
                         ids=lambda s: f"{s[0]}{s[1]}")
def test_blur_matrices_are_symmetric(oracle_mod, spec):
    """n1 and n2 are mutual neighbours, so every single-axis blur B_j is symmetric.  tcamcrf_filter_transposed
    relies on this: it runs the same blur with the axes in the opposite order (include/tcamcrf.h).  The product of
    the blurs is not symmetric, and neither is A."""
    h, w = 19, 37
    planes = _planes(h, w, "natural", seed=3)
    L, _ = lattice_and_filter(oracle_mod, spec, planes, h, w)
    W, B, _ = lm.lattice_matrices(L)
    assert W.shape == (h * w, L.m)
    for j, b in enumerate(B):
        assert abs(b - b.T).max() == 0, f"B_{j} is not symmetric"
        # each vertex: itself plus at most two neighbours at 1/2
        assert b.diagonal().min() == 1.0 and (b.sum(axis=1).A.ravel() <= 2.0).all()
    s = synth.make_segs(1, 2, h, w, seed=1)[0].reshape(2, -1)
    a, at = lm.apply(L, s), lm.apply(L, s, transposed=True)
    assert rel_err(at, a) > 1e-6 or L.d == 1


@pytest.mark.parametrize("spec", [("colour", 2), ("colour", 5), ("xy", 3)], ids=lambda s: f"{s[0]}{s[1]}")
def test_exact_gradient_matches_finite_difference(oracle_mod, spec):
    """crf_grad_exact64 is the gradient of crf_loss64: the loss is quadratic in S, so a central difference is exact
    up to rounding; and the reference's -2 g w AS / N is not, because A is not symmetric."""
    n, k, h, w = 2, 3, 9, 13
    rng = np.random.default_rng(11)
    ops = []
    for i in range(n):
        L, _ = lattice_and_filter(oracle_mod, spec, _planes(h, w, "noise", seed=i), h, w)
        ops.append(lm.LatticeOperator(L))
    s = lm.softmax64(rng.standard_normal((n, k, h, w)))
    v = rng.standard_normal((n, k, h, w))
    g, weight = 0.7, 1e-3

    def loss(x):
        ax = np.stack([ops[i].apply(x[i].reshape(k, -1)) for i in range(n)]).reshape(x.shape)
        return lm.crf_loss64(x, ax, n, weight)

    AS = np.stack([ops[i].apply(s[i].reshape(k, -1)) for i in range(n)]).reshape(s.shape)
    AtS = np.stack([ops[i].apply(s[i].reshape(k, -1), transposed=True) for i in range(n)]).reshape(s.shape)
    grad = lm.crf_grad_exact64(AS, AtS, n, g, weight)
    directional = g * (loss(s + v) - loss(s - v)) / 2.0
    got = (grad * v).sum()
    assert abs(got - directional) <= 1e-10 * abs(directional)
    approx = (lm.crf_grad_reference64(AS, n, g, weight) * v).sum()
    assert abs(approx - directional) > 1e-6 * abs(directional)


def test_logits_chain_rule_matches_finite_difference():
    """logits_grad64 is the chain rule of crf_loss64(softmax64(z)) for a FIXED G = d loss / d S."""
    rng = np.random.default_rng(5)
    z = 3.0 * rng.standard_normal((2, 4, 3, 5))
    G = rng.standard_normal(z.shape)
    dz = lm.logits_grad64(lm.softmax64(z), G)
    e = 1e-6
    for idx in [(0, 0, 0, 0), (1, 3, 2, 4), (0, 2, 1, 3)]:
        zp, zm = z.copy(), z.copy()
        zp[idx] += e
        zm[idx] -= e
        fd = ((lm.softmax64(zp) - lm.softmax64(zm)) * G).sum() / (2 * e)
        assert abs(fd - dz[idx]) < 1e-8
    # the gradient of a softmax sums to zero over the classes
    assert np.abs(dz.sum(axis=1)).max() < 1e-14
