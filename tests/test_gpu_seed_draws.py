"""GPU suite (-m gpu): the seeder's in-kernel Exp(1) draws (TCAMSeeder(rng_parity=False)) against the float64
restatement oracle/seed_draws.py -- the Philox words bit for bit, every draw within 2 float32 ulps, the selection
pick for pick wherever float64 does not call it a near-tie -- and the distribution of the picks against the exact
inclusion probabilities of torch.multinomial(replacement=False), on both seeding paths."""
import numpy as np
import pytest
from scipy import stats

from oracle import seed_draws as sd
from tcam_wsol_video_b200 import synth

pytestmark = pytest.mark.gpu

BITS = sd.KERNEL_BITS
AMBIGUOUS = 2.0 ** -20   # relative gap of two float64 scores below which float32 scores may order them either way


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    assert torch.cuda.is_available()
    return torch


def _lib():
    from tcam_wsol_video_b200 import _lib
    return _lib, _lib.load()


def _stream(torch):
    return torch.cuda.current_stream().cuda_stream


def _within_ulps(got, want, n):
    """|got - want| <= n float32 ulps of want (want in float64)."""
    return np.abs(got.astype(np.float64) - want) <= n * np.spacing(np.abs(want).astype(np.float32)).astype(np.float64)


def _seeder(**kw):
    from tcam_wsol_video_b200.tcam_seeding import TCAMSeeder
    base = dict(seed_tech="seed_weighted", min_=1, max_=1, max_p=0.6, min_p=0.1, fg_erode_k=11, fg_erode_iter=0,
                ksz=3, support_background=True, multi_label_flag=False, seg_ignore_idx=-255, cuda_id=0,
                roi_method="roi_all", p_min_area_roi=0.05, use_roi=True, rng_parity=False)
    base.update(kw)
    return TCAMSeeder(**base)


def _cams(torch, b, t, h, w, seed, quantised=False):
    """[B,T,H,W] CAM-like maps (bilinear upsampling of low-res noise), optionally quantised to 5 levels so that many
    values tie at the n-th candidate; roi = temporal max >= 0.5."""
    low = torch.from_numpy(synth.make_low_res_cams(b, t, 7, 7, seed=seed)).squeeze(2)
    cams = torch.nn.functional.interpolate(low, size=(h, w), mode="bilinear", align_corners=False)
    if quantised:
        cams = torch.round(cams * 4) / 4
    roi = (cams.amax(dim=1, keepdim=True) >= 0.5).long()
    return cams.contiguous(), roi


def _expected(cams_max, roi, rng, *, max_p, min_p, k_fg, k_bg, weighted, draws=None):
    """float64 picks [B,2,kmax] (-1 = unused), the ambiguity flag of every (sample, side) (two adjacent scores among
    the first k + 1 closer than AMBIGUOUS but not equal) and the number of (sample, side) with an exact tie there.
    draws: None -> the in-kernel Philox draws of rng; else a function (b, side, n) -> the n draws of the candidates in
    row-major order."""
    b_n = cams_max.shape[0]
    kmax = max(k_fg, k_bg, 1)
    picks = np.full((b_n, 2, kmax), -1, dtype=np.int64)
    ambiguous = np.zeros((b_n, 2), dtype=bool)
    ties = 0
    for b in range(b_n):
        fg, bg, wts = sd.candidates(cams_max[b], None if roi is None else roi[b], max_p=max_p, min_p=min_p,
                                    max_=k_fg, min_=k_bg)
        for side, (cand, k) in enumerate(((fg, k_fg), (bg, k_bg))):
            if cand.size == 0 or k == 0:
                continue
            vals = wts if (side == 0 and weighted) else np.ones(cand.size)
            q = sd.exp_draw_f64(sd.seed_words(rng, b, side, cand), BITS) if draws is None else draws(b, side, cand.size)
            got, gaps = sd.select_f64(cand, vals, q, k)
            picks[b, side, :got.size] = got
            ambiguous[b, side] = ((gaps > 0) & (gaps < AMBIGUOUS)).any()
            ties += int((gaps == 0).any())
    return picks, ambiguous, ties


def _compare(sel, picks, ambiguous, what):
    """Every (sample, side) whose picks differ must be a float64 near-tie; returns (cases, ambiguous cases)."""
    differ = (sel != picks).any(axis=2)
    wrong = np.argwhere(differ & ~ambiguous)
    assert wrong.size == 0, f"{what}: (sample, side) {wrong[:5].tolist()}: kernel {sel[tuple(wrong[0])].tolist()} " \
                            f"vs float64 {picks[tuple(wrong[0])].tolist()}"
    return differ.size, int(ambiguous.sum())


def _fused(torch, cams, roi, rng_words, *, max_p, min_p, k_fg, k_bg, weighted):
    """tcam_seed_fused with the given Philox key words (no draws passed in, counts computed in the kernel)."""
    _l, lib = _lib()
    b, t, h, w = cams.shape
    kmax = max(k_fg, k_bg, 1)
    dev = torch.device("cuda", 0)
    cams_d = cams.to(dev).contiguous()
    roi_d = None if roi is None else roi.to(dev).reshape(b, h * w).contiguous()
    rng = torch.tensor(rng_words, dtype=torch.int32, device=dev)
    cam_max = torch.empty((b, h, w), dtype=torch.float32, device=dev)
    sel = torch.empty((b, 2, kmax), dtype=torch.int32, device=dev)
    assert lib.tcam_seed_fused_supported(h * w, kmax) == 1
    _l.check(lib.tcam_seed_fused(cams_d.data_ptr(), t, None if roi_d is None else roi_d.data_ptr(), None, None, None,
                                 rng.data_ptr(), float(np.float32(max_p)), int(max_p * h * w) if k_fg > 0 else 0,
                                 int(min_p * h * w) if k_bg > 0 else 0, k_fg, k_bg, int(weighted), b, h, w, 3, -255,
                                 cam_max.data_ptr(), sel.data_ptr(), kmax, None, _stream(torch)), "tcam_seed_fused")
    return sel.cpu().numpy().astype(np.int64), cam_max.cpu().numpy()


def test_philox_words_and_draws_vs_numpy(torch_cuda):
    """tcam_debug_seed_draws (the device functions seed_fused_kernel calls) against the numpy Philox: every word bit
    for bit over B = 64 samples x 2 sides x 224^2 pixels, every draw within 2 ulps of float64 -log(u)."""
    torch = torch_cuda
    _l, lib = _lib()
    b_n, hw = 64, 224 * 224
    torch.manual_seed(2024)
    keys = [(0, 0), (2 ** 31 - 2, 2 ** 31 - 2)] + \
        [tuple(torch.randint(0, 2 ** 31 - 1, (2,), dtype=torch.int32).tolist()) for _ in range(2)]
    words = torch.empty(b_n * 2 * hw, dtype=torch.int32, device="cuda")
    draws = torch.empty(b_n * 2 * hw, dtype=torch.float32, device="cuda")
    bs = np.repeat(np.arange(2 * b_n, dtype=np.uint64), hw)
    pix = np.tile(np.arange(hw, dtype=np.uint64), 2 * b_n)
    for key in keys:
        rng = torch.tensor(key, dtype=torch.int32, device="cuda")
        _l.check(lib.tcam_debug_seed_draws(rng.data_ptr(), b_n, hw, words.data_ptr(), draws.data_ptr(), _stream(torch)),
                 "tcam_debug_seed_draws")
        got_w = words.cpu().numpy().view(np.uint32)
        got_d = draws.cpu().numpy()
        want_w = sd.philox4x32_10((pix, bs, 0x5EED, 0), key)[0]
        assert np.array_equal(got_w, want_w), (key, int(np.argmax(got_w != want_w)))
        assert np.array_equal(sd.seed_words(key, 3, 1, np.arange(hw)), want_w[7 * hw:8 * hw])
        want_d = sd.exp_draw_f64(want_w, BITS)
        ok = _within_ulps(got_d, want_d, 2)
        assert ok.all(), (key, got_d[~ok][:4].tolist(), want_d[~ok][:4].tolist())


def test_exp_transform_exhaustive(torch_cuda):
    """tcam_debug_exp_draws on one word per value the transform can see (m = word >> (32 - bits), random low bits):
    every draw finite and > 0, within 2 ulps of float64 -log((m + 0.5) / 2^bits), non-increasing in m."""
    torch = torch_cuda
    _l, lib = _lib()
    n = 1 << BITS
    m = np.arange(n, dtype=np.uint32)
    low = np.random.default_rng(5).integers(0, 1 << (32 - BITS), size=n, dtype=np.uint32)
    words = (m << np.uint32(32 - BITS)) | low
    words_d = torch.from_numpy(words.view(np.int32)).cuda()
    draws_d = torch.empty(n, dtype=torch.float32, device="cuda")
    _l.check(lib.tcam_debug_exp_draws(words_d.data_ptr(), n, draws_d.data_ptr(), _stream(torch)), "tcam_debug_exp_draws")
    got = draws_d.cpu().numpy()
    want = sd.exp_draw_f64(words, BITS)
    bad = np.flatnonzero(~(np.isfinite(got) & (got > 0)))
    assert bad.size == 0, f"{bad.size} draws not finite and > 0, first at m = {bad[:4].tolist()}: {got[bad[:4]].tolist()}"
    ok = _within_ulps(got, want, 2)
    assert ok.all(), f"{int((~ok).sum())} draws beyond 2 ulps, first at m = {np.flatnonzero(~ok)[:4].tolist()}"
    assert (np.diff(got) <= 0).all(), np.flatnonzero(np.diff(got) > 0)[:4]


# (k_fg, k_bg, weighted, use_roi, quantised)
SELECT_CONFIGS = [(1, 1, True, True, False),      # README recipe
                  (3, 5, False, True, False),
                  (4, 3, True, False, True),
                  (32, 32, True, True, True),      # kSeedFusedMaxK
                  (32, 32, False, False, False)]
SELECT_SHAPES = [(32, 5, 224, 224), (8, 1, 37, 53), (64, 1, 8, 5)]   # 37 x 53: HW % 4 != 0; 8 x 5: n_cand < k
EDGE_KEYS = [(0, 0), (2 ** 31 - 2, 2 ** 31 - 2)]                        # the first configs' keys; then random ones


def test_fused_selection_vs_float64(torch_cuda):
    """seed_fused_kernel's picks against top-k of val / draw in float64 with the same Philox words, over shapes, k,
    weighted / uniform sampling, quantised CAMs, an empty roi, roi = None and a flat sample.  A (sample, side) may differ
    only where two adjacent float64 scores among the first k + 1 are closer than 2^-20 relative, and such near-ties
    must stay below 0.1 % of the cases."""
    torch = torch_cuda
    max_p, min_p = 0.6, 0.1
    key_rng = np.random.default_rng(77)
    cases = amb = exact = 0
    for ci, (k_fg, k_bg, weighted, use_roi, quantised) in enumerate(SELECT_CONFIGS):
        for si, (b, t, h, w) in enumerate(SELECT_SHAPES):
            cams, roi = _cams(torch, b, t, h, w, seed=10 * ci + si, quantised=quantised)
            cams[1] = -1.0                                   # flat: no seeds at all
            roi[2] = 0                                       # empty roi: no fg candidates
            rng = EDGE_KEYS[ci] if ci < len(EDGE_KEYS) else tuple(int(x) for x in key_rng.integers(0, 2 ** 31 - 1, 2))
            r = roi if use_roi else None
            sel, cam_max = _fused(torch, cams, r, rng, max_p=max_p, min_p=min_p, k_fg=k_fg, k_bg=k_bg, weighted=weighted)
            assert np.array_equal(cam_max, cams.amax(dim=1).numpy())
            picks, ambiguous, ties = _expected(cam_max, None if r is None else r[:, 0].numpy(), rng, max_p=max_p,
                                               min_p=min_p, k_fg=k_fg, k_bg=k_bg, weighted=weighted)
            assert (sel[1] == -1).all() and (use_roi is False or (sel[2, 0] == -1).all())
            c, a = _compare(sel, picks, ambiguous, f"config {ci} shape {(b, t, h, w)}")
            cases, amb, exact = cases + c, amb + a, exact + ties
    print(f"fused path: {cases} (sample, side) cases, {amb} float64 near-ties, {exact} with an exact tie")
    assert amb <= 0.001 * cases, (amb, cases)


def test_fused_selection_through_the_seeder(torch_cuda):
    """The same comparison through TCAMSeeder(rng_parity=False).forward_stack: the key words are the two that _select
    draws from torch's CUDA generator, replayed here after the same torch.manual_seed."""
    torch = torch_cuda
    b, t, h, w = 32, 5, 224, 224
    cams, roi = _cams(torch, b, t, h, w, seed=3)
    seeder = _seeder(max_=4, min_=3)
    torch.manual_seed(8)
    seeds, cam_max = seeder.forward_stack(cams.cuda(), roi.cuda(), sparse=True)
    torch.manual_seed(8)
    rng = torch.randint(0, 2 ** 31 - 1, (2,), dtype=torch.int32, device="cuda").tolist()
    picks, ambiguous, _ = _expected(cam_max.cpu().numpy(), roi[:, 0].numpy(), rng, max_p=0.6, min_p=0.1, k_fg=4, k_bg=3,
                                    weighted=True)
    _compare(seeds.sel.cpu().numpy().astype(np.int64), picks, ambiguous, "TCAMSeeder.forward_stack")


def test_u_rounding_to_one_regression(torch_cuda):
    """Key (2770, 12345), sample 0, background: pixel 2490's word is 0xffffff31, whose top 24 bits are all ones --
    with u = (m + 0.5) / 2^24 computed in float32 that u rounded to 1.0, the draw to 0 and the score to -inf, so the
    pixel could never be picked.  Its true draw is ~6e-8 against 1.97 for the only other candidate (pixel 0)."""
    torch = torch_cuda
    rng = (2770, 12345)
    word = int(sd.seed_words(rng, 0, 1, 2490))
    assert word >> 8 == 0xFFFFFF
    assert sd.exp_draw_f64(sd.seed_words(rng, 0, 1, 0), 24) == pytest.approx(1.966, abs=1e-3)
    cams = torch.full((1, 1, 64, 64), 0.5)
    cams.view(-1)[[0, 2490]] = 0.0
    sel, _ = _fused(torch, cams, None, rng, max_p=0.0, min_p=2 / 4096, k_fg=0, k_bg=1, weighted=False)
    assert sel[0, 0, 0] == -1
    assert sel[0, 1, 0] == 2490, sel[0, 1].tolist()


# ((B, T, H, W), k_fg, k_bg, weighted): 224^2 and 37 x 53 take the shared-memory select kernel, 640^2 the other one
TWO_KERNEL_CASES = [((32, 5, 224, 224), 1, 1, True), ((64, 1, 37, 53), 5, 3, False), ((64, 1, 8, 5), 32, 32, True),
                    ((2, 1, 640, 640), 32, 32, True)]


def test_two_kernel_path_selection_vs_float64(torch_cuda, monkeypatch):
    """rng_parity=False on the two-kernel path (tcam_seed_select: the fused kernel refused, or a frame above its limit):
    the draws are torch's exponential_ over b*2*h*w slots, candidate r of (sample, side) uses slot (2b + side)*HW + r.
    Replayed from the generator, the picks must match float64 top-k under the same near-tie rule."""
    torch = torch_cuda
    _l, lib = _lib()
    monkeypatch.setattr(lib, "tcam_seed_fused_supported", lambda hw, kmax: 0)
    cases = amb = exact = 0
    for i, ((b, t, h, w), k_fg, k_bg, weighted) in enumerate(TWO_KERNEL_CASES):
        cams, roi = _cams(torch, b, t, h, w, seed=40 + i, quantised=i == 1)
        if b > 2:
            cams[1] = 0.75                                   # flat: no seeds at all
        seeder = _seeder(max_=k_fg, min_=k_bg, seed_tech="seed_weighted" if weighted else "seed_uniform")
        torch.manual_seed(100 + i)
        seeds, cam_max = seeder.forward_stack(cams.cuda(), roi.cuda(), sparse=True)
        torch.manual_seed(100 + i)
        q = torch.empty(b * 2 * h * w, dtype=torch.float32, device="cuda").exponential_(1).cpu().numpy()
        hw = h * w
        picks, ambiguous, ties = _expected(cam_max.cpu().numpy(), roi[:, 0].numpy(), None, max_p=0.6, min_p=0.1,
                                           k_fg=k_fg, k_bg=k_bg, weighted=weighted,
                                           draws=lambda bb, side, n: q[(2 * bb + side) * hw:(2 * bb + side) * hw + n])
        c, a = _compare(seeds.sel.cpu().numpy().astype(np.int64), picks, ambiguous, f"two-kernel case {i}")
        cases, amb, exact = cases + c, amb + a, exact + ties
    print(f"two-kernel path: {cases} (sample, side) cases, {amb} float64 near-ties, {exact} with an exact tie")
    assert amb <= 0.001 * cases, (amb, cases)


FG_WEIGHTS = np.array([0.1, 0.15, 0.25, 0.4, 0.6, 1.0], dtype=np.float32)   # 10x span


def _distribution_cams(torch, b):
    """B identical 8x8 CAMs: 6 foreground candidates (max_p = 6/64) with FG_WEIGHTS, 5 background candidates
    (min_p = 5/64, the 5 lowest values), everything else in between."""
    cam = np.linspace(0.09, 0.06, 64, dtype=np.float32)
    fg_pix = np.array([3, 12, 21, 30, 45, 60])
    bg_pix = np.array([0, 17, 38, 50, 63])
    cam[fg_pix] = FG_WEIGHTS
    cam[bg_pix] = np.array([0.01, 0.02, 0.03, 0.04, 0.05], dtype=np.float32)
    cams = torch.from_numpy(np.broadcast_to(cam.reshape(1, 1, 8, 8), (b, 1, 8, 8)).copy())
    return cams, fg_pix, bg_pix


def _check_distribution(sels, fg_pix, bg_pix, k_fg, k_bg, weights, what):
    """sels: the [B,2,kmax] picks of consecutive calls on B identical samples.  Checks the pick frequencies against
    inclusion_probabilities (5.5 sigma), independence of neighbouring samples (mean overlap of their pick sets = sum of
    pi^2, 5.5 sigma) and of the fg and bg picks of a sample (chi-square p > 1e-6), and that calls do not repeat."""
    calls, b = len(sels), sels[0].shape[0]
    for c in range(1, calls):
        assert not np.array_equal(sels[c], sels[c - 1]), what
    sel = np.concatenate(sels)                                                 # [calls*B, 2, kmax]
    n = sel.shape[0]
    for side, pix, k, pi in ((0, fg_pix, k_fg, sd.inclusion_probabilities(weights, k_fg)),
                             (1, bg_pix, k_bg, sd.inclusion_probabilities(np.ones(bg_pix.size), k_bg))):
        picks = sel[:, side, :k]
        assert np.isin(picks, pix).all() and (sel[:, side, k:] == -1).all(), what
        assert (np.sort(picks, axis=1)[:, 1:] != np.sort(picks, axis=1)[:, :-1]).all(), what   # distinct
        onehot = (picks[:, :, None] == pix[None, None, :]).any(axis=1)                         # [n, candidates]
        freq = onehot.sum(axis=0)
        sigma = np.sqrt(n * pi * (1 - pi))
        assert (np.abs(freq - n * pi) <= 5.5 * sigma).all(), (what, side, freq.tolist(), (n * pi).tolist())
        # neighbours within a call, as disjoint pairs (0,1), (2,3), ... and (1,2), (3,4), ...: overlap of the sets
        per_call = onehot.reshape(calls, b, -1)
        for first in (0, 1):
            left, right = per_call[:, first:b - 1:2], per_call[:, first + 1::2]
            overlap = (left & right[:, :left.shape[1]]).sum(axis=2).reshape(-1).astype(np.float64)
            se = overlap.std() / np.sqrt(overlap.size)
            assert abs(overlap.mean() - (pi ** 2).sum()) <= 5.5 * se, (what, side, first, overlap.mean(), (pi ** 2).sum())
    # fg and bg of one sample: contingency table of the first fg pick and the first bg pick
    table = np.zeros((fg_pix.size, bg_pix.size))
    np.add.at(table, (np.searchsorted(fg_pix, sel[:, 0, 0]), np.searchsorted(bg_pix, sel[:, 1, 0])), 1)
    p = stats.chi2_contingency(table)[1]
    assert p > 1e-6, (what, p, table.tolist())


@pytest.mark.parametrize("path", ["fused", "two_kernel"])
def test_pick_distribution(torch_cuda, monkeypatch, path):
    """B = 4096 identical samples per call, 5 calls with a fixed torch seed, weighted fg (k = 1 and k = 3) and uniform
    bg (k = 2), through TCAMSeeder(rng_parity=False): see _check_distribution.  The seed is fixed, so the test is
    deterministic; it is aimed at plumbing errors (offsets, correlated streams, one side's weights on the other), the
    last bits are the other tests' job."""
    torch = torch_cuda
    if path == "two_kernel":
        _l, lib = _lib()
        monkeypatch.setattr(lib, "tcam_seed_fused_supported", lambda hw, kmax: 0)
    b, calls = 4096, 5
    cams, fg_pix, bg_pix = _distribution_cams(torch, b)
    cams = cams.cuda()
    weights = (FG_WEIGHTS + np.float32(1e-8)).astype(np.float64)   # the kernel's float32 cam + 1e-8
    for k_fg in (1, 3):
        seeder = _seeder(max_=k_fg, min_=2, max_p=6 / 64, min_p=5 / 64, use_roi=False)
        torch.manual_seed(1000 + k_fg)
        sels = [seeder.forward_stack(cams, None, sparse=True)[0].sel.cpu().numpy() for _ in range(calls)]
        _check_distribution(sels, fg_pix, bg_pix, k_fg, 2, weights, f"{path} k_fg={k_fg}")
