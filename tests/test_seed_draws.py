"""CPU suite: the float64 restatement of the seeder's in-kernel draws (oracle/seed_draws.py) against published
known answers, against oracle/seeding.py and against a Monte-Carlo of the sampling it describes."""
import numpy as np
import pytest
import torch

from oracle import seed_draws as sd
from oracle import seeding


@pytest.mark.parametrize("counter,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
])
def test_philox_known_answers(counter, key, want):
    """Random123's known-answer vectors for Philox4x32-10 (kat_vectors), scalar and broadcast over an array."""
    got = sd.philox4x32_10(counter, key)
    assert tuple(int(x) for x in got) == want
    wide = sd.philox4x32_10([np.full(3, c, dtype=np.uint32) for c in counter], key)
    assert all(np.array_equal(w, np.full(3, v, dtype=np.uint32)) for w, v in zip(wide, want))


def test_seed_words_counter_layout():
    """seed_words = word 0 of Philox at (pixel, 2b + side, 0x5eed, 0), vectorised over pixels and samples."""
    rng = (2770, 12345)
    pix = np.arange(5000)
    for b, side in ((0, 0), (0, 1), (7, 1)):
        want = sd.philox4x32_10((pix, np.full_like(pix, 2 * b + side), 0x5EED, 0), rng)[0]
        assert np.array_equal(sd.seed_words(rng, b, side, pix), want)
    assert int(sd.seed_words(rng, 0, 1, 2490)) == 0xFFFFFF31   # the draw that rounded to u = 1 before bits = 23


def test_exp_draw_f64_edges():
    top = np.uint32(0xFFFFFFFF)
    for bits in (23, 24):
        assert sd.exp_draw_f64(top, bits) == pytest.approx(2.0 ** -(bits + 1), rel=1e-12)   # -log(1 - 2^-(bits+1))
        assert sd.exp_draw_f64(np.uint32(0), bits) == pytest.approx((bits + 1) * np.log(2.0), rel=1e-15)
    # the low 32 - bits bits of the word are ignored; draws decrease with m
    w = (np.arange(1 << 10, dtype=np.uint32) << np.uint32(22)) | np.uint32(0x2A5A5)
    d = sd.exp_draw_f64(w, 10)
    assert np.array_equal(d, sd.exp_draw_f64(w & np.uint32(0xFFC00000), 10))
    assert (np.diff(d) < 0).all() and (d > 0).all()


@pytest.mark.parametrize("use_roi", [True, False])
def test_candidates_match_the_seeding_restatement(use_roi):
    """Quantised CAMs (most n-th values tie): the candidate sets are what sample_fg / sample_bg draw from -- with
    max_ >= n both pick every candidate."""
    g = torch.Generator().manual_seed(4)
    for trial in range(6):
        h, w = (13, 17) if trial % 2 else (24, 20)
        cam = torch.randint(0, 4, (h, w), generator=g).float() / 4
        roi = (torch.rand((h, w), generator=g) > 0.4).long() if use_roi else None
        if trial == 5 and use_roi:
            roi[:] = 0                                   # empty roi: no fg candidates
        max_p, min_p = 0.3 + 0.05 * trial, 0.1 + 0.03 * trial
        fg, bg, wts = sd.candidates(cam.numpy(), None if roi is None else roi.numpy(), max_p=max_p, min_p=min_p,
                                    max_=1, min_=1)
        big = h * w
        want_fg = seeding.sample_fg(cam, roi, torch.zeros((h, w), dtype=torch.long), max_p, big, seeding.SEED_UNIFORM)
        want_bg = seeding.sample_bg(cam, torch.zeros((h, w), dtype=torch.long), min_p, big)
        assert np.array_equal(fg, want_fg.reshape(-1).nonzero().flatten().numpy())
        assert np.array_equal(bg, want_bg.reshape(-1).nonzero().flatten().numpy())
        n_fg = int(max_p * (roi.sum() if roi is not None else h * w))
        assert fg.size == n_fg and bg.size == int(min_p * h * w)
        score = (cam * roi if roi is not None else cam) + 1e-8
        assert np.array_equal(wts, score.reshape(-1)[fg].numpy())
    flat = np.full((8, 8), 0.25, dtype=np.float32)
    assert all(x.size == 0 for x in sd.candidates(flat, None, max_p=0.5, min_p=0.5, max_=1, min_=1))
    fg, bg, _ = sd.candidates(np.arange(64, dtype=np.float32).reshape(8, 8), None, max_p=0.5, min_p=0.5, max_=0,
                              min_=1)
    assert fg.size == 0 and bg.size == 32


def test_select_f64_order_ties_and_gaps():
    pixels = np.array([9, 3, 5, 7])
    picks, gaps = sd.select_f64(pixels, np.ones(4), np.array([0.5, 0.25, 0.5, 2.0]), 3)
    assert picks.tolist() == [3, 5, 9]                   # scores 4, 2, 2, 0.5: the tie goes to the lower pixel
    assert gaps.tolist() == [0.5, 0.0, 0.75]
    picks, gaps = sd.select_f64(pixels, np.array([1.0, 1.0, 8.0, 1.0]), np.ones(4), 9)   # k > n
    assert picks.tolist() == [5, 3, 7, 9] and gaps.size == 3


@pytest.mark.parametrize("weights,k", [([1, 2, 3, 4, 5, 10], 1), ([1, 2, 3, 4, 5, 10], 3),
                                       ([0.1, 0.15, 0.25, 0.4, 0.6, 1.0, 0.3, 0.2], 2), ([1, 1, 1, 1, 1], 2)])
def test_inclusion_probabilities_vs_exponential_race(weights, k):
    """Exact inclusion probabilities against a float64 Monte-Carlo of the exponential race (top-k of w / E,
    E ~ Exp(1)); each vector sums to k."""
    w = np.asarray(weights, dtype=np.float64)
    pi = sd.inclusion_probabilities(w, k)
    assert pi.sum() == pytest.approx(k, abs=1e-12)
    assert ((pi > 0) & (pi <= 1 + 1e-12)).all()
    n_mc = 200_000
    e = np.random.default_rng(12).exponential(size=(n_mc, w.size))
    top = np.argsort(-(w / e), axis=1, kind="stable")[:, :k]
    freq = np.bincount(top.reshape(-1), minlength=w.size) / n_mc
    sigma = np.sqrt(pi * (1 - pi) / n_mc)
    assert (np.abs(freq - pi) <= 5.5 * sigma + 1e-12).all(), (freq, pi)
    if np.allclose(w, w[0]):
        assert np.allclose(pi, k / w.size)
