"""oracle/seed_draws.py -- TEST INFRASTRUCTURE ONLY.

Float64 restatement of the seeder's in-kernel random draws (``TCAMSeeder(rng_parity=False)``, csrc/seed.cuh:
``seed_philox_word`` / ``exp1_from_word`` inside ``seed_fused_kernel``) and of the selection they drive, so that the
kernel can be compared with what it is meant to compute:

  philox4x32_10          Philox4x32-10 (Salmon et al., SC'11; Random123), vectorised over uint32 arrays
  seed_words             the kernel's counter layout: (pixel, 2*b + side, 0x5eed, 0), keyed by (rng[0], rng[1])
  exp_draw_f64           the Exp(1) draw -log(u) in float64 from the exact uniform u = (m + 0.5) / 2^bits,
                         m = word >> (32 - bits); the kernel uses bits = KERNEL_BITS
  candidates             the fg / bg candidate pixels of one sample, from oracle/seeding.py (_SFG / _SBG semantics)
  select_f64             top-k of val / draw in float64, ties to the lowest pixel index
  inclusion_probabilities  exact inclusion probabilities of successive sampling without replacement
                         (torch.multinomial(replacement=False)), by enumeration of the ordered k-tuples

Everything but ``candidates`` is numpy only.
"""
from __future__ import annotations

import itertools

import numpy as np

KERNEL_BITS = 23   # bits of the word exp1_from_word keeps: u = (2m + 1) * 2^-24 = (m + 0.5) / 2^23, m = word >> 9

_M0, _M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
_W0, _W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
_MASK = np.uint64(0xFFFFFFFF)
_SEED_TAG = 0x5EED


def philox4x32_10(counter, key):
    """counter: 4 uint32 arrays (broadcastable), key: 2 uint32 words or arrays -> 4 uint32 arrays."""
    c0, c1, c2, c3 = np.broadcast_arrays(*[np.asarray(c, dtype=np.uint64) & _MASK for c in counter])
    k0, k1 = [np.asarray(k, dtype=np.uint64) & _MASK for k in key]
    for _ in range(10):
        p0 = _M0 * c0   # < 2^64: the 64-bit product gives mulhi and mullo
        p1 = _M1 * c2
        c0, c1, c2, c3 = (p1 >> np.uint64(32)) ^ c1 ^ k0, p1 & _MASK, (p0 >> np.uint64(32)) ^ c3 ^ k1, p0 & _MASK
        k0 = (k0 + _W0) & _MASK
        k1 = (k1 + _W1) & _MASK
    return tuple(x.astype(np.uint32) for x in (c0, c1, c2, c3))


def seed_words(rng, b, side, pixel):
    """The word seed_fused_kernel draws from for (sample b, side 0 fg / 1 bg, pixel): first output word of Philox at
    counter (pixel, 2b + side, 0x5eed, 0) keyed by the two generator words rng (int32 values >= 0)."""
    pixel = np.asarray(pixel, dtype=np.uint64)
    bs = np.asarray(b, dtype=np.uint64) * np.uint64(2) + np.asarray(side, dtype=np.uint64)
    key = (np.uint64(int(rng[0]) & 0xFFFFFFFF), np.uint64(int(rng[1]) & 0xFFFFFFFF))
    return philox4x32_10((pixel, bs, np.uint64(_SEED_TAG), np.uint64(0)), key)[0]


def exp_draw_f64(word, bits=KERNEL_BITS):
    """-log(u) in float64, u = (m + 0.5) / 2^bits exactly, m = word >> (32 - bits).  1 - u is exact too, so log1p
    keeps full relative accuracy for u near 1, where the smallest draws (the ones that decide a pick) come from."""
    m = np.asarray(word, dtype=np.uint32).astype(np.uint64) >> np.uint64(32 - bits)
    one_minus_u = (np.float64(2.0 ** bits) - m.astype(np.float64) - 0.5) / 2.0 ** bits
    return -np.log1p(-one_minus_u)


def candidates(cam, roi, *, max_p, min_p, max_, min_):
    """(fg, bg) candidate pixel indices of one sample [h,w] in row-major order, exactly the sets _SFG / _SBG draw
    from (oracle/seeding.py: float32 cam*roi + 1e-8 or cam + 1e-8, stable sort, the first n; n = int(max_p * roi.sum())
    as a float32 product, int(max_p*h*w) without a roi, int(min_p*h*w) for the background; none for a flat CAM), and
    the float32 fg scores of the fg candidates (the weights of seed_weighted)."""
    import torch

    from . import seeding

    cam = torch.as_tensor(np.asarray(cam, dtype=np.float32))
    roi = None if roi is None else torch.as_tensor(np.asarray(roi, dtype=np.int64))
    none = np.zeros(0, dtype=np.int64)
    fg, bg, w = none, none, np.zeros(0, dtype=np.float32)
    if cam.min() == cam.max():                                       # _OneSample: no seeds for a flat CAM
        return fg, bg, w
    n, _cam, tmp = seeding.fg_candidates(cam, roi, max_p)
    if n > 0 and max_ > 0:
        fg = torch.nonzero(tmp.reshape(-1)).flatten().numpy()
        w = _cam.reshape(-1)[fg].numpy().astype(np.float32)
    n, tmp = seeding.bg_candidates(cam, min_p)
    if n > 0 and min_ > 0:
        bg = torch.nonzero(tmp.reshape(-1)).flatten().numpy()
    return fg, bg, w


def select_f64(pixels, vals, draws, k):
    """Top-k of vals / draws in float64 (torch.multinomial without replacement given the Exp(1) draws), ties to the
    lowest pixel.  Returns (picks: the k chosen pixels in the order the kernel writes them, gaps: relative differences
    (s_j - s_{j+1}) / s_j of adjacent scores among the first k + 1 in that order).  A gap at the rounding level of
    float32 scores makes the order ambiguous, not wrong.  A gap of exactly 0 comes from two candidates with the same
    value and the same draw (the draws take 2^KERNEL_BITS values): the kernel's float32 scores tie too and it takes
    the lower pixel, like this function."""
    pixels = np.asarray(pixels, dtype=np.int64)
    scores = np.asarray(vals, dtype=np.float64) / np.asarray(draws, dtype=np.float64)
    order = np.lexsort((pixels, -scores))
    k = min(int(k), pixels.size)
    top = scores[order[:k + 1]]
    gaps = (top[:-1] - top[1:]) / top[:-1] if top.size > 1 else np.zeros(0)
    return pixels[order[:k]], gaps


def inclusion_probabilities(weights, k):
    """P(i is among the k picks) when k items are drawn one after another without replacement, each with probability
    proportional to its weight among those left (torch.multinomial(weights, k, replacement=False)).  Exact sum over
    the ordered k-tuples: meant for n <= 8, k <= 3."""
    w = np.asarray(weights, dtype=np.float64)
    n = w.size
    assert 1 <= k <= n
    total = w.sum()
    pi = np.zeros(n)
    for tup in itertools.permutations(range(n), k):
        p, left = 1.0, total
        for i in tup:
            p *= w[i] / left
            left -= w[i]
        pi[list(tup)] += p
    return pi
