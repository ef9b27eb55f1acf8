"""oracle/lattice_matrix.py -- the permutohedral filter as a sparse float64 matrix.  TEST INFRASTRUCTURE ONLY.

A lattice (``oracle.Lattice``: offset, bary, nbr, M) fixes the whole filter of one frame as a linear operator:

    A  = alpha * W * B_d ... B_0 * W^T,        A^T = alpha * W * B_0^T ... B_d^T * W^T

* W is P x M with W[p, offset[p, r]] = bary[p, r] (splat = W^T, slice = W);
* B_j = I + (N1_j + N2_j) / 2 over all M vertices, the padding-only vertices of the reference's ghost pixels
  included; N1_j[v, nbr[j, v, 0]] = 1, and a missing neighbour (-1) adds nothing;
* alpha = 1 / (1 + 2^-d).

This is ``Permutohedral::compute`` (permutohedral.cpp:507-572) with every operation in float64 and no rounding
order, so it is the reference against which both the float32 C restatement (permuto_oracle.c) and the CUDA
kernels are measured.  The loss helpers restate dense_crf_loss.py:56-74 and the fused-softmax chain rule.
"""
from __future__ import annotations

from typing import List, Tuple

import numpy as np
import scipy.sparse as sp


def lattice_matrices(L) -> Tuple[sp.csr_matrix, List[sp.csr_matrix], float]:
    """(W [P, M], [B_0 .. B_d] each [M, M], alpha) in float64."""
    d, p, m = L.d, L.n, L.m
    rows = np.repeat(np.arange(p), d + 1)
    W = sp.csr_matrix((L.bary[:p].astype(np.float64).ravel(), (rows, L.offset[:p].ravel())), shape=(p, m))
    eye = sp.identity(m, dtype=np.float64, format="csr")
    B = []
    for j in range(d + 1):
        nb = L.nbr[j]
        rr, cc = [], []
        for side in (0, 1):
            ok = nb[:, side] >= 0
            rr.append(np.nonzero(ok)[0])
            cc.append(nb[ok, side])
        r, c = np.concatenate(rr), np.concatenate(cc)
        B.append((eye + sp.csr_matrix((np.full(len(r), 0.5), (r, c)), shape=(m, m))).tocsr())
    alpha = 1.0 / (1.0 + 2.0 ** -d)
    return W, B, alpha


class LatticeOperator:
    """The matrices of one lattice, kept for repeated applications."""

    def __init__(self, L):
        self.W, self.B, self.alpha = lattice_matrices(L)

    def apply(self, planes, transposed: bool = False) -> np.ndarray:
        """A S (or A^T S) for planes [K, P]; float64 [K, P]."""
        v = self.W.T @ np.asarray(planes, dtype=np.float64).reshape(-1, self.W.shape[0]).T   # [M, K]
        if transposed:
            for b in reversed(self.B):
                v = b.T @ v
        else:
            for b in self.B:
                v = b @ v
        return (self.alpha * (self.W @ v)).T


def apply(L, planes, transposed: bool = False) -> np.ndarray:
    """A S or A^T S in float64 for planes [K, P] through the lattice L."""
    return LatticeOperator(L).apply(planes, transposed)


def softmax64(logits, axis: int = 1) -> np.ndarray:
    z = np.asarray(logits, dtype=np.float64)
    z = z - z.max(axis=axis, keepdims=True)
    e = np.exp(z)
    return e / e.sum(axis=axis, keepdims=True)


def crf_loss64(segs, AS, n_norm: float, weight: float = 1.0) -> float:
    """weight * (-sum(segs * AS) / n_norm) (dense_crf_loss.py:63-64, 118-122)."""
    return float(weight * (-(np.asarray(segs, np.float64) * np.asarray(AS, np.float64)).sum() / n_norm))


def crf_grad_reference64(AS, n_norm: float, grad_out: float = 1.0, weight: float = 1.0) -> np.ndarray:
    """The reference's backward -2 * g * w * AS / N (dense_crf_loss.py:73), which treats A as symmetric."""
    return -2.0 * grad_out * weight * np.asarray(AS, np.float64) / n_norm


def crf_grad_exact64(AS, AtS, n_norm: float, grad_out: float = 1.0, weight: float = 1.0) -> np.ndarray:
    """The true gradient of crf_loss64: -(g * w / N) (A + A^T) S."""
    return -(grad_out * weight / n_norm) * (np.asarray(AS, np.float64) + np.asarray(AtS, np.float64))


def logits_grad64(probs, G, axis: int = 1) -> np.ndarray:
    """Chain rule through softmax: dz = p * (G - sum_j p_j G_j)."""
    p = np.asarray(probs, np.float64)
    G = np.asarray(G, np.float64)
    return p * (G - (p * G).sum(axis=axis, keepdims=True))
