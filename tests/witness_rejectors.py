"""The correspondence rejectors of PCL 1.10 (MedianDistance, OneToOne, Trimmed, Distance) restated a SECOND time, in numpy,
from the semantics in include/pe_b200.h : peb_rejector (not from tests/rejector_oracle.cpp : reject_chain), plus witness.ICP
with a rejector chain.  TEST INFRASTRUCTURE, like tests/witness.py.

Order statistics by np.partition, the one-to-one and trimmed orders by np.lexsort; float32 where PCL computes in float."""
from __future__ import annotations

import numpy as np

import witness as W

F = np.float32
DISTANCE, MEDIAN_DISTANCE, ONE_TO_ONE, TRIMMED = range(4)


def median_score(src: np.ndarray, tgt: np.ndarray) -> np.ndarray:
    """(src - tgt).squaredNorm() of two Vector4f (w = 1 on both sides) with Eigen's 4-lane association (v0 + v2) + (v1 + v3)."""
    d = np.asarray(src, F)[:, :3] - np.asarray(tgt, F)[:, :3]
    return ((d[:, 0] * d[:, 0] + d[:, 2] * d[:, 2]) + (d[:, 1] * d[:, 1] + F(0))).astype(F)


def reject(q, m, d2, score, chain) -> np.ndarray:
    """Positions of the pairs the chain leaves, in the order it leaves them (q: source, m: target, d2, score per pair)."""
    q, m = np.asarray(q, np.int64), np.asarray(m, np.int64)
    d2, score = np.asarray(d2, F), np.asarray(score, F)
    idx = np.arange(len(q))
    for r in chain:
        kind, value = r[0], float(r[1]) if len(r) > 1 else 0.0
        min_corr = int(r[2]) if len(r) > 2 else 0
        if kind == DISTANCE:
            idx = idx[d2[idx] < F(value * value)]
        elif kind == MEDIAN_DISTANCE:
            if len(idx) == 0:
                continue
            s = score[idx].astype(np.float64)
            med = np.partition(s, len(s) // 2)[len(s) // 2]
            idx = idx[s <= med * value]
        elif kind == ONE_TO_ONE:
            o = idx[np.lexsort((q[idx], d2[idx], m[idx]))]  # by target, then distance, then source
            first = np.ones(len(o), bool)
            first[1:] = m[o][1:] != m[o][:-1]
            idx = o[first]
        elif kind == TRIMMED:
            ratio = F(min(1.0, max(0.0, float(F(value)))))
            n_keep = max(int(np.floor(ratio * F(len(idx)))), min_corr)
            if n_keep < len(idx):
                idx = idx[np.lexsort((q[idx], d2[idx]))][:max(n_keep, 0)]
        else:
            raise ValueError(f"unknown rejector kind {kind}")
    return idx


class ICP(W.ICP):
    """witness.ICP whose correspondences also go through a rejector chain ((kind, value[, min_corr]) tuples)."""

    def __init__(self, target, normals=None, chain=()):
        super().__init__(target, normals)
        self.chain = list(chain)

    def correspondences(self, work, valid, max_corr_dist, rejector_max_dist):
        q, m, d2 = super().correspondences(work, valid, max_corr_dist, rejector_max_dist)
        k = reject(q, m, d2, median_score(work[q], self.tgt[m]), self.chain)
        return q[k], m[k], d2[k]
