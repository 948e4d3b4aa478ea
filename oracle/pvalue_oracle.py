"""Oracle for the exact null distribution of the scan's Float16 score (csrc/pvalue.cu).  TEST INFRASTRUCTURE ONLY.

The library computes the survival function by a gather over ordered values with a binary search per base; this oracle runs the
forward form instead: the probability mass over all 65 536 Float16 bit patterns, pushed through each column with numpy float16
adds and np.add.at, then a reverse cumulative sum over the non-NaN values in value order (-0 merged with +0).  brute_survival
enumerates all 4^m windows for short PWMs.
"""
from __future__ import annotations

import itertools

import numpy as np

from .scan_oracle import _eff_table

_BITS = np.arange(65536, dtype=np.uint32).astype(np.uint16)
_VALS = _BITS.view(np.float16)
_NONNAN = ~np.isnan(_VALS)
# rank of every non-NaN pattern in value order (-Inf = 0, -0 and +0 share a rank, +Inf = NV - 1)
_RANK = np.where(_BITS & 0x8000, 0xFC00 - _BITS.astype(np.int64), _BITS.astype(np.int64) + 0x7C00)
NV = 63489


def eff_tables(pwm):
    """(forward, reverse) effective tables (4, m) float16 of a (4, m) PWM: the scan's Inf * 0 = NaN rule, reverse(pwm)."""
    p = np.asarray(pwm, np.float16)
    return _eff_table(p), _eff_table(p[::-1, ::-1])


def _survival_from_pmf(pmf):
    """pmf over bit patterns -> (65536,) S(t) = P(score >= t) by bit pattern, NaN at the NaN patterns."""
    by_rank = np.zeros(NV)
    np.add.at(by_rank, _RANK[_NONNAN], pmf[_NONNAN])
    S = np.cumsum(by_rank[::-1].astype(np.longdouble))[::-1].astype(np.float64)
    out = np.full(65536, np.nan)
    out[_NONNAN] = S[_RANK[_NONNAN]]
    return out


def survival(tab, bg):
    """Forward DP: tab (4, m) float16 effective table, bg (4,) -> (65536,) float64 survival by bit pattern."""
    tab = np.asarray(tab, np.float16)
    bg = np.asarray(bg, np.float64)
    pmf = np.zeros(65536)
    pmf[0] = 1.0                                             # the scan starts from s = +0
    for j in range(tab.shape[1]):
        new = np.zeros(65536)
        for b in range(4):
            with np.errstate(invalid="ignore", over="ignore"):
                nb = (_VALS + tab[b, j]).astype(np.float16).view(np.uint16)
            np.add.at(new, nb, pmf * bg[b])
        pmf = new
    return _survival_from_pmf(pmf)


def brute_survival(tab, bg):
    """The same by enumerating all 4^m windows (m <= 8): Float16 sums in column order from +0, float64 probabilities."""
    tab = np.asarray(tab, np.float16)
    bg = np.asarray(bg, np.float64)
    m = tab.shape[1]
    seqs = np.array(list(itertools.product(range(4), repeat=m)), np.int64).reshape(-1, m)
    s = np.zeros(len(seqs), np.float16)
    pr = np.ones(len(seqs))
    for j in range(m):
        with np.errstate(invalid="ignore", over="ignore"):
            s = (s + tab[seqs[:, j], j]).astype(np.float16)
        pr = pr * bg[seqs[:, j]]
    pmf = np.zeros(65536)
    np.add.at(pmf, s.view(np.uint16), pr)
    return _survival_from_pmf(pmf)


def rank(bits):
    """value-order rank of Float16 bit patterns (NaN patterns give meaningless ranks)."""
    return _RANK[np.asarray(bits, np.uint16)]


def dense_scores(tab, codes):
    """(N, L - m + 1) float16 scores of every window of equal-length code rows under one effective table."""
    tab = np.asarray(tab, np.float16)
    m = tab.shape[1]
    N, L = codes.shape
    s = np.zeros((N, max(L - m + 1, 0)), np.float16)
    for j in range(m):
        with np.errstate(invalid="ignore", over="ignore"):
            s = (s + tab[codes[:, j:j + s.shape[1]], j]).astype(np.float16)
    return s
