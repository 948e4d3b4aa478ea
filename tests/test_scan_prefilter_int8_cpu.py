"""The tensor-core scan (csrc/scan_tc.cuh) multiplies an int8 table Q, the exact integer form of the real-valued filter D_real that
tests/test_scan_prefilter_cpu.py checks (column 0 = entries minus t' rounded up to Float16, then the remaining columns):

    Q[j][b] = ceil(2^e * f[j][b]) + k[j],   sum_j k[j] = 0,   Q in [-128, 127]

so that the int32 window sum is >= 2^e * D_real, and every true hit (D_real > 0) gives a sum >= 1.  The library exposes the table
(mb200_scan_prefilter_int8, host arithmetic only); these tests check the inequality and the hit implication exhaustively over all
4^len windows for short motifs and on windows biased towards the threshold for long ones, that nothing was rounded down, and that
the rounding up keeps the candidates per hit of the benchmark's scan (500 PWMs of length 8-40) low."""
import itertools

import numpy as np
import pytest

from motifs_jl_b200 import _lib, synth

f16 = np.float16


def seq_f16(vals):
    """left-to-right Float16 running sum of the rows of vals (n_windows, len)"""
    s = np.zeros(vals.shape[0], f16)
    for j in range(vals.shape[1]):
        s = (s.astype(np.float32) + vals[:, j].astype(np.float32)).astype(f16)
    return s


def real_filter(cols, thr):
    """the real-valued filter f (len, 4) float64 and t, or None when the slot is disabled"""
    E, tp, col0, possible = _lib.scan_prefilter_bound(cols, thr)
    if not possible:
        return None
    f = cols.astype(np.float64).copy()
    f[0] = col0.astype(np.float64)
    return f


def check(cols, thr, idx):
    """cols (len, 4) float16, idx (n_windows, len) base indices -> (true hits, real-filter candidates, int8 candidates)"""
    n = cols.shape[0]
    vals = cols[np.arange(n)[None, :], idx]
    hit = seq_f16(vals).astype(np.float64) > max(float(f16(thr)), 0.0)
    f = real_filter(cols, thr)
    q8 = _lib.scan_prefilter_int8(cols, thr)
    if f is None:
        assert q8 is None and not hit.any()
        return 0, 0, 0
    e, k, Q = q8
    Q = Q.astype(np.int64)
    s = 2.0 ** e
    assert k.sum() == 0
    assert Q.min() >= -128 and Q.max() <= 127
    assert (Q - k[:, None] >= np.ceil(s * f)).all(), "an entry was rounded down"
    D = f[np.arange(n)[None, :], idx].sum(axis=1)                                  # exact in float64
    DQ = Q[np.arange(n)[None, :], idx].sum(axis=1)
    assert (DQ >= s * D).all()
    assert (DQ[hit] > 0).all(), "a true hit is not a candidate of the int8 filter"
    return int(hit.sum()), int((D > 0).sum()), int((DQ > 0).sum())


@pytest.mark.parametrize("seed", range(6))
def test_exhaustive_short_motifs(seed):
    rng = np.random.default_rng(seed)
    for length in (1, 2, 3, 5, 8, 9):
        cm = synth.random_count_matrices(1, length, length, 100 * seed + length)[0]
        pwm = synth.motifs_from_count_matrices([cm]).pwms[0]                       # (4, len) float16
        if seed % 2:
            pwm = (pwm.astype(np.float32) * rng.choice([0.03, 7.0, 16.0, 40.0])).astype(f16)
        cols = np.ascontiguousarray(pwm.T)
        idx = np.array(list(itertools.product(range(4), repeat=length)), np.int64)
        best = float(cols.astype(np.float32).max(axis=1).sum())
        for frac in (0.0, 0.3, 0.7, 0.95, 1.0, 1.2):
            h, c16, c8 = check(cols, f16(frac * best), idx)
            assert c8 >= c16 >= h


@pytest.mark.parametrize("seed", range(5))
def test_sampled_long_motifs_near_the_threshold(seed):
    rng = np.random.default_rng(10 + seed)
    scale = (1.0, 0.03, 7.0, 16.0, 40.0)[seed]
    for length in (16, 33, 40, 64):
        cm = synth.random_count_matrices(1, length, length, 7 * seed + length)[0]
        pwm = synth.motifs_from_count_matrices([cm]).pwms[0]
        pwm = (pwm.astype(np.float32) * scale).astype(f16)
        cols = np.ascontiguousarray(pwm.T)
        w = cols.astype(np.float64)
        pr = np.exp2(np.clip((w - w.max(axis=1, keepdims=True)) / max(scale, 1e-3), -30, 0) * rng.choice([0.5, 1.0, 2.0]))
        pr /= pr.sum(axis=1, keepdims=True)
        mix = 0.7 * pr + 0.3 * 0.25
        idx = np.stack([rng.choice(4, size=100_000, p=mix[j]) for j in range(length)], axis=1)
        best = float(w.max(axis=1).sum())
        total = 0
        for frac in (0.2, 0.5, 0.7, 0.9):
            h, c16, c8 = check(cols, f16(frac * best), idx)
            total += h
        assert total > 0


def test_very_negative_entries_do_not_coarsen_the_table():
    """log-odds near -Inf in one column only: entries that cannot reach a positive window are raised, not the scale lowered"""
    cm = synth.random_count_matrices(1, 20, 20, 5)[0]
    cols = np.ascontiguousarray(synth.motifs_from_count_matrices([cm]).pwms[0].T)
    best = float(cols.astype(np.float32).max(axis=1).sum())
    e0 = _lib.scan_prefilter_int8(cols, f16(0.7 * best))[0]
    cols[3, 1] = f16(-3000.0)
    idx = np.random.default_rng(0).integers(0, 4, size=(50_000, 20))
    idx[::2, 3] = 1
    check(cols, f16(0.7 * best), idx)
    assert _lib.scan_prefilter_int8(cols, f16(0.7 * best))[0] == e0


def test_disabled_slot():
    cols = np.full((5, 4), -1.0, f16)
    assert _lib.scan_prefilter_int8(cols, f16(0.5)) is None


def test_candidates_per_hit_of_the_benchmark_scan():
    """bench.py's scan sweep: 500 PWMs of length 8-40 (columns 1000 x Dirichlet(0.3)), both strands, 0.7 x the best score, on
    40 000 uniform random positions.  The FP16 filter had ~1.05 candidates per hit; the int8 rounding up costs < 1.5x that, far
    inside the candidate list (10x the hits of a batch)."""
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(500, 8, 40, 4))
    thr = synth.stated_thresholds(ms, 0.7)
    rng = np.random.default_rng(1)
    npos = 40_000
    seq = rng.integers(0, 4, npos + 40)
    hits = c16 = c8 = 0
    for k in range(500):
        pwm = np.asarray(ms.pwms[k], f16)
        for cols in (np.ascontiguousarray(pwm.T), np.ascontiguousarray(pwm[::-1, ::-1].T)):
            idx = np.lib.stride_tricks.sliding_window_view(seq, cols.shape[0])[:npos]
            h, a, b = check(cols, thr[k], idx)
            hits += h; c16 += a; c8 += b
    assert hits > 500
    assert c8 <= 1.5 * hits, (hits, c16, c8)
