"""Host-side mirror of the reference's scan / threshold / count / Fisher entry points (SURVEY §8a part 2).

Function names, argument meaning and result conventions follow the reference (paths under its src/):
  get_pos_scores_arr, gpu_scan, scan_w_gpu!      inference/_h3_1_alignment.jl:57-112
  motifs_prep, countmat2pfm, freq2pwm            inference/_s1_make_motifs.jl:68-76,185-190
  get_best_thresh, filter_position_by_best_thresh!, filter_positions_scores_usecomp!
                                                 inference/_s2_filter_pos_w_scores.jl:90-138
  pvalue2score                                   inference/_h2_Touzet.jl:170-187
  get_uniq_pos, get_uniq_counts, get_union_ranges, get_total_occupied_positions
                                                 inference/_h4_overlap_ratio.jl:5-15,40-79
  active_counts_position, fisher_pvec, get_fisher_p_values   inference/_h7_fisher.jl:1-44
  pvec_from_test_data                            render/pvec_calculations.jl:1-22

Like the reference, results are 1-BASED (sequence numbers and start positions) and grouped as
`positions[m][n]` dictionaries; the C ABI underneath is 0-based.  All scoring happens in
libmotifs_b200 on the GPU — this module only marshals and post-processes (Float64 statistics on K values).
Julia's `!` suffix is spelled `_` (scan_w_gpu_ = scan_w_gpu!).
"""
from __future__ import annotations

import math
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

from . import _lib

f16, f32 = np.float16, np.float32

# inference/_0_const.jl
max_pwm_length_Touzet2 = 15
pvalue_Touzet_large, pvalue_Touzet_mid, pvalue_Touzet_small = 0.0001, 0.0001, 0.0003
score_thresh_increment = f16(0.5)
_granularity_ = 1e-1
effective_pos_ic_thresh = 0.5
mv_avg_window = 3


# ---------------------------------------------------------------------------------------------
# motifs struct (inference/_s1_make_motifs.jl:1-18) — the fields the hot path reads and writes
# ---------------------------------------------------------------------------------------------
@dataclass
class Motifs:
    pwms: List[np.ndarray]                                  # each (4, len) float16
    lens: np.ndarray                                        # int64
    cmats: Optional[List[np.ndarray]] = None
    pfms: Optional[List[np.ndarray]] = None
    effective_segments: Optional[List[List[range]]] = None  # 1-based inclusive ranges, as Julia UnitRange
    max_effective_lens: Optional[np.ndarray] = None
    max_scores: Optional[np.ndarray] = None
    min_scores: Optional[np.ndarray] = None
    score_thresh: Optional[np.ndarray] = None               # float16
    positions: Optional[List[Dict[int, np.ndarray]]] = None
    scores: Optional[List[Dict[int, np.ndarray]]] = None
    use_comp: Optional[List[Dict[int, np.ndarray]]] = None
    positions_bg: Optional[List[Dict[int, np.ndarray]]] = None
    scores_bg: Optional[List[Dict[int, np.ndarray]]] = None
    use_comp_bg: Optional[List[Dict[int, np.ndarray]]] = None
    # library-side occurrence counts of the last filtered scan, keyed (bg, test) -> (K,4) int64
    _counts: dict = field(default_factory=dict)

    @property
    def num_motifs(self) -> int:
        return len(self.pwms)


def countmat2pfm(count_matrix, ps=f16(0.01)):
    """Float16((cnt + ps) ./ (colsum + 4ps)) — _s1_make_motifs.jl:68-74 (all Float16 arithmetic)."""
    cm = np.asarray(count_matrix, f16)
    colsum = np.zeros(cm.shape[1], f16)
    for a in range(cm.shape[0]):
        colsum = (colsum + cm[a]).astype(f16)
    with np.errstate(all="ignore"):
        return ((cm + f16(ps)).astype(f16) / (colsum + f16(f16(4) * f16(ps))).astype(f16)[None, :]).astype(f16)


def freq2pwm(pfm, bg):
    """log2.(pfm ./ bg), bg Float32 — _s1_make_motifs.jl:76; stored as Float16."""
    with np.errstate(all="ignore"):
        return np.log2(np.asarray(pfm, f16).astype(f32) / np.asarray(bg, f32).reshape(4, 1)).astype(f32).astype(f16)


def cmat2ic(cmat, bg=(0.25, 0.25, 0.25, 0.25), ps=f16(0.0001)):
    """inference/_h0_trim.jl:1-5: Float16 frequencies, Float64 information content per column."""
    c = (np.asarray(cmat, f16) + f16(ps)).astype(f16)
    colsum = np.zeros(c.shape[1], f16)
    for a in range(4):
        colsum = (colsum + c[a]).astype(f16)
    with np.errstate(all="ignore"):
        freq = (c / colsum[None, :]).astype(f16).astype(np.float64)
        return (freq * np.log2(freq / np.asarray(bg, np.float64).reshape(4, 1))).sum(axis=0)


def get_high_ic_segments(ic_vec, m=mv_avg_window, ic_threshold=effective_pos_ic_thresh):
    """_s1_make_motifs.jl:24-48: moving average (window m) > threshold -> maximal runs, 1-based inclusive ranges."""
    v = np.asarray(ic_vec, np.float64)
    n = len(v)
    h = m // 2
    mv = np.array([v[max(0, i - h):min(n, i + h + 1)].mean() for i in range(n)])
    bits = np.concatenate([[False], mv > ic_threshold, [False]])
    d = np.diff(bits.astype(np.int8))
    starts = np.nonzero(d > 0)[0] + 1
    ends = np.nonzero(d < 0)[0]
    return [range(int(s), int(e) + 1) for s, e in zip(starts, ends)]


def countmats2motifs(count_mats, bg) -> Motifs:
    """_s1_make_motifs.jl:100-125 (without the empty-segment filter's re-indexing side effects)."""
    pfms = [countmat2pfm(c) for c in count_mats]
    pwms = [freq2pwm(p, bg) for p in pfms]
    segs = [get_high_ic_segments(cmat2ic(c)) for c in count_mats]
    keep = [i for i, s in enumerate(segs) if len(s) > 0]
    return Motifs(pwms=[pwms[i] for i in keep], lens=np.array([pwms[i].shape[1] for i in keep], np.int64),
                  cmats=[np.asarray(count_mats[i], f16) for i in keep], pfms=[pfms[i] for i in keep],
                  effective_segments=[segs[i] for i in keep],
                  max_effective_lens=np.array([max(len(r) for r in segs[i]) for i in keep], np.int64))


def motifs_prep(ms: Motifs):
    K = ms.num_motifs
    return [dict() for _ in range(K)], [dict() for _ in range(K)], [dict() for _ in range(K)]


def pack_pwms(ms: Motifs):
    """pwms = zeros(Float16, K, 4, maxlen); pwms[i,:,1:len_i] = ms.pwms[i]  (_h3_1_alignment.jl:65-69).
    Returned in Julia memory order, i.e. numpy shape (maxlen, 4, K)."""
    K = ms.num_motifs
    maxlen = int(np.max(ms.lens))
    out = np.zeros((maxlen, 4, K), f16)
    for k, p in enumerate(ms.pwms):
        out[: p.shape[1], :, k] = np.asarray(p, f16).T
    return out


def _which(data, bg=False, test=False):
    """data_(data; test) / data_bg(data; test)  (_h3_1_alignment.jl:54-55)."""
    if bg:
        return data.seqs_bg_test if test else data.seqs_bg
    return data.seqs_test if test else data.seqs


def _scan_raw(ms: Motifs, data, *, fwd, rc, bg, test, thresh=None, want_hits=True, want_counts=False):
    seqs = _which(data, bg=bg, test=test)
    return seqs.ctx.scan(seqs, pack_pwms(ms), ms.lens, thresh, fwd=fwd, rc=rc, want_hits=want_hits, want_counts=want_counts)


def get_pos_scores_arr(ms: Motifs, data, rc=False, bg=False, test=False):
    """-> (found_record (n,3) uint32 rows (motif, seq, pos) 1-based, score_record float16).
    The reference returns records in `findall` order of a (K, Nb, 4L) tensor per batch of 5000; the order
    here is (seq, motif, pos), which builds the same per-(motif, seq) lists in modify_w_found!."""
    hits, _ = _scan_raw(ms, data, fwd=not rc, rc=rc, bg=bg, test=test)
    rec = np.stack([hits["motif"].astype(np.uint32) + 1, hits["seq"] + 1, hits["pos"] + 1], axis=1).astype(np.uint32)
    return rec, hits["score_f16"].view(f16)


def _hits_to_dicts(hits, K):
    positions, scores, use_comp = [dict() for _ in range(K)], [dict() for _ in range(K)], [dict() for _ in range(K)]
    if len(hits) == 0:
        return positions, scores, use_comp
    order = np.argsort(hits["motif"], kind="stable")           # keeps (seq, comp, pos) order inside a motif
    h = hits[order]
    key = h["motif"].astype(np.int64) * (1 << 32) + h["seq"].astype(np.int64)
    cut = np.nonzero(np.diff(key))[0] + 1
    starts = np.concatenate([[0], cut])
    ends = np.concatenate([cut, [len(h)]])
    pos1 = h["pos"].astype(np.int64) + 1
    sc = h["score_f16"].view(f16)
    cp = h["comp"].astype(bool)
    for s, e in zip(starts, ends):
        m, n = int(h["motif"][s]), int(h["seq"][s]) + 1
        positions[m][n] = pos1[s:e].copy()
        scores[m][n] = sc[s:e].copy()
        use_comp[m][n] = cp[s:e].copy()
    return positions, scores, use_comp


def gpu_scan(ms: Motifs, data, bg=False, test=False):
    """Forward pass then reverse(pwm) pass, merged per (motif, seq) — _h3_1_alignment.jl:89-99.  One library
    call scores both strands; per (motif, seq) the lists hold forward hits (ascending) then rc hits."""
    hits, _ = _scan_raw(ms, data, fwd=True, rc=True, bg=bg, test=test)
    return _hits_to_dicts(hits, ms.num_motifs)


def scan_w_gpu_(ms: Motifs, data, bg=False):
    positions, scores, use_comp = gpu_scan(ms, data, bg=bg)
    if bg:
        ms.positions_bg, ms.scores_bg, ms.use_comp_bg = positions, scores, use_comp
    else:
        ms.positions, ms.scores, ms.use_comp = positions, scores, use_comp


# ---------------------------------------------------------------------------------------------
# Touzet p-value -> score (inference/_h2_Touzet.jl), Float64; tiny (PWM segments of <= 15 columns)
# ---------------------------------------------------------------------------------------------
def pvalue2score(pwm, pval, eps=_granularity_, bg=(0.25, 0.25, 0.25, 0.25)):
    assert 0 <= pval <= 1, "pvalue must be in [0,1]"
    p = np.asarray(pwm, np.float64)
    assert p.shape[0] == 4, "The input matrix must have only 4 rows"
    b = np.asarray(bg).astype(np.float64)
    m = p.shape[1]
    delta = p.max(axis=0) - p.min(axis=0)
    p = p[:, np.argsort(-delta, kind="stable")]                 # min_score_range
    pe = np.floor(p / eps) * eps                                # round_pwm
    colmax, colmin = pe.max(axis=0), pe.min(axis=0)
    # suffix best / worst scores, accumulated left to right like sum(generator) in best_score/worst_score
    def suffix(vals, i):
        s = 0.0
        for x in vals[i:]:
            s += x
        return s
    alpha = suffix(colmin, 0)
    keys = np.array([0.0])
    vals = np.array([1.0])
    for i in range(m):
        bs, ws = (suffix(colmax, i + 1), suffix(colmin, i + 1)) if i + 1 < m else (0.0, 0.0)
        t = keys[:, None] + pe[None, :, i]                      # (n, 4): score-major, base-minor = reference order
        w = vals[:, None] * b[None, :]
        ok = (alpha - bs <= t) & (t <= math.inf - ws)
        t, w = t[ok], w[ok]
        # accumulate equal keys in encounter order (Q[i][t] += ...)
        order = np.argsort(t, kind="stable")
        t, w = t[order], w[order]
        uniq, start = np.unique(t, return_index=True)
        acc = np.zeros(len(uniq))
        idx = np.searchsorted(uniq, t)
        for j in range(len(t)):                                 # sequential to keep the reference's add order
            acc[idx[j]] += w[j]
        keys, vals = uniq, acc
    q_sum = 0.0
    for v in vals:
        q_sum += v
    largest = None
    for k, v in zip(keys, vals):                                # find_largest_alpha
        if q_sum >= pval:
            largest = k
        else:
            return float(k)
        q_sum -= v
    return None if largest is None else float(largest)


def get_pvalue(pwm):
    n = pwm.shape[1]
    if 9 < n <= 11:
        return pvalue_Touzet_mid
    if n <= 9:
        return pvalue_Touzet_small
    return pvalue_Touzet_large


# ---------------------------------------------------------------------------------------------
# Fisher exact test, right tail (HypothesisTests.FisherExactTest(a, c, b, d), tail=:right)
# ---------------------------------------------------------------------------------------------
def fisher_right(a, c, b, d):
    """P[X >= a], X ~ Hypergeometric(a+c successes, b+d failures, a+b draws).  Float64: probability ratios
    pmf(x+1)/pmf(x) accumulated in log space around the mode and normalised by their own sum (no lgamma of large
    arguments), ~1e-12 relative to Rmath's phyper that the reference reaches through HypothesisTests."""
    a, c, b, d = int(a), int(c), int(b), int(d)
    succ, fail, draws = a + c, b + d, a + b
    hi = min(draws, succ)
    lo = max(0, draws - fail)
    if a <= lo:
        return 1.0
    if a > hi:
        return 0.0
    tot = succ + fail
    mean = draws * succ / tot
    sigma = math.sqrt(max(draws * (succ / tot) * (fail / tot), 1.0))
    w = int(60 * sigma) + 100
    x_lo = max(lo, int(mean) - w)
    x_hi = min(hi, max(int(mean), a) + w)
    if a < x_lo:
        return 1.0
    x = np.arange(x_lo, x_hi, dtype=np.float64)               # ratios pmf(x+1)/pmf(x)
    logratio = np.log((succ - x) * (draws - x)) - np.log((x + 1.0) * (fail - draws + x + 1.0))
    logr = np.concatenate([[0.0], np.cumsum(logratio)])
    logr -= logr.max()
    r = np.exp(logr)
    total = r.sum()
    k = a - x_lo
    upper = r[k:].sum()
    if upper <= 0.5 * total:
        return float(upper / total)
    return float(1.0 - r[:k].sum() / total)


# Loader's saddle-point binomial pmf ("Fast and accurate computation of binomial probabilities", 2000), as R's dbinom computes it:
# ~1e-15 relative for every n, where lgamma differences lose digits at n ~ 1e6.
def _stirlerr(n):
    """log(n!) - log(sqrt(2 pi n) (n/e)^n) for integer n >= 1."""
    if n <= 15:
        return math.lgamma(n + 1.0) - (n + 0.5) * math.log(n) + n - 0.5 * math.log(2.0 * math.pi)
    nn = float(n) * n
    s0, s1, s2, s3, s4 = 1.0 / 12, 1.0 / 360, 1.0 / 1260, 1.0 / 1680, 1.0 / 1188
    if n > 500:
        return (s0 - s1 / nn) / n
    if n > 80:
        return (s0 - (s1 - s2 / nn) / nn) / n
    if n > 35:
        return (s0 - (s1 - (s2 - s3 / nn) / nn) / nn) / n
    return (s0 - (s1 - (s2 - (s3 - s4 / nn) / nn) / nn) / nn) / n


def _bd0(x, m):
    """x log(x/m) + m - x, without cancellation when x is close to m."""
    if abs(x - m) < 0.1 * (x + m):
        v = (x - m) / (x + m)
        s = (x - m) * v
        ej = 2.0 * x * v
        v *= v
        j = 1
        while True:
            ej *= v
            s1 = s + ej / (2 * j + 1)
            if s1 == s:
                return s1
            s, j = s1, j + 1
    return x * math.log(x / m) + m - x


def _binom_pmf(x, n, p, q):
    if x == 0:
        return math.exp(-_bd0(n, n * q) - n * p if p < 0.1 else n * math.log(q))
    if x == n:
        return math.exp(-_bd0(n, n * p) - n * q if q < 0.1 else n * math.log(p))
    lc = _stirlerr(n) - _stirlerr(x) - _stirlerr(n - x) - _bd0(x, n * p) - _bd0(n - x, n * q)
    lf = math.log(2.0 * math.pi) + math.log(x) + math.log1p(-x / n)
    return math.exp(lc - 0.5 * lf)


def binom_right(k, n, p):
    """P[X >= k], X ~ Binomial(n, p), in Float64 (~1e-12 relative wherever it is above 1e-300).  The tail away from the mode is
    summed from its first term by the ratios pmf(x+1)/pmf(x); a tail that holds the mode is 1 minus the other tail."""
    k, n, p = int(k), int(n), float(p)
    if k <= 0:
        return 1.0
    if k > n or p <= 0.0:
        return 0.0
    if p >= 1.0:
        return 1.0
    q = 1.0 - p
    mode = int((n + 1) * p)
    if k > mode:                                        # right tail: terms fall from x = k on
        x0, step, ratio = k, 1, p / q
    else:                                               # 1 - P[X <= k-1]: terms fall from x = k-1 down
        x0, step, ratio = k - 1, -1, q / p
    t0 = _binom_pmf(x0, n, p, q)
    total, last, x = t0, t0, x0
    while last > 1e-18 * total:
        hi = min(n - x, 4096) if step > 0 else min(x, 4096)
        if hi <= 0:
            break
        xs = x + step * np.arange(hi, dtype=np.float64)           # the terms x+step .. x+step*hi
        r = ((n - xs) / (xs + 1.0) if step > 0 else xs / (n - xs + 1.0)) * ratio
        terms = last * np.cumprod(r)
        total += float(terms.sum())
        last = float(terms[-1])
        x += step * hi
    return float(total) if step > 0 else float(max(0.0, 1.0 - total))


def fisher_pvec(activate_counts, activate_counts_bg, data, test=False):
    """_h7_fisher.jl:21-36."""
    asum = (data.N_test if test else data.N) * data.L
    out = np.zeros(len(activate_counts), np.float64)
    for i, (a, b) in enumerate(zip(activate_counts, activate_counts_bg)):
        a, b = int(a), int(b)
        out[i] = 1.0 if (a == 0 and b == 0) else fisher_right(a, asum - a, b, asum - b)
    return out


# ---------------------------------------------------------------------------------------------
# thresholds and filtering (inference/_s2_filter_pos_w_scores.jl)
# ---------------------------------------------------------------------------------------------
def _all_scores(sdict):
    return np.concatenate(list(sdict.values())) if sdict else np.zeros(0, f16)


def get_best_thresh(scores, bg_scores, max_score, min_score, max_eff_len, eff_pos, pwm, asum, bg):
    """_s2_filter_pos_w_scores.jl:90-114.  scores / bg_scores: dict seq -> float16 array."""
    if any(len(r) < max_pwm_length_Touzet2 for r in eff_pos):
        best = 0.0
        for r in eff_pos:
            if len(r) > max_pwm_length_Touzet2 or len(r) <= 1:
                continue
            sub = np.asarray(pwm, f16)[:, r.start - 1: r.stop - 1]
            best += pvalue2score(sub, get_pvalue(sub), bg=bg)
        return best
    # Fisher sweep: counts of scores > t come from one sorted array each instead of re-scanning the dicts
    sc = np.sort(_all_scores(scores).astype(f32))
    bsc = np.sort(_all_scores(bg_scores).astype(f32))
    best_thresh, t, best_p = min_score, min_score, f32(1)
    while t < max_score:
        a = len(sc) - int(np.searchsorted(sc, f32(t), side="right"))
        b = len(bsc) - int(np.searchsorted(bsc, f32(t), side="right"))
        p = fisher_right(a, asum - a, b, asum - b)
        if p < best_p:
            best_p, best_thresh = p, t
        t = f16(t + score_thresh_increment)
    return best_thresh


def get_max_score(scores, scores_bg):
    v = np.concatenate([_all_scores(scores), _all_scores(scores_bg)])
    return f16(-np.inf) if v.size == 0 else f16(v.max())


def get_min_score(scores, scores_bg):
    v = np.concatenate([_all_scores(scores), _all_scores(scores_bg)])
    return f16(np.inf) if v.size == 0 else f16(v.min())


def filter_position_by_best_thresh_(positions, scores, use_comp, best_thresh):
    """keep score .> thresh (Float16 vs Float16) — _s2_filter_pos_w_scores.jl:116-125."""
    if positions is None or scores is None or use_comp is None:
        return
    t = f16(best_thresh)
    for k in list(positions.keys()):
        mask = scores[k] > t
        positions[k], scores[k], use_comp[k] = positions[k][mask], scores[k][mask], use_comp[k][mask]


def filter_positions_scores_usecomp_(ms: Motifs, data, bg):
    """_s2_filter_pos_w_scores.jl:127-138."""
    K = ms.num_motifs
    ms.max_scores = np.array([get_max_score(ms.scores[i], ms.scores_bg[i]) for i in range(K)], f16)
    ms.min_scores = np.array([get_min_score(ms.scores[i], ms.scores_bg[i]) for i in range(K)], f16)
    ms.score_thresh = np.zeros(K, f16)
    for i in range(K):
        with np.errstate(over="ignore"):
            ms.score_thresh[i] = f16(get_best_thresh(ms.scores[i], ms.scores_bg[i], ms.max_scores[i], ms.min_scores[i],
                                                     ms.max_effective_lens[i], ms.effective_segments[i], ms.pwms[i],
                                                     data.N * data.L, bg))
    for i in range(K):
        filter_position_by_best_thresh_(ms.positions[i], ms.scores[i], ms.use_comp[i], ms.score_thresh[i])
        filter_position_by_best_thresh_(ms.positions_bg[i], ms.scores_bg[i], ms.use_comp_bg[i], ms.score_thresh[i])


# ---------------------------------------------------------------------------------------------
# occurrence counts (inference/_h4_overlap_ratio.jl, _h7_fisher.jl)
# ---------------------------------------------------------------------------------------------
def get_uniq_pos(positions_i):
    return {k: np.array(list(dict.fromkeys(v.tolist())), np.int64) for k, v in positions_i.items()}


def active_counts_position(positions):
    return np.array([float(sum(len(v) for v in p.values())) for p in positions], np.float64)


def get_uniq_counts(ms: Motifs):
    return (active_counts_position([get_uniq_pos(p) for p in ms.positions]),
            active_counts_position([get_uniq_pos(p) for p in ms.positions_bg]))


def union_ranges(ranges):
    """_h4_overlap_ratio.jl:48-56 — including its loop bound: `eachindex(@view ranges[2:end])` is 1..n-1 and
    indexes the unsliced array, so the range with the largest start is never merged in when n >= 2."""
    if len(ranges) == 0:
        return []
    ranges = sorted(ranges, key=lambda r: r[0])
    out = [ranges[0]]
    for i in range(1, len(ranges)):
        r = ranges[i - 1]
        if out[-1][1] >= r[0]:
            out[-1] = (out[-1][0], r[1])
        else:
            out.append(r)
    return out


def union_pos(positions_arr_k, length):
    return union_ranges([(int(p), int(p) + length - 1) for p in positions_arr_k])


def get_union_ranges(positions_i, len_i):
    return {k: union_pos(v, int(len_i)) for k, v in positions_i.items()}


def get_total_occupied_positions(position_ranges):
    return sum(e - s + 1 for rs in position_ranges.values() for s, e in rs)


def get_fisher_p_values(ms: Motifs, data, test=False):
    tot = [get_total_occupied_positions(get_union_ranges(p, l)) for p, l in zip(ms.positions, ms.lens)]
    tot_bg = [get_total_occupied_positions(get_union_ranges(p, l)) for p, l in zip(ms.positions_bg, ms.lens)]
    return fisher_pvec(tot, tot_bg, data, test=test)


def scan_counts(ms: Motifs, data, bg=False, test=False, thresh=None):
    """Fused variant used once thresholds are known: the library applies score > thresh in the kernel and returns
    per-motif {n_hits, unique starts, union_ranges coverage, true coverage} without materialising hits."""
    _, counts = _scan_raw(ms, data, fwd=True, rc=True, bg=bg, test=test, thresh=thresh, want_hits=False, want_counts=True)
    return counts


def scan_hist(ms: Motifs, data, bg=False, test=False):
    """(K, 32768) histogram of the Float16 bit patterns of every hit score (score > 0, both strands) of one data set."""
    seqs = _which(data, bg=bg, test=test)
    return _lib.scan_hist(seqs.ctx, seqs, pack_pwms(ms), ms.lens)


def get_best_thresh_hist(h_fg, h_bg, eff_pos, pwm, asum, bg, ctx=None):
    """get_best_thresh (_s2_filter_pos_w_scores.jl:90-114) from the score histograms of the foreground and background scans
    instead of the hit dictionaries: identical result, no hit lists.  With a ctx the Touzet DP runs in the library
    (mb200_pvalue2score, bit-identical to pvalue2score below and ~100x faster than the interpreter)."""
    if any(len(r) < max_pwm_length_Touzet2 for r in eff_pos):
        best = 0.0
        for r in eff_pos:
            if len(r) > max_pwm_length_Touzet2 or len(r) <= 1:
                continue
            sub = np.asarray(pwm, f16)[:, r.start - 1: r.stop - 1]
            if ctx is not None:
                best += _lib.pvalue2score(ctx, sub, get_pvalue(sub), _granularity_, bg)
            else:
                best += pvalue2score(sub, get_pvalue(sub), bg=bg)
        return best
    both = np.nonzero((h_fg + h_bg)[: 0x7C01])[0]                       # positive finite halves and +Inf, ascending in value
    if len(both) == 0:
        return f16(np.inf)                                               # get_min_score of nothing (:24-36)
    min_score = np.array([both[0]], np.uint16).view(f16)[0]
    max_score = np.array([both[-1]], np.uint16).view(f16)[0]
    tail_fg = np.concatenate([np.cumsum(h_fg[::-1].astype(np.int64))[::-1], [0]])   # tail[b] = hits with pattern >= b
    tail_bg = np.concatenate([np.cumsum(h_bg[::-1].astype(np.int64))[::-1], [0]])
    best_thresh, t, best_p = min_score, min_score, f32(1)
    while t < max_score:
        b = int(np.array([t], f16).view(np.uint16)[0])
        a_, b_ = int(tail_fg[b + 1]), int(tail_bg[b + 1])                # scores strictly greater than t
        p = fisher_right(a_, asum - a_, b_, asum - b_)
        if p < best_p:
            best_p, best_thresh = p, t
        t = f16(t + score_thresh_increment)
    return best_thresh


def filter_positions_scores_usecomp_fused_(ms: Motifs, data, bg):
    """filter_positions_scores_usecomp! without hit lists: thresholds from two histogram scans, then the filtered occurrence counts
    from two fused counting scans.  Sets ms.score_thresh / max_scores / min_scores; returns (counts_fg, counts_bg) as (K,4) arrays."""
    K = ms.num_motifs
    h_fg, h_bg = scan_hist(ms, data), scan_hist(ms, data, bg=True)
    ms.score_thresh = np.zeros(K, f16)
    for i in range(K):
        with np.errstate(over="ignore"):
            ms.score_thresh[i] = f16(get_best_thresh_hist(h_fg[i], h_bg[i], ms.effective_segments[i], ms.pwms[i], data.N * data.L, bg, ctx=data.seqs.ctx))
    return scan_counts(ms, data, thresh=ms.score_thresh), scan_counts(ms, data, bg=True, thresh=ms.score_thresh)


def pvec_from_test_data(ms: Motifs, data, no_olap=False):
    """render/pvec_calculations.jl:1-22 — test-set scans filtered by ms.score_thresh, union coverage, Fisher.
    The scan, the filter and both counts are one fused library call per data set."""
    if no_olap:
        raise NotImplementedError("no_olap=true is never set by the reference's shipping path (render.jl:78)")
    c = scan_counts(ms, data, bg=False, test=True, thresh=ms.score_thresh)
    cb = scan_counts(ms, data, bg=True, test=True, thresh=ms.score_thresh)
    pvec = fisher_pvec(c[:, 2], cb[:, 2], data, test=True)
    return pvec, c[:, 1].astype(np.float64)
