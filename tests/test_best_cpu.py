"""Host statistics of the best-site scan: the binomial tail, best-site AUC, CentriMo central enrichment and the fragment -> record
reduction of records.best_sites.  No GPU needed."""
import numpy as np
import pytest
from scipy import stats

from motifs_jl_b200 import _lib, inference, records


@pytest.mark.parametrize("n", [0, 1, 2, 7, 40, 1000, 54321, 1_000_000])
def test_binom_right_matches_scipy(n):
    rng = np.random.default_rng(n)
    for p in (0.0, 1.0, 1e-7, 1e-3, 0.02, 0.25, 0.5, 0.6, 0.97, 1 - 1e-6):
        ks = {0, 1, n, n + 1, max(n - 1, 0), int(n * p), int(n * p) + 1} | set(rng.integers(0, n + 1, 12).tolist())
        for k in sorted(ks):
            ref = float(stats.binom.sf(k - 1, n, p))
            got = inference.binom_right(k, n, p)
            if ref >= 1e-300:
                assert abs(got - ref) <= 1e-9 * ref, (k, n, p, got, ref)
            else:
                assert got < 1e-290, (k, n, p, got, ref)


def _sites(score, found, lengths=None, pos=None):
    score = np.asarray(score, np.float16)
    found = np.asarray(found, bool)
    R, K = score.shape
    return records.BestSites([f"r{i}" for i in range(R)], np.full(R, 100, np.int64) if lengths is None else np.asarray(lengths, np.int64),
                             np.where(found, score, 0).astype(np.float16),
                             np.where(found, 0 if pos is None else pos, -1).astype(np.int64), np.zeros((R, K), np.uint8), found)


def test_best_site_auc_matches_pair_count_and_mannwhitney():
    rng = np.random.default_rng(3)
    fg = _sites(rng.integers(-4, 5, (60, 4)) * 0.5, rng.random((60, 4)) < 0.8)
    bg = _sites(rng.integers(-5, 4, (45, 4)) * 0.5, rng.random((45, 4)) < 0.6)
    fg.score[0, 0] = -np.inf                                       # a found -Inf ranks above records without a site
    bg.score[1, 0] = -np.inf
    fg.found[0, 0] = bg.found[1, 0] = True
    auc = records.best_site_auc(fg, bg)
    for k in range(4):
        a = np.where(fg.found[:, k], fg.score[:, k].astype(np.float64), -1e300)
        b = np.where(bg.found[:, k], bg.score[:, k].astype(np.float64), -1e300)
        a[np.isneginf(a)], b[np.isneginf(b)] = -1e299, -1e299
        brute = ((a[:, None] > b[None, :]).sum() + 0.5 * (a[:, None] == b[None, :]).sum()) / (len(a) * len(b))
        mw = stats.mannwhitneyu(a, b).statistic / (len(a) * len(b))
        assert auc[k] == pytest.approx(brute, abs=1e-12) and auc[k] == pytest.approx(mw, abs=1e-12)
    none = _sites(np.zeros((5, 1)), np.zeros((5, 1)))
    assert records.best_site_auc(none, none)[0] == 0.5                # everything ties


def _centrimo_direct(pos, found, L, m):
    """every window enumerated over start positions, scipy's binomial tail"""
    starts = np.arange(L - m + 1)
    d = np.abs(2 * starts + m - L)
    radii = sorted({int(x) for x in d if x < L - m})
    N = int(found.sum())
    if not radii or N == 0:
        return 0, 0, N, 0.0, 1.0, 1.0
    bestp, best = 2.0, None
    pd = np.abs(2 * pos[found] + m - L)
    for r in radii:
        nr = int((d <= r).sum())
        k = int((pd <= r).sum())
        p = float(stats.binom.sf(k - 1, N, nr / len(starts)))
        if p < bestp:
            bestp, best = p, (nr, k, N * nr / len(starts))
    return best[0], best[1], N, best[2], bestp, min(1.0, bestp * len(radii))


@pytest.mark.parametrize("L", [200, 201])
def test_central_enrichment_matches_direct_enumeration(L):
    rng = np.random.default_rng(L)
    R = 300
    lens = np.array([8, 11, 20, 199, L - 1, L, L + 3])                # both parities of L - m; L - m <= 1 and no start at all
    K = len(lens)
    pos = np.zeros((R, K), np.int64)
    found = rng.random((R, K)) < 0.9
    for k, m in enumerate(lens):
        npos = max(L - m + 1, 1)
        centre = (L - m) // 2
        central = np.clip(centre + rng.integers(-6, 7, R), 0, npos - 1)
        pos[:, k] = np.where(rng.random(R) < 0.3 * (k % 2), central, rng.integers(0, npos, R))
        if L - m < 0:
            found[:, k] = False
    best = records.BestSites([""] * R, np.full(R, L), np.zeros((R, K), np.float16), np.where(found, pos, -1), np.zeros((R, K), np.uint8), found)
    ce = records.central_enrichment(best, lens)
    for k, m in enumerate(lens):
        w, kk, n, e, p, pa = _centrimo_direct(pos[:, k], found[:, k], L, int(m))
        assert (ce.window[k], ce.k[k], ce.n[k]) == (w, kk, n), k
        assert ce.expected[k] == pytest.approx(e, rel=1e-12)
        assert ce.p[k] == pytest.approx(p, rel=1e-9) and ce.p_adj[k] == pytest.approx(pa, rel=1e-9)
    assert ce.p[1] < 1e-10                                            # the centred motif
    assert ce.window[4] == ce.window[5] == ce.window[6] == 0 and ce.p_adj[4] == 1.0


def test_central_enrichment_rejects_unequal_lengths_and_handles_no_sites():
    best = _sites(np.zeros((3, 1)), np.ones((3, 1)), lengths=[100, 100, 120])
    with pytest.raises(ValueError, match=r"\[100, 120\]"):
        records.central_enrichment(best, [8])
    none = _sites(np.zeros((4, 1)), np.zeros((4, 1)))
    ce = records.central_enrichment(none, [8])
    assert ce.window[0] == 0 and ce.p[0] == ce.p_adj[0] == 1.0 and ce.n[0] == 0


def test_fragment_to_record_reduction():
    h = lambda x: np.float16(x).view(np.uint16)
    fb = np.zeros((6, 2), _lib.BEST_DTYPE)
    # record 0: fragments 0 (start 0) and 1 (start 50) and 2 (start 90); record 1: fragment 3; record 2: fragments 4, 5 (no sites)
    fb[0, 0] = (10, h(3.0), 1, 1); fb[1, 0] = (0, h(3.0), 0, 1); fb[2, 0] = (1, h(2.5), 0, 1)       # equal scores: lower record pos (10)
    fb[0, 1] = (7, h(-1.0), 1, 1); fb[1, 1] = (0, h(-0.5), 1, 1)                                    # higher score wins over position
    fb[3, 0] = (4, h(-np.inf), 0, 1); fb[3, 1] = (0xFFFFFFFF, 0, 0, 0)
    frag_record = np.array([0, 0, 0, 1, 2, 2])
    frag_start = np.array([0, 50, 90, 0, 0, 30])
    score, pos, comp, found = records.reduce_fragment_best(frag_record, frag_start, fb, 4)
    assert found.tolist() == [[True, True], [True, False], [False, False], [False, False]]
    assert pos.tolist() == [[10, 50], [4, -1], [-1, -1], [-1, -1]]
    assert comp.tolist() == [[1, 1], [0, 0], [0, 0], [0, 0]]
    assert score[0].tolist() == [3.0, -0.5] and np.isneginf(score[1, 0]) and score[1, 1] == 0
    # same score and record position on both strands (two fragments cannot overlap, but one fragment's record may): forward wins
    fb2 = np.zeros((2, 1), _lib.BEST_DTYPE)
    fb2[0, 0] = (5, h(1.0), 1, 1); fb2[1, 0] = (5, h(1.0), 0, 1)
    _, pos2, comp2, _ = records.reduce_fragment_best(np.array([0, 0]), np.array([0, 0]), fb2, 1)
    assert pos2[0, 0] == 5 and comp2[0, 0] == 0
