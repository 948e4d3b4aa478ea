"""Host logic of the spacing analysis (records.spacing): anchors from record best sites, the (quadrant, gap) binning and the
SpaMo enrichment test.  No device needed."""
import numpy as np
import pytest
from scipy import stats

from motifs_jl_b200 import records


def _rec(lengths, frags):
    """Records with the given record lengths and fragments (record, start, length); bases are not needed here"""
    fr = np.array(frags, np.int64).reshape(-1, 3)
    return records.Records([f"r{i}" for i in range(len(lengths))], np.array(lengths, np.int64), fr[:, 0].copy(), fr[:, 1].copy(),
                           fr[:, 2].copy(), np.zeros(int(fr[:, 2].sum()), np.uint8))


def test_anchor_mapping_drops_cut_flanks():
    # record 0: one fragment [0, 100); record 1: fragments [0, 40) and [45, 120) (an N run at 40..44); record 2: [10, 60)
    rec = _rec([100, 120, 60], [(0, 0, 100), (1, 0, 40), (1, 45, 75), (2, 10, 50)])
    W, m = 10, 8
    # primary 0 best sites, per record: flank inside; flank crosses the N run; flank touching the record's start (valid)
    pos = np.array([[50, 0], [36, 60], [20, 42]], np.int64)
    score = np.full((3, 2), np.float16(3.0))
    comp = np.zeros((3, 2), np.uint8)
    found = np.ones((3, 2), bool)
    frag, ok = records.spacing_anchors(rec, score, pos, comp, found, [m, m], None, W)
    # (0,0): [40, 68) in fragment 0; (0,1): [-10, 18) leaves the record; (1,0): [26, 54) crosses the N run;
    # (1,1): [50, 78) in fragment 2; (2,0): [10, 38) touches the fragment's start; (2,1): [32, 60) touches the record end
    assert ok.tolist() == [[True, False], [False, True], [True, True]]
    assert frag.tolist() == [[0, -1], [-1, 2], [3, 3]]
    # one base further on either side is dropped
    frag2, ok2 = records.spacing_anchors(rec, score, np.array([[50, 0], [36, 60], [19, 43]]), comp, found, [m, m], None, W)
    assert ok2[2].tolist() == [False, False]
    # record-end rule: the flank must not pass the record's length even when a fragment were longer (it cannot be)
    assert not records.spacing_anchors(rec, score, np.array([[83, 0], [0, 0], [0, 0]]), comp, found, [m, m], None, W)[1][0, 0]


def test_anchor_hit_rule():
    rec = _rec([200], [(0, 0, 200)])
    pos = np.full((1, 5), 100, np.int64)
    score = np.array([[1.0, 0.0, -1.0, 2.0, 2.0]], np.float16)
    found = np.array([[True, True, True, True, False]])
    comp = np.zeros((1, 5), np.uint8)
    _, ok = records.spacing_anchors(rec, score, pos, comp, found, [8] * 5, None, 20)
    assert ok.tolist() == [[True, False, False, True, False]]
    thr = np.array([0.5, -3, -3, np.nan, np.inf], np.float16)
    _, ok = records.spacing_anchors(rec, score, pos, comp, found, [8] * 5, thr, 20)
    assert ok.tolist() == [[True, False, False, False, False]]
    _, ok = records.spacing_anchors(rec, score, pos, comp, found, [8] * 5, np.full(5, 1.0, np.float16), 20)
    assert ok.tolist() == [[False, False, False, True, False]]        # > 1.0, not >=


@pytest.mark.parametrize("c_p", [0, 1])
def test_quadrant_and_gap(c_p):
    a, m_p, m_k = 100, 10, 6
    # left site ending 3 bases before the primary, right site starting 5 bases after it
    sl, sr = a - 3 - m_k, a + m_p + 5
    for c_k in (0, 1):
        ql, gl = records.spacing_bin(a, m_p, c_p, sl, m_k, c_k)
        qr, gr = records.spacing_bin(a, m_p, c_p, sr, m_k, c_k)
        assert (int(gl), int(gr)) == (3, 5)
        same = 0 if c_k == c_p else 2
        # downstream: right of a forward primary, left of a reverse one
        assert int(qr) == same + (1 if c_p == 0 else 0)
        assert int(ql) == same + (0 if c_p == 0 else 1)
    # adjacent sites have gap 0; all four quadrants are reached
    q, g = records.spacing_bin([a] * 4, m_p, c_p, [a - m_k, a + m_p, a - m_k, a + m_p], m_k, [c_p, c_p, 1 - c_p, 1 - c_p])
    assert g.tolist() == [0, 0, 0, 0] and sorted(q.tolist()) == [0, 1, 2, 3]


def _sp(hist):
    P, K, _, W = hist.shape
    return records.Spacing([], W, hist.astype(np.int64), np.zeros(P, np.int64), np.zeros((0, P), np.int64), np.zeros((0, P), np.int64))


def test_enrichment_against_scipy_and_bonferroni():
    rng = np.random.default_rng(3)
    P, K, W = 2, 3, 30
    lens = np.array([6, 12, 31])                                         # the last one does not fit in the margin
    hist = np.zeros((P, K, 4, W), np.int64)
    for p in range(P):
        for k in range(2):
            G = W - lens[k] + 1
            hist[p, k, :, :G] = rng.poisson(3, (4, G))
            hist[p, k, 1, 7] += 25 * (p + 1)
    hist[1, 0] = 0                                                       # no counted site
    e = records.spacing_enrichment(_sp(hist), lens)
    for p in range(P):
        for k in range(K):
            G = W - lens[k] + 1
            n = int(hist[p, k].sum())
            if G < 1 or n == 0:
                assert e.n[p, k] == n and e.q[p, k] == -1 and e.p[p, k] == 1.0 and e.p_adj[p, k] == 1.0
                continue
            B = 4 * G
            flat = hist[p, k, :, :G].reshape(-1)
            top = int(flat.max())
            i = int(np.nonzero(flat == top)[0][0])
            assert (e.n[p, k], e.count[p, k], e.q[p, k], e.gap[p, k]) == (n, top, i // G, i % G)
            ref = stats.binom.sf(top - 1, n, 1.0 / B)
            assert e.p[p, k] == pytest.approx(ref, rel=1e-9)
            assert e.p_adj[p, k] == pytest.approx(min(1.0, ref * B * K), rel=1e-9)
    assert (e.q[0, :2] == 1).all() and (e.gap[0, :2] == 7).all() and e.p_adj[0, 0] < 1e-6


def test_enrichment_tie_rule():
    W, lens = 20, np.array([5])
    hist = np.zeros((1, 1, 4, W), np.int64)
    hist[0, 0, 2, 3] = 4
    hist[0, 0, 1, 9] = 4
    hist[0, 0, 1, 4] = 4
    hist[0, 0, 0, 0] = 1
    e = records.spacing_enrichment(_sp(hist), lens)
    assert (e.q[0, 0], e.gap[0, 0], e.count[0, 0], e.n[0, 0]) == (1, 4, 4, 13)     # lowest q, then lowest gap
    hist[0, 0, 0, W - 1] = 9                                             # past W - m_k: not a bin (never filled by the device)
    e = records.spacing_enrichment(_sp(hist), lens)
    assert (e.q[0, 0], e.gap[0, 0], e.n[0, 0]) == (1, 4, 13)
