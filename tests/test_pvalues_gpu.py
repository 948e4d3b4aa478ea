"""Exact p-values of the scan's Float16 score on the device (mb200_pvtab_*, Context.score_null, records.scan_fasta_pvalues,
records.best_site_pvalues): the survival tables against the forward-DP oracle and enumeration, thresholds, lookups, calibration
on sequences drawn from the background, and the FASTA entry points against a dense enumeration of every window."""
import numpy as np
import pytest
import scipy.stats

import motifs_jl_b200 as mb
from motifs_jl_b200 import _lib, inference, records, synth
from oracle import pvalue_oracle as po
from oracle import scan_oracle as so

pytestmark = pytest.mark.gpu

UNIFORM = np.full(4, 0.25)
SKEWED = np.array([0.35, 0.1, 0.2, 0.35])
ALL_BITS = np.arange(65536, dtype=np.uint32).astype(np.uint16)
NONNAN = ~np.isnan(ALL_BITS.view(np.float16))


def _edge_pwms():
    rng = np.random.default_rng(3)
    out = [rng.normal(0, 2, (4, 1)), rng.normal(0, 2, (4, 7)), rng.normal(0, 1, (4, 6))]
    out[2][:, 2] = 0                                          # a zero column
    ninf = rng.normal(0, 1, (4, 5))
    ninf[1, 3] = -np.inf                                      # -Inf entry: the rest of its column is NaN
    big = rng.normal(0, 1, (4, 6))
    big[0, 1], big[3, 2], big[2, 4], big[1, 0] = 60000, 60000, -60000, -60000
    pinf = rng.normal(0, 1, (4, 4))
    pinf[2, 1] = np.inf
    out += [ninf, big, pinf, np.round(rng.normal(0, 1, (4, 8)) * 8) / 8]
    return [p.astype(np.float16) for p in out]


def _random_pwms(lengths, seed):
    rng = np.random.default_rng(seed)
    return [rng.normal(0, 1.5, (4, int(m))).astype(np.float16) for m in lengths]


def _realistic(K, lo, hi, seed):
    return list(synth.motifs_from_count_matrices(synth.random_count_matrices(K, lo, hi, seed)).pwms)


def _check_tables(null, pwms, bg, brute=True):
    for k, pwm in enumerate(pwms):
        for c, tab in enumerate(po.eff_tables(pwm)):
            got, exp = null.survival(k, c), po.survival(tab, bg)
            assert np.array_equal(np.isnan(got), ~NONNAN)
            g, e = got[NONNAN], exp[NONNAN]
            assert np.array_equal(g == 0, e == 0), (k, c)
            pos = e > 0
            assert np.max(np.abs(g[pos] - e[pos]) / e[pos]) <= 1e-12, (k, c)
            if brute and pwm.shape[1] <= 8:
                b = po.brute_survival(tab, bg)[NONNAN]
                assert np.array_equal(g == 0, b == 0)
                assert np.max(np.abs(g[b > 0] - b[b > 0]) / b[b > 0]) <= 1e-12, (k, c)


@pytest.mark.parametrize("bg", [UNIFORM, SKEWED], ids=["uniform", "skewed"])
def test_tables_lengths_1_to_30(ctx, bg):
    pwms = _random_pwms(np.random.default_rng(1).permutation(np.arange(1, 31)), 5)
    pw, lens = so.pack_pwms(pwms)
    null = ctx.score_null(pw, lens, bg)
    try:
        _check_tables(null, pwms, bg)
    finally:
        null.free()


@pytest.mark.parametrize("bg", [UNIFORM, SKEWED], ids=["uniform", "skewed"])
def test_tables_edge_and_realistic_pwms(ctx, bg):
    pwms = _edge_pwms() + _realistic(6, 8, 30, 7)
    pw, lens = so.pack_pwms(pwms)
    null = ctx.score_null(pw, lens, bg)
    try:
        _check_tables(null, pwms, bg)
    finally:
        null.free()


def test_builds_are_bit_identical(ctx):
    pwms = _realistic(40, 6, 30, 11) + _edge_pwms()
    pw, lens = so.pack_pwms(pwms)
    a, b = ctx.score_null(pw, lens, SKEWED), ctx.score_null(pw, lens, SKEWED)
    try:
        for k in range(len(pwms)):
            for c in (0, 1):
                assert np.array_equal(a.survival(k, c).view(np.uint64), b.survival(k, c).view(np.uint64))
    finally:
        a.free(); b.free()


def test_thresholds_follow_the_rule(ctx):
    pwms = _edge_pwms() + _realistic(5, 8, 20, 3)
    pw, lens = so.pack_pwms(pwms)
    K = len(pwms)
    null = ctx.score_null(pw, lens, SKEWED)
    try:
        S = {(k, c): null.survival(k, c) for k in range(K) for c in (0, 1)}
        s_inf = np.array([S[(k, 0)][0x7C00] for k in range(K)])
        assert s_inf.max() > 0                                  # the overflow / +Inf PWMs put mass on +Inf
        below = np.where(s_inf > 0, s_inf / 2, 1e-300)
        vals = ALL_BITS.view(np.float16)[NONNAN]
        for pv in [np.zeros(K), np.ones(K), np.full(K, 1e-4), np.full(K, 1e-3), np.full(K, 0.5), below,
                   np.random.default_rng(0).uniform(0, 1, K)]:
            th = null.thresholds(pv)
            assert th.shape == (K, 2) and th.dtype == np.float16
            for k in range(K):
                for c in (0, 1):
                    s = S[(k, c)][NONNAN]
                    # the rule holds for every score above -Inf; at s* = -Inf the threshold is -Inf itself
                    above = vals > -np.inf
                    assert np.array_equal((vals > th[k, c])[above], (s <= pv[k])[above]), (k, c, pv[k], th[k, c])
                    if pv[k] < S[(k, c)][0x7C00]:
                        assert th[k, c] == np.inf
                    if S[(k, c)][0xFC00] <= pv[k]:
                        assert th[k, c] == -np.inf
    finally:
        null.free()


def test_lookup_equals_table(ctx):
    pwms = _edge_pwms() + _realistic(3, 8, 12, 5)
    pw, lens = so.pack_pwms(pwms)
    K = len(pwms)
    null = ctx.score_null(pw, lens, UNIFORM)
    try:
        rng = np.random.default_rng(9)
        n = 300_000
        bits = rng.integers(0, 65536, n).astype(np.uint16)
        bits[:6] = [0x8000, 0x0000, 0x7C00, 0xFC00, 0x7E00, 0xFE01]   # -0, +0, +Inf, -Inf, NaNs
        motif = rng.integers(0, K, n).astype(np.uint16)
        comp = rng.integers(0, 2, n).astype(np.uint8)
        got = null.pvalues(motif, comp, bits)
        tabs = np.stack([np.stack([null.survival(k, c) for c in (0, 1)]) for k in range(K)])
        exp = tabs[motif, comp, bits]
        assert np.array_equal(np.isnan(got), np.isnan(exp)) and np.array_equal(got[~np.isnan(got)], exp[~np.isnan(exp)])
        assert np.isnan(got[4]) and np.isnan(got[5])
        assert got[0] == tabs[motif[0], comp[0], 0]
        assert len(null.pvalues([], [], np.zeros(0, np.uint16))) == 0
        for m in (1, 7, 165, 4097):                             # any count, odd ones included
            part = null.pvalues(motif[-m:], comp[-m:], bits[-m:])
            assert np.array_equal(part.view(np.uint64), got[-m:].view(np.uint64))
    finally:
        null.free()


def test_calibration_on_background_sequences(ctx):
    bg = np.array([0.3, 0.2, 0.2, 0.3])
    rng = np.random.default_rng(2024)
    N, L, p0 = 2000, 1000, 1e-3
    ascii = np.frombuffer(b"ACGT", np.uint8)[rng.choice(4, size=(N, L), p=bg)]
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(6, 8, 20, 17))
    pw, lens = inference.pack_pwms(ms), ms.lens
    null = ctx.score_null(pw, lens, bg)
    seqs = ctx.seqs_from_ascii(ascii)
    try:
        th = null.thresholds(p0)
        assert np.all(th > 0)                                   # the scan's score > 0 rule plays no part
        for c in (0, 1):
            _, counts = ctx.scan(seqs, pw, lens, np.ascontiguousarray(th[:, c]), fwd=c == 0, rc=c == 1, want_hits=False)
            s_star = np.nextafter(th[:, c], np.float16(np.inf))
            prob = null.pvalues(np.arange(len(lens)), np.full(len(lens), c), s_star)
            assert np.all(prob <= p0) and np.all(prob > p0 / 20)
            n_win = N * (L - lens + 1)
            mean, sd = n_win * prob, np.sqrt(n_win * prob * (1 - prob))
            assert np.all(np.abs(counts[:, 0] - mean) <= 5 * sd), (c, counts[:, 0], mean, sd)
    finally:
        seqs.free(); null.free()


# ---- FASTA entry points against a dense enumeration of every window --------------------------------------------------------
def _write_fasta(path, names, seqs, width=60):
    with open(path, "w") as fh:
        for n, s in zip(names, seqs):
            fh.write(f">{n} peak\n")
            for i in range(0, len(s), width):
                fh.write(s[i:i + width] + "\n")


@pytest.fixture(scope="module")
def peaks_fasta(tmp_path_factory):
    """Records of different lengths with N runs, an IUPAC code, soft-masked bases and planted sites of the first motif."""
    rng = np.random.default_rng(31)
    site = "TGACGTCA"
    names, seqs = [], []
    for i, L in enumerate((4000, 1200, 333, 17, 0, 2600, 90, 45, 700, 1500)):
        s = bytearray(np.frombuffer(b"ACGT", np.uint8)[rng.choice(4, L, p=[0.3, 0.2, 0.2, 0.3])].tobytes())
        if L > 40:
            p, q = sorted(int(x) for x in rng.integers(0, L, 2))
            s[p:min(q, p + 150)] = b"N" * (min(q, p + 150) - p)
            s[:4] = b"NNNN"; s[L // 2] = ord("R"); s[10:30] = s[10:30].lower()
        for p in rng.integers(0, max(L - len(site), 1), L // 200):
            s[int(p):int(p) + len(site)] = site.encode()
        names.append(f"peak{i}"); seqs.append(s.decode())
    path = tmp_path_factory.mktemp("pv") / "peaks.fa"
    _write_fasta(path, names, seqs)
    pwms = list(synth.motifs_from_count_matrices([synth.count_matrix_from_sites([site] * 30)] +
                                                 synth.random_count_matrices(3, 6, 14, 8)).pwms)
    pwms.append(np.full((4, 6), -0.5, np.float16))             # every window scores -3: threshold below 0 (clamped)
    return str(path), pwms


def _dense_oracle(rec, pwms, bg, p0):
    """every window of every fragment: (record, pos, motif, comp, score bits, p) with p <= p0 and score > 0"""
    off = rec.frag_offsets
    tabs = [po.eff_tables(p) for p in pwms]
    S = [[po.survival(t, bg) for t in tt] for tt in tabs]
    out = []
    for f in range(len(rec.frag_len)):
        codes = so.ascii_to_codes(rec.bases[off[f]: off[f + 1]][None, :])
        for k in range(len(pwms)):
            for c in (0, 1):
                s = po.dense_scores(tabs[k][c], codes)[0]
                bits = s.view(np.uint16)
                p = S[k][c][bits]
                sel = np.nonzero((p <= p0) & (s > 0))[0]
                for i in sel.tolist():
                    out.append((int(rec.frag_record[f]), int(rec.frag_start[f]) + i, k, c, int(bits[i]), float(p[i])))
    out.sort(key=lambda t: (t[0], t[2], t[3], t[1]))
    return out, S


def test_scan_fasta_pvalues_equals_dense_enumeration(ctx, peaks_fasta):
    path, pwms = peaks_fasta
    rec = records.read_records(path)
    p0 = 1e-3
    res = records.scan_fasta_pvalues(ctx, path, pwms, p0)
    bg = records.base_background(rec)
    assert np.array_equal(res.bg, bg)
    exp, S = _dense_oracle(rec, pwms, bg, p0)
    h = res.hits
    assert len(h) == len(exp) > 20
    assert np.array_equal(h["record"], [e[0] for e in exp]) and np.array_equal(h["pos"], [e[1] for e in exp])
    assert np.array_equal(h["motif"], [e[2] for e in exp]) and np.array_equal(h["comp"], [e[3] for e in exp])
    assert np.array_equal(h["score_f16"], [e[4] for e in exp])
    ep = np.array([e[5] for e in exp])
    assert np.allclose(res.pvalue, ep, rtol=1e-12, atol=0)
    lens = np.array([p.shape[1] for p in pwms])
    n_tests = 2 * np.array([np.maximum(0, rec.frag_len - m + 1).sum() for m in lens])
    assert np.array_equal(res.n_tests, n_tests)
    for k in range(len(pwms)):
        sel = h["motif"] == k
        n = int(sel.sum())
        q = scipy.stats.false_discovery_control(np.concatenate([ep[sel], np.ones(n_tests[k] - n)]))[:n]
        assert np.allclose(res.qvalue[sel], q, rtol=1e-10, atol=0)
    # a slot is clamped (threshold below 0) exactly when P(score > 0) = S(+0) <= p0: the planted motif's windows with two
    # mismatches score below 0 while P(at most one mismatch) < p0, so it is clamped; the constant PWM scores -3 everywhere
    clamped = np.array([[S[k][c][0x0000] <= p0 for c in (0, 1)] for k in range(len(pwms))])
    assert np.array_equal(res.clamped, clamped) and np.array_equal(res.clamped, res.thresh < 0)
    assert clamped[0].all() and clamped[-1].all() and not clamped[1:-1].any()
    assert not np.any(h["motif"] == len(pwms) - 1)
    for k in range(len(pwms)):                                 # the thresholds are the rule's
        for c in (0, 1):
            v = ALL_BITS.view(np.float16)[NONNAN]
            assert np.array_equal(v > res.thresh[k, c], S[k][c][NONNAN] <= p0)


def test_best_site_pvalues_against_oracle(ctx, peaks_fasta):
    path, pwms = peaks_fasta
    rec = records.read_records(path)
    best = records.best_sites(ctx, rec, pwms)
    bg = records.base_background(rec)
    site_p, seq_p = records.best_site_pvalues(ctx, rec, best, pwms)
    R, K = best.found.shape
    assert site_p.shape == seq_p.shape == (R, K)
    assert np.array_equal(np.isnan(site_p), ~best.found) and np.array_equal(np.isnan(seq_p), ~best.found)
    S = [[po.survival(t, bg) for t in po.eff_tables(p)] for p in pwms]
    lens = np.array([p.shape[1] for p in pwms])
    for r in range(R):
        fr = rec.frag_record == r
        for k in range(K):
            if not best.found[r, k]:
                continue
            e = S[k][best.comp[r, k]][best.score[r, k].view(np.uint16)]
            assert abs(site_p[r, k] - e) <= 1e-12 * e
            n = 2 * int(np.maximum(0, rec.frag_len[fr] - lens[k] + 1).sum())
            assert np.isclose(seq_p[r, k], -np.expm1(n * np.log1p(-e)), rtol=1e-12, atol=0)


def test_invalid_arguments_leave_context_usable(ctx):
    pwms = _realistic(3, 6, 10, 2)
    pw, lens = so.pack_pwms(pwms)
    pw16 = np.ascontiguousarray(pw).view(np.uint16)
    L = ctx._lib
    h = mb._lib.C.c_void_p()
    P = _lib._ptr

    def create(pw_, ln, K, maxlen, bg):
        return L.mb200_pvtab_create(ctx._h, P(pw_), P(ln), K, maxlen, P(bg), mb._lib.C.byref(h))

    ok_bg = np.full(4, 0.25)
    bad = [create(pw16, lens, len(lens), pw.shape[0], np.array([0.5, 0.5, 0.5, -0.5])),
           create(pw16, lens, len(lens), pw.shape[0], np.array([0.25, 0.25, 0.25, np.nan])),
           create(pw16, lens, len(lens), pw.shape[0], np.array([0.25, 0.25, 0.25, np.inf])),
           create(pw16, lens, len(lens), pw.shape[0], np.array([0.25, 0.25, 0.25, 0.2501])),
           create(pw16, lens, 0, pw.shape[0], ok_bg),
           create(pw16, np.array([0, 6, 6], np.int64), 3, pw.shape[0], ok_bg),
           create(pw16, np.array([pw.shape[0] + 1, 6, 6], np.int64), 3, pw.shape[0], ok_bg),
           create(None, lens, len(lens), pw.shape[0], ok_bg),
           create(pw16, lens, len(lens), pw.shape[0], None),
           L.mb200_pvtab_create(ctx._h, P(pw16), P(lens), len(lens), pw.shape[0], P(ok_bg), None)]
    assert bad == [_lib.E_INVALID] * len(bad)
    null = ctx.score_null(pw, lens, np.array([0.25, 0.25, 0.25, 0.25 + 5e-7]))  # within 1e-6 of 1
    try:
        for pv in ([0.1, -1e-9, 0.1], [0.1, 1.0 + 1e-9, 0.1], [np.nan, 0.1, 0.1]):
            with pytest.raises(mb.MB200Error) as e:
                null.thresholds(pv)
            assert e.value.code == _lib.E_INVALID
        for m, c in ((3, 0), (0, 2)):
            with pytest.raises(mb.MB200Error) as e:
                null.pvalues([m], [c], [0x3C00])
            assert e.value.code == _lib.E_INVALID
        for k, c in ((3, 0), (-1, 0), (0, 2)):
            with pytest.raises(mb.MB200Error) as e:
                null.survival(k, c)
            assert e.value.code == _lib.E_INVALID
        out = np.zeros(6, np.uint16)
        assert L.mb200_pvtab_thresholds(ctx._h, null._h, None, P(out)) == _lib.E_INVALID
        assert L.mb200_pvtab_thresholds(ctx._h, None, P(np.zeros(3)), P(out)) == _lib.E_INVALID
        assert L.mb200_pvtab_lookup(ctx._h, null._h, None, None, None, 1, None) == _lib.E_INVALID
        assert L.mb200_pvtab_survival(ctx._h, null._h, 0, 0, None) == _lib.E_INVALID
        assert L.mb200_pvtab_destroy(ctx._h, None) == _lib.E_INVALID
        # the context and the table still work
        th = null.thresholds(1e-3)
        assert th.shape == (3, 2) and np.isfinite(null.pvalues([0], [1], th[0, 1:2])).all()
    finally:
        null.free()
    a = synth.random_ascii(50, 100, 1)
    seqs = ctx.seqs_from_ascii(a)
    hits, counts = ctx.scan(seqs, pw, lens)
    ohits, ocounts = so.scan(pw, lens, so.ascii_to_codes(a), None)
    assert len(hits) == len(ohits) and np.array_equal(counts, ocounts)
    seqs.free()
