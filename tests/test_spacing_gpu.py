"""Secondary-motif spacings around primary sites (mb200_seqs_windows, mb200_scan_spacing, records.spacing) checked bit-exact
against an oracle written from the definitions: both margins sliced on the host, dense Float16 window scores (sequential adds in
numpy's float16 on oracle/scan_oracle.py's effective tables, NaN windows dropped), the best window of the two margins together
(highest score, lowest row position, forward strand), the hit rule of mb200_scan and the (quadrant, gap) binning."""
import ctypes
import os

import numpy as np
import pytest

from motifs_jl_b200 import _lib, records, synth
from oracle import scan_oracle as so

pytestmark = pytest.mark.gpu

NONE = 0xFFFFFFFF
FIELDS = ("pos", "score_f16", "comp", "found")


def _ord(bits):
    b = np.asarray(bits, np.int64)
    return np.where(b & 0x8000, ~b & 0xFFFF, b | 0x8000)


def _dense(pwm, codes, rc):
    pwm = np.asarray(pwm, np.float16)
    n, L = codes.shape
    m = pwm.shape[1]
    npos = L - m + 1
    if npos <= 0:
        return None
    tab = so._eff_table(pwm[::-1, ::-1] if rc else pwm)
    s = np.zeros((n, npos), np.float16)
    with np.errstate(invalid="ignore", over="ignore"):
        for j in range(m):
            s = (s + tab[codes[:, j:j + npos], j]).astype(np.float16)
    return s


def _hit(score_bits, t):
    """mb200_scan's rule on Float16 bits: score > 0 and score > t (t None: > 0; NaN t: never)"""
    s = np.asarray(score_bits, np.uint16).view(np.float16)
    ok = s > np.float16(0)
    if t is not None:
        t = np.float16(t)
        ok &= (not np.isnan(t)) & (s > t)
    return ok


def oracle_spacing(rows, anchors, n_primary, pwm_list, thresh, margin):
    """(hist (P, K, 4, W) int64, sites (n, K) BEST_DTYPE) from the definitions"""
    W, K, n = margin, len(pwm_list), len(anchors)
    hist = np.zeros((n_primary, K, 4, W), np.int64)
    sites = np.zeros((n, K), _lib.BEST_DTYPE)
    sites["pos"] = NONE
    if n == 0:
        return hist, sites
    a = anchors["start"].astype(np.int64)
    m_p = anchors["len"].astype(np.int64)
    c_p = anchors["comp"].astype(np.int64)
    left = so.ascii_to_codes(np.stack([rows[r][s - W: s] for r, s in zip(anchors["row"], a)]))
    right = so.ascii_to_codes(np.stack([rows[r][s + l: s + l + W] for r, s, l in zip(anchors["row"], a, m_p)]))
    for k, pwm in enumerate(pwm_list):
        m_k = pwm.shape[1]
        best = np.zeros(n, np.int64)
        for side, codes in ((0, left), (1, right)):
            for rc in (0, 1):
                s = _dense(pwm, codes, rc)
                if s is None:
                    continue
                u = np.arange(s.shape[1], dtype=np.int64)[None, :]
                pos = (a - W)[:, None] + u if side == 0 else (a + m_p)[:, None] + u
                key = np.where(np.isnan(s), 0, (_ord(s.view(np.uint16)) << 34) | ((0xFFFFFFFF - pos) << 1) | (1 - rc))
                best = np.maximum(best, key.max(axis=1))
        f = best != 0
        o = best >> 34
        bits = np.where(f, np.where(o & 0x8000, o & 0x7FFF, ~o & 0xFFFF), 0).astype(np.uint16)
        pos = np.where(f, 0xFFFFFFFF - ((best >> 1) & 0xFFFFFFFF), NONE)
        comp = np.where(f, 1 - (best & 1), 0)
        counted = f & _hit(bits, None if thresh is None else thresh[k])
        sites["pos"][:, k], sites["score_f16"][:, k], sites["comp"][:, k], sites["found"][:, k] = pos, bits, comp, counted
        for i in np.nonzero(counted)[0]:
            s_ = int(pos[i])
            on_left = s_ < a[i]
            g = a[i] - (s_ + m_k) if on_left else s_ - (a[i] + m_p[i])
            downstream = (not on_left) if c_p[i] == 0 else on_left
            q = 2 * int(comp[i] != c_p[i]) + int(downstream)
            assert 0 <= g <= W - m_k
            hist[anchors["primary"][i], k, q, g] += 1
    return hist, sites


def _same(got, exp):
    assert got.shape == exp.shape
    for f in FIELDS:
        bad = np.argwhere(got[f] != exp[f])
        assert len(bad) == 0, (f, bad[:5].tolist(), got[tuple(bad[0])], exp[tuple(bad[0])])


def _rows(lengths, seed):
    rng = np.random.default_rng(seed)
    return [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(n))].copy() for n in lengths]


def _store(ctx, rows, ragged):
    if not ragged:
        return ctx.seqs_from_ascii(np.stack(rows))
    off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    return ctx.seqs_from_ragged(np.concatenate(rows), off)


def _anchors(rows, n, margin, plens, seed, touch=True):
    """n anchors with random rows, primaries and strands whose flanks fit; the first ones touch a row's start and end"""
    rng = np.random.default_rng(seed)
    an = np.zeros(n, _lib.ANCHOR_DTYPE)
    ok_rows = [r for r in range(len(rows)) if len(rows[r]) >= 2 * margin + max(plens)]
    for i in range(n):
        p = int(rng.integers(0, len(plens)))
        r = ok_rows[int(rng.integers(0, len(ok_rows)))]
        hi = len(rows[r]) - plens[p] - margin
        s = margin if (touch and i == 0) else hi if (touch and i == 1) else int(rng.integers(margin, hi + 1))
        an[i] = (r, s, plens[p], p, int(rng.integers(0, 2)), 0)
    return an


def _pw(pwm_list):
    return so.pack_pwms(pwm_list)


def _check(ctx, rows, seqs, an, P, pwms, thresh, margin):
    pw, lens = _pw(pwms)
    hist, sites = ctx.scan_spacing(seqs, an, P, pw, lens, thresh, margin=margin, want_sites=True)
    eh, es = oracle_spacing(rows, an, P, pwms, thresh, margin)
    _same(sites, es)
    assert np.array_equal(hist.astype(np.int64), eh)
    # the histogram is the bincount of the counted sites
    i, k = np.nonzero(sites["found"])
    q, g = records.spacing_bin(an["start"][i], an["len"][i], an["comp"][i], sites["pos"][i, k].astype(np.int64), lens[k], sites["comp"][i, k])
    bc = np.zeros_like(eh)
    np.add.at(bc, (an["primary"][i].astype(np.int64), k, q, g), 1)
    assert np.array_equal(bc, eh)
    h2, s2 = ctx.scan_spacing(seqs, an, P, pw, lens, thresh, margin=margin)
    assert s2 is None and np.array_equal(h2, hist)
    return hist, sites


# ---- window gather -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ragged", [False, True])
def test_windows_equal_host_slices(ctx, ragged):
    rows = _rows([2100] * 7, 1) if not ragged else _rows([2100, 1, 17, 2047, 150, 2000, 33], 1)
    s = _store(ctx, rows, ragged)
    for length in (1, 15, 16, 17, 150, 2000):
        rr, ss = [], []
        for r, row in enumerate(rows):
            L = len(row)
            if L < length:
                continue
            for o in range(16):                                          # every start offset mod 16
                st = min(o + 16 * (r % 3), L - length)
                rr.append(r); ss.append(st)
            rr.append(r); ss.append(L - length)                          # ends on the row's last base
        w = ctx.seqs_windows(s, rr, ss, length)
        try:
            got = w.to_ascii()
            assert got.shape == (len(rr), length) and (w.lengths == length).all()
            exp = np.stack([rows[r][st: st + length] for r, st in zip(rr, ss)])
            assert np.array_equal(got, exp), length
        finally:
            w.free()
    lib, h = ctx._lib, ctypes.c_void_p()
    for rr, ss, ln in (([0], [len(rows[0]) - 9], 10), ([0], [-1], 5), ([len(rows)], [0], 1), ([-1], [0], 1), ([0], [0], 0)):
        r_, s_ = np.array(rr, np.int64), np.array(ss, np.int64)
        rc = lib.mb200_seqs_windows(ctx._h, s._h, _lib._ptr(r_), _lib._ptr(s_), 1, ln, ctypes.byref(h))
        assert rc == _lib.E_INVALID and not h.value
    if ragged:                                                            # a ragged row's own length is the limit
        r_, s_ = np.array([1], np.int64), np.array([0], np.int64)
        assert lib.mb200_seqs_windows(ctx._h, s._h, _lib._ptr(r_), _lib._ptr(s_), 1, 2, ctypes.byref(h)) == _lib.E_INVALID
    s.free()


# ---- spacing against the oracle ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("ragged", [False, True])
def test_spacing_matches_oracle(ctx, ragged):
    margin = 80
    rows = _rows([400] * 12, 2) if not ragged else _rows([400, 183, 90, 260, 1000, 177, 400, 301], 2)
    # 30 short secondaries, 2 of 65-75 columns, 1 longer than the margin.  Sorted by length in groups of 16: the first group runs
    # in scan_kernel<·, true>, the two groups holding motifs over 64 columns in scan_long_kernel<true>
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(30, 6, 30, 3) + synth.random_count_matrices(2, 65, 75, 4)
                                          + synth.random_count_matrices(1, 81, 90, 5))
    thr = synth.stated_thresholds(ms, 0.3)
    thr[1], thr[2], thr[3] = np.float16(np.inf), np.float16(np.nan), np.float16(-2.0)
    an = _anchors(rows, 300, margin, [8, 12, 20], 6)
    s = _store(ctx, rows, ragged)
    try:
        for t in (None, thr):
            hist, sites = _check(ctx, rows, s, an, 3, ms.pwms, t, margin)
            assert ctx.last_timing()[1]["scan"] == 2                   # one batch: scan_kernel once and scan_long_kernel once
            assert not hist[:, -1].any() and (sites["pos"][:, -1] == NONE).all()       # longer than the margin: no window
            assert hist.sum() > 100 and set(np.unique(an["comp"])) == {0, 1}
        assert not hist[:, 1].any() and not hist[:, 2].any()                 # +Inf / NaN thresholds count nothing
        # every counted site is a hit mb200_scan reports in its source row, with the same score bits
        pw, lens = _pw(ms.pwms)
        hits, _ = ctx.scan(s, pw, lens, thr, want_counts=False)
        keys = set(zip(hits["seq"].tolist(), hits["motif"].tolist(), hits["pos"].tolist(), hits["comp"].tolist(), hits["score_f16"].tolist()))
        i, k = np.nonzero(sites["found"])
        assert len(i) > 50
        for ii, kk in zip(i.tolist(), k.tolist()):
            b = sites[ii, kk]
            assert (int(an["row"][ii]), kk, int(b["pos"]), int(b["comp"]), int(b["score_f16"])) in keys
        # flanks touching the row's ends are valid; one base further is not
        lib = ctx._lib
        pwu = np.ascontiguousarray(pw).view(np.uint16)
        h = np.zeros((3, len(lens), 4, margin), np.uint32)
        for bad in ((0, margin - 1), (1, len(rows[an["row"][1]]) - int(an["len"][1]) - margin + 1)):
            b = an[[bad[0]]].copy()
            b["start"] = bad[1]
            rc = lib.mb200_scan_spacing(ctx._h, s._h, _lib._ptr(b), 1, 3, margin, _lib._ptr(pwu), _lib._ptr(lens), len(lens), pw.shape[0],
                                        None, _lib._ptr(h), None)
            assert rc == _lib.E_INVALID
    finally:
        s.free()


def test_spacing_ties(ctx):
    """an equal site in both margins goes to the left one; a palindromic secondary to the forward strand"""
    margin, site = 40, b"GATTACAGG"
    rows = _rows([200] * 8, 7)
    pal = b"GCATATGC"                                                    # reverse complement of itself
    for r in rows:
        r[100:110] = np.frombuffer(b"CCCCCCCCCC", np.uint8)              # the primary's site
        r[70:79] = np.frombuffer(site, np.uint8)                         # left margin [60, 100)
        r[125:134] = np.frombuffer(site, np.uint8)                       # right margin [110, 150)
        r[80:88] = np.frombuffer(pal, np.uint8)
        r[135:143] = np.frombuffer(pal, np.uint8)
    site_pwm = np.array([[2 if c == b else -1 for b in "ACGT"] for c in site.decode()], np.float16).T
    pal_pwm = np.array([[2 if c == b else -1 for b in "ACGT"] for c in pal.decode()], np.float16).T
    assert np.array_equal(pal_pwm[::-1, ::-1], pal_pwm)
    an = np.zeros(8, _lib.ANCHOR_DTYPE)
    an["row"], an["start"], an["len"], an["comp"] = np.arange(8), 100, 10, np.arange(8) % 2
    for ragged in (False, True):
        s = _store(ctx, rows, ragged)
        try:
            hist, sites = _check(ctx, rows, s, an, 1, [site_pwm, pal_pwm], None, margin)
        finally:
            s.free()
        assert (sites["pos"][:, 0] == 70).all() and (sites["comp"][:, 0] == 0).all()
        assert (sites["pos"][:, 1] == 80).all() and (sites["comp"][:, 1] == 0).all()
        assert hist[0, 0, 0, 100 - 79] == 4 and hist[0, 0, 3, 100 - 79] == 4   # same strand upstream (fwd primary); opposite downstream (rc)


def test_spacing_non_finite_entries(ctx):
    margin = 60
    rows = _rows([300] * 10, 8)
    rng = np.random.default_rng(9)
    base = [rng.normal(0, 1, (4, 10)).astype(np.float16) for _ in range(5)]
    base[0][2, 3] = np.inf
    base[1][0, 4] = -np.inf
    base[2][1, 0] = np.inf
    base[2][2, 0] = -np.inf                                              # every window NaN
    base[3][0, 5] = -np.inf
    base[4][3, 9] = np.nan
    an = _anchors(rows, 120, margin, [10, 7], 10)
    for ragged in (False, True):
        s = _store(ctx, rows, ragged)
        try:
            for t in (None, np.array([0.5, -1, 0, np.inf, 0.25], np.float16)):
                hist, sites = _check(ctx, rows, s, an, 2, base, t, margin)
                assert not sites["found"][:, 2].any() and (sites["pos"][:, 2] == NONE).all()
                assert hist[:, 0].sum() > 0
        finally:
            s.free()


def test_spacing_errors_and_empty(ctx):
    rows = _rows([300] * 4, 11)
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(5, 6, 12, 12))
    pw, lens = _pw(ms.pwms)
    pwu = np.ascontiguousarray(pw).view(np.uint16)
    s = _store(ctx, rows, False)
    an = _anchors(rows, 10, 50, [8], 13)
    lib = ctx._lib
    try:
        hist, sites = ctx.scan_spacing(s, an[:0], 2, pw, lens, margin=50, want_sites=True)
        assert hist.shape == (2, 5, 4, 50) and not hist.any() and sites.shape == (0, 5)

        def call(a, P=1, margin=50, h=True):
            hh = np.zeros(max(P, 1) * 5 * 4 * max(margin, 1), np.uint32)
            return lib.mb200_scan_spacing(ctx._h, s._h, _lib._ptr(a), len(a), P, margin, _lib._ptr(pwu), _lib._ptr(lens), 5, pw.shape[0],
                                          None, _lib._ptr(hh) if h else None, None)
        assert call(an) == _lib.OK
        for kw in ({"margin": 0}, {"margin": 65537}, {"P": 0}, {"P": 65536}, {"h": False}):
            assert call(an, **kw) == _lib.E_INVALID, kw
        for field, val in (("primary", 1), ("comp", 2), ("len", 0), ("row", 4), ("row", -1), ("start", 49), ("start", 300 - 8 - 50 + 1)):
            b = an.copy()
            b[field][3] = val
            assert call(b) == _lib.E_INVALID, (field, val)
        # a histogram that cannot fit on the device (65 535 x 50 x 4 x 65 536 counters, 3.4 TB)
        long_row = ctx.seqs_from_ascii(_rows([140_000], 14)[0][None, :])
        try:
            ms50 = synth.motifs_from_count_matrices(synth.random_count_matrices(50, 6, 12, 15))
            pw50, lens50 = _pw(ms50.pwms)
            pw50u = np.ascontiguousarray(pw50).view(np.uint16)
            big = np.zeros(1, _lib.ANCHOR_DTYPE)
            big[0] = (0, 70_000, 8, 0, 0, 0)
            hh = np.zeros(4, np.uint32)                                  # never written: the call fails before any copy
            rc = lib.mb200_scan_spacing(ctx._h, long_row._h, _lib._ptr(big), 1, 65535, 65536, _lib._ptr(pw50u), _lib._ptr(lens50), 50,
                                        pw50.shape[0], None, _lib._ptr(hh), None)
            assert rc == _lib.E_NOMEM
        finally:
            long_row.free()
        assert call(an) == _lib.OK                                       # the context still works
    finally:
        s.free()


# ---- batches, determinism --------------------------------------------------------------------------------------------------
def test_spacing_batches(ctx):
    """margin 2000 and 500 PWMs: about 8 300 anchors a batch under the 8 GB key budget, so 20 000 anchors take three batches"""
    margin = 2000
    rows = list(synth.random_ascii(2500, 4200, 14))
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(500, 8, 40, 15))
    pw, lens = _pw(ms.pwms)
    thr = synth.stated_thresholds(ms, 0.5)
    an = _anchors(rows, 20_000, margin, [8, 12], 16, touch=False)
    s = ctx.seqs_from_ascii(np.stack(rows))
    try:
        hist, sites = ctx.scan_spacing(s, an, 2, pw, lens, thr, margin=margin, want_sites=True)
        t, n = ctx.last_timing()
        # every secondary has <= 40 columns: one scan_kernel launch per batch.  The batch size below is the key budget's
        # arithmetic (8 GiB of 32-bit keys per 16 positions and slot; 500 PWMs = 32 groups of 32 slots); the launch counts pin it,
        # so the boundary anchors picked from it are the library's batch boundaries
        W = (margin - int(lens.min()) + 1 + 31) // 32
        per_batch = (8 << 30) // (W * 1024 * 4 * 2) // 2
        assert n["scan"] == -(-len(an) // per_batch) >= 3
        assert n["pack"] == 1 and t["pack"] > 0 and t["count"] > 0
        for m, batches in ((per_batch, 1), (per_batch + 1, 2)):
            ctx.scan_spacing(s, an[:m], 2, pw, lens, thr, margin=margin)
            assert ctx.last_timing()[1]["scan"] == batches, m
        parts = [an[:7000], an[7000:13001], an[13001:]]
        tot = sum(ctx.scan_spacing(s, p, 2, pw, lens, thr, margin=margin)[0].astype(np.int64) for p in parts)
        assert np.array_equal(tot, hist.astype(np.int64)) and hist.sum() > 0
        pick = np.array([0, 1, per_batch - 1, per_batch, per_batch + 1, 2 * per_batch - 1, 2 * per_batch, 19_999], np.int64)
        _, small = ctx.scan_spacing(s, an[pick], 2, pw, lens, thr, margin=margin, want_sites=True)
        _same(sites[pick], small)
        _, es = oracle_spacing(rows, an[pick[:4]], 2, ms.pwms[:60], thr[:60], margin)
        _same(sites[pick[:4], :60], es)
    finally:
        s.free()


def test_spacing_deterministic_and_scans_after(ctx):
    rows = _rows([600] * 300, 17)
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(40, 6, 24, 18))
    pw, lens = _pw(ms.pwms)
    thr = synth.stated_thresholds(ms, 0.5)
    s = _store(ctx, rows, False)
    an = _anchors(rows, 3000, 150, [10, 14], 19)
    try:
        hits0, c0 = ctx.scan(s, pw, lens, thr)
        tc0 = _lib.scan_last_path(ctx)
        b0 = ctx.scan_best(s, pw, lens)
        h1, s1 = ctx.scan_spacing(s, an, 2, pw, lens, thr, margin=150, want_sites=True)
        h2, s2 = ctx.scan_spacing(s, an, 2, pw, lens, thr, margin=150, want_sites=True)
        assert h1.tobytes() == h2.tobytes() and s1.tobytes() == s2.tobytes() and h1.sum() > 0
        hits1, c1 = ctx.scan(s, pw, lens, thr)
        assert tc0 == 1 and _lib.scan_last_path(ctx) == 1
        assert hits1.tobytes() == hits0.tobytes() and np.array_equal(c1, c0)
        assert ctx.scan_best(s, pw, lens).tobytes() == b0.tobytes()
    finally:
        s.free()


# ---- end to end on a FASTA peak set ---------------------------------------------------------------------------------------
def _rc(s):
    return s[::-1].translate(str.maketrans("ACGT", "TGCA"))


def _write_fasta(path, names, seqs, width=60):
    with open(path, "w") as fh:
        for n, s in zip(names, seqs):
            fh.write(f">{n} peak\n")
            for i in range(0, len(s), width):
                fh.write(s[i:i + width] + "\n")


def test_spacing_end_to_end(ctx, tmp_path):
    R, L, W = 3000, 500, 150
    prim, sec = "GGACTTAGCATG", "TTGCCAAGTC"
    assert _rc(prim) != prim and _rc(sec) != sec
    rng = np.random.default_rng(21)
    seqs, planted, cut = [], np.zeros(R, bool), np.zeros(R, bool)
    for i in range(R):
        s = list("".join(rng.choice(list("ACGT"), L)))
        if rng.random() < 0.4:                                           # primary, 7 bp, secondary: on either strand
            unit = prim + "".join(rng.choice(list("ACGT"), 7)) + sec
            planted[i] = True
            if rng.random() < 0.5:
                s[244 - 7 - len(sec): 244 + len(prim)] = _rc(unit)       # the primary still starts at 244, now on strand 1
            else:
                s[244: 244 + len(unit)] = unit
        else:
            s[244: 244 + len(prim)] = prim if rng.random() < 0.5 else _rc(prim)
        if i % 100 == 7:                                                 # an N run inside the flank
            s[130:134] = "NNNN"
            cut[i] = True
        elif i % 100 == 9:                                               # an N run outside it
            s[20:26] = "NNNNNN"
        seqs.append("".join(s))
    path = os.path.join(tmp_path, "peaks.fa")
    _write_fasta(path, [f"peak{i}" for i in range(R)], seqs)
    rec = records.read_records(path)
    cms = [synth.count_matrix_from_sites([prim] * 30), synth.count_matrix_from_sites([sec] * 30)]
    primary = synth.motifs_from_count_matrices(cms[:1])
    secondary = synth.motifs_from_count_matrices(cms + synth.random_count_matrices(1, 10, 10, 22))      # primary (homotypic), composite partner, decoy
    sthr = synth.stated_thresholds(secondary, 0.6)
    sp = records.spacing(ctx, rec, primary.pwms, secondary.pwms, secondary_thresh=sthr, margin=W, want_sites=True)
    # anchors: best site a hit with its whole flank inside the peak and free of N
    bs = records.best_sites(ctx, rec, primary.pwms)
    m = len(prim)
    exp = [bool(bs.found[i, 0]) and float(bs.score[i, 0]) > 0 and bs.pos[i, 0] >= W and bs.pos[i, 0] + m + W <= L and
           "N" not in seqs[i][bs.pos[i, 0] - W: bs.pos[i, 0] + m + W] for i in range(R)]
    assert sp.n_anchors[0] == sum(exp) and not np.asarray(exp)[cut].any() and sum(exp) > R - 60
    assert (sp.pos[:, 0] >= 0).tolist() == exp
    e = records.spacing_enrichment(sp, secondary.lens)
    assert (e.q[0, 1], e.gap[0, 1]) == (1, 7) and e.p_adj[0, 1] < 1e-20
    assert e.p_adj[0, 2] > 1e-3
    # both orientations of the composite land in the (same strand, downstream, 7) bin
    i = np.nonzero(sp.sites["found"][:, 0, 1])[0]
    q, g = records.spacing_bin(sp.pos[i, 0], m, sp.comp[i, 0], sp.sites["pos"][i, 0, 1], len(sec), sp.sites["comp"][i, 0, 1])
    top = i[(q == 1) & (g == 7)]
    assert set(sp.comp[top, 0].tolist()) == {0, 1} and min(np.bincount(sp.comp[top, 0])) > 200
    assert sp.hist[0, 1, 1, 7] == len(top)
    # a k = 1 shuffle of the same peaks: nothing enriched
    sh = records.shuffle_records(ctx, rec, 1, seed=23)
    e2 = records.spacing_enrichment(records.spacing(ctx, sh, primary.pwms, secondary.pwms, secondary_thresh=sthr, margin=W), secondary.lens)
    assert (e2.p_adj >= 1e-3).all(), e2.p_adj
