"""Best site per (row, motif) (mb200_scan_best, records.best_sites) checked bit-exact (pos, comp, score bits, found) against an
oracle: dense Float16 window scores, sequential adds in numpy's float16 (the table form of oracle/scan_oracle.py's numpy twin,
itself checked against the C literal form of greedy_search! where the score is positive), with the valid starts sliced, NaN
windows dropped and the tie rule applied (highest score, lowest position, forward strand)."""
import os

import numpy as np
import pytest

from motifs_jl_b200 import _lib, records, synth
from oracle import scan_oracle as so

pytestmark = pytest.mark.gpu

FIELDS = ("pos", "score_f16", "comp", "found")
NONE = 0xFFFFFFFF


def _ord(bits):
    b = np.asarray(bits, np.int64)
    return np.where(b & 0x8000, ~b & 0xFFFF, b | 0x8000)


def _dense(pwm, codes, rc):
    """(n, L - m + 1) float16 scores of one motif and strand, or None when no window fits"""
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


def oracle_best(pwm_list, rows, strands=3, check_literal=False):
    """(N, K) BEST_DTYPE for rows (a list of ASCII uint8 arrays of any lengths), each length group scored on its own"""
    N, K = len(rows), len(pwm_list)
    out = np.zeros((N, K), _lib.BEST_DTYPE)
    out["pos"] = NONE
    L = np.array([len(r) for r in rows], np.int64)
    for Ln in np.unique(L):
        idx = np.nonzero(L == Ln)[0]
        if Ln == 0:
            continue
        codes = so.ascii_to_codes(np.stack([rows[i] for i in idx]))
        if check_literal:
            pw, lens = so.pack_pwms(pwm_list)
        for k, pwm in enumerate(pwm_list):
            best = np.zeros(len(idx), np.int64)
            for rc in (0, 1):
                if not (strands >> rc) & 1:
                    continue
                s = _dense(pwm, codes, rc)
                if s is None:
                    continue
                if check_literal:                                   # C literal form: max(score, 0) on every valid start
                    lit = so.pos_scores(pw[:, :, k:k + 1], lens[k:k + 1], codes, rc)[0, :, : s.shape[1]]
                    with np.errstate(invalid="ignore"):
                        pos_part = np.where(s > 0, s, np.float16(0)).astype(np.float16)
                    assert np.array_equal(lit.view(np.uint16), pos_part.view(np.uint16))
                bits = s.view(np.uint16)
                p = np.arange(s.shape[1], dtype=np.int64)[None, :]
                key = np.where(np.isnan(s), 0, (_ord(bits) << 34) | ((0xFFFFFFFF - p) << 1) | (1 - rc))
                best = np.maximum(best, key.max(axis=1))
            f = best != 0
            o = best >> 34
            out["found"][idx, k] = f
            out["pos"][idx, k] = np.where(f, 0xFFFFFFFF - ((best >> 1) & 0xFFFFFFFF), NONE)
            out["comp"][idx, k] = np.where(f, 1 - (best & 1), 0)
            out["score_f16"][idx, k] = np.where(f, np.where(o & 0x8000, o & 0x7FFF, ~o & 0xFFFF), 0)
    return out


def _same(got, exp):
    assert got.shape == exp.shape
    for f in FIELDS:
        bad = np.argwhere(got[f] != exp[f])
        assert len(bad) == 0, (f, bad[:5].tolist(), got[tuple(bad[0])], exp[tuple(bad[0])])


def _pw(pwm_list):
    return so.pack_pwms(pwm_list)


def _rows(lengths, seed):
    rng = np.random.default_rng(seed)
    return [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(n))].copy() for n in lengths]


def _ragged(ctx, rows):
    off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    return ctx.seqs_from_ragged(np.concatenate(rows) if rows else np.zeros(0, np.uint8), off)


def _motifs(seed, n=24, lo=8, hi=40):
    cms = [synth.count_matrix_from_sites(["TGACGTCA"] * 40), synth.count_matrix_from_sites(["AAAAAAAAAAAA"] * 40)] + \
        synth.random_count_matrices(n, lo, hi, seed)
    return synth.motifs_from_count_matrices(cms)


@pytest.mark.parametrize("fwd,rc", [(True, True), (True, False), (False, True)])
def test_fixed_store_planted(ctx, fwd, rc):
    a = synth.planted_gapped(300, 200, 31)
    ms = _motifs(32, n=30, lo=6, hi=30)
    pw, lens = _pw(ms.pwms)
    s = ctx.seqs_from_ascii(a)
    got = ctx.scan_best(s, pw, lens, fwd=fwd, rc=rc)
    s.free()
    exp = oracle_best(ms.pwms, list(a), (1 if fwd else 0) | (2 if rc else 0), check_literal=True)
    _same(got, exp)
    assert got["found"].all()
    if fwd and rc:
        assert (got["comp"] == 1).any() and (got["comp"] == 0).any()
    else:
        assert (got["comp"] == (0 if fwd else 1)).all()


LENGTHS_A = [0, 3, 16, 17, 31, 32, 100, 160, 255, 37, 1, 64, 200, 256, 0, 129, 48, 7, 250, 95] * 6
LENGTHS_B = [250, 5, 0, 33, 128, 249, 80, 17, 112, 9, 190] * 8


@pytest.mark.parametrize("lengths,seed", [(LENGTHS_A, 1), (LENGTHS_B, 2)])
def test_ragged_rows_equal_their_own_scan(ctx, lengths, seed):
    """empty rows, rows shorter than every motif, multiples of 16 and not; the poly-A motif would score best in the padding"""
    rows = _rows(lengths, seed)
    ms = _motifs(seed + 20, n=20, lo=4, hi=40)
    pw, lens = _pw(ms.pwms)
    s = _ragged(ctx, rows)
    got = ctx.scan_best(s, pw, lens)
    s.free()
    exp = oracle_best(ms.pwms, rows)
    _same(got, exp)
    L = np.array(lengths)
    assert not got["found"][L == 0].any()
    pa = got[:, 1]                                                      # poly-A (12 columns)
    assert (pa["found"] == (L >= 12)).all()
    assert (pa["pos"][L >= 12] + 12 <= L[L >= 12]).all()


def _int_pwm(cols):
    return np.asarray(cols, np.float16).T.copy()                       # cols: list of [A, C, G, T] -> (4, len)


def test_ties(ctx):
    rng = np.random.default_rng(5)
    site = b"GATTACAGG"
    rows = _rows([120] * 6, 6)
    for r in rows:
        r[20:29] = np.frombuffer(site, np.uint8)
        r[77:86] = np.frombuffer(site, np.uint8)
    # the site motif: +2 per matching base, -1 otherwise (integers: every sum exact)
    site_pwm = _int_pwm([[2 if c == b else -1 for b in "ACGT"] for c in site.decode()])
    # palindromic integer PWM: reverse(pwm) == pwm, so both strands give the same bits at every start
    half = rng.integers(-3, 4, (3, 4))
    pal_cols = list(half) + [[1, 0, 0, 1]] + [c[::-1] for c in half[::-1]]
    pal = _int_pwm(pal_cols)
    assert np.array_equal(pal[::-1, ::-1], pal)
    flat = np.full((4, 7), np.float16(0.5))                            # every window scores 3.5
    pwms = [site_pwm, pal, flat]
    pw, lens = _pw(pwms)
    s = _ragged(ctx, rows)
    got = ctx.scan_best(s, pw, lens)
    s.free()
    _same(got, oracle_best(pwms, rows))
    assert (got["pos"][:, 0] == 20).all() and (got["comp"][:, 0] == 0).all()
    assert (got["comp"][:, 1] == 0).all()
    assert (got["pos"][:, 2] == 0).all() and (got["comp"][:, 2] == 0).all()
    assert (got["score_f16"][:, 2] == np.float16(3.5).view(np.uint16)).all()


def test_non_finite_entries(ctx):
    rows = _rows([90, 150, 47, 200, 5], 7)
    rng = np.random.default_rng(8)
    base = [rng.normal(0, 1, (4, 10)).astype(np.float16) for _ in range(5)]
    base[0][2, 3] = np.inf                                             # windows without G at column 3 are NaN (Inf * 0)
    base[1][0, 4] = -np.inf                                            # the same with -Inf
    base[2][1, 0] = np.inf
    base[2][2, 0] = -np.inf                                            # column 0: every window NaN
    base[3][0, 5] = -np.inf                                            # windows with A at column 5 are -Inf, the others NaN
    base[4][3, 9] = np.nan                                             # NaN unless T at column 9 ... and then NaN too: all NaN
    pw, lens = _pw(base)
    s = _ragged(ctx, rows)
    got = ctx.scan_best(s, pw, lens)
    s.free()
    _same(got, oracle_best(base, rows))
    found = got["found"][:4]
    assert found[:, 0].all() and not got["found"][:, 2].any() and not got["found"][:, 4].any()
    assert (got["pos"][:, 2] == NONE).all() and (got["score_f16"][:, 2] == 0).all()
    assert got["found"][:4, 1].all() and (got["score_f16"][:4, 1] == 0xFC00).all()      # a -Inf best score
    assert got["found"][:4, 3].all() and (got["score_f16"][:4, 3] == 0xFC00).all()
    assert not got["found"][4].any()                                   # 5 bases: no window of 10 columns


def test_long_pwms_mixed_with_short(ctx):
    rows = _rows([300, 70, 0, 200, 66, 65, 299, 150, 12, 288], 9)
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(3, 65, 120, 10) + synth.random_count_matrices(6, 8, 30, 11))
    pw, lens = _pw(ms.pwms)
    s = _ragged(ctx, rows)
    for fwd, rc in ((True, True), (False, True), (True, False)):
        got = ctx.scan_best(s, pw, lens, fwd=fwd, rc=rc)
        _same(got, oracle_best(ms.pwms, rows, (1 if fwd else 0) | (2 if rc else 0)))
    s.free()


def test_row_over_131072_positions(ctx):
    """the reducer cuts a row into chunks of 1024 position blocks; the best site sits in the last one"""
    site = "TGACGTCATTGACGTCA"
    rows = _rows([140_003, 5000, 0, 17, 131_088], 12)
    rows[0][139_950:139_950 + len(site)] = np.frombuffer(site.encode(), np.uint8)
    rows[4][131_088 - len(site):] = np.frombuffer(site.encode(), np.uint8)
    ms = synth.motifs_from_count_matrices([synth.count_matrix_from_sites([site] * 30)] + synth.random_count_matrices(5, 8, 30, 13))
    pw, lens = _pw(ms.pwms)
    s = _ragged(ctx, rows)
    got = ctx.scan_best(s, pw, lens)
    s.free()
    _same(got, oracle_best(ms.pwms, rows))
    assert got["pos"][0, 0] == 139_950 and got["pos"][4, 0] == 131_088 - len(site)


def test_batches_equal_small_stores(ctx):
    """40 000 x 2000 bp against 500 PWMs needs about 20 GB of keys: three batches under the 8 GB budget"""
    a = synth.random_ascii(40_000, 2000, 14)
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(500, 8, 40, 15))
    pw, lens = _pw(ms.pwms)
    s = ctx.seqs_from_ascii(a)
    got = ctx.scan_best(s, pw, lens)
    t, n = ctx.last_timing()
    assert n["scan"] >= 3
    pick = np.array([0, 1, 2, 9_000, 16_643, 16_644, 16_645, 27_000, 33_287, 33_288, 39_998, 39_999], np.int64)   # 16 644 rows a batch
    g = s.gather(pick)
    small = ctx.scan_best(g, pw, lens)
    g.free()
    s.free()
    _same(got[pick], small)
    _same(small[:6], oracle_best(ms.pwms, list(a[pick[:6]])))


def test_async_upload(ctx):
    a = synth.planted_gapped(3000, 300, 16)
    ms = _motifs(17, n=12)
    pw, lens = _pw(ms.pwms)
    s = ctx.seqs_from_ascii(a)
    exp = ctx.scan_best(s, pw, lens)
    s.free()
    buf = np.ascontiguousarray(a)
    sa = ctx.seqs_from_host_ptr(buf.ctypes.data, a.shape[0], a.shape[1], wait=False)
    got = ctx.scan_best(sa, pw, lens)
    sa.free()
    assert got.tobytes() == exp.tobytes()
    _same(got[:50], oracle_best(ms.pwms, list(a[:50])))


def test_consistent_with_scan_hits(ctx):
    rows = _rows(LENGTHS_B, 18)
    ms = _motifs(19, n=16)
    pw, lens = _pw(ms.pwms)
    s = _ragged(ctx, rows)
    best = ctx.scan_best(s, pw, lens)
    hits, _ = ctx.scan(s, pw, lens, None, want_counts=False)
    s.free()
    sc = hits["score_f16"].view(np.float16).astype(np.float32)
    bsc = best["score_f16"].view(np.float16).astype(np.float32)
    checked = 0
    for n in range(len(rows)):
        for k in range(len(lens)):
            b = best[n, k]
            if not b["found"] or not bsc[n, k] > 0:
                continue
            sel = (hits["seq"] == n) & (hits["motif"] == k)
            top = sc[sel].max()
            h = hits[sel][sc[sel] == top]
            h = h[np.lexsort((h["comp"], h["pos"]))][0]
            assert (b["pos"], b["comp"], b["score_f16"]) == (h["pos"], h["comp"], h["score_f16"])
            checked += 1
    assert checked > 100


def test_errors_and_tensor_core_scan_after(ctx):
    a = synth.planted_gapped(200, 150, 20)
    ms = _motifs(21, n=10)
    pw, lens = _pw(ms.pwms)
    s = ctx.seqs_from_ascii(a)
    ctx.scan_best(s, pw, lens)
    out = np.zeros((s.N, len(lens)), _lib.BEST_DTYPE)
    lib = ctx._lib
    pwu = np.ascontiguousarray(pw).view(np.uint16)
    for flags, ptr in ((_lib.SCAN_FWD | _lib.SCAN_RC | _lib.SCAN_REDUCE, out), (_lib.SCAN_FWD | _lib.SCAN_WANT_HITS, out),
                       (_lib.SCAN_FWD | _lib.SCAN_WANT_COUNTS, out), (0, out), (_lib.SCAN_FWD | _lib.SCAN_RC, None)):
        rc = lib.mb200_scan_best(ctx._h, s._h, _lib._ptr(pwu), _lib._ptr(lens), len(lens), pw.shape[0], flags, _lib._ptr(ptr))
        assert rc == _lib.E_INVALID, flags
    ctx.scan_best(s, pw, lens)
    thr = synth.stated_thresholds(ms, 0.5)
    hits, counts = ctx.scan(s, pw, lens, thr)
    assert _lib.scan_last_path(ctx) == 1
    oh, oc = so.scan(pw, lens, so.ascii_to_codes(a), thr)
    assert len(hits) == len(oh) > 0 and np.array_equal(counts, oc)
    for f in ("seq", "pos", "motif", "score_f16", "comp"):
        assert np.array_equal(hits[f], oh[f])
    _, c2 = ctx.scan(s, pw, lens, thr, want_hits=False)
    assert np.array_equal(c2, oc)
    s.free()


# ---- records.best_sites and the statistics on it --------------------------------------------------------------------------
def _write_fasta(path, names, seqs, width=60):
    with open(path, "w") as fh:
        for n, s in zip(names, seqs):
            fh.write(f">{n} peak\n")
            for i in range(0, len(s), width):
                fh.write(s[i:i + width] + "\n")


def test_best_sites_fasta_matches_per_fragment_oracle(ctx, tmp_path):
    rng = np.random.default_rng(22)
    names, seqs = [], []
    for i, L in enumerate((5000, 1200, 333, 17, 0, 2600, 90, 45)):
        s = bytearray(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)].tobytes())
        for _ in range(3):
            if L > 20:
                p, q = sorted(int(x) for x in rng.integers(0, L, 2))
                s[p:min(q, p + 200)] = b"N" * (min(q, p + 200) - p)
        if L > 40:
            s[:5] = b"NNNNN"; s[-3:] = b"nnn"; s[L // 2] = ord("R")
            s[10:30] = s[10:30].lower()
        for p in rng.integers(0, max(L - 8, 1), L // 300):
            if L >= 8:
                s[p:p + 8] = b"TGACGTCA"
        names.append(f"rec{i}")
        seqs.append(s.decode())
    path = os.path.join(tmp_path, "g.fa")
    _write_fasta(path, names, seqs)
    ms = _motifs(23, n=8)
    bs = records.best_sites(ctx, path, ms.pwms)
    assert bs.names == names and bs.lengths.tolist() == [len(x) for x in seqs]
    frags = []                                                          # (record, start, bases)
    for ri, s in enumerate(seqs):
        u = s.upper()
        i = 0
        while i < len(u):
            if u[i] in "ACGT":
                j = i
                while j < len(u) and u[j] in "ACGT":
                    j += 1
                frags.append((ri, i, np.frombuffer(u[i:j].encode(), np.uint8)))
                i = j
            else:
                i += 1
    fb = oracle_best(ms.pwms, [f[2] for f in frags])
    # per record and motif, brute force over its fragments: highest score, then lowest record position, then forward
    R, K = len(seqs), len(ms.pwms)
    found, pos = np.zeros((R, K), bool), np.full((R, K), -1, np.int64)
    comp, score = np.zeros((R, K), np.uint8), np.zeros((R, K), np.uint16)
    for r in range(R):
        for k in range(K):
            cands = [(int(_ord(b["score_f16"])), -(f[1] + int(b["pos"])), -int(b["comp"]), int(b["score_f16"]))
                     for f, b in zip(frags, fb[:, k]) if f[0] == r and b["found"]]
            if cands:
                o, npos, ncomp, bits = max(cands)
                found[r, k], pos[r, k], comp[r, k], score[r, k] = True, -npos, -ncomp, bits
    assert np.array_equal(bs.found, found) and np.array_equal(bs.pos, pos) and np.array_equal(bs.comp, comp)
    assert np.array_equal(bs.score.view(np.uint16), score)
    assert bs.found[0].all() and not bs.found[4].any()
    assert sum(f[0] == 0 for f in frags) > 1                            # record 0 is cut into several fragments
    # every position is in record coordinates: the window lies on A/C/G/T of the record
    for r in range(len(seqs)):
        for k in range(len(ms.pwms)):
            if bs.found[r, k]:
                w = seqs[r][bs.pos[r, k]: bs.pos[r, k] + ms.pwms[k].shape[1]].upper()
                assert set(w) <= set("ACGT")


def test_central_enrichment_and_auc_end_to_end(ctx, tmp_path):
    rng = np.random.default_rng(24)
    R, L = 2000, 500
    site = "TGACGTCATCGA"
    rows = synth.random_ascii(R, L, 25).copy()
    planted = rng.random(R) < 0.6
    for r in np.nonzero(planted)[0]:
        c = L // 2 + int(rng.integers(-10, 11))                        # site centre within +-10 bp of the peak centre
        p = c - len(site) // 2
        s = site if rng.random() < 0.5 else site[::-1].translate(str.maketrans("ACGT", "TGCA"))
        rows[r, p:p + len(site)] = np.frombuffer(s.encode(), np.uint8)
    path = os.path.join(tmp_path, "peaks.fa")
    _write_fasta(path, [f"peak{i}" for i in range(R)], [bytes(r).decode() for r in rows])
    # control: a random PWM that does not resemble the planted site (one that does, such as seed 26's, is centrally enriched for real)
    ms = synth.motifs_from_count_matrices([synth.count_matrix_from_sites([site] * 40)] + synth.random_count_matrices(1, 10, 10, 27))
    lens = ms.lens
    rec = records.read_records(path)
    fg = records.best_sites(ctx, rec, ms.pwms)
    bg = records.best_sites(ctx, records.shuffle_records(ctx, rec, 2, seed=27), ms.pwms)
    assert fg.found.all() and bg.found.all()
    ce = records.central_enrichment(fg, lens)
    auc = records.best_site_auc(fg, bg)
    assert ce.p_adj[0] < 1e-10 and ce.k[0] > ce.expected[0] * 3
    # 40 % of the peaks carry no site and score like the background, so the AUC of the whole set is about 0.6 + 0.4 / 2
    assert auc[0] > 0.75
    sub = lambda b, m: records.BestSites([], b.lengths[m], b.score[m], b.pos[m], b.comp[m], b.found[m])
    assert records.best_site_auc(sub(fg, planted), bg)[0] > 0.9
    assert ce.p_adj[1] > 1e-3 and 0.4 < auc[1] < 0.6
