"""Ragged stores (rows of different lengths, mb200_seqs_from_ascii_ragged) and scan_fasta.  A scan of a ragged store must return
exactly what the same scan returns for each row on its own: checked bit-exact (positions, strands, Float16 score bits, counts)
against the oracle run on each group of equal-length rows."""
import os

import numpy as np
import pytest

import motifs_jl_b200 as mb
from motifs_jl_b200 import _lib, inference, loadfasta, records, synth
from oracle import scan_oracle as so

pytestmark = pytest.mark.gpu

FIELDS = ("seq", "pos", "motif", "score_f16", "comp")


def _rows(lengths, seed):
    rng = np.random.default_rng(seed)
    return [np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(n))].copy() for n in lengths]


def _plant(rows, site, seed, every=3):
    rng = np.random.default_rng(seed)
    s = np.frombuffer(site.encode(), np.uint8)
    for r in rows[::every]:
        if len(r) >= len(s):
            p = int(rng.integers(0, len(r) - len(s) + 1))
            r[p:p + len(s)] = s
    return rows


def _ragged(ctx, rows):
    off = np.concatenate([[0], np.cumsum([len(r) for r in rows])]).astype(np.int64)
    return ctx.seqs_from_ragged(np.concatenate(rows) if rows else np.zeros(0, np.uint8), off)


def _oracle(pw, lens, rows, thr, strands=3, want_hits=True):
    """the oracle on every group of equal-length rows, hits re-numbered to the row index and sorted (seq, motif, comp, pos)"""
    K = pw.shape[2]
    counts = np.zeros((K, 4), np.int64)
    parts = []
    L = np.array([len(r) for r in rows])
    for n in np.unique(L):
        if n == 0:
            continue
        idx = np.nonzero(L == n)[0]
        h, c = so.scan(pw, lens, so.ascii_to_codes(np.stack([rows[i] for i in idx])), thr, strands, want_hits=want_hits)
        counts += c
        if want_hits:
            h = h.copy()
            h["seq"] = idx[h["seq"]]
            parts.append(h)
    if not want_hits:
        return None, counts
    h = np.concatenate(parts) if parts else np.zeros(0, so.HIT_DTYPE)
    return h[np.lexsort((h["pos"], h["comp"], h["motif"], h["seq"]))], counts


def _same_hits(h, oh):
    assert len(h) == len(oh)
    for f in FIELDS:
        assert np.array_equal(h[f], oh[f]), f


def _check(ctx, rows, ms, thr=None, tc=None):
    pw, lens = so.pack_pwms(ms.pwms)
    seqs = _ragged(ctx, rows)
    assert np.array_equal(seqs.lengths, [len(r) for r in rows])
    oh, oc = _oracle(pw, lens, rows, thr)
    h, c = ctx.scan(seqs, pw, lens, thr)
    if tc is not None:
        assert _lib.scan_last_path(ctx) == tc
    _same_hits(h, oh)
    assert np.array_equal(c, oc)
    _, c2 = ctx.scan(seqs, pw, lens, thr, want_hits=False)
    if tc is not None:
        assert _lib.scan_last_path(ctx) == tc
    assert np.array_equal(c2, oc)
    if thr is not None:
        h3, c3 = ctx.scan(seqs, pw, lens, thr, tensor=False)
        assert _lib.scan_last_path(ctx) == 0
        _same_hits(h3, oh)
        assert np.array_equal(c3, oc)
    seqs.free()
    return oh, oc


# lengths: empty rows, rows shorter than every PWM, multiples of 16 and not; the longest row a multiple of 16 (256) or not (250)
LENGTHS_A = [0, 3, 16, 17, 31, 32, 100, 160, 255, 37, 1, 64, 200, 256, 0, 129, 48, 7, 250, 95] * 6
LENGTHS_B = [250, 5, 0, 33, 128, 249, 80, 17, 112, 9, 190] * 8


def _motifs(seed, n=24, lo=8, hi=40):
    cms = [synth.count_matrix_from_sites(["TGACGTCA"] * 40), synth.count_matrix_from_sites(["AAAAAAAAAAAA"] * 40)] + \
        synth.random_count_matrices(n, lo, hi, seed)
    return synth.motifs_from_count_matrices(cms)


@pytest.mark.parametrize("lengths,seed", [(LENGTHS_A, 1), (LENGTHS_B, 2)])
def test_ragged_thresholded_tensor_and_simt(ctx, lengths, seed):
    """thresholded scans on the tensor-core path (and tensor=False); the poly-A motif would match the zero padding everywhere"""
    rows = _plant(_rows(lengths, seed), "TGACGTCA", seed + 10)
    ms = _motifs(seed + 20)
    oh, oc = _check(ctx, rows, ms, synth.stated_thresholds(ms, 0.5), tc=1)
    assert len(oh) > 0 and oc[0, 0] > 0


@pytest.mark.parametrize("lengths,seed", [(LENGTHS_A, 3), (LENGTHS_B, 4)])
def test_ragged_score_positive(ctx, lengths, seed):
    rows = _rows(lengths, seed)
    ms = _motifs(seed + 20, n=10, lo=1, hi=64)
    _check(ctx, rows, ms, None, tc=0)


def test_ragged_long_pwm(ctx):
    """PWMs longer than 64 columns take scan_long_kernel; rows shorter and longer than them"""
    rows = _rows([300, 70, 0, 200, 66, 65, 299, 150, 12, 288], 5)
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(3, 65, 120, 6) + synth.random_count_matrices(6, 8, 30, 7))
    for p in ms.pwms[:3]:
        p[:] = (p / np.float16(8)).astype(np.float16)
        p[:, ::3] = np.abs(p[:, ::3])
    _, oc = _check(ctx, rows, ms)
    assert oc[:3, 0].sum() > 0
    _check(ctx, rows, ms, synth.stated_thresholds(ms, 0.4))


def test_ragged_row_over_131072_positions(ctx):
    """one row long enough for the blocked counting of chromosome-scale sequences (more than 4096 mask words)"""
    rows = _plant(_rows([140_003, 5000, 0, 17, 131_000, 131_088], 8), "TGACGTCATTGACGTCA", 9, every=1)
    ms = synth.motifs_from_count_matrices([synth.count_matrix_from_sites(["TGACGTCATTGACGTCA"] * 30)] + synth.random_count_matrices(8, 8, 40, 10))
    pw, lens = so.pack_pwms(ms.pwms)
    thr = synth.stated_thresholds(ms, 0.6)
    seqs = _ragged(ctx, rows)
    for t in (thr, None):
        _, oc = _oracle(pw, lens, rows, t, want_hits=False)
        for tensor in (True, False):
            _, c = ctx.scan(seqs, pw, lens, t, want_hits=False, tensor=tensor)
            assert np.array_equal(c, oc)
    seqs.free()


def test_ragged_scan_hist(ctx):
    rows = _rows(LENGTHS_A, 11)
    ms = _motifs(12, n=8)
    pw, lens = so.pack_pwms(ms.pwms)
    seqs = _ragged(ctx, rows)
    got = _lib.scan_hist(ctx, seqs, pw, lens)
    seqs.free()
    exp = np.zeros_like(got)
    L = np.array([len(r) for r in rows])
    for n in np.unique(L[L > 0]):
        s = ctx.seqs_from_ascii(np.stack([rows[i] for i in np.nonzero(L == n)[0]]))
        exp += _lib.scan_hist(ctx, s, pw, lens)
        s.free()
    assert np.array_equal(got, exp)
    # and the histogram counts the oracle's hits
    oh, _ = _oracle(pw, lens, rows, None)
    assert int(got.sum()) == len(oh)


def test_equal_lengths_ragged_equals_fixed(ctx):
    a = synth.planted_gapped(300, 120, 13)
    rows = [r.copy() for r in a]
    ms = _motifs(14, n=12)
    pw, lens = so.pack_pwms(ms.pwms)
    thr = synth.stated_thresholds(ms, 0.5)
    r, f = _ragged(ctx, rows), ctx.seqs_from_ascii(a)
    assert (r.N, r.Lb) == (f.N, f.Lb) and np.array_equal(r.download(), f.download())
    for t in (thr, None):
        for wh in (True, False):
            hr, cr = ctx.scan(r, pw, lens, t, want_hits=wh)
            hf, cf = ctx.scan(f, pw, lens, t, want_hits=wh)
            assert np.array_equal(cr, cf) and (not wh or hr.tobytes() == hf.tobytes())
    assert np.array_equal(_lib.scan_hist(ctx, r, pw, lens), _lib.scan_hist(ctx, f, pw, lens))
    cr, tr = r.base_counts()
    cf, tf = f.base_counts()
    assert np.array_equal(cr, cf) and np.array_equal(tr, tf)
    assert np.array_equal(r.to_ascii(), f.to_ascii())
    for k in (1, 2, 3, 4):
        sr, sf = r.shuffle(k, 77, first_stream=5), f.shuffle(k, 77, first_stream=5)
        assert np.array_equal(sr.download(), sf.download())
        sr.free(); sf.free()
    r.free(); f.free()


def _kmers(row, k):
    return sorted(row[i:i + k].tobytes() for i in range(len(row) - k + 1))


@pytest.mark.parametrize("lengths", [LENGTHS_A[:40], [70_000, 300, 0, 5, 66_000, 1, 65_536, 65_537]])
def test_ragged_shuffle(ctx, lengths):
    rows = _rows(lengths, 15)
    s = _ragged(ctx, rows)
    ks = (1, 2, 3, 4) if max(lengths) <= 65536 else (1,)
    for k in ks:
        sh = s.shuffle(k, 123, first_stream=0)
        assert np.array_equal(sh.lengths, lengths)
        out = sh.to_ascii()
        words = sh.download()
        for i, (row, n) in enumerate(zip(rows, lengths)):
            got = out[i, :n]
            assert not out[i, n:].any()                                      # to_ascii writes 0 past the row
            if n % 16:
                assert words[i, n // 16] >> np.uint32(2 * (n % 16)) == 0      # the padding stays zero
            assert not words[i, (n + 15) // 16:].any()
            assert _kmers(got, k) == _kmers(row, k)                        # k-mer counts preserved
            if i % 7 == 0 or n > 65536:
                alone = ctx.seqs_from_ascii(row[None, :]) if n else None
                if alone is not None:
                    a2 = alone.shuffle(k, 123, first_stream=i)
                    assert np.array_equal(a2.to_ascii()[0], got)               # row i = that row shuffled alone on stream i
                    a2.free(); alone.free()
        c, t = sh.base_counts()
        assert c.sum() == sum(lengths) and t.sum() == sum(max(n - 1, 0) for n in lengths)
        sh.free()
    if max(lengths) > 65536:
        with pytest.raises(mb.MB200Error) as e:
            s.shuffle(2, 1)
        assert e.value.code == _lib.E_UNSUPPORTED
    s.free()


def test_ragged_gather_and_base_counts(ctx):
    rows = _rows(LENGTHS_B, 16)
    s = _ragged(ctx, rows)
    idx = np.array([3, 0, 10, 10, 2], np.int64)
    g = s.gather(idx)
    assert np.array_equal(g.lengths, [len(rows[i]) for i in idx])
    exp = _ragged(ctx, [rows[i] for i in idx])
    assert np.array_equal(g.download(), exp.download()) and np.array_equal(g.to_ascii(), exp.to_ascii())
    c, t = s.base_counts()
    allb = np.concatenate(rows)
    assert np.array_equal(c, [(allb == ord(x)).sum() for x in "ACGT"])
    tt = np.zeros((4, 4), np.int64)
    codes = {ord(x): i for i, x in enumerate("ACGT")}
    for r in rows:
        for a_, b_ in zip(r[:-1], r[1:]):
            tt[codes[a_], codes[b_]] += 1
    assert np.array_equal(t, tt)
    g.free(); exp.free(); s.free()


def test_ragged_bad_symbol_and_empty(ctx):
    rows = _rows([10, 20, 5], 17)
    rows[1][4] = ord("N")
    with pytest.raises(mb.MB200Error) as e:
        _ragged(ctx, rows)
    assert e.value.code == _lib.E_BAD_SEQUENCE
    s = _ragged(ctx, [np.zeros(0, np.uint8)] * 3)
    pw, lens = so.pack_pwms(_motifs(18, n=2).pwms)
    h, c = ctx.scan(s, pw, lens)
    assert len(h) == 0 and not c.any()
    s.free()


def test_ragged_count_matrices(ctx):
    rows = _rows([40, 12, 70], 19)
    s = _ragged(ctx, rows)
    lens = np.array([8, 10], np.int64)
    ok = np.zeros(3, _lib.SITE_DTYPE)
    ok[:] = [(0, 0, 32, 0), (1, 1, 2, 1), (0, 2, 62, 0)]                    # windows end exactly at the row's end or inside it
    got = _lib.count_matrices(ctx, s, ok, lens)
    assert got[0].sum() == 16 and got[1].sum() == 10
    bad = ok.copy()
    bad[1] = (1, 1, 3, 0)                                                    # ends one base past row 1 (12 bases), inside Lb = 70
    with pytest.raises(mb.MB200Error) as e:
        _lib.count_matrices(ctx, s, bad, lens)
    assert e.value.code == _lib.E_INVALID
    s.free()


def test_csc_rejects_ragged_store(ctx):
    from motifs_jl_b200 import model as mdl
    hp = mdl.Hyperparam()
    rows = _rows([100] * 11 + [60], 20)
    s = _ragged(ctx, rows)
    assert s.Lb == 100
    m = _lib.CscModel(ctx, hp, 100)
    idx = np.arange(hp.batch_size) % s.N
    for call in (lambda: m.loss_grad(s, idx), lambda: m.step_begin(s, idx)):
        with pytest.raises(mb.MB200Error) as e:
            call()
        assert e.value.code == _lib.E_UNSUPPORTED
    m.free()
    mf = _lib.CscModel(ctx, hp, 100, forward_only=True)
    for shard in (None, (0, 1)):
        with pytest.raises(mb.MB200Error) as e:
            mf.codes(s, 0, hp.batch_size, shard=shard)
        assert e.value.code == _lib.E_UNSUPPORTED
    mf.free(); s.free()


# ---- scan_fasta ---------------------------------------------------------------------------------------------------------
def _write_fasta(path, names, seqs, width=60):
    with open(path, "w") as fh:
        for n, s in zip(names, seqs):
            fh.write(f">{n} some description\n")
            for i in range(0, len(s), width):
                fh.write(s[i:i + width] + "\n")


def _genome_like(seed):
    rng = np.random.default_rng(seed)
    recs = []
    for L in (5000, 1200, 333, 17, 0, 2600, 90):
        s = bytearray(np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, L)].tobytes())
        for _ in range(3):                                                   # N runs (also at the ends) and IUPAC letters
            if L > 20:
                p, q = sorted(int(x) for x in rng.integers(0, L, 2))
                s[p:min(q, p + 200)] = b"N" * (min(q, p + 200) - p)
        if L > 40:
            s[:5] = b"NNNNN"; s[-3:] = b"nnn"; s[L // 2] = ord("R")
            s[10:30] = s[10:30].lower()                                      # soft-masked bases are scanned
        site = b"TGACGTCA"
        for p in rng.integers(0, max(L - 8, 1), L // 150):
            if L >= 8:
                s[p:p + 8] = site
        recs.append(s.decode())
    return [f"rec{i}" for i in range(len(recs))], recs


def test_scan_fasta_matches_per_fragment_oracle(ctx, tmp_path):
    names, seqs = _genome_like(21)
    path = os.path.join(tmp_path, "g.fa")
    _write_fasta(path, names, seqs)
    ms = _motifs(22, n=10)
    thr = synth.stated_thresholds(ms, 0.5)
    res = records.scan_fasta(ctx, path, ms.pwms, thr)
    assert res.names == names
    # per-fragment oracle, mapped to record coordinates
    pw, lens = so.pack_pwms(ms.pwms)
    frags = []
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
    frags = [f for f in frags if len(f[2]) >= lens.min()]
    oh, oc = _oracle(pw, lens, [f[2] for f in frags], thr)
    assert np.array_equal(res.counts, oc)
    assert res.S == sum(len(f[2]) for f in frags)
    rec = np.array([frags[i][0] for i in oh["seq"]], np.int64)
    pos = np.array([frags[i][1] for i in oh["seq"]], np.int64) + oh["pos"]
    o = np.lexsort((pos, oh["comp"], oh["motif"], rec))
    assert len(res.hits) == len(oh) > 0
    assert np.array_equal(res.hits["record"], rec[o]) and np.array_equal(res.hits["pos"], pos[o])
    for f in ("motif", "comp", "score_f16"):
        assert np.array_equal(res.hits[f], oh[f][o])
    # one bucket per distinct length: same result
    res0 = records.scan_fasta(ctx, path, ms.pwms, thr, max_padding=0)
    assert res0.hits.tobytes() == res.hits.tobytes() and np.array_equal(res0.counts, res.counts) and res0.S == res.S
    # a shuffled background: p-values for every motif, deterministic in the seed
    r1 = records.scan_fasta(ctx, path, ms.pwms, thr, background=2, seed=5, want_hits=False)
    r2 = records.scan_fasta(ctx, records.read_records(path), ms.pwms, thr, background=2, seed=5, want_hits=False)
    assert r1.hits is None and r1.S_bg == r1.S and np.array_equal(r1.counts_bg, r2.counts_bg)
    assert np.array_equal(r1.pvalues, r2.pvalues) and r1.pvalues[0] < 1e-3


def test_scan_fasta_shuffle_uses_fragment_streams(ctx, tmp_path):
    names, seqs = _genome_like(23)
    path = os.path.join(tmp_path, "g.fa")
    _write_fasta(path, names, seqs)
    rec = records.read_records(path)
    a = records.shuffle_records(ctx, rec, 2, seed=9)
    b = records.shuffle_records(ctx, rec, 2, seed=9, chunk_bases=3000)          # other chunks, same fragments and streams
    assert np.array_equal(a.bases, b.bases)
    off = rec.frag_offsets
    f = int(np.argmax(rec.frag_len))
    row = rec.bases[off[f]:off[f + 1]]
    s = ctx.seqs_from_ascii(row[None, :])
    sh = s.shuffle(2, 9, first_stream=f)
    assert np.array_equal(sh.to_ascii()[0], a.bases[off[f]:off[f + 1]])
    sh.free(); s.free()


def test_scan_fasta_pvalues_equal_pvec_from_test_data(ctx, tmp_path):
    a = synth.planted_gapped(800, 100, 24)
    data = loadfasta.FASTA_DNA([bytes(r).decode() for r in a], ctx, rng=np.random.default_rng(3))
    bg = loadfasta.get_data_bg(data)
    ms = synth.motifs_from_count_matrices([synth.count_matrix_from_sites(["TGACGT"] * 40), synth.count_matrix_from_sites(["ACGTCA"] * 40)]
                                          + synth.random_count_matrices(4, 8, 20, 25), bg)
    ms.score_thresh = synth.stated_thresholds(ms, 0.5)
    pvec, _ = inference.pvec_from_test_data(ms, data)
    fg_path, bg_path = os.path.join(tmp_path, "fg.fa"), os.path.join(tmp_path, "bg.fa")
    loadfasta.write_fasta(fg_path, data.ascii_test)
    loadfasta.write_fasta(bg_path, data.ascii_bg_test)
    res = records.scan_fasta(ctx, fg_path, ms, background=bg_path, want_hits=False)
    assert res.S == res.S_bg == data.N_test * data.L
    assert np.array_equal(res.pvalues, pvec)
    assert pvec[0] < 1e-3
    data.free()
