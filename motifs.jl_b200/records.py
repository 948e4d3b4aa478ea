"""Scan FASTA files as they are: peak sets with peaks of different widths, genomes with chromosomes, N runs and unplaced contigs.

`read_records` keeps every record of a FASTA file (mb200_records_read: no cap, no length or N filter).  The scan runs over each
record's N-free FRAGMENTS, the maximal runs of A/C/G/T; N, IUPAC codes and '-' are not scanned.  `bucket_fragments` packs the
fragments into ragged stores (mb200_seqs_from_ascii_ragged), and `scan_fasta` scans them and maps the hits back to record
coordinates.

Bucketing rule (INTEGRATION.md gives it to the Julia host as well): fragments shorter than the shortest PWM are dropped (no start
position fits); the others are sorted by length, longest first, ties by fragment index, and cut greedily into buckets so that
the padding of every bucket is at most `max_padding` (1/8) of the positions its store scans (n_rows x longest row).  The scan's
cost follows the padded positions, so a store never spends more than 1/8 of its time on padding.
"""
from __future__ import annotations

import ctypes as C
import os
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import _lib, inference

RECORD_HIT_DTYPE = np.dtype([("record", "<i8"), ("pos", "<i8"), ("motif", "<u2"), ("comp", "u1"), ("score_f16", "<u2")])


@dataclass
class Records:
    """The records of one FASTA file.  Fragment f is bases[frag_offsets[f]:frag_offsets[f+1]], found at
    [frag_start[f], frag_start[f] + frag_len[f]) of record frag_record[f] (0-based)."""
    names: List[str]
    lengths: np.ndarray          # (R,) int64 record lengths (every sequence byte counts, N included)
    frag_record: np.ndarray      # (F,) int64
    frag_start: np.ndarray       # (F,) int64
    frag_len: np.ndarray         # (F,) int64
    bases: np.ndarray            # uint8 "ACGT", the fragments concatenated

    @property
    def frag_offsets(self) -> np.ndarray:
        return np.concatenate([[0], np.cumsum(self.frag_len)]).astype(np.int64)


@dataclass
class ScanResult:
    """hits: RECORD_HIT_DTYPE sorted by (record, motif, comp, pos), positions 0-based in record coordinates (None without hits).
    counts: (K, 4) int64 as mb200_scan returns them, summed over fragments: {hits, unique starts, coverage with the reference's
    union_ranges quirk (the last interval of every (motif, fragment) with >= 2 hits dropped), true coverage}.
    S: scanned positions = the summed length of the scanned fragments.  With a background: its counts, its S and the right-tail
    Fisher p-value of every motif on column 2 (1.0 when neither side has a hit), as pvec_from_test_data computes them."""
    hits: Optional[np.ndarray]
    counts: np.ndarray
    S: int
    names: List[str]
    counts_bg: Optional[np.ndarray] = None
    S_bg: Optional[int] = None
    pvalues: Optional[np.ndarray] = None


def read_records(path) -> Records:
    lib = _lib.load()
    h = C.c_void_p()
    rc = lib.mb200_records_read(os.fsencode(path), C.byref(h))
    if rc != _lib.OK:
        raise _lib.MB200Error(rc, f"mb200_records_read({path}) failed")
    try:
        nr, nf, nb, nn = C.c_int64(), C.c_int64(), C.c_int64(), C.c_int64()
        lib.mb200_records_counts(h, C.byref(nr), C.byref(nf), C.byref(nb), C.byref(nn))
        names = np.zeros(nn.value, np.uint8)
        lengths = np.zeros(nr.value, np.int64)
        lib.mb200_records_names(h, _lib._ptr(names), _lib._ptr(lengths))
        rec, start, ln = (np.zeros(nf.value, np.int64) for _ in range(3))
        bases = np.zeros(nb.value, np.uint8)
        lib.mb200_records_fragments(h, _lib._ptr(rec), _lib._ptr(start), _lib._ptr(ln), _lib._ptr(bases))
    finally:
        lib.mb200_records_free(h)
    name_list = [b.decode("utf-8", "replace") for b in names.tobytes().split(b"\0")[: nr.value]]
    return Records(name_list, lengths, rec, start, ln, bases)


def bucket_fragments(frag_len, min_len: int, max_padding: float = 1.0 / 8) -> List[np.ndarray]:
    """Fragment indices per ragged store (see the module docstring).  Deterministic; every fragment of at least min_len bases lands
    in exactly one bucket; in each bucket n * longest - sum(lengths) <= max_padding * n * longest.  max_padding = 0 gives one
    bucket per distinct length."""
    L = np.asarray(frag_len, np.int64)
    idx = np.nonzero(L >= max(int(min_len), 1))[0]
    order = idx[np.lexsort((idx, -L[idx]))]
    Ls = L[order].tolist()
    keep = 1.0 - float(max_padding)
    out, i, n = [], 0, len(order)
    while i < n:
        lmax, tot, j = Ls[i], Ls[i], i + 1
        # fragments come longest first: once one does not fit, no later one does
        while j < n and tot + Ls[j] >= keep * (j - i + 1) * lmax:
            tot += Ls[j]
            j += 1
        out.append(order[i:j])
        i = j
    return out


def _pwm_args(motifs_or_pwms, thresh):
    if isinstance(motifs_or_pwms, inference.Motifs):
        ms = motifs_or_pwms
        th = ms.score_thresh if thresh is None else thresh
    else:
        pwms = [np.asarray(p, np.float16) for p in motifs_or_pwms]
        ms = inference.Motifs(pwms=pwms, lens=np.array([p.shape[1] for p in pwms], np.int64))
        th = thresh
    th = None if th is None else np.ascontiguousarray(th, np.float16)
    return inference.pack_pwms(ms), np.ascontiguousarray(ms.lens, np.int64), th


def _scan_records(ctx, rec: Records, pw, lens, thr, want_hits, max_padding):
    K = len(lens)
    counts = np.zeros((K, 4), np.int64)
    off = rec.frag_offsets
    S, parts = 0, []
    for b in bucket_fragments(rec.frag_len, int(lens.min()), max_padding):
        ls = rec.frag_len[b]
        ascii = np.concatenate([rec.bases[off[f]: off[f + 1]] for f in b])
        seqs = ctx.seqs_from_ragged(ascii, np.concatenate([[0], np.cumsum(ls)]))
        try:
            hits, c = ctx.scan(seqs, pw, lens, thr, want_hits=want_hits, want_counts=True)
        finally:
            seqs.free()
        counts += c
        S += int(ls.sum())
        if want_hits and len(hits):
            frag = b[hits["seq"].astype(np.int64)]
            h = np.zeros(len(hits), RECORD_HIT_DTYPE)
            h["record"] = rec.frag_record[frag]
            h["pos"] = rec.frag_start[frag] + hits["pos"].astype(np.int64)
            h["motif"], h["comp"], h["score_f16"] = hits["motif"], hits["comp"], hits["score_f16"]
            parts.append(h)
    hits = None
    if want_hits:
        hits = np.concatenate(parts) if parts else np.zeros(0, RECORD_HIT_DTYPE)
        hits = hits[np.lexsort((hits["pos"], hits["comp"], hits["motif"], hits["record"]))]
    return ScanResult(hits, counts, S, list(rec.names))


def shuffle_records(ctx, rec: Records, k: int, seed: int = 0, chunk_bases: int = 1 << 28) -> Records:
    """The same records with every fragment shuffled on the device (k-mer counts preserved, mb200_seqs_shuffle); fragment f draws
    from random stream f, so its background does not depend on how the fragments are grouped.  Fragments are shuffled in index
    order, in ragged stores of at most chunk_bases padded positions (a longer fragment alone)."""
    off = rec.frag_offsets
    L = rec.frag_len
    out = np.empty_like(rec.bases)
    F, i0 = len(L), 0
    while i0 < F:
        i1, lmax = i0 + 1, int(L[i0])
        while i1 < F and (i1 - i0 + 1) * max(lmax, int(L[i1])) <= chunk_bases:
            lmax = max(lmax, int(L[i1]))
            i1 += 1
        s = ctx.seqs_from_ragged(rec.bases[off[i0]: off[i1]], off[i0: i1 + 1] - off[i0])
        try:
            sh = s.shuffle(k, seed, first_stream=i0)
            try:
                rows = sh.to_ascii()
            finally:
                sh.free()
        finally:
            s.free()
        out[off[i0]: off[i1]] = rows[np.arange(rows.shape[1])[None, :] < L[i0:i1, None]]
        i0 = i1
    return Records(list(rec.names), rec.lengths.copy(), rec.frag_record.copy(), rec.frag_start.copy(), L.copy(), out)


def scan_fasta(ctx, path_or_records, motifs_or_pwms, thresh=None, *, want_hits=True, background=None, seed=0,
               max_padding: float = 1.0 / 8) -> ScanResult:
    """Scan every N-free fragment of a FASTA file (a path or a Records) with both strands of every PWM.

    motifs_or_pwms: an inference.Motifs (its pwms, lens and, when thresh is None, score_thresh) or a list of (4, len) PWMs.
    thresh: K Float16 thresholds (a hit needs score > 0 and score > thresh) or None (score > 0).
    background: None; an int k = a k-mer-preserving shuffle of the same fragments (fragment f on random stream f of `seed`);
    or another FASTA path / Records, scanned the same way.  With a background the result carries its counts and S and the
    Fisher p-values.  max_padding: the bucketing bound (bucket_fragments)."""
    rec = path_or_records if isinstance(path_or_records, Records) else read_records(path_or_records)
    pw, lens, thr = _pwm_args(motifs_or_pwms, thresh)
    res = _scan_records(ctx, rec, pw, lens, thr, want_hits, max_padding)
    if background is None:
        return res
    if isinstance(background, (int, np.integer)) and not isinstance(background, bool):
        bg_rec = shuffle_records(ctx, rec, int(background), seed)
    else:
        bg_rec = background if isinstance(background, Records) else read_records(background)
    bg = _scan_records(ctx, bg_rec, pw, lens, thr, False, max_padding)
    res.counts_bg, res.S_bg = bg.counts, bg.S
    a_, b_ = res.counts[:, 2], bg.counts[:, 2]
    res.pvalues = np.array([1.0 if (a == 0 and b == 0) else inference.fisher_right(a, res.S - a, b, bg.S - b)
                            for a, b in zip(a_.tolist(), b_.tolist())], np.float64)
    return res


# ---- best site per (record, motif), and the statistics built on it ------------------------------------------------------
@dataclass
class BestSites:
    """The best site of every (record, motif): the highest score over every window of the record's N-free fragments on both
    strands, ties to the lowest record position, then to the forward strand (comp = 0).  score: Float16, exactly mb200_scan's
    score of that window; pos: 0-based start in record coordinates, -1 when found is False (no fragment holds a window of the
    motif, or every window is NaN; score and comp are 0 then)."""
    names: List[str]
    lengths: np.ndarray          # (R,) int64 record lengths
    score: np.ndarray            # (R, K) float16
    pos: np.ndarray              # (R, K) int64
    comp: np.ndarray             # (R, K) uint8
    found: np.ndarray            # (R, K) bool


def _h16_ord(bits):
    """Float16 bit patterns -> integers in the order of their values (-0 ties +0)."""
    b = np.asarray(bits, np.uint16).astype(np.int64)
    b = np.where(b == 0x8000, 0, b)
    return np.where(b & 0x8000, ~b & 0xFFFF, b | 0x8000)


def reduce_fragment_best(frag_record, frag_start, fbest, n_records):
    """Fragment best sites (F, K) _lib.BEST_DTYPE -> record best sites: (score (R,K) float16, pos (R,K) int64, comp, found).
    Same rule as the kernel's, in record coordinates: highest score, then lowest record position, then forward."""
    F, K = fbest.shape
    R = int(n_records)
    found = fbest["found"].astype(bool)
    rec = np.broadcast_to(np.asarray(frag_record, np.int64)[:, None], (F, K))[found]
    mot = np.broadcast_to(np.arange(K, dtype=np.int64)[None, :], (F, K))[found]
    pos = (np.asarray(frag_start, np.int64)[:, None] + fbest["pos"].astype(np.int64))[found]
    key = (_h16_ord(fbest["score_f16"][found]).astype(np.uint64) << np.uint64(48)) | \
          (((np.uint64(1 << 47) - np.uint64(1) - pos.astype(np.uint64)) << np.uint64(1))) | \
          (np.uint64(1) - fbest["comp"][found].astype(np.uint64))
    best = np.zeros(R * K, np.uint64)
    np.maximum.at(best, rec * K + mot, key)
    best = best.reshape(R, K)
    f = best != 0
    o = (best >> np.uint64(48)).astype(np.int64)
    bits = np.where(o & 0x8000, o & 0x7FFF, ~o & 0xFFFF).astype(np.uint16)
    score = np.where(f, bits, 0).astype(np.uint16).view(np.float16)
    p = np.where(f, np.int64((1 << 47) - 1) - ((best >> np.uint64(1)) & np.uint64((1 << 47) - 1)).astype(np.int64), -1)
    comp = np.where(f, 1 - (best & np.uint64(1)).astype(np.int64), 0).astype(np.uint8)
    return score, p, comp, f


def best_sites(ctx, path_or_records, motifs_or_pwms, *, max_padding: float = 1.0 / 8) -> BestSites:
    """Best site of every (record, motif) of a FASTA file (a path or a Records): the fragments are scanned in the buckets of
    scan_fasta (mb200_scan_best on both strands) and reduced to records on the host.  motifs_or_pwms: an inference.Motifs or a
    list of (4, len) PWMs (thresholds play no part)."""
    rec = path_or_records if isinstance(path_or_records, Records) else read_records(path_or_records)
    pw, lens, _ = _pwm_args(motifs_or_pwms, None)
    K = len(lens)
    fbest = np.zeros((len(rec.frag_len), K), _lib.BEST_DTYPE)
    off = rec.frag_offsets
    for b in bucket_fragments(rec.frag_len, int(lens.min()), max_padding):
        ls = rec.frag_len[b]
        seqs = ctx.seqs_from_ragged(np.concatenate([rec.bases[off[f]: off[f + 1]] for f in b]), np.concatenate([[0], np.cumsum(ls)]))
        try:
            fbest[b] = ctx.scan_best(seqs, pw, lens)
        finally:
            seqs.free()
    score, pos, comp, found = reduce_fragment_best(rec.frag_record, rec.frag_start, fbest, len(rec.names))
    return BestSites(list(rec.names), rec.lengths.copy(), score, pos, comp, found)


def best_site_auc(fg: BestSites, bg: BestSites) -> np.ndarray:
    """(K,) float64: the probability that a foreground record's best score beats a background record's, ties counted 1/2
    (Mann-Whitney U / (n1 n2)), from average ranks.  Records without a site rank below every found score and tie with each
    other.  NaN for a motif when either side has no records."""
    n1, n2 = fg.found.shape[0], bg.found.shape[0]
    K = fg.found.shape[1]
    out = np.full(K, np.nan)
    if n1 == 0 or n2 == 0:
        return out
    for k in range(K):
        key = np.concatenate([np.where(fg.found[:, k], _h16_ord(fg.score[:, k].view(np.uint16)), 0),
                              np.where(bg.found[:, k], _h16_ord(bg.score[:, k].view(np.uint16)), 0)])
        u, inv, cnt = np.unique(key, return_inverse=True, return_counts=True)
        first = np.concatenate([[0], np.cumsum(cnt)[:-1]])
        avg = first + (cnt + 1) / 2.0                       # 1-based average rank of each distinct key
        r1 = avg[inv[:n1]].sum()
        out[k] = (r1 - n1 * (n1 + 1) / 2.0) / (n1 * n2)
    return out


@dataclass
class CentralEnrichment:
    """Per motif, the central window with the smallest binomial p-value (CentriMo): it holds `window` start positions and `k` of
    the `n` found best sites, `expected` = n * window / (L - m + 1); p = P[Binom(n, window / (L - m + 1)) >= k], p_adj = min(1,
    p * number of windows tried).  window = 0, p = p_adj = 1 when there is no window (L - m <= 1) or no site."""
    window: np.ndarray           # (K,) int64
    k: np.ndarray                # (K,) int64
    n: np.ndarray                # (K,) int64
    expected: np.ndarray         # (K,) float64
    p: np.ndarray                # (K,) float64
    p_adj: np.ndarray            # (K,) float64


def central_enrichment(best: BestSites, lens) -> CentralEnrichment:
    """CentriMo's central enrichment test on summit-centred peaks of one length L.  A start p of a motif of length m lies at
    doubled offset d = 2p + m - L from the centre; for every r in {|d|} below L - m the window {p : |d| <= r} holds r + 1 starts
    and is tested against the uniform null over all L - m + 1 starts (N runs included).  lens: the K motif lengths."""
    L_all = np.unique(np.asarray(best.lengths, np.int64))
    if len(L_all) > 1:
        raise ValueError(f"central_enrichment needs records of one length (summit-centred peaks); found lengths {L_all.tolist()}")
    lens = np.asarray(lens, np.int64)
    K = len(lens)
    res = CentralEnrichment(np.zeros(K, np.int64), np.zeros(K, np.int64), np.zeros(K, np.int64), np.zeros(K), np.ones(K), np.ones(K))
    if len(L_all) == 0:
        return res
    L = int(L_all[0])
    for k in range(K):
        m = int(lens[k])
        f = best.found[:, k]
        N = int(f.sum())
        res.n[k] = N
        if L - m <= 1 or N == 0:
            continue
        npos = L - m + 1
        d = np.abs(2 * best.pos[f, k] + m - L)
        radii = np.arange((L - m) % 2, L - m, 2)        # every |d| below L - m (all of one parity)
        cum = np.cumsum(np.bincount(d, minlength=L - m + 1))
        best_p, best_i = 2.0, 0
        for i, r in enumerate(radii.tolist()):
            p = inference.binom_right(int(cum[r]), N, (r + 1) / npos)
            if p < best_p:
                best_p, best_i = p, i
        r = int(radii[best_i])
        res.window[k], res.k[k] = r + 1, int(cum[r])
        res.expected[k] = N * (r + 1) / npos
        res.p[k], res.p_adj[k] = best_p, min(1.0, best_p * len(radii))
    return res


# ---- secondary-motif spacing around primary sites (SpaMo) ----------------------------------------------------------------
SPACING_SITE_DTYPE = np.dtype([("pos", "<i8"), ("score", "<f2"), ("comp", "u1"), ("found", "?")])


@dataclass
class Spacing:
    """Spacings of secondary motifs around the record best sites of primary motifs (`spacing`).  An anchor is a record whose best
    site of primary p (at pos[r, p] on strand comp[r, p], record coordinates) is a hit (score > 0 and > the primary's threshold)
    with its whole flank [pos - margin, pos + m_p + margin) inside one N-free fragment.  hist[p, k, q, g] counts the anchors of p
    whose best site of secondary k in the two margins is a hit at gap g in quadrant q, in the primary's orientation: 0 same strand
    upstream, 1 same strand downstream, 2 opposite strand upstream, 3 opposite strand downstream.  pos / comp are -1 for records
    that are not anchors of p.  sites (with want_sites): the best window of every (record, primary, secondary) in record
    coordinates, found = counted; pos = -1 where there is no anchor or no window."""
    names: List[str]
    margin: int
    hist: np.ndarray             # (P, K, 4, margin) int64
    n_anchors: np.ndarray        # (P,) int64
    pos: np.ndarray              # (R, P) int64
    comp: np.ndarray             # (R, P) int64
    sites: Optional[np.ndarray] = None      # (R, P, K) SPACING_SITE_DTYPE


def spacing_bin(a, m_p, c_p, s, m_k, c_k):
    """(q, g) of a secondary site at s (length m_k, strand c_k) next to a primary site at a (length m_p, strand c_p), as
    mb200_scan_spacing bins it (element-wise over arrays).  Left of the primary (s < a): g = a - (s + m_k); right: g = s -
    (a + m_p).  Downstream is the right side for c_p = 0 and the left side for c_p = 1; q = 2 (c_k != c_p) + downstream."""
    a, m_p, c_p, s, m_k, c_k = (np.asarray(x, np.int64) for x in (a, m_p, c_p, s, m_k, c_k))
    left = s < a
    g = np.where(left, a - (s + m_k), s - (a + m_p))
    down = (left == (c_p != 0)).astype(np.int64)
    return 2 * (c_k != c_p).astype(np.int64) + down, g


def _hit_mask(score, thresh):
    """score > 0 and > thresh (float16, NaN threshold: never), the hit rule of mb200_scan, per column."""
    s = np.asarray(score, np.float16)
    ok = s > np.float16(0)
    if thresh is not None:
        t = np.asarray(thresh, np.float16)
        ok &= ~np.isnan(t)[None, :] & (s > np.where(np.isnan(t), np.float16(0), t)[None, :])
    return ok


def spacing_anchors(rec: Records, score, pos, comp, found, primary_lens, primary_thresh, margin: int):
    """Record best sites of the primaries -> anchors.  Returns (frag (R, P) int64 fragment holding the flank, -1 for no anchor,
    and the (R, P) bool anchor mask).  A best site counts when it is a hit and [pos - margin, pos + m_p + margin) lies inside
    one fragment (no N run, no record end)."""
    R, P = np.shape(pos)
    m = np.asarray(primary_lens, np.int64)[None, :]
    ok = np.asarray(found, bool) & _hit_mask(score, primary_thresh)
    lo = np.asarray(pos, np.int64) - margin
    hi = np.asarray(pos, np.int64) + m + margin
    frag = np.full((R, P), -1, np.int64)
    if len(rec.frag_len) and R:
        coff = np.concatenate([[0], np.cumsum(rec.lengths)]).astype(np.int64)
        gstart = coff[rec.frag_record] + rec.frag_start             # increasing: fragments come in record order
        rr = np.broadcast_to(np.arange(R, dtype=np.int64)[:, None], (R, P))
        f = np.searchsorted(gstart, coff[rr] + lo, side="right") - 1
        fc = np.clip(f, 0, len(gstart) - 1)
        inside = (f >= 0) & (lo >= 0) & (rec.frag_record[fc] == rr) & (rec.frag_start[fc] <= lo) & \
                 (hi <= rec.frag_start[fc] + rec.frag_len[fc])
        ok &= inside
        frag = np.where(ok, fc, -1)
    else:
        ok[:] = False
    return frag, ok


def spacing(ctx, path_or_records, primary, secondary, *, primary_thresh=None, secondary_thresh=None, margin: int = 150,
            want_sites: bool = False, max_padding: float = 1.0 / 8) -> Spacing:
    """SpaMo-style spacing analysis of a FASTA peak set (a path or a Records).  The primaries' record best sites (best_sites)
    that are hits with a whole flank become anchors; the fragments holding them are bucketed as in scan_fasta (only those
    fragments), and one mb200_scan_spacing call per bucket finds the best site of every secondary in both margins of each
    anchor and adds it to the device histogram.  primary / secondary: an inference.Motifs (its score_thresh is the threshold
    when none is given) or a list of (4, len) PWMs.  spacing_enrichment tests the histogram."""
    rec = path_or_records if isinstance(path_or_records, Records) else read_records(path_or_records)
    ppw, plens, pthr = _pwm_args(primary, primary_thresh)
    spw, slens, sthr = _pwm_args(secondary, secondary_thresh)
    margin = int(margin)
    if margin < 1:
        raise ValueError("margin must be >= 1")
    P, K, R = len(plens), len(slens), len(rec.names)
    bs = best_sites(ctx, rec, primary, max_padding=max_padding)
    frag, ok = spacing_anchors(rec, bs.score, bs.pos, bs.comp, bs.found, plens, None if pthr is None else pthr.view(np.float16),
                               margin)
    hist = np.zeros((P, K, 4, margin), np.int64)
    sites = None
    if want_sites:
        sites = np.zeros((R, P, K), SPACING_SITE_DTYPE)
        sites["pos"] = -1
    has = np.zeros(len(rec.frag_len), bool)
    has[frag[ok]] = True
    off = rec.frag_offsets
    for b in bucket_fragments(np.where(has, rec.frag_len, 0), 1, max_padding):
        row_of = np.full(len(rec.frag_len), -1, np.int64)
        row_of[b] = np.arange(len(b))
        sel = ok & (row_of[np.maximum(frag, 0)] >= 0)
        rr, pp = np.nonzero(sel)
        f = frag[rr, pp]
        an = np.zeros(len(rr), _lib.ANCHOR_DTYPE)
        an["row"] = row_of[f]
        an["start"] = bs.pos[rr, pp] - rec.frag_start[f]
        an["len"] = plens[pp]
        an["primary"] = pp
        an["comp"] = bs.comp[rr, pp]
        ls = rec.frag_len[b]
        seqs = ctx.seqs_from_ragged(np.concatenate([rec.bases[off[g]: off[g + 1]] for g in b]), np.concatenate([[0], np.cumsum(ls)]))
        try:
            h, st = ctx.scan_spacing(seqs, an, P, spw, slens, sthr, margin=margin, want_sites=want_sites)
        finally:
            seqs.free()
        hist += h
        if want_sites:
            w = st["pos"] != np.uint32(0xFFFFFFFF)
            out = sites[rr, pp]
            out["pos"] = np.where(w, rec.frag_start[f][:, None] + st["pos"].astype(np.int64), -1)
            out["score"] = st["score_f16"].view(np.float16)
            out["comp"] = st["comp"]
            out["found"] = st["found"].astype(bool)
            sites[rr, pp] = out
    pos = np.where(ok, bs.pos, -1)
    comp = np.where(ok, bs.comp.astype(np.int64), -1)
    return Spacing(list(rec.names), margin, hist, ok.sum(axis=0).astype(np.int64), pos, comp, sites)


@dataclass
class SpacingEnrichment:
    """Per (primary, secondary): the most populated (quadrant, gap) bin among the B = 4 (margin - m_k + 1) bins where a
    secondary of length m_k fits (ties: lowest q, then lowest gap), its count of the n counted sites, p = P[Binom(n, 1/B) >=
    count] (SpaMo's uniform null) and p_adj = min(1, p * B * K), Bonferroni over bins and secondaries.  q = gap = -1, p = p_adj =
    1 where n = 0 or the secondary does not fit in the margin."""
    n: np.ndarray                # (P, K) int64
    q: np.ndarray                # (P, K) int64
    gap: np.ndarray              # (P, K) int64
    count: np.ndarray            # (P, K) int64
    p: np.ndarray                # (P, K) float64
    p_adj: np.ndarray            # (P, K) float64


def spacing_enrichment(sp: Spacing, secondary_lens) -> SpacingEnrichment:
    P, K, _, W = sp.hist.shape
    lens = np.asarray(secondary_lens, np.int64)
    if lens.shape != (K,):
        raise ValueError("secondary_lens must hold K lengths")
    res = SpacingEnrichment(np.zeros((P, K), np.int64), np.full((P, K), -1, np.int64), np.full((P, K), -1, np.int64),
                            np.zeros((P, K), np.int64), np.ones((P, K)), np.ones((P, K)))
    for k in range(K):
        G = W - int(lens[k]) + 1
        if G < 1:
            continue
        B = 4 * G
        for p in range(P):
            h = sp.hist[p, k, :, :G]
            n = int(h.sum())
            res.n[p, k] = n
            if n == 0:
                continue
            i = int(np.argmax(h.reshape(-1)))               # first maximum in (q, gap) order
            q, g = divmod(i, G)
            c = int(h[q, g])
            pv = inference.binom_right(c, n, 1.0 / B)
            res.q[p, k], res.gap[p, k], res.count[p, k] = q, g, c
            res.p[p, k], res.p_adj[p, k] = pv, min(1.0, pv * B * K)
    return res


# ---- exact p-values and q-values of scan hits and best sites (FIMO-style) ------------------------------------------------
def base_background(rec: Records) -> np.ndarray:
    """(4,) float64 A/C/G/T frequencies of the records' fragments, averaged with their reverse complement (A = T, C = G): the
    default background of scan_fasta_pvalues and best_site_pvalues.  Both strands are scanned, so the null of either strand
    should not depend on which strand the file happens to hold."""
    code = np.full(256, 4, np.int64)
    for i, c in enumerate(b"ACGT"):
        code[c] = i
    n = np.bincount(code[np.asarray(rec.bases, np.uint8)], minlength=5)[:4].astype(np.float64)
    n = n + n[::-1]
    if n.sum() == 0:
        raise ValueError("the records hold no A/C/G/T bases: no background")
    return n / n.sum()


def _windows_per(frag_len, lens):
    """(F, K) int64: windows of every motif on one strand of every fragment, max(0, L_f - m_k + 1)."""
    return np.maximum(0, np.asarray(frag_len, np.int64)[:, None] - np.asarray(lens, np.int64)[None, :] + 1)


def bh_qvalues(p, n_tests) -> np.ndarray:
    """Benjamini-Hochberg q-values of hits with p-values p among n_tests >= len(p) tests whose other p-values are larger:
    q_(i) = min(1, min_{j >= i} p_(j) n_tests / j) over the hits sorted by p (ties share the q of the last of them)."""
    p = np.asarray(p, np.float64)
    q = np.empty(len(p))
    if len(p) == 0:
        return q
    o = np.argsort(p, kind="stable")
    s = p[o] * float(n_tests) / np.arange(1, len(p) + 1)
    q[o] = np.minimum(1.0, np.minimum.accumulate(s[::-1])[::-1])
    return q


def sidak(site_p, n) -> np.ndarray:
    """1 - (1 - site_p)^n, evaluated as -expm1(n log1p(-site_p)) (stable for small site_p): the probability that the best of n
    independent windows scores at least as high as a site of p-value site_p (CentriMo's and AME's correction)."""
    site_p = np.asarray(site_p, np.float64)
    with np.errstate(divide="ignore", invalid="ignore"):
        return -np.expm1(np.asarray(n, np.float64) * np.log1p(-site_p))


@dataclass
class PValueScan:
    """Hits of scan_fasta_pvalues: RECORD_HIT_DTYPE sorted by (record, motif, comp, pos) with p-value <= the requested one.
    pvalue: exact P(score >= the hit's score) of one window of its strand under bg; qvalue: Benjamini-Hochberg per motif over
    n_tests[k] windows (both strands of every fragment).  thresh: (K, 2) per-strand Float16 thresholds (score > thresh <=> p <=
    the requested p); clamped: slots whose threshold is below 0, where the scan's score > 0 rule drops sites with p small
    enough but score <= 0."""
    hits: np.ndarray
    pvalue: np.ndarray           # (n,) float64
    qvalue: np.ndarray           # (n,) float64
    n_tests: np.ndarray          # (K,) int64
    thresh: np.ndarray           # (K, 2) float16
    bg: np.ndarray               # (4,) float64
    names: List[str]
    clamped: np.ndarray          # (K, 2) bool


def scan_fasta_pvalues(ctx, path_or_records, motifs_or_pwms, pvalue: float = 1e-4, *, bg=None,
                       max_padding: float = 1.0 / 8) -> PValueScan:
    """Scan a FASTA file (a path or a Records) "at p < pvalue": every window on either strand whose exact p-value under a
    background of independent bases is at most pvalue, with Benjamini-Hochberg q-values per motif.

    The null tables come from Context.score_null (exact for the scan's Float16 score).  The fragments are scanned as in
    scan_fasta at the per-motif threshold min(fwd, rc) of the two strands' thresholds; each hit's p-value is looked up on its
    own strand and hits with p > pvalue (the strand with the higher threshold) are dropped.  The q-values are exact from the
    hits alone: every unreported window has a larger p-value and counts as p = 1.  The scan reports only score > 0, so on a
    clamped slot (threshold < 0, i.e. pvalue above P(score > 0)) sites with p <= pvalue and score <= 0 are missing; their q
    values then treat them as p = 1 (conservative).  bg: (4,) A/C/G/T frequencies, default base_background(records)."""
    rec = path_or_records if isinstance(path_or_records, Records) else read_records(path_or_records)
    pw, lens, _ = _pwm_args(motifs_or_pwms, None)
    K = len(lens)
    bg = base_background(rec) if bg is None else np.asarray(bg, np.float64)
    null = ctx.score_null(pw, lens, bg)
    try:
        thresh = null.thresholds(float(pvalue))
        res = _scan_records(ctx, rec, pw, lens, np.minimum(thresh[:, 0], thresh[:, 1]), True, max_padding)
        hits = res.hits
        p = null.pvalues(hits["motif"], hits["comp"], hits["score_f16"])
    finally:
        null.free()
    keep = p <= pvalue
    hits, p = hits[keep], p[keep]
    n_tests = 2 * _windows_per(rec.frag_len, lens).sum(axis=0).astype(np.int64)
    q = np.empty(len(p))
    order = np.argsort(hits["motif"], kind="stable")          # the hits of each motif, as one slice of `order`
    cut = np.searchsorted(hits["motif"][order], np.arange(K + 1))
    for k in np.nonzero(np.diff(cut))[0]:
        idx = order[cut[k]: cut[k + 1]]
        q[idx] = bh_qvalues(p[idx], n_tests[k])
    return PValueScan(hits, p, q, n_tests, thresh, bg, list(rec.names), thresh < np.float16(0))


def best_site_pvalues(ctx, path_or_records, best: BestSites, motifs_or_pwms, *, bg=None):
    """(site_p, seq_p), both (R, K) float64, NaN where the record has no site of the motif.  site_p: the exact p-value of the best
    site's score on its strand; seq_p = -expm1(n log1p(-site_p)), the probability that the best of the record's n windows (both
    strands of its fragments) scores at least as high, with the Sidak correction CentriMo and AME use.  best: best_sites of the
    same records and motifs; bg: default base_background(records)."""
    rec = path_or_records if isinstance(path_or_records, Records) else read_records(path_or_records)
    pw, lens, _ = _pwm_args(motifs_or_pwms, None)
    R, K = best.found.shape
    bg = base_background(rec) if bg is None else np.asarray(bg, np.float64)
    r, k = np.nonzero(best.found)
    null = ctx.score_null(pw, lens, bg)
    try:
        p = null.pvalues(k, best.comp[r, k], best.score[r, k].view(np.uint16))
    finally:
        null.free()
    site_p = np.full((R, K), np.nan)
    site_p[r, k] = p
    n = np.zeros((R, K), np.int64)
    np.add.at(n, np.asarray(rec.frag_record, np.int64), 2 * _windows_per(rec.frag_len, lens))
    seq_p = np.full((R, K), np.nan)
    seq_p[r, k] = sidak(p, n[r, k])
    return site_p, seq_p
