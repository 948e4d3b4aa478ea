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
