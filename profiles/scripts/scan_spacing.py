"""Cost of the spacing scan (mb200_scan_spacing) on a peak set, against returning the best-site records of the same flank store.

Workload: --peaks summit-centred peaks of 500 bp (random bases) with a planted composite in 40 % of them (primary 0's consensus at
230, secondary 0's consensus 7 bp downstream on the same strand); 10 primaries (primary 0 from its planted sites, 9 from
synth.random_count_matrices(9, 8, 20, 7)); config 4's 500 PWMs as secondaries, built as bench.py builds them
(synth.random_count_matrices(500, 8, 40, 4)) with synth.stated_thresholds(ms, 0.7) as secondary thresholds; margin 150.  Anchors
are every (peak, primary) whose best site (mb200_scan_best of the peaks) scores > 0 with its whole flank inside the peak.

Timed, best of --reps after a warm-up, host clock around calls that end in a device synchronise:
  spacing:      ctx.scan_spacing (window gather + scan + reduce + spacing kernel + one histogram copy);
  best_records: the same flank store (ctx.seqs_windows, rows 2i / 2i + 1 = the margins of anchor i) through ctx.scan_best, its
                2 x anchors x K 8-byte records returned to a new pageable host array (what the spacing histogram replaces).
The device split (mb200_last_timing: pack = window gather, scan, count = reduce + spacing, d2h) is from the last timed rep.  Card
name and power limit are read before and after, in the same run.
Run from the repository root on the GPU:  python profiles/scripts/scan_spacing.py  -> one JSON line."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "scripts"))
import bench  # noqa: E402
import motifs_jl_b200 as mb  # noqa: E402
from motifs_jl_b200 import _lib, inference, synth  # noqa: E402
from scan_ragged import LUT, gpu_info  # noqa: E402

MARGIN = 150
PRIM = "GGACTTAGCATG"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--peaks", type=int, default=100_000)
    ap.add_argument("--secondaries", type=int, default=500)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    ctx = mb.Context(0)
    out = {"gpu": gpu_info(), "peaks": args.peaks, "peak_bp": 500, "primaries": 10, "secondaries": args.secondaries, "margin": MARGIN,
           "timing": f"best of {args.reps} reps after a warm-up; host clock around synchronising calls"}
    sec, _, _ = bench.make_motifs(args.secondaries)
    sthr = synth.stated_thresholds(sec, 0.7)
    prim = synth.motifs_from_count_matrices([synth.count_matrix_from_sites([PRIM] * 30)] + synth.random_count_matrices(9, 8, 20, 7))
    rng = np.random.default_rng(2026)
    a = LUT[rng.integers(0, 4, (args.peaks, 500), dtype=np.uint8)]
    cons = "".join("ACGT"[i] for i in np.asarray(sec.cmats[0], np.float32).argmax(axis=0))
    unit = np.frombuffer((PRIM + "ACGTACG" + cons).encode(), np.uint8)
    planted = rng.random(args.peaks) < 0.4
    a[planted, 230: 230 + len(unit)] = unit
    s = ctx.seqs_from_ascii(a)
    ppw, plens = inference.pack_pwms(prim), np.asarray(prim.lens, np.int64)
    spw, slens = inference.pack_pwms(sec), np.asarray(sec.lens, np.int64)
    best = ctx.scan_best(s, ppw, plens)
    n, p = np.nonzero((best["found"] == 1) & (best["score_f16"].view(np.float16) > 0) & (best["pos"].astype(np.int64) >= MARGIN) &
                      (best["pos"].astype(np.int64) + plens[None, :] + MARGIN <= 500))
    an = np.zeros(len(n), _lib.ANCHOR_DTYPE)
    an["row"], an["start"], an["len"], an["primary"], an["comp"] = n, best["pos"][n, p], plens[p], p, best["comp"][n, p]
    A, K = len(an), len(slens)
    out["anchors"] = A
    out["flank_bases"] = 2 * A * MARGIN

    def spacing():
        t0 = time.perf_counter()
        h, _ = ctx.scan_spacing(s, an, 10, spw, slens, sthr, margin=MARGIN)
        return time.perf_counter() - t0, ctx.last_timing()[0], h

    rows = np.repeat(an["row"], 2)
    starts = np.stack([an["start"] - MARGIN, an["start"] + an["len"]], axis=1).reshape(-1)

    def records():
        t0 = time.perf_counter()
        w = ctx.seqs_windows(s, rows, starts, MARGIN)
        t1 = time.perf_counter()
        r = ctx.scan_best(w, spw, slens)
        t2 = time.perf_counter()
        w.free()
        return t2 - t0, t1 - t0, ctx.last_timing()[0], r.nbytes

    spacing()
    ts, split, hist = [], None, None
    for _ in range(args.reps):
        t, split, hist = spacing()
        ts.append(t)
    records()
    tr, tg, rsplit, rbytes = [], [], None, 0
    for _ in range(args.reps):
        t, g, rsplit, rbytes = records()
        tr.append(t)
        tg.append(g)
    e = min(ts)
    q, g = np.unravel_index(np.argmax(hist[0, 0]), hist[0, 0].shape)
    out["spacing"] = {"call_s": round(e, 4), "flank_gbp_s": round(2 * A * MARGIN / e / 1e9, 3),
                      "device_ms": {k: round(split[k], 2) for k in ("pack", "scan", "count", "d2h", "total")},
                      "d2h_bytes": int(hist.nbytes),
                      "call_over_scan_kernel": round(e * 1e3 / split["scan"], 3),
                      "count_plus_d2h_share": round((split["count"] + split["d2h"]) / (e * 1e3), 4),
                      "planted_top_bin": [int(q), int(g), int(hist[0, 0, q, g])]}
    out["best_records"] = {"call_s": round(min(tr), 4), "gather_s": round(min(tg), 4),
                           "flank_gbp_s": round(2 * A * MARGIN / min(tr) / 1e9, 3),
                           "device_ms": {k: round(rsplit[k], 2) for k in ("scan", "count", "d2h", "total")},
                           "d2h_bytes": int(rbytes)}
    out["records_over_spacing"] = round(min(tr) / e, 3)
    s.free()
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
