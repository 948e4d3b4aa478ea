"""Cost of exact p-values (csrc/pvalue.cu): survival-table build, lookups, and scan_fasta_pvalues against scan_fasta.

Workloads:
  build:  Context.score_null for --motifs PWMs of lengths 8-30 (synth.random_count_matrices(K, 8, 30, 4)), both strands, skewed
          background (0.3, 0.2, 0.2, 0.3).  Bytes per column step: a slot-column reads S_j and writes S_{j+1}, 63 489 float64 each
          (unique bytes; each thread gathers 4 values of S_j, mostly from L2), against 7.7 TB/s.
  lookup: ScoreNull.pvalues of --hits random (motif, strand, Float16 score) triples, host arrays in and out.
  e2e:    --peaks records of 500 bp (one fragment each, bases drawn from the background), the same PWMs:
          records.scan_fasta_pvalues(p = 1e-4) against records.scan_fasta at the same score thresholds (per motif the smaller
          of the two strands' thresholds, what scan_fasta_pvalues scans at), both from in-memory Records.
Timed, best of --reps after a warm-up, host clock around calls that end in a device synchronise.  Card name and power limit
are read before and after, in the same run.
Run from the repository root on the GPU:  python profiles/scripts/scan_pvalues.py  -> one JSON line."""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "scripts"))
import motifs_jl_b200 as mb  # noqa: E402
from motifs_jl_b200 import inference, records, synth  # noqa: E402
from scan_ragged import gpu_info  # noqa: E402

NV = 63489
BG = np.array([0.3, 0.2, 0.2, 0.3])


def best_of(fn, reps):
    fn()
    ts, r = [], None
    for _ in range(reps):
        t0 = time.perf_counter()
        r = fn()
        ts.append(time.perf_counter() - t0)
    return min(ts), r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--motifs", type=int, default=500)
    ap.add_argument("--hits", type=int, default=10_000_000)
    ap.add_argument("--peaks", type=int, default=100_000)
    ap.add_argument("--pvalue", type=float, default=1e-4)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    ctx = mb.Context(0)
    out = {"gpu": gpu_info(), "motifs": args.motifs, "lens": "8-30", "bg": BG.tolist(),
           "timing": f"best of {args.reps} reps after a warm-up; host clock around synchronising calls"}
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(args.motifs, 8, 30, 4))
    pw, lens = inference.pack_pwms(ms), np.asarray(ms.lens, np.int64)

    def build():
        n = ctx.score_null(pw, lens, BG)
        n.free()
    t, _ = best_of(build, args.reps)
    slot_cols = 2 * int(lens.sum())
    unique = slot_cols * 2 * NV * 8
    out["build"] = {"call_s": round(t, 4), "slots": 2 * args.motifs, "slot_columns": slot_cols, "column_steps": int(lens.max()),
                    "unique_bytes": unique, "unique_tb_s": round(unique / t / 1e12, 3),
                    "share_of_7.7_tb_s": round(unique / t / 7.7e12, 4), "table_bytes": 2 * args.motifs * NV * 8}

    null = ctx.score_null(pw, lens, BG)
    rng = np.random.default_rng(5)
    m = rng.integers(0, args.motifs, args.hits).astype(np.uint16)
    c = rng.integers(0, 2, args.hits).astype(np.uint8)
    s = rng.integers(0, 0x7C00, args.hits).astype(np.uint16)
    t, p = best_of(lambda: null.pvalues(m, c, s), args.reps)
    out["lookup"] = {"hits": args.hits, "call_s": round(t, 4), "mhits_s": round(args.hits / t / 1e6, 1)}
    thresh = null.thresholds(args.pvalue)
    null.free()

    L = 500
    bases = np.frombuffer(b"ACGT", np.uint8)[rng.choice(4, size=args.peaks * L, p=BG)]
    ar = np.arange(args.peaks, dtype=np.int64)
    rec = records.Records([f"peak{i}" for i in range(args.peaks)], np.full(args.peaks, L, np.int64), ar,
                          np.zeros(args.peaks, np.int64), np.full(args.peaks, L, np.int64), bases)
    thr = np.minimum(thresh[:, 0], thresh[:, 1])
    t_scan, r_scan = best_of(lambda: records.scan_fasta(ctx, rec, ms.pwms, thr), args.reps)
    t_pv, r_pv = best_of(lambda: records.scan_fasta_pvalues(ctx, rec, ms.pwms, args.pvalue, bg=BG), args.reps)
    assert np.array_equal(r_pv.thresh, thresh)
    out["e2e"] = {"peaks": args.peaks, "peak_bp": L, "pvalue": args.pvalue,
                  "scan_fasta_s": round(t_scan, 4), "scan_fasta_hits": int(len(r_scan.hits)),
                  "scan_fasta_pvalues_s": round(t_pv, 4), "hits_p_le_pvalue": int(len(r_pv.hits)),
                  "added_s": round(t_pv - t_scan, 4), "ratio": round(t_pv / t_scan, 3),
                  "clamped_slots": int(r_pv.clamped.sum())}
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
