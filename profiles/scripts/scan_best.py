"""Throughput of the best-site scan (mb200_scan_best) against the counts-only score > 0 scan of the same stores.

Both run the SIMT scan kernel family (scan_kernel), so the ratio is the cost of the best-site epilogue, the 32-bit keys (twice
the hit-mask bytes) and the reducer, against the mask epilogue and the counting kernel.  Config 4's 500 PWMs of length 8-40
(bench.make_motifs).  Two workloads:
  peaks500: --fixed-peaks peaks of 500 bp in one fixed-length store (summit-centred peaks, the input of central enrichment);
  peaks:    --peaks peaks of log-uniform length 100-2000 bp (scan_ragged.py's peak workload), bucketed by records.bucket_fragments.
Timed: every store of a workload, host clock around library calls that end in a device synchronise; the two modes alternate
rep by rep after one warm-up pass of each, best of --reps.  Rates are real bases (padding excluded) per second.  The device-side
split of the best-site scan (mb200_last_timing: scan kernel, reducer, copies) is summed over the stores of the last rep.
Run from the repository root on the GPU:  python profiles/scripts/scan_best.py  -> one JSON line."""
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
from motifs_jl_b200 import inference  # noqa: E402
from scan_ragged import LUT, gpu_info, peaks, stores  # noqa: E402


def run(ctx, st, pw, lens, mode):
    ms = {"scan": 0.0, "count": 0.0, "d2h": 0.0}
    t0 = time.perf_counter()
    for s, _, _ in st:
        if mode == "best":
            ctx.scan_best(s, pw, lens)
        else:
            ctx.scan(s, pw, lens, None, want_hits=False)
        t, _ = ctx.last_timing()
        for k in ms:
            ms[k] += t[k]
    return time.perf_counter() - t0, ms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--fixed-peaks", type=int, default=100_000)
    ap.add_argument("--peaks", type=int, default=200_000)
    ap.add_argument("--motifs", type=int, default=500)
    ap.add_argument("--reps", type=int, default=5)
    args = ap.parse_args()
    ctx = mb.Context(0)
    ms, _, _ = bench.make_motifs(args.motifs)
    pw, mlen = inference.pack_pwms(ms), ms.lens
    rng = np.random.default_rng(2024)
    out = {"gpu": gpu_info(), "motifs": args.motifs,
           "timing": f"best of {args.reps} alternating reps after a warm-up of each mode; host clock around synchronising calls"}
    fixed = LUT[rng.integers(0, 4, (args.fixed_peaks, 500), dtype=np.uint8)]
    fl, fb = peaks(args.peaks, rng)
    workloads = (("peaks500", lambda: [(ctx.seqs_from_ascii(fixed), fixed.size, fixed.size)]),
                 ("peaks", lambda: stores(ctx, fl, fb, int(mlen.min()))))
    for name, make in workloads:
        st = make()
        real = sum(x[1] for x in st)
        for mode in ("best", "counts"):
            run(ctx, st, pw, mlen, mode)
        tb, tc, split, csplit = [], [], None, None
        for _ in range(args.reps):
            t, split = run(ctx, st, pw, mlen, "best")
            tb.append(t)
            t, csplit = run(ctx, st, pw, mlen, "counts")
            tc.append(t)
        for s, _, _ in st:
            s.free()
        out[name] = {"stores": len(st), "real_bases": real,
                     "best_s": round(min(tb), 4), "counts_s": round(min(tc), 4),
                     "best_gbp_s": round(real / min(tb) / 1e9, 3), "counts_gbp_s": round(real / min(tc) / 1e9, 3),
                     "time_ratio": round(min(tb) / min(tc), 3),
                     "best_device_ms": {"scan": round(split["scan"], 2), "reduce": round(split["count"], 2), "d2h": round(split["d2h"], 2)},
                     "counts_device_ms": {"scan": round(csplit["scan"], 2), "count": round(csplit["count"], 2)}}
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
