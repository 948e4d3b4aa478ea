"""Throughput of scans over ragged stores (the stores scan_fasta builds) against a fixed-length 200 bp store of the same bases.

Config 4's PWM set and thresholds (bench.make_motifs: 500 PWMs of length 8-40).  Two workloads:
  genome: 24 chromosomes with the length proportions of GRCh38 chr1..22, X, Y scaled to --genome-bp, plus 200 contigs of
          20-200 kb; 10 kb telomere N runs at both ends, a centromere N run of 1.5 % of each chromosome, and one scattered
          1-10 kb N run per 2 Mbp.  The N-free fragments are bucketed by records.bucket_fragments.
  peaks:  --peaks peaks of log-uniform length 100-2000 bp, bucketed the same way.
Each is compared with its bases cut into 200 bp rows of one fixed-length store, in the same process.  Timed: counts-only
thresholded scans (mb200_scan) of all stores of a workload, host clock around calls that end in a device synchronise; the
uploads are not timed.  Rates are REAL bases (padding excluded) per second; best of --reps after one warm-up pass.
Run from the repository root on the GPU:  python profiles/scripts/scan_ragged.py  -> one JSON line."""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import motifs_jl_b200 as mb  # noqa: E402
from motifs_jl_b200 import inference, records  # noqa: E402

GRCH38_MBP = [248.96, 242.19, 198.30, 190.21, 181.54, 170.81, 159.35, 145.14, 138.39, 133.80, 135.09, 133.28, 114.36, 107.04,
              101.99, 90.34, 83.26, 80.37, 58.62, 64.44, 46.71, 50.82, 156.04, 57.23]
LUT = np.frombuffer(b"ACGT", np.uint8)


def fragments_of(seq_list):
    """N-free runs of every sequence -> (lengths, concatenated bases) in record order"""
    lens, parts = [], []
    for s in seq_list:
        ok = np.concatenate([[False], s != ord("N"), [False]])
        d = np.flatnonzero(np.diff(ok.astype(np.int8)))
        for a, b in zip(d[0::2], d[1::2]):
            lens.append(b - a)
            parts.append(s[a:b])
    return np.array(lens, np.int64), np.concatenate(parts)


def genome(total_bp, rng):
    scale = total_bp / (sum(GRCH38_MBP) * 1e6)
    seqs = []
    for mbp in GRCH38_MBP:
        L = int(mbp * 1e6 * scale)
        s = LUT[rng.integers(0, 4, L, dtype=np.uint8)]
        s[:10_000] = ord("N"); s[-10_000:] = ord("N")
        c0, cl = int(0.4 * L), int(0.015 * L)
        s[c0:c0 + cl] = ord("N")
        for p in rng.integers(10_000, L - 20_000, L // 2_000_000):
            s[p:p + int(rng.integers(1000, 10_001))] = ord("N")
        seqs.append(s)
    for L in rng.integers(20_000, 200_001, 200):
        seqs.append(LUT[rng.integers(0, 4, int(L), dtype=np.uint8)])
    return fragments_of(seqs)


def peaks(n, rng):
    lens = np.exp(rng.uniform(np.log(100), np.log(2000), n)).astype(np.int64)
    return lens, LUT[rng.integers(0, 4, int(lens.sum()), dtype=np.uint8)]


def stores(ctx, lens, bases, minlen):
    off = np.concatenate([[0], np.cumsum(lens)])
    out = []
    for b in records.bucket_fragments(lens, minlen):
        ls = lens[b]
        asc = np.concatenate([bases[off[f]:off[f + 1]] for f in b])
        out.append((ctx.seqs_from_ragged(asc, np.concatenate([[0], np.cumsum(ls)])), int(ls.sum()), len(b) * int(ls.max())))
    return out


def timed(ctx, st, pw, lens, thr, reps):
    def one():
        c = np.zeros((len(lens), 4), np.int64)
        for s, _, _ in st:
            c += ctx.scan(s, pw, lens, thr, want_hits=False)[1]
        return c
    counts = one()                                                  # warm-up (and the tensor-core path's CTA balance)
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        c = one()
        ts.append(time.perf_counter() - t0)
        assert np.array_equal(c, counts)
    return min(ts), float(np.median(ts)), counts


def gpu_info():
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=60)
        return r.stdout.strip().splitlines()[0]
    except Exception as e:                                          # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genome-bp", type=int, default=1_000_000_000)
    ap.add_argument("--peaks", type=int, default=200_000)
    ap.add_argument("--motifs", type=int, default=500)
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    ctx = mb.Context(0)
    ms, thr, _ = bench.make_motifs(args.motifs)
    pw, mlen = inference.pack_pwms(ms), ms.lens
    rng = np.random.default_rng(2024)
    out = {"gpu": gpu_info(), "motifs": args.motifs, "timing": f"best of {args.reps} after a warm-up, counts-only thresholded scans"}
    for name, (fl, fb) in (("genome", genome(args.genome_bp, rng)), ("peaks", peaks(args.peaks, rng))):
        st = stores(ctx, fl, fb, int(mlen.min()))
        real = sum(x[1] for x in st)
        padded = sum(x[2] for x in st)
        t, tmed, _ = timed(ctx, st, pw, mlen, thr, args.reps)
        for s, _, _ in st:
            s.free()
        nfix = int(real // 200)
        fixed = ctx.seqs_from_ascii(fb[: nfix * 200].reshape(nfix, 200))
        tf, tfmed, _ = timed(ctx, [(fixed, nfix * 200, nfix * 200)], pw, mlen, thr, args.reps)
        fixed.free()
        r_rag, r_fix = real / t, nfix * 200 / tf
        out[name] = {"fragments": len(fl), "stores": len(st), "real_bases": real, "padded_positions": padded,
                     "ragged_s": round(t, 4), "ragged_median_s": round(tmed, 4), "ragged_gbp_s": round(r_rag / 1e9, 3),
                     "fixed200_rows": nfix, "fixed200_s": round(tf, 4), "fixed200_median_s": round(tfmed, 4),
                     "fixed200_gbp_s": round(r_fix / 1e9, 3), "ratio": round(r_rag / r_fix, 3)}
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
