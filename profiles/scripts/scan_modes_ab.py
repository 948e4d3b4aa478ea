"""A/B of two builds of the library on the scan modes bench.py does not time, on ONE box (box-to-box variation is ~15 %).

  python profiles/scripts/scan_modes_ab.py OTHER_LIB > scan_modes_ab.json

runs this script with --one in four processes, the other build (MB200_LIBRARY=OTHER_LIB) and this tree's build alternating: old,
new, old, new.  Every process runs every workload once as a warm-up and then --reps times; it reports a hash of the outputs, the
launch counts per timing slot of the last call (mb200_last_timing; summed over the stores of a ragged workload) and the best
whole-call time (host clock around calls that end in a device synchronise).  The parent checks that hashes and launch counts are
equal in all four processes and prints one JSON line.  Workloads (inputs seeded, so every process scans the same bases):
  hits_tc:     config 4's 500 PWMs and thresholds (bench.make_motifs) over 1 M x 200 bp, hit list + counts: the serial
               tensor-core loop, then count, prefix sum, emit and clear;
  hits_simt:   10 of those PWMs without thresholds (score > 0) over 500 000 x 200 bp, hit list + counts: scan_kernel;
  hist:        the 500 PWMs over 100 000 x 200 bp, mb200_scan_hist;
  best:        scan_best.py's peaks500 workload, 100 000 x 500 bp, mb200_scan_best with the 500 PWMs;
  spacing:     scan_spacing.py's workload (100 000 peaks of 500 bp, 10 primaries, 500 secondaries, margin 150), mb200_scan_spacing;
  ragged:      scan_ragged.py's peak set (200 000 peaks of 100-2000 bp, bucketed into ragged stores), thresholded counts: the
               pipelined tensor-core loop on ragged stores.
Card name, power limit and maximum SM clock are read before and after, in the same run."""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles", "scripts"))


def digest(*arrays):
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()[:16]


def workloads(ctx):
    """name -> function that runs the workload once and returns (output hash, launches, extra)"""
    import bench
    from motifs_jl_b200 import _lib, inference, synth
    from scan_ragged import LUT, peaks, stores

    ms, thr, _ = bench.make_motifs(500)
    pw, lens = inference.pack_pwms(ms), np.asarray(ms.lens, np.int64)
    rng = np.random.default_rng(2027)
    out = {}

    s1 = ctx.seqs_from_ascii(LUT[rng.integers(0, 4, (1_000_000, 200), dtype=np.uint8)])

    def hits_tc():
        h, c = ctx.scan(s1, pw, lens, thr)
        return digest(h, c), ctx.last_timing()[1], {"hits": int(len(h)), "path": _lib.scan_last_path(ctx)}
    out["hits_tc"] = hits_tc

    ms10 = synth.motifs_from_count_matrices(ms.cmats[:10])
    pw10, lens10 = inference.pack_pwms(ms10), np.asarray(ms10.lens, np.int64)
    s2 = ctx.seqs_from_ascii(LUT[rng.integers(0, 4, (500_000, 200), dtype=np.uint8)])

    def hits_simt():
        h, c = ctx.scan(s2, pw10, lens10, None)
        return digest(h, c), ctx.last_timing()[1], {"hits": int(len(h)), "path": _lib.scan_last_path(ctx)}
    out["hits_simt"] = hits_simt

    s3 = ctx.seqs_from_ascii(LUT[rng.integers(0, 4, (100_000, 200), dtype=np.uint8)])

    def hist():
        return digest(_lib.scan_hist(ctx, s3, pw, lens)), ctx.last_timing()[1], {}
    out["hist"] = hist

    s4 = ctx.seqs_from_ascii(LUT[rng.integers(0, 4, (100_000, 500), dtype=np.uint8)])

    def best():
        return digest(ctx.scan_best(s4, pw, lens)), ctx.last_timing()[1], {}
    out["best"] = best

    # scan_spacing.py's anchors: every (peak, primary) whose best site scores > 0 with its whole flank inside the peak
    margin, prim_site = 150, "GGACTTAGCATG"
    sthr = synth.stated_thresholds(ms, 0.7)
    prim = synth.motifs_from_count_matrices([synth.count_matrix_from_sites([prim_site] * 30)] + synth.random_count_matrices(9, 8, 20, 7))
    a = LUT[rng.integers(0, 4, (100_000, 500), dtype=np.uint8)]
    cons = "".join("ACGT"[i] for i in np.asarray(ms.cmats[0], np.float32).argmax(axis=0))
    unit = np.frombuffer((prim_site + "ACGTACG" + cons).encode(), np.uint8)
    a[rng.random(len(a)) < 0.4, 230: 230 + len(unit)] = unit
    s5 = ctx.seqs_from_ascii(a)
    plens = np.asarray(prim.lens, np.int64)
    pb = ctx.scan_best(s5, inference.pack_pwms(prim), plens)
    n, p = np.nonzero((pb["found"] == 1) & (pb["score_f16"].view(np.float16) > 0) & (pb["pos"].astype(np.int64) >= margin) &
                      (pb["pos"].astype(np.int64) + plens[None, :] + margin <= 500))
    an = np.zeros(len(n), _lib.ANCHOR_DTYPE)
    an["row"], an["start"], an["len"], an["primary"], an["comp"] = n, pb["pos"][n, p], plens[p], p, pb["comp"][n, p]

    def spacing():
        h, _ = ctx.scan_spacing(s5, an, 10, pw, lens, sthr, margin=margin)
        return digest(h), ctx.last_timing()[1], {"anchors": int(len(an))}
    out["spacing"] = spacing

    fl, fb = peaks(200_000, rng)
    st = stores(ctx, fl, fb, int(lens.min()))

    def ragged():
        c, launches = np.zeros((len(lens), 4), np.int64), {}
        for s, _, _ in st:
            c += ctx.scan(s, pw, lens, thr, want_hits=False)[1]
            for k, v in ctx.last_timing()[1].items():
                launches[k] = launches.get(k, 0) + v
        return digest(c), launches, {"stores": len(st), "path": _lib.scan_last_path(ctx)}
    out["ragged"] = ragged
    return out


def one(reps):
    import motifs_jl_b200 as mb
    ctx = mb.Context(0)
    res = {}
    for name, run in workloads(ctx).items():
        h0, _, _ = run()                                            # warm-up (and the tensor-core path's CTA balance)
        ts = []
        for _ in range(reps):
            t0 = time.perf_counter()
            h, launches, extra = run()
            ts.append((time.perf_counter() - t0) * 1e3)
            if h != h0:
                raise RuntimeError(f"{name}: outputs differ between calls of one build")
        res[name] = {"hash": h, "launches": launches, "best_ms": round(min(ts), 2), **extra}
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("other_lib", nargs="?")
    ap.add_argument("--one", action="store_true", help="measure the library MB200_LIBRARY selects (this tree's by default)")
    ap.add_argument("--reps", type=int, default=3)
    args = ap.parse_args()
    if args.one:
        print(json.dumps(one(args.reps)))
        return
    if not args.other_lib:
        ap.error("give the other build's library")
    from scan_ragged import gpu_info
    out = {"gpu": gpu_info(), "old": os.path.basename(args.other_lib), "new": "this tree's build", "runs": []}
    for side in ("old", "new", "old", "new"):
        env = dict(os.environ)
        env.pop("MB200_LIBRARY", None)
        if side == "old":
            env["MB200_LIBRARY"] = os.path.abspath(args.other_lib)
        r = subprocess.run([sys.executable, os.path.abspath(__file__), "--one", "--reps", str(args.reps)], env=env,
                           capture_output=True, text=True)
        if r.returncode:
            sys.exit(f"{side} run failed:\n{r.stderr[-4000:]}")
        out["runs"].append({"side": side, **json.loads(r.stdout.strip().splitlines()[-1])})
    runs = out["runs"]
    out["equal"] = {w: all(r[w]["hash"] == runs[0][w]["hash"] and r[w]["launches"] == runs[0][w]["launches"] for r in runs)
                    for w in runs[0] if w != "side"}
    out["best_ms"] = {w: {side: [r[w]["best_ms"] for r in runs if r["side"] == side] for side in ("old", "new")} for w in out["equal"]}
    out["gpu_after"] = gpu_info()
    print(json.dumps(out))
    sys.exit(0 if all(out["equal"].values()) else 1)


if __name__ == "__main__":
    main()
