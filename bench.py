#!/usr/bin/env python
"""bench.py — the hot path on synthetic input of BASELINE.json's shapes; prints ONE JSON line (rank 0).

  python bench.py --gpus 1 --steps 3 --warmup 3
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
      bench.py --gpus N --steps K --warmup W
  python bench.py --impl reference ...     # the CPU restatement of the reference on the host cores
  python bench.py ... --dump-outputs bench_outputs/a   # also writes the last timed step's outputs as <name>.npy (compare two builds)

BASELINE.json's metric has two halves and the line carries both, plus one nested row per remaining GPU config:
  * top level  — scanned bp/s on configs[3], the scan sweep: 500 PWMs (len 8-40) over 10M x 200 bp (2 Gbp), forward +
    reverse strands, fused threshold, per-motif occurrence counts.  A "step" is one pass of the scan over all sequences.
    At N>1 the sequences are sharded over ranks (strong scaling: total work fixed), no data-path collective; the per-motif
    counts are summed once per step by ONE all-reduce inside the library (MB200_SCAN_REDUCE).  Every rank generates the SAME
    global data set (seeded per 1 Mi-sequence chunk) and takes its slice, so `checks.counts_sha` must be identical at every N.
    Inputs exceed L2 (0.5 GB packed), no flush needed.
  * "training" — training sequences/s on configs[1] (20k x 100 bp, batch 6 per rank, AdaBelief): optimiser steps of the
    unrolled CSC network (forward + hand-derived reverse pass + update), one all-reduce of the 30 433 gradients per step
    inside mb200_csc_adabelief_step at N>1 (weak scaling: every rank adds a batch of 6).
  * "config3_training" — configs[2]: 200k x 200 bp data-parallel training, same step; at N>1 the line carries the in-line check
    "all-reduced gradient == mean of the per-rank gradients".
  * "config5_long_scan" — configs[4]: one 250 Mbp sequence + its 1-mer shuffle, 50 PWMs, tiled scan, counts, Fisher (rank 0).
"""
import argparse
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CHUNK = 1 << 20                                   # sequences per seeded chunk of the global scan data set
FP32_SIMT_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12   # 148 SMs x 128 FMA lanes x 2 flop x 1.965 GHz


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3,
                    help="timed steps of every timed loop: scan passes, bench steps of --train-steps / --c3-steps optimiser steps (10 of the "
                         "64-group row, 200 of the 16-group row), code-retrieval calls, score > 0 scans, config-5 steps, and their end-to-end legs")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="all", choices=["all", "both", "scan", "train", "config3", "config5"])
    ap.add_argument("--nseq", type=int, default=10_000_000)
    ap.add_argument("--seqlen", type=int, default=200)
    ap.add_argument("--motifs", type=int, default=500)
    ap.add_argument("--train-nseq", type=int, default=20_000)
    ap.add_argument("--train-seqlen", type=int, default=100)
    ap.add_argument("--train-steps", type=int, default=1500, help="optimiser steps per timed bench step")
    ap.add_argument("--c3-nseq", type=int, default=200_000)
    ap.add_argument("--c3-seqlen", type=int, default=200)
    ap.add_argument("--c3-steps", type=int, default=600, help="optimiser steps of the config-3 row")
    ap.add_argument("--c3-groups", type=int, default=1, help="batches of 6 per rank and optimiser step in the config-3 row")
    ap.add_argument("--c5-bp", type=int, default=250_000_000)
    ap.add_argument("--c5-motifs", type=int, default=50)
    ap.add_argument("--c5-check-bp", type=int, default=10_000_000, help="prefix of the config-5 sequence the oracle re-counts")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="target CPU time of each cpu_baseline sample")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what each timed path returned in its last step as DIR/<name>.npy (float32 or "
                         "float64, at most 64 MB in all); the inputs depend on the arguments only, so two builds can be compared file by file")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


OUTPUTS = {}                                      # name -> what a timed path returned in its last step (--dump-outputs), rank 0
DUMP_MAX_BYTES = 64 << 20
CODES_MAX_ROWS = 1_900_000                        # 30.4 MB of float32 per code-retrieval path (two paths + the rest < 64 MB)


def code_records(recs, n_seqs):
    """code records as (n, 4) float32 rows (seq, fil, position, magnitude), sorted, so that two builds compare row by row; exact
    while sequence indices stay below 2^24.  When the library's bound of 64 records per sequence could exceed CODES_MAX_ROWS, only
    the records of every k-th sequence are kept: a choice by content, so the kept rows stay comparable whatever the record count."""
    a = np.stack([recs["seq"], recs["fil"], recs["position"], np.ascontiguousarray(recs["mag_f16"]).view(np.float16)], axis=1).astype(np.float32)
    k = -(-64 * n_seqs // CODES_MAX_ROWS)
    if k > 1:
        a = a[np.asarray(recs["seq"]) % k == 0]
    return a[np.lexsort(a.T[::-1])]


def dump_outputs(d):
    total = sum(a.nbytes for a in OUTPUTS.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed {DUMP_MAX_BYTES}")
    os.makedirs(d, exist_ok=True)
    for name, a in OUTPUTS.items():
        assert a.dtype in (np.float32, np.float64), (name, a.dtype)
        np.save(os.path.join(d, f"{name}.npy"), a)


class ClockSampler:
    """nvidia-smi clocks during the timed region (B200_PROFILING.md recipe)."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.t.join(timeout=2)
        sm = [float(r[0]) for r in self.rows if len(r) >= 6 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 6 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(sm)}


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


def load_expected():
    """hashes of the global count tables baked from an N=1 run (tests/golden/bench_expected.json): the only hardware proof that
    sharding + the in-library reduce return what one GPU returns."""
    try:
        return json.load(open(os.path.join(ROOT, "tests", "golden", "bench_expected.json")))
    except Exception:
        return {}


def sha_of(a):
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()[:16]


# ------------------------------------------------------------------------------------------------------------------
# scan half
# ------------------------------------------------------------------------------------------------------------------
def make_motifs(K, seed=4):
    """SURVEY §8d cfg 4: K count matrices (len U{8..40}, columns 1000 x Dirichlet(0.3)), pfm/pwm per B0 with bg = 0.25; thresholds
    per B4: Touzet p-value thresholds (mb200_pvalue2score) where get_best_thresh takes that branch — some effective segment
    shorter than 15 (_s2_filter_pos_w_scores.jl:91-98) — else 0.7 x the best possible score (stated)."""
    from motifs_jl_b200 import synth, inference, _lib
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(K, 8, 40, seed))
    thr = synth.stated_thresholds(ms, 0.7)
    n_touzet = 0
    bg = np.full(4, 0.25)
    for k in range(K):
        segs = ms.effective_segments[k]
        if any(len(r) < inference.max_pwm_length_Touzet2 for r in segs):
            best, ok = 0.0, True
            for r in segs:
                if len(r) > inference.max_pwm_length_Touzet2 or len(r) <= 1:
                    continue
                sub = np.asarray(ms.pwms[k], np.float16)[:, r.start - 1: r.stop - 1]
                sc = _lib.pvalue2score(None, sub, inference.get_pvalue(sub), inference._granularity_, bg)
                if sc is None:
                    ok = False
                    break
                best += sc
            if ok and best > 0:
                thr[k] = np.float16(best)
                n_touzet += 1
    return ms, thr, n_touzet


def cells_per_seq(lens, Lb):
    lens = np.asarray(lens, np.int64)
    return int(2 * ((Lb - lens + 1).clip(min=0) * lens).sum())


def scan_config(args, n_touzet=None):
    return {"workload": f"scan sweep: {args.motifs} PWMs (len 8-40) x {args.nseq} seqs x {args.seqlen} bp, fwd+rc, fused threshold, counts",
            "baseline_config_index": 3, "n_seqs": args.nseq, "seq_len": args.seqlen, "n_motifs": args.motifs,
            "thresholds": "Touzet p-value threshold where get_best_thresh takes that branch (an effective segment < 15), else 0.7 x max score (Float16)",
            "data_seeding": f"global data set seeded per chunk of {CHUNK} sequences (identical at every N)",
            "l2": "inputs larger than L2 (no flush needed)", "parallelism": f"seq-shard x{args.gpus}"}


def train_config(nseq, Lb, world, opt_steps, index, groups=1):
    return {"workload": f"CSC training: {nseq} seqs x {Lb} bp (planted gapped motif), {groups} batch(es) of 6 per rank and optimiser step, "
                        f"M=50 K=24 h=12 q=32, 6 XYZ + 3 DF passes, AdaBelief",
            "baseline_config_index": index, "n_seqs": nseq, "seq_len": Lb, "global_batch": 6 * groups * world, "groups_per_rank": groups,
            "optimizer_steps_per_bench_step": opt_steps, "parallelism": f"dp{world}",
            "l2": "working set (<20 MB) is L2 resident by design" if groups == 1 else "working set (~14 MB per group) exceeds L2: no flush needed"}


def oracle_threads():
    """all host cores for the CPU arm, whatever OMP_NUM_THREADS the launcher exported (torchrun sets 1)."""
    from oracle import scan_oracle as so
    cores = os.cpu_count() or 1
    return so.set_threads(cores)


def cpu_scan_rate(pw, lens, thr, ascii_rows, target_s):
    """oracle (CPU port) scan+filter+counts on a bounded sample, all host threads; returns (bp/s, sample, threads, seconds)."""
    from oracle import scan_oracle as so
    threads = oracle_threads()
    codes = so.ascii_to_codes(ascii_rows)
    probe = min(len(codes), 16 * threads)
    t0 = time.perf_counter()
    so.scan(pw, lens, codes[:probe], thr, want_hits=False)
    dt = time.perf_counter() - t0
    n = int(min(len(codes), max(probe, probe * target_s / max(dt, 1e-6))))
    t0 = time.perf_counter()
    so.scan(pw, lens, codes[:n], thr, want_hits=False)
    dt = time.perf_counter() - t0
    return n * codes.shape[1] / dt, n, threads, dt


def cpu_train_rate(ascii_rows, flat, target_s):
    """oracle (PyTorch-CPU position-space restatement + autograd) loss/gradient/AdaBelief steps on the host cores."""
    import torch
    from oracle import csc_oracle as co, scan_oracle as so
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    hp = co.Hyperparam()
    codes = so.ascii_to_codes(ascii_rows)
    n = co.n_params(hp)
    p = flat.astype(np.float32).copy()
    mt, st = np.zeros(n), np.zeros(n)
    rng = np.random.default_rng(0)
    steps, t0 = 0, time.perf_counter()
    while True:
        idx = rng.permutation(len(codes))[:hp.batch_size]
        _, g, _ = co.loss_and_grad(codes[idx], p, hp)
        pn, mt, st = co.adabelief_step(p[:n].astype(np.float64), g[:n].astype(np.float64), mt, st, t=steps + 1)
        p[:n] = pn.astype(np.float32)
        steps += 1
        dt = time.perf_counter() - t0
        if dt >= target_s or steps >= 400:
            break
    return hp.batch_size * steps / dt, steps, torch.get_num_threads(), dt


def gen_scan_rows(torch, dev, n_lo, n_hi, Lb, seed0=4):
    """rows [n_lo, n_hi) of the GLOBAL data set: chunk c (CHUNK sequences) is drawn from a generator seeded seed0 + c, whichever rank
    needs it, so every world size scans the same 2 Gbp."""
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    out = torch.empty((n_hi - n_lo, Lb), dtype=torch.uint8, device=dev)
    for c in range(n_lo // CHUNK, (n_hi + CHUNK - 1) // CHUNK):
        g = torch.Generator(device=dev)
        g.manual_seed(seed0 + 7919 * c)
        rows = lut[torch.randint(0, 4, (CHUNK, Lb), device=dev, generator=g, dtype=torch.int64)]
        lo, hi = max(n_lo, c * CHUNK), min(n_hi, (c + 1) * CHUNK)
        out[lo - n_lo: hi - n_lo] = rows[lo - c * CHUNK: hi - c * CHUNK]
        del rows
    return out


def bench_scan(args, ctx, torch, dist, world, rank, local, dev, stream):
    from motifs_jl_b200 import inference, _lib as mblib
    K, Lb = args.motifs, args.seqlen
    n_lo, n_hi = args.nseq * rank // world, args.nseq * (rank + 1) // world
    n_local = n_hi - n_lo
    ms, thr, n_touzet = make_motifs(K)
    pw, lens = inference.pack_pwms(ms), ms.lens
    ascii_dev = gen_scan_rows(torch, dev, n_lo, n_hi, Lb)
    ascii_host = torch.empty((n_local, Lb), dtype=torch.uint8, pin_memory=True)
    ascii_host.copy_(ascii_dev)
    torch.cuda.synchronize()
    seqs = ctx.seqs_from_device_ptr(ascii_dev.data_ptr(), n_local, Lb)
    del ascii_dev

    def step_resident():
        _, c = ctx.scan(seqs, pw, lens, thr, want_hits=False, want_counts=True, reduce=True)      # counts summed over ranks inside the call
        return c

    def step_e2e():
        s2 = ctx.seqs_from_host_ptr(ascii_host.data_ptr(), n_local, Lb, wait=False)     # H2D of this step's input + pack, overlapping the scan
        _, c = ctx.scan(s2, pw, lens, thr, want_hits=False, want_counts=True, reduce=True)
        s2.free()
        return c

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t_scan = t_cnt = 0.0
        n_launch = nk = 0
        timed.t_verify = 0.0
        e0.record(stream)
        for _ in range(steps):
            res = fn()
            t, l = ctx.last_timing()
            t_scan += t["scan"]; t_cnt += t["count"]; nk += l["scan"]; timed.t_verify += t["emit"]
            n_launch += sum(l.values())
        e1.record(stream)
        barrier()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        return float(tt.item()) / steps, res, t_scan, t_cnt, nk, n_launch

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    ms_step, counts, t_scan, t_cnt, n_scan_launch, n_launch = timed(step_resident, args.steps, args.warmup)
    if rank == 0:
        OUTPUTS["scan_counts"] = counts.astype(np.float64)
    t_verify = timed.t_verify
    scan_path = mblib.scan_last_path(ctx)                                     # 1: tcgen05 pre-filter + exact re-scoring, 0: SIMT scan_kernel
    clocks = sampler.stop() if rank == 0 else None
    ms_e2e, counts2, *_ = timed(step_e2e, max(1, args.steps), 1)
    assert np.array_equal(counts, counts2)
    # reference semantics without a threshold (hit = score > 0, _h3_1_alignment.jl:33,82 — what scan_w_gpu! and the histogram scans
    # of render_result! run): SIMT scan_kernel, counts only, on a bounded slice of this rank's shard
    n_gt0 = min(n_local, max(1, 1_000_000 // world))
    s_gt0 = ctx.seqs_from_host_ptr(ascii_host.data_ptr(), n_gt0, Lb)
    ctx.scan(s_gt0, pw, lens, None, want_hits=False, want_counts=True)
    barrier()
    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    g0.record(stream)
    for _ in range(args.steps):
        ctx.scan(s_gt0, pw, lens, None, want_hits=False, want_counts=True, reduce=True)
    g1.record(stream)
    barrier()
    tg = torch.tensor([g0.elapsed_time(g1) / args.steps], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(tg, op=dist.ReduceOp.MAX)
    ms_gt0 = float(tg.item())
    s_gt0.free()
    total_bp = args.nseq * Lb
    out = None
    if rank == 0:
        peaks = load_peaks()
        hbm_peak = float(peaks.get("hbm_gbs", 6650.0))
        launches_per_step = n_scan_launch / args.steps
        bytes_per_launch = (n_local * Lb / 4.0) / launches_per_step + float(2 * 4 * lens.sum() * 2)
        ms_per_launch = t_scan / max(1, n_scan_launch)
        ach = bytes_per_launch / (ms_per_launch * 1e-3) / 1e9
        cells_rate = cells_per_seq(lens, Lb) * n_local / ((t_scan / args.steps) * 1e-3)
        sm_mhz = (clocks or {}).get("sm_mhz") or float(peaks.get("sm_max_mhz", 1965.0))
        alu_peak = 148 * 4 * (512.0 / 28.0) * sm_mhz * 1e6             # cells/s when the ALU pipe is saturated (see DESIGN.md 3.1)
        key = f"scan_n{args.nseq}_l{Lb}_k{K}"
        exp = load_expected().get(key)
        csha = sha_of(counts)
        out = {"metric": "scanned_bp_per_sec", "value": total_bp / (ms_step / 1e3), "unit": "bp/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
               "dtype": "f16", "data": "synthetic", "config": scan_config(args),
               "e2e": {"value": total_bp / (ms_e2e / 1e3), "unit": "bp/s", "ms_per_step": ms_e2e,
                       "h2d_bytes_per_step": int(n_local * Lb + pw.nbytes + lens.nbytes + 2 * K), "d2h_bytes_per_step": int(K * 4 * 8)},
               "gpu_launches": int(n_launch), "clocks": clocks,
               "roofline": {"bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                            "traffic": 30760.0 * (n_local / launches_per_step) if (Lb == 200 and K == 500) else None,
                            "traffic_source": "ncu --set full of one launch, profiles/r01_scan_v2_ncu_full_summary.csv: dram read+write = 30.76 KB per sequence "
                                              "(hit-mask writes), scaled to this launch's sequences; not re-measured in this run",
                            "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback", "kernel": "scan_kernel",
                            "ms_per_launch": ms_per_launch, "kernel_share_of_step": (t_scan / args.steps) / ms_step,
                            "count_kernel_share_of_step": (t_cnt / args.steps) / ms_step,
                            "note": "2-bit packing makes the scan table-lookup bound, not HBM bound (SURVEY §8d): see binding",
                            "binding": {"bound": "alu-issue", "what": "per PWM cell: 1/2 PRMT (entry select) + 1/2 HADD2/HFMA2 (one sequential Float16 add); the 8 PRMT + ~4 HADD2 per column "
                                                "share the ALU pipe (1 instr / 2 clk / SM sub-partition): ~28 clk per 512 cells",
                                        "cells_per_s": cells_rate, "achieved": cells_rate / 1e12, "peak": alu_peak / 1e12, "unit": "Tcell/s",
                                        "frac": cells_rate / alu_peak, "peak_source": "148 SM x 4 sub-partitions x 512 cells / 28 clk x SM clock under load"}},
               "checks": {"counts_sum": [int(x) for x in counts.sum(axis=0)], "counts_sha": csha, "counts_sha_expected_from_n1": exp,
                          "counts_match_n1": (csha == exp) if exp else None, "touzet_thresholds": int(n_touzet)},
               "scan_score_gt0": {"metric": "scanned_bp_per_sec", "value": n_gt0 * world * Lb / (ms_gt0 / 1e3), "unit": "bp/s", "ms": ms_gt0,
                                  "kernel": "scan_kernel (SIMT, bit-exact HADD2 chain)",
                                  "sample": f"{n_gt0} sequences per rank x {Lb} bp, all {K} PWMs, both strands, hit = score > 0 (no threshold), counts only"}}
        if scan_path == 1:
            # dominant kernel: k_scan_tc (csrc/scan_tc.cuh), a one-hot GEMM on the tensor cores.  Algorithmic flops (SURVEY §8d): 8 per PWM
            # cell = 2 (multiply-add) x 4 (one-hot bases), cells = strands x N x sum_k (Lb - len_k + 1) len_k; the launch also computes the
            # zero padding of K to the longest motif of a 256-slot block and the windows that straddle two sequences, which are not counted.
            tf_peak = float(peaks.get("bf16_tflops_sustained", peaks.get("bf16_tflops", 1413.0)))
            flops_per_launch = 8.0 * cells_per_seq(lens, Lb) * n_local / launches_per_step
            tf = flops_per_launch / (ms_per_launch * 1e-3) / 1e12
            hbm = dict(out["roofline"]); hbm.pop("binding", None); hbm.pop("traffic", None); hbm.pop("traffic_source", None); hbm["kernel"] = "k_scan_tc"
            hbm["note"] = "algorithmic HBM bytes (0.25 B/bp + tables) over the same kernel time: the scan is not HBM bound (SURVEY §8d)"
            out["roofline"] = {"bound": "tensor", "achieved": tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": tf / tf_peak,
                               "traffic": 54.8 * (n_local / launches_per_step) if (Lb == 200 and K == 500) else None,
                               "traffic_source": "ncu --set full of one launch (profiles/r01_scan_tc_ncu_full_summary.csv): dram read + write = 15.96 MB for 291 271 "
                                                 "sequences = 54.8 B per sequence (algorithmic: 50 B packed sequence + the tables once), scaled to this launch's "
                                                 "sequences; not re-measured in this run",
                               "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained (kernel timed inside a long step)" if peaks else "fallback",
                               "kernel": "k_scan_tc", "ms_per_launch": ms_per_launch,
                               "kernel_share_of_step": (t_scan / args.steps) / ms_step,
                               "verify_kernel_share_of_step": (t_verify / args.steps) / ms_step,
                               "count_kernel_share_of_step": (t_cnt / args.steps) / ms_step,
                               "algorithmic_flops_per_launch": flops_per_launch,
                               "note": "FP16 one-hot GEMM pre-filter (FP32 accumulate in TMEM), candidates re-scored with the reference's sequential Float16 adds: "
                                       "hit sets identical to the SIMT kernel; cells/s below counts useful PWM cells only",
                               "cells_per_s": cells_rate, "hbm": hbm}
        if world == 1 and not args.no_cpu_baseline:
            from oracle import scan_oracle as so                              # cpu_baseline leg: the checker, timed on the host cores
            sample = ascii_host[: min(n_local, 20000)].numpy()
            rate, n, threads, dt = cpu_scan_rate(pw, lens, thr, sample, args.cpu_seconds)
            out["cpu_baseline"] = {"value": rate, "unit": "bp/s", "cores": threads, "kind": "port", "seconds": dt,
                                   "sample": f"first {n} of {args.nseq} sequences x {Lb} bp, all {K} PWMs, both strands (oracle/scan_oracle.c, OpenMP, {threads} threads)"}
            _, oc = so.scan(pw, lens, so.ascii_to_codes(sample[:n]), thr, want_hits=False)
            s3 = ctx.seqs_from_ascii(sample[:n])
            _, gc = ctx.scan(s3, pw, lens, thr, want_hits=False)
            out["checks"]["sample_counts_match_oracle"] = bool(np.array_equal(oc, gc))
            out["checks"]["oracle_sample_seqs"] = int(n)
            s3.free()
    seqs.free()
    del ascii_host
    return out


# ------------------------------------------------------------------------------------------------------------------
# training half (configs[1] and configs[2])
# ------------------------------------------------------------------------------------------------------------------
def flops_per_seq(Lb):
    """SURVEY §8d: algorithmic FLOP per sequence of forward + reverse pass, counting the F-layer contractions only (A6/A7/A9/A11)."""
    c = Lb - 7; l = c - 11
    mac = 7 * l * 24 * 12 * 100 + 14 * c * 100 * 24 * 12 + 3 * 12 * 100 * 24 * l
    return 3.0 * 2.0 * mac


def bench_train(args, ctx, torch, dist, world, rank, local, dev, name, N, Lb, opt_steps, index, groups=1, e2e_leg=True, extras=True, warm_mult=50):
    from motifs_jl_b200 import model as mdl, synth
    from motifs_jl_b200._lib import CscModel
    hp = mdl.Hyperparam()
    a = synth.planted_gapped(N, Lb, index + 1)                            # SURVEY §8d: seed 2 for config 2 (index 1), seed 3 for config 3
    n_train = N - int(np.floor((1 - 0.9) * N))                            # loadfasta/helpers.jl:144
    a = a[:n_train]
    pinned = torch.from_numpy(a).pin_memory()
    cdl = mdl.ucdl(hp, np.random.default_rng(2))
    side = torch.cuda.Stream(device=dev)                                  # the library launches (kernels AND its NCCL calls) on this stream
    ctx.set_stream(side.cuda_stream)
    out = None
    with torch.cuda.stream(side):
        seqs = ctx.seqs_from_host_ptr(pinned.data_ptr(), n_train, Lb)
        model = CscModel(ctx, hp, Lb, n_groups=groups)
        model.set_params(cdl.flat)
        model.broadcast_params(0)
        rng = np.random.default_rng(1234)                                 # same permutation stream on every rank
        nb = hp.batch_size * groups
        per_step = nb * world
        state = {"perm": rng.permutation(n_train), "pos": 0, "loss": None, "l1": None}

        def next_idx():
            if state["pos"] + per_step > n_train:
                state["perm"], state["pos"] = rng.permutation(n_train), 0
            lo = state["pos"] + rank * nb
            state["pos"] += per_step
            return state["perm"][lo: lo + nb]

        def opt_step():
            model.step_begin(seqs, next_idx())                            # H2D: the sequence indices; forward + reverse pass
            state["loss"], state["l1"] = model.adabelief_step()           # ONE all-reduce of the gradients (in-library NCCL) + update + D2H of loss, l1

        checks = {}
        if world > 1:
            # in-line proof of the data-parallel step: the gradient the update consumed == mean over ranks of the local gradients
            idx = next_idx()
            _, g_local = model.loss_grad(seqs, idx)
            g_all = ctx.comm_allgather(g_local)
            model.step_begin(seqs, idx)
            model.adabelief_step()
            g_avg = model.get_grads()
            ref = g_all.astype(np.float64).mean(axis=0)
            err = float(np.abs(g_avg - ref).max() / max(np.abs(ref).max(), 1e-30))
            checks["allreduced_grad_vs_mean_of_rank_grads_rel_err"] = err
            checks["allreduced_grad_is_mean"] = bool(err <= 1e-6)
            p_all = ctx.comm_allgather(model.get_params())
            checks["params_identical_on_all_ranks"] = bool((p_all == p_all[0]).all())
        for _ in range(max(3, min(args.warmup, 3) * warm_mult)):          # >= 3 warm-up iterations of the step (graph capture included)
            opt_step()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = ctx.last_timing()[1]["csc"]
        n_bench = args.steps
        e0.record(side)
        t0 = time.perf_counter()
        for _ in range(n_bench * opt_steps):
            opt_step()
        e1.record(side)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        launches = int(ctx.last_timing()[1]["csc"] - l0)
        if rank == 0:
            OUTPUTS[f"{name}_loss_l1"] = np.array([state["loss"], state["l1"]], np.float32)
            OUTPUTS[f"{name}_params"] = model.get_params()
        tt = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        ms_bench_step = float(tt.item()) / n_bench
        n_opt = n_bench * opt_steps
        ms_opt = ms_bench_step / opt_steps
        ms_e2e_opt = None
        if e2e_leg:
            # end-to-end leg: every optimiser step ships ITS batch from host memory (the reference's `S |> gpu`, train.jl:41):
            # ASCII rows -> 2 bit/base -> one H2D copy -> step -> D2H of loss and l1
            def opt_step_host():
                model.step_begin_host(a[next_idx()])
                state["loss"], state["l1"] = model.adabelief_step()

            for _ in range(50):
                opt_step_host()
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            f0.record(side)
            for _ in range(args.steps * opt_steps):
                opt_step_host()
            f1.record(side)
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t2 = torch.tensor([f0.elapsed_time(f1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(t2, op=dist.ReduceOp.MAX)
            ms_e2e_opt = float(t2.item()) / (args.steps * opt_steps)
        if rank == 0:
            peaks = load_peaks()
            seq_s = nb * world * opt_steps / (ms_bench_step / 1e3)
            tf = flops_per_seq(Lb) * seq_s / 1e12
            tf_peak = float(peaks.get("bf16_tflops_sustained", 1413.0))
            out = {"metric": "training_sequences_per_sec", "value": seq_s, "unit": "seq/s", "n_gpus": world, "steps": n_bench,
                   "ms_per_step": ms_bench_step, "ms_per_optimizer_step": ms_opt, "higher_is_better": True,
                   "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": train_config(N, Lb, world, opt_steps, index, groups),
                   "gpu_launches": launches, "kernels_per_optimizer_step": launches / n_opt,
                   "roofline": {"bound": "latency", "achieved": tf, "peak": tf_peak, "unit": "TFLOP/s", "frac": tf / tf_peak,
                                "peak_source": "MEASURED_PEAKS.json bf16_tflops_sustained" if peaks else "fallback",
                                "fp32_simt_peak_tflops": FP32_SIMT_TFLOPS, "frac_of_fp32_simt_peak": tf / FP32_SIMT_TFLOPS,
                                "algorithmic_flops_per_seq": flops_per_seq(Lb), "kernels_per_optimizer_step": launches / n_opt,
                                "us_per_kernel": 1e3 * ms_opt / max(1.0, launches / n_opt),
                                "traffic": 586752.0 if (groups == 1 and Lb == 100) else None,
                                "traffic_source": "ncu --set full of one k_csc_fused_fwd launch (the dominant kernel, 59 % of the step): dram read + write = 0.587 MB "
                                                  "(profiles/r02_csc_fused_fwd_ncu_full_summary.csv); the working set is L2 resident" if (groups == 1 and Lb == 100) else None,
                                "note": "a batch of 6 is a dependent chain of small fp32 ops (SURVEY §8d): the step is bound by launch / dependency latency, "
                                        "neither by HBM nor by the tensor pipe; achieved = algorithmic F-layer flops (fwd + reverse = 3 x fwd) x seq/s"},
                   "final_loss": state["loss"], "final_l1_F": state["l1"], "wall_s": wall, "optimizer_steps_timed": n_opt, "checks": checks}
            if ms_e2e_opt is not None:
                # value: sequences resident in HBM, a step ships the indices.  e2e: every step ships its sequences from the host.
                out["e2e"] = {"value": nb * world / (ms_e2e_opt / 1e3), "unit": "seq/s", "ms_per_optimizer_step": ms_e2e_opt,
                              "h2d_bytes_per_step": int(opt_steps * nb * ((Lb + 15) // 16) * 4),
                              "d2h_bytes_per_step": int(opt_steps * 8),
                              "note": "per optimiser step: the ASCII rows packed to 2 bit/base on the host, one H2D copy, loss + l1 read back"}
            if extras and world == 1 and not args.no_cpu_baseline:
                rate, steps, cores, dt = cpu_train_rate(a[:2000], cdl.flat, args.cpu_seconds)
                out["cpu_baseline"] = {"value": rate, "unit": "seq/s", "cores": cores, "kind": "port", "seconds": dt,
                                       "sample": f"{steps} optimiser steps of batch 6 (oracle/csc_oracle.py, PyTorch-CPU fp32 + autograd, {cores} threads)"}
        p_trained = model.get_params()
        model.free()
        if extras:
            # code retrieval (inference/_1_code_retrieval.jl:33-56) over the training set with the parameters training just produced: 1024 batches of
            # 6 per launch sequence, fp32 (the parity path) and with the dense contraction on the tcgen05 BF16 kernel (stated tolerance); with a
            # communicator the batches are sharded over the ranks and the records all-gathered
            res = {}
            for tag, tc in (("fp32", False), ("tensor_cores_bf16", True)):
                n_dec = n_train - n_train % hp.batch_size
                G = max(1, min(1024, -(-(n_dec // hp.batch_size) // world)))
                mc = CscModel(ctx, hp, Lb, n_groups=G, forward_only=True, tensor_cores=tc)
                mc.set_params(p_trained)
                recs = mc.codes(seqs, shard="comm" if world > 1 else None)                    # warm-up (and the records for the comparison)
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                c0.record(side)
                for _ in range(args.steps):
                    last = mc.codes(seqs, shard="comm" if world > 1 else None)
                c1.record(side)
                if world > 1:
                    dist.barrier()
                torch.cuda.synchronize()
                if rank == 0:
                    OUTPUTS[f"{name}_codes_{tag}"] = code_records(last, n_dec)
                tc_ms = torch.tensor([c0.elapsed_time(c1) / args.steps], dtype=torch.float64, device=dev)
                if world > 1:
                    dist.all_reduce(tc_ms, op=dist.ReduceOp.MAX)
                res[tag] = (recs, float(tc_ms.item()), n_dec)
                mc.free()
            if rank == 0:
                r32, ms32, n_dec = res["fp32"]
                rtc, mstc, _ = res["tensor_cores_bf16"]
                key = lambda r: (r["seq"].astype(np.int64) * 65536 + r["fil"].astype(np.int64)) * 65536 + r["position"].astype(np.int64)
                same = int(np.intersect1d(key(r32), key(rtc)).size)
                out["code_retrieval"] = {"metric": "decoded_sequences_per_sec", "value": n_dec / (ms32 / 1e3), "unit": "seq/s", "ms": ms32,
                                         "records": int(len(r32)), "dtype": "f32",
                                         "sample": f"{n_dec} sequences x {Lb} bp, 6 ADMM_XYZ passes, {world} rank(s), records (position, fil, seq, Float16 magnitude) returned to the host",
                                         "tensor_cores_bf16": {"value": n_dec / (mstc / 1e3), "unit": "seq/s", "ms": mstc, "records": int(len(rtc)),
                                                               "records_also_in_fp32": same, "fraction_of_fp32_records": same / max(1, len(r32)),
                                                               "note": "opt-in (tcgen05 kind::f16, BF16 operands): the top-q projection is discontinuous, so rounded operands move a few codes; the fp32 path is the parity path"}}
        # extra data point (NOT the headline): 16 independent batches of 6 per optimiser step on one GPU — the same arithmetic as
        # 16 data-parallel ranks (global batch 96, gradients averaged), i.e. a different optimisation trajectory than the reference's
        if extras and rank == 0 and world == 1:
            G = 16
            mg = CscModel(ctx, hp, Lb, n_groups=G)
            mg.set_params(cdl.flat)
            r2 = np.random.default_rng(7)
            for _ in range(20):
                mg.step_begin(seqs, r2.permutation(n_train)[:6 * G]); mg.adabelief_step()
            torch.cuda.synchronize()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            nst = 200 * args.steps                                         # bench steps of 200 optimiser steps
            g0.record(side)
            for _ in range(nst):
                mg.step_begin(seqs, r2.permutation(n_train)[:6 * G]); loss_l1 = mg.adabelief_step()
            g1.record(side)
            torch.cuda.synchronize()
            OUTPUTS[f"{name}_batched_groups_loss_l1"] = np.array(loss_l1, np.float32)
            OUTPUTS[f"{name}_batched_groups_params"] = mg.get_params()
            msg = g0.elapsed_time(g1) / nst
            out["batched_groups"] = {"groups_per_step": G, "global_batch": 6 * G, "value": 6 * G / (msg / 1e3), "unit": "seq/s",
                                     "ms_per_optimizer_step": msg,
                                     "note": "each group is a reference batch (own median mask, own D/F updates); gradients averaged over groups"}
            mg.free()
        seqs.free()
    ctx.set_stream(None)
    return out


# ------------------------------------------------------------------------------------------------------------------
# configs[4]: chromosome-length sequence, tiled scan, counts fg + bg, Fisher
# ------------------------------------------------------------------------------------------------------------------
def bench_long_scan(args, ctx, torch, dev, stream):
    """SURVEY §8d cfg 5: one sequence of 250 Mbp with 3 planted motif families every ~50 kb; background = 1-mer shuffle (a permutation,
    drawn on the device by mb200_seqs_shuffle); K = 50 PWMs len 8-40; per-motif hit / unique / coverage counts fg and bg, Fisher.
    Rank 0 only: the reference's union_ranges coverage is defined per sequence (its last interval is dropped, _h4_overlap_ratio.jl:48-56),
    so cutting ONE sequence over ranks would change the counted value."""
    from motifs_jl_b200 import inference, synth
    Lg, K = args.c5_bp, args.c5_motifs
    ms = synth.motifs_from_count_matrices(synth.random_count_matrices(K, 8, 40, 5))
    thr = synth.stated_thresholds(ms, 0.7)
    pw, lens = inference.pack_pwms(ms), ms.lens
    g = torch.Generator(device=dev)
    g.manual_seed(5)
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    seq = torch.empty(Lg, dtype=torch.uint8, device=dev)
    piece = 1 << 26
    for s in range(0, Lg, piece):
        e = min(Lg, s + piece)
        seq[s:e] = lut[torch.randint(0, 4, (e - s,), device=dev, generator=g, dtype=torch.int64)]
    # plant the consensus of motif families 0, 1, 2 every ~50 kb (fixed stride + family-dependent offset)
    for fam in range(3):
        cons = np.asarray(ms.pwms[fam], np.float32).argmax(axis=0)
        site = lut[torch.from_numpy(cons).to(dev)]
        starts = torch.arange(1000 + 17_000 * fam, Lg - 64, 50_000, device=dev)
        idx = (starts[:, None] + torch.arange(len(cons), device=dev)[None, :]).reshape(-1)
        seq[idx] = site.repeat(len(starts))
    host = torch.empty(Lg, dtype=torch.uint8, pin_memory=True)
    host.copy_(seq)
    torch.cuda.synchronize()
    fg = ctx.seqs_from_device_ptr(seq.data_ptr(), 1, Lg)
    del seq
    bg = fg.shuffle(1, seed=5)

    def step():
        _, c = ctx.scan(fg, pw, lens, thr, want_hits=False, want_counts=True)
        _, cb = ctx.scan(bg, pw, lens, thr, want_hits=False, want_counts=True)
        return c, cb

    for _ in range(2):
        step()
    torch.cuda.synchronize()
    n = args.steps
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(n):
        c, cb = step()
    e1.record(stream)
    torch.cuda.synchronize()
    ms_step = e0.elapsed_time(e1) / n
    OUTPUTS["config5_long_scan_fg_counts"] = c.astype(np.float64)
    OUTPUTS["config5_long_scan_bg_counts"] = cb.astype(np.float64)
    # end to end: both sequences from pinned host ASCII each step
    bg_host = torch.from_numpy(bg.to_ascii().reshape(-1)).pin_memory()

    def step_e2e():
        s1 = ctx.seqs_from_host_ptr(host.data_ptr(), 1, Lg, wait=False)
        _, c1 = ctx.scan(s1, pw, lens, thr, want_hits=False, want_counts=True)
        s2 = ctx.seqs_from_host_ptr(bg_host.data_ptr(), 1, Lg, wait=False)
        _, c2 = ctx.scan(s2, pw, lens, thr, want_hits=False, want_counts=True)
        s1.free(); s2.free()
        return c1, c2

    step_e2e()
    torch.cuda.synchronize()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record(stream)
    for _ in range(n):
        c1, c2 = step_e2e()
    f1.record(stream)
    torch.cuda.synchronize()
    ms_e2e = f0.elapsed_time(f1) / n
    assert np.array_equal(c1, c) and np.array_equal(c2, cb)

    class _D:
        N, N_test, L = 1, 1, Lg
    pvec = inference.fisher_pvec(c[:, 2], cb[:, 2], _D())
    out = {"metric": "scanned_bp_per_sec", "value": 2.0 * Lg / (ms_step / 1e3), "unit": "bp/s", "n_gpus": 1, "steps": n, "ms_per_step": ms_step,
           "higher_is_better": True, "dtype": "f16", "data": "synthetic",
           "config": {"workload": f"long-sequence scan: one {Lg} bp sequence + its 1-mer shuffle (device permutation), {K} PWMs (len 8-40), fwd+rc, "
                                  f"fused threshold 0.7 x max, hit / unique / coverage counts, Fisher", "baseline_config_index": 4,
                      "tiling": "the library cuts the sequence into batches of 256-position tiles; windows read across tile borders (motif-length halo), "
                                "a hit belongs to the tile of its start", "parallelism": "rank 0 only (per-sequence coverage quirk)"},
           "e2e": {"value": 2.0 * Lg / (ms_e2e / 1e3), "unit": "bp/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": int(2 * Lg), "d2h_bytes_per_step": int(2 * K * 32)},
           "checks": {"fg_counts_sum": [int(x) for x in c.sum(axis=0)], "bg_counts_sum": [int(x) for x in cb.sum(axis=0)],
                      "planted_families_significant": bool((pvec[:3] < 1e-5).all()), "n_significant_1e-5": int((pvec < 1e-5).sum()),
                      "counts_sha": sha_of(np.concatenate([c, cb]))}}
    exp = load_expected().get(f"long_l{Lg}_k{K}")
    out["checks"]["counts_sha_expected"] = exp
    out["checks"]["counts_match_expected"] = (out["checks"]["counts_sha"] == exp) if exp else None
    if not args.no_cpu_baseline and args.c5_check_bp > 0:
        # oracle equality on a prefix of both sequences (>= 10 Mbp each): same thresholds, counts of that prefix scanned on its own
        from oracle import scan_oracle as so
        oracle_threads()
        nchk = min(Lg, args.c5_check_bp)
        ok = True
        t0 = time.perf_counter()
        for hbuf in (host, bg_host):
            rows = hbuf[:nchk].numpy().reshape(1, nchk)
            _, oc = so.scan(pw, lens, so.ascii_to_codes(rows), thr, want_hits=False)
            sp = ctx.seqs_from_ascii(rows)
            _, gc = ctx.scan(sp, pw, lens, thr, want_hits=False)
            sp.free()
            ok = ok and bool(np.array_equal(oc, gc))
        dt = time.perf_counter() - t0
        out["checks"]["prefix_counts_match_oracle"] = ok
        out["checks"]["oracle_prefix_bp"] = int(nchk)
        out["cpu_baseline"] = {"value": 2.0 * nchk / dt, "unit": "bp/s", "cores": os.cpu_count(), "kind": "port", "seconds": dt,
                               "sample": f"first {nchk} bp of the sequence and of its shuffle, all {K} PWMs (oracle + the GPU re-scan of the same prefix inside the timed span)"}
    fg.free(); bg.free()
    return out


def run_reference(args):
    """--impl reference: the reference cannot run here (Julia absent, CuArray-typed code), so this arm times the oracle's CPU
    restatement of the same path on the host cores (SURVEY §8c/§8d, BASELINE.md §3), bounded sample per step.  torchrun exports
    OMP_NUM_THREADS=1 to its workers: the arm sets its own thread count and prints what OpenMP really used."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cores = os.cpu_count() or 1
    os.environ["OMP_NUM_THREADS"] = str(cores)                                # before libgomp is loaded
    from motifs_jl_b200 import inference, model as mdl, synth
    from oracle import scan_oracle as so
    threads = oracle_threads()
    ms, thr, _ = make_motifs(args.motifs)
    pw, lens = inference.pack_pwms(ms), ms.lens
    per_step_target = max(2.0, min(args.cpu_seconds, 60.0 / max(1, args.steps + args.warmup)))
    sample = synth.random_ascii(min(args.nseq, 20000), args.seqlen, 4)
    _, n, threads, _ = cpu_scan_rate(pw, lens, thr, sample, per_step_target)
    codes = so.ascii_to_codes(sample[:n])
    times = []
    for i in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        so.scan(pw, lens, codes, thr, want_hits=False)
        if i >= args.warmup:
            times.append(time.perf_counter() - t0)
    ms_step = 1e3 * float(np.mean(times))
    value = n * args.seqlen / (ms_step / 1e3)
    out = {"impl": "reference", "metric": "scanned_bp_per_sec", "value": value, "unit": "bp/s", "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
           "vs_baseline": None, "dtype": "f16", "data": "synthetic", "config": scan_config(args),
           "cpu_baseline": {"value": value, "unit": "bp/s", "cores": threads, "kind": "port", "threads_used": threads, "host_cores": cores,
                            "sample_seqs": int(n),
                            "sample": f"{n} of {args.nseq} sequences x {args.seqlen} bp, all {args.motifs} PWMs, both strands, per step"},
           "e2e": {"value": value, "unit": "bp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}
    if args.workload in ("all", "both", "train"):
        a = synth.planted_gapped(2000, args.train_seqlen, 2)
        cdl = mdl.ucdl(mdl.Hyperparam(), np.random.default_rng(2))
        rate, steps, tcores, dt = cpu_train_rate(a, cdl.flat, min(args.cpu_seconds, 20.0))
        out["training"] = {"impl": "reference", "metric": "training_sequences_per_sec", "value": rate, "unit": "seq/s",
                           "config": train_config(args.train_nseq, args.train_seqlen, 1, args.train_steps, 1), "higher_is_better": True,
                           "cpu_baseline": {"value": rate, "unit": "seq/s", "cores": tcores, "kind": "port", "threads_used": tcores,
                                            "sample": f"{steps} optimiser steps of batch 6 in {dt:.1f} s (oracle/csc_oracle.py)"},
                           "e2e": {"value": rate, "unit": "seq/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


def main():
    args = parse()
    if args.impl == "reference":
        return run_reference(args)
    import torch
    import torch.distributed as dist
    import motifs_jl_b200 as mb
    from motifs_jl_b200 import parallel

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)                    # plumbing: barriers, the max-over-ranks of the timings, the id bootstrap
    ctx = mb.Context(local)
    if world > 1:
        parallel.init_comm(ctx)                                           # the library's own communicator carries every data-path collective
    stream = torch.cuda.current_stream()
    wl = args.workload
    out = None
    if wl in ("all", "both", "scan"):
        out = bench_scan(args, ctx, torch, dist, world, rank, local, dev, stream)
    nested = {}
    if wl in ("all", "both", "train"):
        nested["training"] = bench_train(args, ctx, torch, dist, world, rank, local, dev, "training", args.train_nseq, args.train_seqlen,
                                         args.train_steps, 1)
    if wl in ("all", "config3"):
        nested["config3_training"] = bench_train(args, ctx, torch, dist, world, rank, local, dev, "config3_training", args.c3_nseq, args.c3_seqlen,
                                                 args.c3_steps, 2, groups=args.c3_groups, e2e_leg=False, extras=False)
    if wl == "all" and args.c3_groups == 1:
        # the same data-parallel run with 64 reference batches per rank and optimiser step (global batch 384 x ranks): what the ranks are
        # worth once a step carries enough work to fill a GPU (the many-group launch path of the library; DESIGN.md section 3.2)
        nested["config3_training_64groups"] = bench_train(args, ctx, torch, dist, world, rank, local, dev, "config3_training_64groups",
                                                          args.c3_nseq, args.c3_seqlen, 10, 2, groups=64, e2e_leg=False, extras=False, warm_mult=3)
    if wl in ("all", "config5") and rank == 0:
        nested["config5_long_scan"] = bench_long_scan(args, ctx, torch, dev, stream)
    if world > 1:
        dist.barrier()
    if rank == 0:
        if out is None:
            key = next(iter(nested))
            out = nested.pop(key)
            out["warmup"] = args.warmup
        for k, v in nested.items():
            out[k] = v
            out["gpu_launches"] = int(out.get("gpu_launches") or 0) + int((v or {}).get("gpu_launches") or 0)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs)
        print(json.dumps(out), flush=True)
    ctx.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
