# The int8 pre-filter of k_scan_tc against the previous (FP16) build, on ONE box (box-to-box variation is ~15 %), alternating
# old / new / old / new.  Set-up, from the repo root:
#   mkdir -p build_prev/tree && git archive <old commit> | tar -x -C build_prev/tree     (its Python binds the old ABI)
#   make -C build_prev/tree -j8 && cp oracle/liboracle.so build_prev/tree/oracle/
#   make -j8 TCS_PROFILE=1 BUILD=build_prof LIB=build_prof/libmotifs_b200_prof.so build_prof/libmotifs_b200_prof.so
# (build_prev/ and build_prof/ are git-ignored).  Prints the card, the GPU tests, the bench lines of both builds, the candidates and
# hits per scan, the issued int8 MAC rate against the dense INT8 rate, and one TCS_PROFILE=1 role-clock capture of the new kernel.
# Usage: bash profiles/scripts/scan_int8_ab.sh <output directory, relative to the repo root>
set -u
OUT=${1:?usage: scan_int8_ab.sh <output directory>}
mkdir -p $OUT
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm,clocks.sm --format=csv | tee $OUT/card.txt
export MB200_SCAN_TC_STATS=1
timeout 900 python -m pytest tests/test_scan_gpu.py tests/test_golden_gpu.py -x -q -m gpu > $OUT/scan_tests.log 2>&1
echo "scan tests rc $?"; tail -1 $OUT/scan_tests.log
grep -q " passed" $OUT/scan_tests.log && ! grep -q "failed\|error" $OUT/scan_tests.log || exit 1
ROOT=$PWD
for r in 1 2; do
  for side in old new; do
    if [ $side = old ]; then dir=build_prev/tree; else dir=.; fi
    (cd $dir && timeout 900 python bench.py --workload scan --steps 3 --warmup 3 --no-cpu-baseline --dump-outputs $ROOT/$OUT/dump_${side}_$r \
       > $ROOT/$OUT/scan_${side}_$r.json 2> $ROOT/$OUT/scan_${side}_$r.err)
    echo "scan $side $r rc $?"
  done
done
for side in old new; do
  if [ $side = old ]; then dir=build_prev/tree; else dir=.; fi
  (cd $dir && timeout 900 python bench.py --workload config5 --steps 3 --warmup 3 --no-cpu-baseline --dump-outputs $ROOT/$OUT/dump_c5_${side} \
     > $ROOT/$OUT/c5_${side}.json 2> $ROOT/$OUT/c5_${side}.err)
  echo "config5 $side rc $?"
done
OUT=$OUT python - <<'PY'
import json, os, re, glob, numpy as np
OUT = os.environ["OUT"]
def line(p):
    return json.loads(open(p).read().strip().splitlines()[-1])
def stats(p):
    return [l.strip() for l in open(p) if "tensor-core scan" in l]
for side in ("old", "new"):
    vals, steps, launch, e2e = [], [], [], []
    for r in (1, 2):
        d = line(f"{OUT}/scan_{side}_{r}.json")
        vals.append(d["value"]); steps.append(d["ms_per_step"]); launch.append(d["roofline"].get("ms_per_launch"))
        e2e.append(d["e2e"]["value"])
        print(side, r, "value", round(d["value"] / 1e9, 4), "Gbp/s  ms_per_step", round(d["ms_per_step"], 2), "k_scan_tc ms/launch", launch[-1], "kernel", d["roofline"].get("kernel"),
              "e2e", round(d["e2e"]["value"] / 1e9, 4), "checks", {k: d["checks"].get(k) for k in ("counts_sha", "counts_sha_expected_from_n1", "counts_match_n1")})
    print(side, "median value", np.median(vals), "spread", (max(vals) - min(vals)) / np.median(vals), "median e2e", np.median(e2e))
    st = stats(f"{OUT}/scan_{side}_2.err")
    print(side, "last stats line:", st[-1] if st else None)
    c = line(f"{OUT}/c5_{side}.json"); c5 = c.get("config5_long_scan", c)
    print(side, "config5", {k: c5.get(k) for k in ("value", "ms_per_step", "unit")})
for name in ("scan_counts",):
    a = [np.load(p) for p in sorted(glob.glob(f"{OUT}/dump_*_[12]/{name}.npy"))]
    print(name, "identical across all four runs:", all(np.array_equal(a[0], x) for x in a), len(a))
for name in ("config5_long_scan_fg_counts", "config5_long_scan_bg_counts"):
    o, n = np.load(f"{OUT}/dump_c5_old/{name}.npy"), np.load(f"{OUT}/dump_c5_new/{name}.npy")
    print(name, "identical:", np.array_equal(o, n))
# issued int8 MACs over k_scan_tc time (the stats line of the last scan call of the new build) against dense INT8 (4500 TOPS = 2250 T MAC/s)
for l in stats(f"{OUT}/scan_new_2.err")[-1:]:
    m = re.search(r"scan ([0-9.]+) ms.*int8 MACs ([0-9.e+]+)", l)
    ms, macs = float(m.group(1)), float(m.group(2))
    print(f"issued int8 MAC rate {macs / ms / 1e9:.1f} T MAC/s = {macs / ms / 1e9 / 2250:.3f} of dense INT8 (data-sheet 2250 T MAC/s at 1000 W)")
PY
export MB200_LIBRARY=$ROOT/build_prof/libmotifs_b200_prof.so MB200_SCAN_TC_DEBUG=2
timeout 600 python bench.py --steps 1 --warmup 0 --no-cpu-baseline --workload scan --nseq 1000000 > $OUT/tc_dbg.json 2> $OUT/tc_dbg.err
echo "role clocks rc $?"; grep tcdbg $OUT/tc_dbg.err | head -148 | awk 'NR%12==1'; grep "tensor-core" $OUT/tc_dbg.err | tail -2
unset MB200_LIBRARY MB200_SCAN_TC_DEBUG MB200_SCAN_TC_STATS
timeout 1500 python -m pytest tests -m gpu -q > $OUT/gpu_tests.log 2>&1; echo "gpu tests rc $?"; tail -3 $OUT/gpu_tests.log
timeout 600 python -c "import __graft_entry__ as g; g.smoke()" > $OUT/smoke.log 2>&1; echo "smoke rc $?"; tail -4 $OUT/smoke.log
