#!/bin/bash
# One single-GPU session: full GPU suite, bench, ncu launch list of a step, ncu --set full of the layer-1 GEMM and
# the gather.  Outputs under gpurun_out/<tag>_*.
#   usage: bash scripts/gpu_session.sh <tag> [skip-ncu]
cd "$(dirname "$0")/.." || exit 1
tag=${1:-r2}
mkdir -p gpurun_out
O=gpurun_out
t0=$(date +%s)
el() { echo "[t+$(( $(date +%s) - t0 ))s] $*"; }

el "1. GPU test-suite"
timeout 900 python -m pytest tests -m gpu -q --maxfail=25 --tb=short -p no:cacheprovider > $O/${tag}_tests.log 2>&1
tail -5 $O/${tag}_tests.log

el "2. bench"
timeout 400 python bench.py --steps 200 --warmup 20 > $O/${tag}_bench.json 2> $O/${tag}_bench.err
python - <<PY
import json
try:
    d = json.load(open("$O/${tag}_bench.json"))
    print("value %.1f spread %.3f e2e %.1f launches %d  L1 %s  gather frac %.3f  td3 %.1f" % (
        d["value"], d["spread"]["rel"], d["e2e"]["value"], d["gpu_launches"],
        {k: round(v["ms"] * 1e3, 2) for k, v in d["roofline"]["per_tile"].items()}, d["roofline_gather"]["frac"],
        d.get("td3", {}).get("steps_per_sec", 0)))
    print("roofline frac %.3f (single-launch method %.2f us)" % (d["roofline"]["frac"], d["roofline"]["ms_single_launch_between_events"] * 1e3))
except Exception as e:
    print("bench failed:", e); print(open("$O/${tag}_bench.err").read()[-2000:])
PY

el "3. REINFORCE policy gradient against the vocabulary size"
timeout 900 python scripts/bench_reinforce_vocab.py > $O/${tag}_reinforce_vocab.jsonl 2> $O/${tag}_reinforce_vocab.err

if [ "$2" != "skip-ncu" ]; then
el "4. ncu: launch list of the step"
timeout 300 ncu --metrics gpu__time_duration.sum --clock-control none -c 900 --csv --log-file $O/${tag}_launches.csv \
  python bench.py --steps 3 --warmup 3 --repeats 1 --no-cpu-baseline --no-other-algo > $O/${tag}_ncu_bench.log 2>&1
el "5. ncu --set full: layer-1 GEMM, gather"
timeout 300 ncu --set full --clock-control none --import-source on -k regex:tc_gemm -c 2 -f -o $O/${tag}_tc_gemm \
  python scripts/prof_tc.py 64 > $O/${tag}_ncu_tc.log 2>&1
timeout 120 ncu -i $O/${tag}_tc_gemm.ncu-rep --page raw --csv > $O/${tag}_tc_gemm_raw.csv 2>/dev/null
timeout 300 ncu --set full --clock-control none -k regex:frame_gather -c 2 -f -o $O/${tag}_gather \
  python scripts/prof_gather.py > $O/${tag}_ncu_gather.log 2>&1
timeout 120 ncu -i $O/${tag}_gather.ncu-rep --page raw --csv > $O/${tag}_gather_raw.csv 2>/dev/null
timeout 300 ncu --set full --clock-control none -k regex:frame_gather -c 2 -f -o $O/${tag}_gather_big \
  python scripts/prof_gather.py 65536 > $O/${tag}_ncu_gather_big.log 2>&1
timeout 120 ncu -i $O/${tag}_gather_big.ncu-rep --page raw --csv > $O/${tag}_gather_big_raw.csv 2>/dev/null
fi
el "done"
