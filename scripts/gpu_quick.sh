#!/bin/bash
# quick GPU round trip: parity tests (optionally -k filter via $2) + a short bench, its JSON line kept as $OUT/bench_$TAG.json
TAG=${1:-x}; KF=${2:-}; OUT=${OUT:-build/quick}
mkdir -p "$OUT"
if [ -n "$KF" ]; then timeout 900 python -m pytest tests -m gpu -x -q -k "$KF" 2>&1 | tail -15; else timeout 900 python -m pytest tests -m gpu -x -q 2>&1 | tail -15; fi
timeout 300 python bench.py --steps 30 --warmup 5 --no-cpu-baseline > "$OUT/bench_${TAG}.json" 2> "$OUT/bench_${TAG}.err" || tail -5 "$OUT/bench_${TAG}.err"
python - <<P
import json
d=json.load(open("$OUT/bench_${TAG}.json"))
r=d["roofline"]
print("value %.4g ms_step %.4f e2e %.4g dyn_ms %.4f env_ms %.4f frac %.4f k %.3f lane_eff %.3f wd %s" % (d["value"], d["ms_per_step"], d["e2e"]["value"], r["kernel_ms_per_launch"], d["env_kernel"]["ms_per_launch"], r["frac"], r["mean_attempts_per_env_step"], r["warp_divergence"]["lane_efficiency"], d["overlap"]["watchdog"]))
P
