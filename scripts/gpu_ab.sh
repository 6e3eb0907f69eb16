#!/bin/bash
# A/B library variants on the bench workload, interleaved twice: scripts/gpu_ab.sh base base@FWGYM_LONG_DIV=0 ...
# (names under build/variants, scripts/build_variant.sh; NAME@VAR=VALUE sets an environment variable for that arm)
for rep in $(seq 1 ${REPS:-2}); do
for arm in "$@"; do
  name=${arm%%@*}; setting=""; [[ "$arm" == *@* ]] && setting=${arm#*@}
  env $setting FWGYM_LIB=build/variants/libfwgym_$name.so timeout 300 python bench.py --steps 30 --warmup 5 --no-cpu-baseline > gpurun_out/bench_ab_$name.json 2> gpurun_out/bench_ab_$name.err || tail -3 gpurun_out/bench_ab_$name.err
  python - <<P
import json
d=json.load(open("gpurun_out/bench_ab_$name.json")); r=d["roofline"]; wd=r["warp_divergence"]
print("[$arm #$rep] value %.4g (%.1f us/step) e2e %.4g dyn_ms %.4f env_ms %.4f serial %.4f lane_eff %.3f passes %.0f lane_att %.0f watchdog %.0f" % (d["value"], d["ms_per_step"]*1e3, d["e2e"]["value"], r["kernel_ms_per_launch"], d["env_kernel"]["ms_per_launch"], d["overlap"]["serial_ms_per_step"], wd["lane_efficiency"], wd["warp_passes"], wd["lane_attempts"], d["overlap"]["watchdog"]))
P
done
done
