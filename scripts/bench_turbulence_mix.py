#!/usr/bin/env python
"""Cost of per-env Dryden intensities on the benchmark workload (bench.py: 65 536 envs, fixed_wing_config.json,
observation noise std 0.1, fp64 dopri5), three arms on the same GPU in one process:

    uniform   one handle at moderate turbulence (bench.py's own configuration)
    lms       a mixed handle, every reset draws light / moderate / severe with probability 1/3 each
    all4      a mixed handle, every reset draws none / light / moderate / severe with probability 1/4 each

    python scripts/bench_turbulence_mix.py --out profiles/turbulence_mix_b200.json

Each arm: reset, a 200-step untimed burn-in (every env in its first episode, a stationary episode mix), then
`--rounds` rounds of `--steps` timed steps, the arms taking turns round by round so that drift of the shared machine
hits all of them alike.  A step is timed with CUDA events, with a write of a buffer larger than L2 between steps (as
bench.py).  Reported per arm: env-steps/s and us per step (median round), dopri5 attempts per env step and warp passes
per step from fw_counters, and us per attempt (step time / mean attempts per env step), which separates what the
physics asks for (severe gusts, `none` envs) from what the kernels cost per unit of work.  The card's name and power
limit are read in the same process.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

ARMS = {
    "uniform_moderate": {"turbulence": True, "turbulence_intensity": "moderate"},
    "mixed_light_moderate_severe": {"turbulence": True,
                                    "turbulence_intensity": {"values": ["light", "moderate", "severe"]}},
    "mixed_all_four": {"turbulence": True,
                       "turbulence_intensity": {"values": ["none", "light", "moderate", "severe"]}},
}


def card():
    """Name, power limit and max SM clock of GPU 0 (nvidia-smi read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                              "-i", "0"], capture_output=True, text=True, timeout=30).stdout.strip()
        name, power, clock = [x.strip() for x in out.split(",")]
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except Exception as e:   # the numbers below are still valid; the card line says why it is missing
        import torch
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unavailable (%s)" % e}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--burn-in", type=int, default=200)
    ap.add_argument("--steps", type=int, default=300, help="timed steps per round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--out", help="write the JSON result here (also printed)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_turbulence_mix.py measures the GPU: no CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from bench import CONFIG_KW
    from fwgym_b200 import FixedWingVecEnv
    from fwgym_b200.config import DEFAULT_ENV_CONFIG
    dev = torch.device("cuda", 0)
    n = a.envs
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    acts = torch.rand((16, n, 3), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2
    vecs = {}
    for name, sim_kw in ARMS.items():
        v = FixedWingVecEnv(DEFAULT_ENV_CONFIG, n, device=dev, config_kw=CONFIG_KW, sim_config_kw=sim_kw, seed=20261017)
        v.reset()
        for i in range(a.burn_in):
            v.step_tensors(acts[i % 16])
        torch.cuda.synchronize(dev)
        v.reset_counters()
        vecs[name] = v
    rounds = {name: [] for name in ARMS}
    for r in range(a.rounds):
        for name, v in vecs.items():
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
            for k in range(a.steps):
                flush.zero_()
                ev[k][0].record()
                v.step_tensors(acts[(r * a.steps + k) % 16])
                ev[k][1].record()
            torch.cuda.synchronize(dev)
            rounds[name].append(sum(e0.elapsed_time(e1) for e0, e1 in ev) * 1e3 / a.steps)   # us per step
    result = {"workload": "%d envs, fixed_wing_config.json + observation noise std 0.1 (bench.py), fp64 dopri5, "
                          "%d burn-in steps, %d rounds x %d timed steps per arm, arms interleaved by round"
                          % (n, a.burn_in, a.rounds, a.steps),
              "card": card(), "arms": {}}
    for name, v in vecs.items():
        c = v.counters()
        us = float(np.median(rounds[name]))
        att = c["attempts"] / c["env_steps"]
        result["arms"][name] = {
            "sim_config_kw": ARMS[name],
            "kernel_variant": v.kernel_variant(),
            "us_per_step": us,
            "us_per_step_rounds": [round(x, 2) for x in rounds[name]],
            "env_steps_per_s": n / (us * 1e-6),
            "attempts_per_env_step": att,
            "warp_passes_per_step": c["warp_max_attempts"] / (c["env_steps"] / n),
            "lane_efficiency": c["warp_steps"] / (32.0 * c["warp_max_attempts"]),
            "us_per_attempt": us / att,
            "resets_per_step": c["resets"] / (c["env_steps"] / n),
            "watchdog": c["watchdog"],
        }
        v.close()
    line = json.dumps(result, indent=1)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
