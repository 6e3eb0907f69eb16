#!/usr/bin/env python
"""Cost and use of per-env aircraft (include/fwgym.h fw_set_aircraft) on the GPU, two measurements in one process:

    step      the benchmark workload (bench.py: 65 536 envs, fixed_wing_config.json, moderate Dryden gusts,
              observation noise std 0.1, fp64 dopri5) on four handles: the shipped one (no aircraft parameters),
              aircraft_parameters=("mass", "C_prop") with every request NaN (the nominal aircraft on the FwSpecRand
              dynamics kernels), and mass, Jx, Jy, Jz, Jxz and C_prop pinned to a distinct +-20 % variant per env, twice:
              with every inertia tensor that is positive definite (Jx Jz - Jxz^2 > 0; the X8's is close to singular, so
              +-20 % reaches near-singular tensors) and with Jx Jz - Jxz^2 kept at half the nominal value or more.  us
              per step, dopri5 attempts per env step (variants change the physics, so the work) and the most attempts
              one env needed in the last timed step (a stiff airframe is the attempt kernel's tail), arms interleaved
              round by round, a buffer larger than L2 written between steps (as bench.py)
    evaluate  the PID evaluation (examples configuration, turbulence off) of the 100 scenarios of test_set_wind_none on
              16 aircraft variants: one evaluate_on_set(aircraft=...) call (1 600 envs) against 16 evaluate_on_set calls
              on handles built from per-variant parameter files (the way scripts/identify_constants.py flies candidate
              aircraft); wall time including handle creation (host clock around work that ends in a device synchronise),
              the arms alternated `--eval-repeats` times, median

    python scripts/bench_aircraft_variants.py --out profiles/aircraft_variants_b200.json

The card's name and power limit are read in the same process.  Parameter files go to a temporary directory.
"""
import argparse
import functools
import json
import os
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))

PINNED = ("mass", "Jx", "Jy", "Jz", "Jxz", "C_prop")


def variants(params, n, seed, min_det=0.0):
    """n airframes: every PINNED parameter at its nominal value times U(0.8, 1.2), redrawn until Jx Jz - Jxz^2 exceeds
    min_det times its nominal value (and 0)."""
    rs = np.random.RandomState(seed)
    det0 = params["Jx"] * params["Jz"] - params["Jxz"] ** 2
    out = {k: params[k] * rs.uniform(0.8, 1.2, n) for k in PINNED}
    bad = out["Jx"] * out["Jz"] - out["Jxz"] ** 2 <= max(min_det * det0, 0.0)
    while bad.any():
        for k in PINNED:
            out[k][bad] = params[k] * rs.uniform(0.8, 1.2, int(bad.sum()))
        bad = out["Jx"] * out["Jz"] - out["Jxz"] ** 2 <= max(min_det * det0, 0.0)
    return out


def bench_step(a, torch, dev):
    from bench import CONFIG_KW, SIM_KW
    from fwgym_b200 import FixedWingVecEnv
    from fwgym_b200.config import DEFAULT_ENV_CONFIG
    n = a.envs
    gen = torch.Generator(device=dev)
    gen.manual_seed(1)
    acts = torch.rand((16, n, 3), generator=gen, device=dev, dtype=torch.float32) * 2 - 1
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)     # > 126 MB L2
    vecs = {}
    for name, names, min_det in (("shipped", (), None), ("mass_cprop_nan", ("mass", "C_prop"), None),
                                 ("pinned_variants", PINNED, 0.0), ("pinned_variants_det_half", PINNED, 0.5)):
        v = FixedWingVecEnv(DEFAULT_ENV_CONFIG, n, device=dev, config_kw=CONFIG_KW, sim_config_kw=SIM_KW,
                            seed=20261017, aircraft_parameters=names)
        if min_det is not None:
            v.set_aircraft(variants(v.cc.params, n, 5, min_det))
        v.reset()
        for i in range(a.burn_in):
            v.step_tensors(acts[i % 16])
        torch.cuda.synchronize(dev)
        v.reset_counters()
        vecs[name] = v
    rounds = {name: [] for name in vecs}
    for r in range(a.rounds):
        for name, v in vecs.items():
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(a.steps)]
            for k in range(a.steps):
                flush.zero_()
                ev[k][0].record()
                v.step_tensors(acts[(r * a.steps + k) % 16])
                ev[k][1].record()
            torch.cuda.synchronize(dev)
            rounds[name].append(sum(e0.elapsed_time(e1) for e0, e1 in ev) * 1e3 / a.steps)
    out = {"workload": "%d envs, bench.py configuration, %d burn-in steps, %d rounds x %d timed steps per arm, arms "
                       "interleaved by round" % (n, a.burn_in, a.rounds, a.steps), "arms": {}}
    for name, v in vecs.items():
        c = v.counters()
        us = float(np.median(rounds[name]))
        out["arms"][name] = {"kernel_variant": v.kernel_variant(), "us_per_step": us,
                             "us_per_step_rounds": [round(x, 2) for x in rounds[name]],
                             "env_steps_per_s": n / (us * 1e-6), "resets_per_step": c["resets"] / (c["env_steps"] / n),
                             "attempts_per_env_step": c["attempts"] / c["env_steps"],
                             "max_env_attempts_last_step": int(v.last_attempts().max()), "watchdog": c["watchdog"]}
        v.close()
    return out


def bench_evaluate(a, torch):
    from fwgym_b200 import evaluate
    from fwgym_b200.vec_env import FixedWingVecEnv
    cfg = os.path.join(ROOT, "fixed-wing-gym_b200", "params", "fixed_wing_config_examples.json")
    scen = evaluate.load_test_set(os.path.join(ROOT, "tests", "golden", "test_set_wind_none.npz"))
    params = json.load(open(os.path.join(ROOT, "fixed-wing-gym_b200", "params", "x8_param.json")))
    var = variants(params, a.variants, 9)
    air = [{k: float(var[k][j]) for k in PINNED} for j in range(a.variants)]
    tmp = tempfile.mkdtemp(prefix="fwgym_aircraft_")
    files = []
    for j, v in enumerate(air):
        P = dict(params)
        P.update(v)
        files.append(os.path.join(tmp, "variant%d.json" % j))
        json.dump(P, open(files[-1], "w"))
    # warm-up of both paths (module load, allocator) at a small size
    evaluate.evaluate_on_set(scen[:8], cfg, controller="pid", seed=1, aircraft=air[:2])[1].close()
    evaluate.evaluate_on_set(scen[:8], cfg, controller="pid", seed=1)[1].close()

    def one_call():
        res, v = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, aircraft=air)
        v.close()
        return np.concatenate([res[j]["lengths"] for j in range(len(air))])

    def per_file_calls():
        lens = []
        orig = evaluate.FixedWingVecEnv
        try:
            for path in files:
                evaluate.FixedWingVecEnv = functools.partial(FixedWingVecEnv, sim_parameter_path=path)
                r, v = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1)
                lens.append(r["lengths"])
                v.close()
        finally:
            evaluate.FixedWingVecEnv = orig
        return np.concatenate(lens)
    arms = {"one_call_%d_variants" % len(air): one_call, "%d_per_file_calls" % len(air): per_file_calls}
    walls = {name: [] for name in arms}
    lengths = {}
    for _ in range(a.eval_repeats):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            lengths[name] = fn()
            torch.cuda.synchronize()
            walls[name].append(time.perf_counter() - t0)
    a_, b_ = lengths.values()
    out = {"workload": "PID, examples configuration, turbulence off, the %d scenarios of test_set_wind_none on %d "
                       "aircraft variants (mass, Jx, Jy, Jz, Jxz, C_prop at +-20 %%), reward traces kept, handle "
                       "creation included, arms alternated %d times" % (len(scen), len(air), a.eval_repeats),
           "episode_lengths_equal": bool(np.array_equal(a_, b_))}
    for name in arms:
        w = float(np.median(walls[name]))
        out[name] = {"wall_s": w, "wall_s_repeats": [round(x, 3) for x in walls[name]],
                     "scenarios_per_s": len(scen) * len(air) / w, "mean_length": float(np.mean(lengths[name]))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--burn-in", type=int, default=200)
    ap.add_argument("--steps", type=int, default=300, help="timed steps per round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--variants", type=int, default=16)
    ap.add_argument("--eval-repeats", type=int, default=3)
    ap.add_argument("--out", help="write the JSON result here (also printed)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_aircraft_variants.py measures the GPU: no CUDA device")
    import __graft_entry__ as ge
    ge.build()
    from bench_turbulence_mix import card
    result = {"card": card(), "step": bench_step(a, torch, torch.device("cuda", 0)), "evaluate": bench_evaluate(a, torch)}
    line = json.dumps(result, indent=1)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
