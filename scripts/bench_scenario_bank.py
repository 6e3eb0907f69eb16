#!/usr/bin/env python
"""Cost and use of scenario banks (include/fwgym.h fw_bank_t) on the GPU, two measurements in one process:

    step      the benchmark workload (bench.py: 65 536 envs, fixed_wing_config.json, moderate Dryden gusts,
              observation noise std 0.1, fp64 dopri5) on a handle without a bank (env kernel default_turb) and on a
              handle with a bank of 4 N scenarios (default_turb_bank: a banked reset reads ~27 doubles of its scenario
              instead of ~15 Philox draws).  The bank holds the initial states and targets a sampled reset of a 4 N-env
              handle drew, so banked and sampled episodes start from the same distribution.  us per step, arms
              interleaved round by round, a buffer larger than L2 written between steps (as bench.py)
    evaluate  the PID evaluation (examples configuration, turbulence off) of test_set_wind_none tiled to 262 144
              scenarios: one banked evaluate_on_set on 65 536 envs against four 65 536-env evaluate_on_set calls (the
              way to fly that many scenarios without a bank: a handle per call), both keeping the reward traces; the
              two arms alternate `--eval-repeats` times; wall time (host clock around work that ends in a device
              synchronise) and scenarios/s, median over the repeats

    python scripts/bench_scenario_bank.py --out profiles/scenario_bank_b200.json

The card's name and power limit are read in the same process.
"""
import argparse
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "scripts"))


INIT_STATE = ("roll", "pitch", "yaw", "omega_p", "omega_q", "omega_r", "position_n", "position_e", "position_d",
              "velocity_u", "velocity_v", "velocity_w", "elevon_left", "elevon_right", "throttle")


def bank_tables(vec_cls, n_scen, dev, config_kw, sim_kw, cfg):
    """A full bank (every initial state variable and target given: nothing is sampled at a banked reset) holding what
    a sampled reset of an n_scen-env handle without a bank draws: the same distribution as the sampler's."""
    v = vec_cls(cfg, n_scen, device=dev, config_kw=config_kw, sim_config_kw=sim_kw, seed=777)
    v.reset()
    st = {k: x.cpu().numpy() for k, x in v.get_named_state(INIT_STATE).items()}
    tg = v.get_targets().cpu().numpy()
    target = {name: tg[k] for k, name in enumerate(v.target_names)}
    v.close()
    return st, target


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
    for name, bank in (("no_bank", False), ("bank_4n", True)):
        v = FixedWingVecEnv(DEFAULT_ENV_CONFIG, n, device=dev, config_kw=CONFIG_KW, sim_config_kw=SIM_KW,
                            seed=20261017, scenario_bank=bank)
        if bank:
            st, tg = bank_tables(FixedWingVecEnv, 4 * n, dev, CONFIG_KW, SIM_KW, DEFAULT_ENV_CONFIG)
            v.set_scenario_bank(state=st, target=tg)
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
        arm = {"kernel_variant": v.kernel_variant(), "us_per_step": us,
               "us_per_step_rounds": [round(x, 2) for x in rounds[name]], "env_steps_per_s": n / (us * 1e-6),
               "resets_per_step": c["resets"] / (c["env_steps"] / n),
               "attempts_per_env_step": c["attempts"] / c["env_steps"], "watchdog": c["watchdog"]}
        if v.scenario_bank:
            arm["scenarios_left_at_end"] = int(4 * n - int(v.scenario_results()["episodes"].sum())
                                               - int((v.scenario_ids() >= 0).sum()))
        out["arms"][name] = arm
        v.close()
    return out


def bench_evaluate(a, torch):
    from fwgym_b200 import evaluate
    cfg = os.path.join(ROOT, "fixed-wing-gym_b200", "params", "fixed_wing_config_examples.json")
    base = evaluate.load_test_set(os.path.join(ROOT, "tests", "golden", "test_set_wind_none.npz"))
    n, total = a.envs, 4 * a.envs
    scen = [base[i % len(base)] for i in range(total)]
    # warm-up of both paths (module load, allocator) at a small size
    evaluate.evaluate_on_set(scen[:256], cfg, controller="pid", seed=1, num_envs=64)[1].close()
    evaluate.evaluate_on_set(scen[:64], cfg, controller="pid", seed=1)[1].close()

    def banked():
        res, v = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, num_envs=n)
        v.close()
        return res["lengths"]

    def four_calls():
        lens = []
        for j in range(4):
            r, v = evaluate.evaluate_on_set(scen[j * n:(j + 1) * n], cfg, controller="pid", seed=1, env_offset=j * n)
            lens.append(r["lengths"])
            v.close()
        return np.concatenate(lens)
    arms = {"banked_%d_envs" % n: banked, "four_calls_%d_envs" % n: four_calls}
    walls = {name: [] for name in arms}
    lengths = {}
    for _ in range(a.eval_repeats):
        for name, fn in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            lengths[name] = fn()
            torch.cuda.synchronize()
            walls[name].append(time.perf_counter() - t0)
    out = {"workload": "PID, examples configuration, turbulence off, test_set_wind_none tiled to %d scenarios, reward "
                       "traces kept, arms alternated %d times" % (total, a.eval_repeats)}
    for name in arms:
        w = float(np.median(walls[name]))
        out[name] = {"wall_s": w, "wall_s_repeats": [round(x, 3) for x in walls[name]], "scenarios_per_s": total / w,
                     "mean_length": float(np.mean(lengths[name]))}
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=65536)
    ap.add_argument("--burn-in", type=int, default=200)
    ap.add_argument("--steps", type=int, default=300, help="timed steps per round")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--eval-repeats", type=int, default=3)
    ap.add_argument("--out", help="write the JSON result here (also printed)")
    a = ap.parse_args()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("bench_scenario_bank.py measures the GPU: no CUDA device")
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
