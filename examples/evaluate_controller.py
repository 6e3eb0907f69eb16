#!/usr/bin/env python
"""The reference's examples/evaluate_controller.py on the GPU: every scenario of a test set flown at once, one env each
(fwgym_b200.evaluate, SURVEY §8f row 2).

    python examples/evaluate_controller.py tests/golden/test_set_wind_none.npz --PID
    python examples/evaluate_controller.py tests/golden/test_set_wind_none.npz --model-path tests/golden/mlp_controller.npz
    python examples/evaluate_controller.py path/to/test_set.npy --PID --turbulence-intensity moderate
    python examples/evaluate_controller.py tests/golden/test_set_wind_none.npz --PID --turbulence-intensity none light moderate severe

`path_to_file`: the reference's pickled test set (.npy, list of {"state", "target"}) or the plain-array fixture
(.npz).  `--model-path`: an .npz with the arrays of a stable-baselines PPO2 MlpPolicy and its VecNormalize statistics
(oracle/make_golden_policy.py writes one from examples/models/mlp_controller).  Prints the reference's result table
(nan-mean per metric and state, evaluate_controller.py:32-41; one table per level when several turbulence levels are
given: they fly as one batch, each scenario once per level) and optionally saves the result dictionary in the
reference's layout (res[metric][state] = [value per scenario], res["rewards"])."""
import argparse
import os
import sys

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("path_to_file", help="test set (.npy as the reference ships them, or the .npz fixture)")
    ap.add_argument("--PID", dest="use_pid", action="store_true", help="use the PID controller")
    ap.add_argument("--model-path", help=".npz with the MlpPolicy arrays (tests/golden/mlp_controller.npz)")
    ap.add_argument("--env-config-path", help="env configuration JSON (default: the examples configuration)")
    ap.add_argument("--turbulence-intensity", nargs="+", default=["none"], choices=["none", "light", "moderate", "severe"],
                    help="one or more levels; several levels run as one batch (a result table per level)")
    ap.add_argument("--save", help="write the result dictionary to this .npy")
    a = ap.parse_args()
    if not a.use_pid and not a.model_path:
        ap.error("give --PID or --model-path")
    import __graft_entry__ as ge
    ge.build()
    from fwgym_b200 import evaluate
    from fwgym_b200.config import DEFAULT_ENV_CONFIG
    cfg = a.env_config_path or os.path.join(os.path.dirname(DEFAULT_ENV_CONFIG), "fixed_wing_config_examples.json")
    scenarios = evaluate.load_test_set(a.path_to_file)
    controller = "pid" if a.use_pid else dict(np.load(a.model_path))
    levels = a.turbulence_intensity
    res, vec = evaluate.evaluate_on_set(scenarios, cfg, controller=controller,
                                        turbulence_intensity=levels[0] if len(levels) == 1 else levels)
    by_level = {levels[0]: res} if len(levels) == 1 else res
    saved = {}
    for lv, r in by_level.items():
        print("turbulence %s: %d scenarios, mean episode length %.1f steps" % (lv, len(scenarios),
                                                                           float(np.mean(r["lengths"]))))
        for key, val in sorted(evaluate.summarise(r).items()):
            print("\t%-28s %.4f" % (key, val))
        out = {m: r[m] for m in evaluate.DEFAULT_METRICS}
        out["rewards"] = [np.asarray(x) for x in r["rewards"]]
        saved[lv] = out
    if a.save:
        np.save(a.save, saved[levels[0]] if len(levels) == 1 else saved, allow_pickle=True)
    vec.close()
