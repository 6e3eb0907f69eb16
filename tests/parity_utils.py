"""Shared driver for the CUDA-vs-oracle parity tests: N oracle envs (one per global env id) stepped next to the
batched CUDA env on identical actions and identical Philox streams."""
import numpy as np

from oracle import harness

STATE_ROWS = ["q0", "q1", "q2", "q3", "omega_p", "omega_q", "omega_r", "position_n", "position_e", "position_d",
              "velocity_u", "velocity_v", "velocity_w", "elevon_left", "elevon_right", "throttle", "elevon_left_dot",
              "elevon_right_dot", "throttle_dot", "roll", "pitch", "yaw", "Va", "alpha", "beta", "elevator", "aileron"]


def rel_err(a, b, floor=1e-6):
    """|a - b| / (|b| + floor): `rel_err <= tol` is numpy's allclose(a, b, rtol=tol, atol=tol * floor).  With the
    floor of 1e-3 the tests use, the 1e-9 bar reads |a - b| <= 1e-9 |b| + 1e-12 (values near zero - a trimmed aileron
    is the difference of two 0.3 rad elevon deflections - are held to 1e-12 absolute)."""
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    return np.abs(a - b) / (np.abs(b) + floor)


def make_oracles(n, config, config_kw, sim_config_kw, seed, env_offset=0, kind="restated"):
    return [harness.OracleRunner(harness.make_env(kind, config, config_kw, sim_config_kw), seed, env_offset + i)
            for i in range(n)]


def gpu_state(vec):
    rows = vec.state_rows()
    st = vec.get_state().cpu().numpy()
    return np.stack([st[rows.index(r)] for r in STATE_ROWS], axis=1)   # [N, 27]


def run_parity(vec, oracles, actions, check_state=True):
    """Step both for len(actions) steps.  Returns dict of per-step max errors and integer mismatches."""
    import torch
    n = len(oracles)
    vec.enable_f64_outputs(True)
    obs_g = vec.reset()
    obs_o = np.stack([np.asarray(o.reset(), dtype=np.float64).ravel() for o in oracles])
    out = {"obs": [rel_err(vec._obs64.cpu().numpy(), obs_o, 1e-3).max()], "rew": [], "state": [], "done_mismatch": 0,
           "k_mismatch": 0, "term_mismatch": 0, "dones": 0, "k_sum": 0}
    for a in actions:
        at = torch.as_tensor(a, dtype=torch.float64, device=vec.device)
        _, _, done_g, term_g = vec.step_tensors(at)
        res = [o.step(a[i]) for i, o in enumerate(oracles)]
        obs_o = np.stack([np.asarray(r[0], dtype=np.float64).ravel() for r in res])
        rew_o = np.array([r[1] for r in res], dtype=np.float64)
        done_o = np.array([r[2] for r in res])
        k_o = np.array([o.attempts_last() for o in oracles])
        k_g = vec.last_attempts().cpu().numpy()
        done_gh = done_g.cpu().numpy().astype(bool)
        out["obs"].append(rel_err(vec._obs64.cpu().numpy(), obs_o, 1e-3).max())
        out["rew"].append(rel_err(vec._rew64.cpu().numpy(), rew_o, 1e-3).max())
        out["done_mismatch"] += int((done_gh != done_o).sum())
        out["k_mismatch"] += int((k_g != k_o).sum())   # every env, incl. those whose episode ended in this step
        out["k_sum"] += int(k_o.sum())
        out["dones"] += int(done_o.sum())
        if check_state:
            so = np.stack([o.ode_state() for o in oracles])
            out["state"].append(rel_err(gpu_state(vec), so, 1e-3).max())
    return out


# ---- oracle rollouts over all host cores (BASELINE configs[1] at its stated size: 4096 envs x 100 steps) -------------
def oracle_rollout_slice(args):
    """Worker (own process): free-running rollout of the oracle envs with global ids `env_ids` on `actions`
    [T, len(env_ids), 3].  -> dict of per-step arrays: obs [T + 1, n, D], rew / done / k / term [T, n], state [T, n, 27]."""
    config, config_kw, sim_kw, seed, env_ids, actions = args
    orcs = [harness.OracleRunner(harness.make_env("restated", config, config_kw, sim_kw), seed, int(gid))
            for gid in env_ids]
    T = actions.shape[0]
    obs = [np.stack([np.asarray(o.reset(), dtype=np.float64).ravel() for o in orcs])]
    rew, done, k, state, term = [], [], [], [], []
    for t in range(T):
        res = [o.step(actions[t, i]) for i, o in enumerate(orcs)]
        obs.append(np.stack([np.asarray(r[0], dtype=np.float64).ravel() for r in res]))
        rew.append([float(r[1]) for r in res])
        done.append([bool(r[2]) for r in res])
        term.append([str(r[3].get("termination", "")) if r[2] else "" for r in res])
        k.append([o.attempts_last() for o in orcs])
        state.append(np.stack([o.ode_state() for o in orcs]))
    return dict(obs=np.array(obs), rew=np.array(rew), done=np.array(done), k=np.array(k), state=np.array(state),
                term=np.array(term))


def oracle_rollout_ids(config, config_kw, sim_kw, seed, env_ids, actions, procs=None):
    """Free-running oracle rollout of the envs with global ids `env_ids` (any order, need not be contiguous: the Philox
    streams are keyed by the global id) on `actions` [T, len(env_ids), 3].  The envs are split over `procs` spawned
    worker processes (spawn, not fork: the caller holds a CUDA context); the per-step arrays come back in the order of
    `env_ids` along the env axis."""
    import multiprocessing as mp
    import os
    env_ids = np.asarray(env_ids, dtype=np.int64)
    n = len(env_ids)
    procs = min(procs or os.cpu_count() or 1, n)
    bounds = np.linspace(0, n, procs + 1).astype(int)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    old = os.environ.get("PYTHONPATH", "")
    os.environ["PYTHONPATH"] = os.pathsep.join([root, os.path.join(root, "tests")] + ([old] if old else []))
    try:
        ctx = mp.get_context("spawn")
        with ctx.Pool(procs) as pool:
            parts = pool.map(oracle_rollout_slice,
                             [(config, config_kw, sim_kw, seed, env_ids[lo:hi], actions[:, lo:hi])
                              for lo, hi in zip(bounds[:-1], bounds[1:]) if hi > lo], chunksize=1)
    finally:
        os.environ["PYTHONPATH"] = old
    return {key: np.concatenate([p[key] for p in parts], axis=1) for key in parts[0]}


def oracle_rollout_parallel(config, config_kw, sim_kw, seed, actions, procs=None):
    """oracle_rollout_ids over the contiguous envs 0 .. N - 1 of `actions` [T, N, 3]."""
    return oracle_rollout_ids(config, config_kw, sim_kw, seed, np.arange(actions.shape[1]), actions, procs)
