"""Evaluation harness (SURVEY §8f row 2): the batched counterpart of examples/evaluate_controller.py:44-169.

The reference pops the scenarios of a test set one by one onto `num_envs` SubprocVecEnv workers, steps a controller
until each scenario's episode ends and collects, per scenario, the reward trace and the episode metrics.  Scenarios
are independent, so here ALL scenarios run at once, one env each: reset(state=, target=) injects them
(fixed_wing.py:287-315), the controller runs on the device (`DevicePID`: fw_pid_step, or any callable mapping the
env to an action tensor), and every env is followed until its first episode end.  Results use the reference's layout:
res[metric][state] = [value per scenario], res["rewards"] = [trace per scenario].
"""
import ctypes

import numpy as np
import torch

from . import _capi
from .vec_env import FixedWingVecEnv

# evaluate_controller.py:68-76: the overrides every evaluation applies to the env config
EVAL_CONFIG_KW = {"steps_max": 1500, "target": {"on_success": "done", "success_streak_fraction": 1,
                                                "success_streak_req": 100,
                                                "states": {0: {"bound": 5}, 1: {"bound": 5}, 2: {"bound": 2}}}}
DEFAULT_METRICS = ("success", "control_variation", "rise_time", "overshoot", "settling_time")


class DevicePID:
    """pyfly/pid_controller.py PIDController for every env of a FixedWingVecEnv, on the device (fw_pid_step).
    Gains are the reference's defaults; the env must use physical actions (action.scale_space = False)."""

    def __init__(self, vec, **gains):
        self.vec = vec
        g = _capi.STRUCTS["fw_pid_gains_t"]()
        g.k_p_V, g.k_i_V = 0.5, 0.1
        g.k_p_phi, g.k_i_phi, g.k_d_phi = 1.0, 0.0, 0.5
        g.k_p_theta, g.k_i_theta, g.k_d_theta = -4.0, -0.75, -0.1
        g.delta_a_min, g.delta_a_max = float(np.radians(-30)), float(np.radians(30))
        g.delta_e_min, g.delta_e_max = float(np.radians(-30)), float(np.radians(35))
        g.delta_t_min, g.delta_t_max = 0.0, 1.0
        for k, v in gains.items():
            setattr(g, k, float(v))
        self.gains = g
        self.integ = torch.zeros((3, vec.num_envs), dtype=torch.float64, device=vec.device)
        self.actions = torch.zeros((vec.num_envs, 3), dtype=torch.float64, device=vec.device)

    def reset(self, mask=None):
        if mask is None:
            self.integ.zero_()
        else:
            self.integ[:, mask.bool()] = 0.0

    def __call__(self, reset_mask=None):
        """-> actions [N, 3] float64 device tensor for the env's CURRENT state and targets."""
        v = self.vec
        rm = None if reset_mask is None else reset_mask.to(torch.uint8).contiguous()
        _capi.check(v._lib.fw_pid_step(v._h, ctypes.byref(self.gains), v._ptr(self.integ), v._ptr(rm),
                                       v._ptr(self.actions), v._stream()))
        self._keep = rm
        return self.actions


class MlpController:
    """A trained stable-baselines PPO2 MlpPolicy as the reference evaluates it (evaluate_controller.py:92-99,153):
    `model.predict(obs, deterministic=True)` = the mean of the Gaussian head, clipped to the action space, on
    observations normalised by the saved VecNormalize statistics ((obs - mean) / sqrt(var + 1e-8), clip 10) — EXCEPT
    the first observation of every scenario, which the reference takes from `env_method("reset")` and therefore feeds
    to the policy raw (evaluate_controller.py:115).  The policy math runs in float64 on the device (a 12-64-64-3 MLP:
    torch matmuls; the controller is not the hot path) so that the CPU twin in the tests reproduces it to rounding.
    `params`: the arrays of tests/golden/mlp_controller.npz (oracle/make_golden_policy.py)."""

    def __init__(self, vec, params, clip_obs=10.0, eps=1e-8):
        from .ppo import ActorCritic, load_sb2_parameters
        self.vec = vec
        d = vec.device
        net = load_sb2_parameters(ActorCritic(int(np.asarray(params["pi_fc0_w"]).shape[0]), 3), params)
        self.pi = net.pi.to(device=d, dtype=torch.float64)
        self.mean = torch.as_tensor(np.asarray(params["obs_mean"], dtype=np.float64), device=d)
        self.std = torch.sqrt(torch.as_tensor(np.asarray(params["obs_var"], dtype=np.float64), device=d) + eps)
        self.ret_std = float(np.sqrt(float(params["ret_var"]) + eps))
        self.clip = clip_obs
        self.low = torch.as_tensor(np.asarray(vec.action_space.low, dtype=np.float64), device=d)
        self.high = torch.as_tensor(np.asarray(vec.action_space.high, dtype=np.float64), device=d)

    @torch.no_grad()
    def __call__(self, obs, raw_mask=None):
        """obs: [N, obs_dim] device tensor (any float type); raw_mask: bool [N], envs whose observation comes straight
        from reset (fed unnormalised).  -> actions [N, 3] float64."""
        o = obs.reshape(obs.shape[0], -1).to(torch.float64)
        on = torch.clamp((o - self.mean) / self.std, -self.clip, self.clip)
        if raw_mask is not None:
            on = torch.where(raw_mask.reshape(-1, 1), o, on)
        return torch.minimum(torch.maximum(self.pi(on), self.low), self.high)


def load_test_set(path):
    """The reference's test sets are pickled lists of {"state": {...}, "target": {...}} (evaluate_controller.py:62);
    the committed fixture stores the same content as plain arrays (tests/golden/test_set_wind_none.npz)."""
    if path.endswith(".npz"):
        ts = np.load(path)
        skeys, tkeys = [str(k) for k in ts["state_keys"]], [str(k) for k in ts["target_keys"]]
        return [{"state": {k: float(ts["state"][i, j]) for j, k in enumerate(skeys)},
                 "target": {k: float(ts["target"][i, j]) for j, k in enumerate(tkeys)}}
                for i in range(ts["state"].shape[0])]
    return list(np.load(path, allow_pickle=True))


def evaluate_on_set(scenarios, config_path, controller="pid", config_kw=None, metrics=DEFAULT_METRICS,
                    turbulence_intensity="none", device="cuda:0", seed=0, max_steps=None, env_offset=0, num_envs=None,
                    keep_rewards=True, aircraft=None):
    """Run every scenario once (in parallel) under `controller`: "pid", a dict of saved MlpPolicy arrays
    (MlpController), or a callable(vec) -> actions tensor.
    Returns (res, vec_env): res[metric][state] lists in scenario order, res["rewards"], res["lengths"].
    `turbulence_intensity`: one level ("none", "light", "moderate", "severe"), or a list of levels: then the S
    scenarios x L levels fly as ONE batch of L * S envs on a handle with per-env intensities (env j * S + i is scenario i
    at level j, pinned with set_turbulence_intensity) and the first element of the return value is {level: res}.
    `env_offset`: global id of the first env (the Philox streams are keyed by it).
    `num_envs` < scenarios x levels: fly them through a scenario bank on that many envs instead (the reference's pool
    of workers that take scenario after scenario, evaluate_controller.py:80-169): every env starts its next scenario
    when its episode ends, the controller is reset for it, and the results come back in scenario order in the same
    layout.  Envs are reused, so the reference's carry-overs across episodes apply (the goal-achieved latch of the
    success reward).  `keep_rewards=False` drops the per-step reward traces (S x steps_max doubles on the device).
    `aircraft`: a list of V variants, each a dict of model parameters (the names FixedWingVecEnv(aircraft_parameters=)
    takes; parameters a variant leaves out keep their nominal values): the S scenarios x V variants fly as ONE batch (env
    j * S + i is scenario i on variant j) and the first element of the return value is {j: res}.  Not together with a
    list of turbulence levels."""
    levels = None if isinstance(turbulence_intensity, str) else list(turbulence_intensity)
    variants = None if aircraft is None else [dict(v) for v in aircraft]
    if variants is not None and levels is not None:
        raise ValueError("evaluate_on_set flies either several turbulence levels or several aircraft, not both")
    if variants is not None and not variants:
        raise ValueError("aircraft: at least one variant")
    n_scen = len(scenarios)
    reps = len(levels) if levels is not None else (len(variants) if variants is not None else 1)
    n = n_scen * reps
    air_names, air = _aircraft_columns(variants, n_scen)
    if num_envs is not None and int(num_envs) < n:
        if max_steps is not None:
            raise ValueError("max_steps cuts episodes short; a banked evaluation flies every episode to its end")
        return _evaluate_banked(scenarios, config_path, controller, config_kw, metrics, levels, turbulence_intensity,
                                device, seed, env_offset, int(num_envs), keep_rewards, air_names, air)
    kw, sim_kw = _eval_kw(config_kw, controller, levels, turbulence_intensity)
    vec = FixedWingVecEnv(config_path, n, device=device, config_kw=kw, sim_config_kw=sim_kw, seed=seed, metrics=True,
                          auto_reset=True, env_offset=env_offset, aircraft_parameters=air_names)
    if levels is not None:
        vec.set_turbulence_intensity([lv for lv in levels for _ in range(n_scen)])
    if air is not None:
        vec.set_aircraft(air)
    state, target = _scenario_columns(scenarios, reps)
    vec.enable_f64_outputs(True)
    vec.reset(state=state, target=target)
    pid = DevicePID(vec) if controller == "pid" else None
    if isinstance(controller, dict):                     # a saved MlpPolicy: the arrays of mlp_controller.npz
        controller = MlpController(vec, controller)
    first = torch.ones(n, dtype=torch.bool, device=vec.device)
    steps_cap = max_steps or vec.cc.steps_max
    alive = torch.ones(n, dtype=torch.bool, device=vec.device)
    rew_trace = torch.full((steps_cap, n), float("nan"), dtype=torch.float64, device=vec.device)
    lengths = torch.zeros(n, dtype=torch.long, device=vec.device)
    ep_rows = torch.full((n, vec.ep_dim), float("nan"), dtype=torch.float64, device=vec.device)
    for t in range(steps_cap):
        if pid is not None:
            actions = pid()
        elif isinstance(controller, MlpController):
            actions = controller(vec._obs64, first if t == 0 else None)
        else:
            actions = controller(vec)
        _, _, done, _ = vec.step_tensors(actions)
        rew_trace[t] = torch.where(alive, vec._rew64, rew_trace[t])
        fin = alive & done.bool()
        if fin.any():
            ep_rows[fin] = vec.episode_metrics()[fin]
            lengths[fin] = t + 1
            alive = alive & ~fin
            if not alive.any():
                break
    lengths[alive] = min(t + 1, steps_cap)
    rows, tr, ln = ep_rows.cpu().numpy(), rew_trace.cpu().numpy(), lengths.cpu().numpy()
    return _split(vec, metrics, rows, tr, ln, n_scen, levels, variants), vec


def _split(vec, metrics, rows, tr, ln, n_scen, levels, variants):
    """res of one block of S envs, or {level: res} / {variant index: res} of consecutive blocks"""
    keys = levels if levels is not None else (range(len(variants)) if variants is not None else None)
    if keys is None:
        return _results(vec, metrics, rows, tr, ln)
    return {k: _results(vec, metrics, rows[j * n_scen:(j + 1) * n_scen],
                        None if tr is None else tr[:, j * n_scen:(j + 1) * n_scen], ln[j * n_scen:(j + 1) * n_scen])
            for j, k in enumerate(keys)}


def _aircraft_columns(variants, n_scen):
    """-> (aircraft_parameters, {name: value per env}) for V variants x S scenarios (env j * S + i flies variant j; a
    parameter a variant leaves out is NaN = nominal), or ((), None) without variants."""
    if variants is None:
        return (), None
    names = tuple(sorted({k for v in variants for k in v}))
    if not names:
        raise ValueError("aircraft: the variants set no parameter")
    cols = {k: np.repeat(np.array([float(v.get(k, np.nan)) for v in variants]), n_scen) for k in names}
    return names, cols


def _eval_kw(config_kw, controller, levels, turbulence_intensity):
    kw = dict(config_kw or {})
    for k, v in EVAL_CONFIG_KW.items():
        kw[k] = v
    if controller == "pid":
        kw["action"] = {"scale_space": False}          # evaluate_controller.py:78-79
    if levels is None:
        sim_kw = {"turbulence": turbulence_intensity != "none", "turbulence_intensity": turbulence_intensity}
    else:
        sim_kw = {"turbulence": True, "turbulence_intensity": {"values": levels}}
    return kw, sim_kw


def _scenario_columns(scenarios, reps):
    """reset(state=, target=) columns of the scenarios, repeated `reps` times (one block per turbulence level)."""
    state = {}
    for k in sorted(scenarios[0]["state"].keys()):
        v0 = scenarios[0]["state"][k]
        if isinstance(v0, (list, tuple, np.ndarray)):     # "wind": [n, e, d]
            state[k] = np.tile(np.array([s["state"][k] for s in scenarios], dtype=np.float64).T, (1, reps))
        else:
            state[k] = np.tile(np.array([s["state"][k] for s in scenarios], dtype=np.float64), reps)
    target = {k: np.tile(np.array([s["target"][k] for s in scenarios], dtype=np.float64), reps)
              for k in scenarios[0]["target"]}
    return state, target


def _evaluate_banked(scenarios, config_path, controller, config_kw, metrics, levels, turbulence_intensity, device, seed,
                     env_offset, num_envs, keep_rewards, air_names=(), air=None):
    """evaluate_on_set on `num_envs` envs: the S x L scenarios (scenario j * S + i = scenario i at level j, or on
    aircraft variant j) are a scenario bank that the auto-resets consume."""
    n_scen = len(scenarios)
    reps = len(levels) if levels is not None else (len(next(iter(air.values()))) // n_scen if air is not None else 1)
    total = n_scen * reps
    kw, sim_kw = _eval_kw(config_kw, controller, levels, turbulence_intensity)
    vec = FixedWingVecEnv(config_path, num_envs, device=device, config_kw=kw, sim_config_kw=sim_kw, seed=seed,
                          metrics=True, auto_reset=True, env_offset=env_offset, scenario_bank=True,
                          aircraft_parameters=air_names)
    state, target = _scenario_columns(scenarios, reps)
    res = vec.set_scenario_bank(state=state, target=target,
                                turbulence_intensity=None if levels is None else
                                [lv for lv in levels for _ in range(n_scen)], aircraft=air)
    vec.enable_f64_outputs(True)
    vec.reset()                                          # env e starts scenario e
    pid = DevicePID(vec) if controller == "pid" else None
    if isinstance(controller, dict):
        controller = MlpController(vec, controller)
    steps_cap = vec.cc.steps_max
    d = vec.device
    rew_trace = torch.full((steps_cap, total), float("nan"), dtype=torch.float64, device=d) if keep_rewards else None
    ep_t = torch.zeros(num_envs, dtype=torch.long, device=d)      # step of each env's running episode
    new = torch.ones(num_envs, dtype=torch.bool, device=d)        # the env starts a scenario at this step
    # every env flies at most ceil(total / num_envs) scenarios of at most steps_max steps each
    for _ in range(steps_cap * (-(-total // num_envs)) + 1):
        ids = vec.scenario_ids().long()
        if pid is not None:
            actions = pid(new)
        elif isinstance(controller, MlpController):
            actions = controller(vec._obs64, new)
        else:
            actions = controller(vec)
        _, _, done, _ = vec.step_tensors(actions)
        if rew_trace is not None:
            fly = ids >= 0
            rew_trace[ep_t[fly], ids[fly]] = vec._rew64[fly]
        new = done.bool()
        ep_t = torch.where(new, torch.zeros_like(ep_t), ep_t + 1)
        if bool((res["length"] >= 0).all()):
            break
    else:
        raise RuntimeError("banked evaluation did not finish every scenario")
    rows, ln = res["episode"].cpu().numpy(), res["length"].long().cpu().numpy()
    tr = None if rew_trace is None else rew_trace.cpu().numpy()
    variants = None if air is None else [None] * reps
    return _split(vec, metrics, rows, tr, ln, n_scen, levels, variants), vec


def _results(vec, metrics, rows, tr, ln):
    """res[metric][state] lists, rewards, lengths and episode rows of one block of envs (in env order)."""
    res = {m: {} for m in metrics}
    for i in range(len(ln)):
        if not np.isfinite(rows[i][1]):
            continue                       # still flying at max_steps: no episode row, length = max_steps
        info = vec.episode_info(rows[i])
        for m in metrics:
            for st, val in info.get(m, {}).items():
                res[m].setdefault(st, []).append(val)
    res["rewards"] = None if tr is None else [tr[:ln[i], i].copy() for i in range(len(ln))]
    res["lengths"] = ln
    res["episode_rows"], res["episode_columns"] = rows, vec.episode_columns()
    return res


def summarise(res, metrics=DEFAULT_METRICS):
    """The numbers of the reference README's result table: nan-mean per metric and state."""
    out = {}
    for m in metrics:
        for st, vals in res.get(m, {}).items():
            out["%s_%s" % (m, st)] = float(np.nanmean(np.asarray(vals, dtype=np.float64)))
    return out
