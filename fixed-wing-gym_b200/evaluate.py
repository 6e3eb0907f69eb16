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
                    turbulence_intensity="none", device="cuda:0", seed=0, max_steps=None, env_offset=0):
    """Run every scenario once (in parallel) under `controller`: "pid", a dict of saved MlpPolicy arrays
    (MlpController), or a callable(vec) -> actions tensor.
    Returns (res, vec_env): res[metric][state] lists in scenario order, res["rewards"], res["lengths"].
    `turbulence_intensity`: one level ("none", "light", "moderate", "severe"), or a list of levels: then the S
    scenarios x L levels fly as ONE batch of L * S envs on a handle with per-env intensities (env j * S + i is scenario i
    at level j, pinned with set_turbulence_intensity) and the first element of the return value is {level: res}.
    `env_offset`: global id of the first env (the Philox streams are keyed by it)."""
    levels = None if isinstance(turbulence_intensity, str) else list(turbulence_intensity)
    n_scen = len(scenarios)
    n = n_scen if levels is None else n_scen * len(levels)
    kw = dict(config_kw or {})
    for k, v in EVAL_CONFIG_KW.items():
        kw[k] = v
    if controller == "pid":
        kw["action"] = {"scale_space": False}          # evaluate_controller.py:78-79
    if levels is None:
        sim_kw = {"turbulence": turbulence_intensity != "none", "turbulence_intensity": turbulence_intensity}
    else:
        sim_kw = {"turbulence": True, "turbulence_intensity": {"values": levels}}
    vec = FixedWingVecEnv(config_path, n, device=device, config_kw=kw, sim_config_kw=sim_kw, seed=seed, metrics=True,
                          auto_reset=True, env_offset=env_offset)
    if levels is not None:
        vec.set_turbulence_intensity([lv for lv in levels for _ in range(n_scen)])
    reps = 1 if levels is None else len(levels)
    skeys = sorted(scenarios[0]["state"].keys())
    state = {}
    for k in skeys:
        v0 = scenarios[0]["state"][k]
        if isinstance(v0, (list, tuple, np.ndarray)):     # "wind": [n, e, d]
            state[k] = np.tile(np.array([s["state"][k] for s in scenarios], dtype=np.float64).T, (1, reps))
        else:
            state[k] = np.tile(np.array([s["state"][k] for s in scenarios], dtype=np.float64), reps)
    target = {k: np.tile(np.array([s["target"][k] for s in scenarios], dtype=np.float64), reps)
              for k in scenarios[0]["target"]}
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
    if levels is None:
        return _results(vec, metrics, rows, tr, ln), vec
    return {lv: _results(vec, metrics, rows[j * n_scen:(j + 1) * n_scen], tr[:, j * n_scen:(j + 1) * n_scen],
                         ln[j * n_scen:(j + 1) * n_scen]) for j, lv in enumerate(levels)}, vec


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
    res["rewards"] = [tr[:ln[i], i].copy() for i in range(len(ln))]
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
