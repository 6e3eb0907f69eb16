"""Batched VecEnv over torch CUDA tensors — the reference-facing host mirror of the hot path.

`FixedWingVecEnv` steps N independent `FixedWingAircraft` (fixed_wing.py:13-437) per call through libfwgym.so.  It
duck-types the stable-baselines VecEnv surface the reference's scripts use (train_rl_controller.py:223-225,
evaluate_controller.py:80-154): num_envs, observation_space/action_space (shape/low/high/dtype), reset(), step(),
step_async()/step_wait(), seed(), get_attr(), set_attr(), env_method(), close(); finished envs auto-reset and return
the post-reset observation, the terminal one is infos[i]["terminal_observation"].  Tensors stay on the device;
`infos` is materialised lazily.  PyTorch is plumbing here (device memory, streams); all compute is in the CUDA library.
"""
import ctypes

import numpy as np
import torch

from . import _capi, scenario_bank
from .config import TURB_LEVELS, CompiledConfig

TERM_NAMES = {0: None, 1: "steps", 2: "success", 3: "numeric"}
N_INIT_ROWS = _capi.DEFINES["FW_N_SV"] + 3
WIND_KEYS = ("wind_n", "wind_e", "wind_d")


class Box:
    """Minimal gym.spaces.Box stand-in (shape / low / high / dtype), float32 like fixed_wing.py:176-183."""

    def __init__(self, low, high, dtype=np.float32):
        self.low = np.asarray(low, dtype=dtype)
        self.high = np.asarray(high, dtype=dtype)
        self.shape = self.low.shape
        self.dtype = np.dtype(dtype)

    def sample(self, rng=None):
        rng = rng or np.random
        lo = np.clip(self.low, -1, 1)
        hi = np.clip(self.high, -1, 1)
        return rng.uniform(lo, hi).astype(self.dtype)


def term_name(code):
    if code >= _capi.DEFINES["FW_TERM_FAIL_BASE"]:
        return _capi.SV_ORDER[code - _capi.DEFINES["FW_TERM_FAIL_BASE"]]
    return TERM_NAMES.get(int(code))


class VecInfos:
    """List-like `infos`: dict i is built on first access (one device->host copy for the whole batch)."""

    def __init__(self, env, done, term, term_obs, targets, ep_out=None):
        self._env, self._done, self._term, self._term_obs, self._targets = env, done, term, term_obs, targets
        self._ep_out = ep_out
        self._host = None
        self._ep_host = None

    def __len__(self):
        return self._env.num_envs

    def _materialise(self):
        if self._host is None:
            self._host = (self._done.cpu().numpy(), self._term.cpu().numpy(), self._targets.cpu().numpy(),
                          None if self._term_obs is None else self._term_obs.cpu().numpy())
        return self._host

    def __getitem__(self, i):
        done, term, tgt, tobs = self._materialise()
        info = {"target": {n: float(tgt[k, i]) for k, n in enumerate(self._env.target_names)}}
        if done[i]:
            info["termination"] = term_name(int(term[i]))
            if tobs is not None:
                info["terminal_observation"] = tobs[i].reshape(self._env.cc.obs_shape)
            if self._ep_out is not None:
                info.update(self._env.episode_info(self._episode_rows()[i]))
        return info

    def _episode_rows(self):
        """Episode-metric rows of the envs that finished in this step: one gather on the device, one copy."""
        if self._ep_host is None:
            idx = torch.nonzero(self._done).flatten()
            rows = self._ep_out[idx].cpu().numpy()
            self._ep_host = {int(e): rows[j] for j, e in enumerate(idx.cpu().numpy())}
        return self._ep_host

    def __iter__(self):
        return (self[i] for i in range(len(self)))


class FixedWingVecEnv:
    def __init__(self, config_path=None, num_envs=1, device="cuda:0", sampler=None, sim_config_path=None,
                 sim_parameter_path=None, config_kw=None, sim_config_kw=None, seed=0, precision="fp64",
                 env_offset=0, auto_reset=True, keep_terminal_obs=False, metrics=False, info_keywords=(),
                 scenario_bank=False, aircraft_parameters=()):
        """`aircraft_parameters`: names of model parameters that may differ per env (set_aircraft): the live model
        parameters but ar, rho, g, Jx, Jy, Jz, Jxz (CompiledConfig.AIRCRAFT_PARAMS).  Not together with
        simulator-parameter randomisation, and b only with turbulence off."""
        if sampler is not None:
            raise NotImplementedError("adaptive sampler hook is out of scope (SURVEY §2 #18)")
        self._lib = _capi.lib()   # raises if the CUDA extension is not built: no fallback
        if not torch.cuda.is_available():
            raise _capi.FwError("FixedWingVecEnv needs a CUDA device (B200, sm_100a); there is no CPU path")
        self.device = torch.device(device)
        self.num_envs = int(num_envs)
        self.env_offset = int(env_offset)
        self.auto_reset = bool(auto_reset)
        self.keep_terminal_obs = bool(keep_terminal_obs)
        self.metrics = bool(metrics)
        self.info_keywords = tuple(info_keywords)
        self.scenario_bank = bool(scenario_bank)   # keep the scenario-bank rows: set_scenario_bank
        self.cc = CompiledConfig(config_path, sim_config_path, sim_parameter_path, config_kw, sim_config_kw, precision,
                                 metrics=self.metrics, scenario_bank=self.scenario_bank,
                                 aircraft_parameters=aircraft_parameters)
        self.cfg = self.cc.cfg
        self.target_names = list(self.cc._target_props_init["states"].keys())
        self.observation_space = Box(self.cc.observation_low, self.cc.observation_high)
        self.action_space = Box(self.cc.action_space_low, self.cc.action_space_high)
        self._h = ctypes.c_void_p()
        pod = self.cc.pod()
        _capi.check(self._lib.fw_create(ctypes.byref(pod), self.num_envs, self.env_offset,
                                        self.device.index or 0, ctypes.byref(self._h)))
        self.obs_dim = self._lib.fw_obs_dim(self._h)
        self.launches_per_step = self._lib.fw_launches_per_step(self._h)
        n, d = self.num_envs, self.device
        self._obs = torch.zeros((n, self.obs_dim), dtype=torch.float32, device=d)
        self._rew = torch.zeros(n, dtype=torch.float32, device=d)
        self._done = torch.zeros(n, dtype=torch.uint8, device=d)
        self._term = torch.zeros(n, dtype=torch.int32, device=d)
        self._term_obs = torch.zeros((n, self.obs_dim), dtype=torch.float32, device=d) if keep_terminal_obs else None
        self._obs64 = self._rew64 = None
        self._actions = None
        self._ep_out = None
        self._turb_noise = None
        self._bank = None
        if self.metrics:
            self.ep_dim = self._lib.fw_episode_dim(self._h)
            self._ep_out = torch.full((n, self.ep_dim), float("nan"), dtype=torch.float64, device=d)
            _capi.check(self._lib.fw_set_episode_out(self._h, self._ptr(self._ep_out)))
        self.training = True
        self.config_version = 0   # bumped by seed() / set_curriculum_level(): captured CUDA graphs must be re-captured
        self._target_row0 = self.state_rows().index("target0")
        self._steps_row = self.state_rows().index("steps_count")
        self.seed(seed)

    # ------------------------------------------------------------------------------------------------ plumbing
    def _stream(self):
        return ctypes.c_void_p(torch.cuda.current_stream(self.device).cuda_stream)

    @staticmethod
    def _ptr(t):
        return ctypes.c_void_p(0 if t is None else t.data_ptr())

    def enable_f64_outputs(self, on=True):
        """Also write float64 observations / rewards (parity checks; the reference returns float64)."""
        if on:
            self._obs64 = torch.zeros((self.num_envs, self.obs_dim), dtype=torch.float64, device=self.device)
            self._rew64 = torch.zeros(self.num_envs, dtype=torch.float64, device=self.device)
        else:
            self._obs64 = self._rew64 = None

    def _shape_obs(self, o):
        return o.view((self.num_envs,) + tuple(self.cc.obs_shape))

    # ---------------------------------------------------------------------------------------------------- API
    def seed(self, seed=None):
        seed = 0 if seed is None else int(seed)
        _capi.check(self._lib.fw_seed(self._h, ctypes.c_uint64(seed & 0xFFFFFFFFFFFFFFFF)))
        self._seed = seed
        self.config_version += 1   # the key is a kernel parameter: a captured graph would replay the old one
        return [seed + self.env_offset + i for i in range(self.num_envs)] if self.num_envs <= 64 else [seed]

    def reset(self, indices=None, state=None, target=None, turbulence_noise=None):
        """Reset all envs (or `indices`).  `state` / `target`: dict name -> scalar or array over the reset envs,
        like FixedWingAircraft.reset(state=, target=) (fixed_wing.py:287-315).  `turbulence_noise`: the reference's
        `**sim_reset_kw` pass-through to PyFly.reset (fixed_wing.py:287,308): unscaled standard-normal samples of the four
        Dryden noise streams for the episodes that start now, [4, T] (the same for every reset env) or [n_reset, 4, T];
        later auto-resets go back to the env's own Philox stream."""
        n, d = self.num_envs, self.device
        mask = None
        idx = None
        if indices is not None:
            idx = torch.as_tensor(np.atleast_1d(indices), dtype=torch.long, device=d)
            mask = torch.zeros(n, dtype=torch.uint8, device=d)
            mask[idx] = 1
        init_state = init_target = None
        if state:
            init_state = torch.full((N_INIT_ROWS, n), float("nan"), dtype=torch.float64, device=d)
            st = dict(state)
            if "wind" in st:
                for k, v in zip(WIND_KEYS, st.pop("wind")):
                    st[k] = v
            for name, val in st.items():
                if name in WIND_KEYS:
                    row = _capi.DEFINES["FW_N_SV"] + WIND_KEYS.index(name)
                elif name in _capi.SV_NAMES:
                    row = _capi.sv_id(name)
                else:
                    continue
                v = torch.as_tensor(np.asarray(val, dtype=np.float64), device=d)
                if idx is None:
                    init_state[row, :] = v
                else:
                    init_state[row, idx] = v
        if target:
            init_target = torch.full((_capi.DEFINES["FW_MAX_TARGETS"], n), float("nan"), dtype=torch.float64, device=d)
            for name, val in target.items():
                row = self.target_names.index(name)
                v = torch.as_tensor(np.asarray(val, dtype=np.float64), device=d)
                if idx is None:
                    init_target[row, :] = v
                else:
                    init_target[row, idx] = v
        noise, noise_len = None, 0
        if turbulence_noise is not None:
            tn = torch.as_tensor(np.asarray(turbulence_noise, dtype=np.float64), device=d)
            if tn.dim() == 2:
                tn = tn.unsqueeze(0)
            if tn.dim() != 3 or tn.shape[1] != 4:
                raise ValueError("turbulence_noise must have shape [4, T] or [n_reset, 4, T]")
            noise_len = int(tn.shape[2])
            noise = torch.zeros((4, noise_len, n), dtype=torch.float64, device=d)   # C-ABI layout [4, T, N]
            if idx is None:
                noise[:] = tn.expand(n, 4, noise_len).permute(1, 2, 0)
            else:
                noise[:, :, idx] = tn.expand(len(idx), 4, noise_len).permute(1, 2, 0)
            if indices is not None and self._turb_noise is not None and self._turb_noise.shape[1] == noise_len:
                keep = torch.ones(n, dtype=torch.bool, device=d)
                keep[idx] = False
                noise[:, :, keep] = self._turb_noise[:, :, keep]    # other envs may still be reading their columns
            self._turb_noise = noise    # the library reads it until those episodes end
        _capi.check(self._lib.fw_reset(self._h, self._ptr(mask), self._ptr(init_state), self._ptr(init_target),
                                       self._ptr(noise), noise_len, self._ptr(self._obs), self._ptr(self._obs64),
                                       self._stream()))
        return self._shape_obs(self._obs)

    def step_tensors(self, actions, out=None):
        """Device-only step: (obs, reward, done, term_code) tensors, no host synchronisation.
        actions: [N, 3] float32 or float64 CUDA tensor (float64 is upcast-free and used for parity).
        out: optional (obs, rew, done, term) device tensors to write instead of the env's own (HostStepper)."""
        if actions.device != self.device:
            actions = actions.to(self.device, non_blocking=True)
        if actions.dtype not in (torch.float32, torch.float64):
            actions = actions.float()
        actions = actions.contiguous()
        if actions.shape != (self.num_envs, 3):
            raise ValueError("actions must have shape (%d, 3)" % self.num_envs)
        obs, rew, done, term = out if out is not None else (self._obs, self._rew, self._done, self._term)
        _capi.check(self._lib.fw_step(self._h, self._ptr(actions), 1 if actions.dtype == torch.float64 else 0,
                                      self._ptr(obs), self._ptr(rew), self._ptr(done),
                                      self._ptr(term), self._ptr(self._obs64), self._ptr(self._rew64),
                                      self._ptr(self._term_obs), 1 if self.auto_reset else 0, self._stream()))
        self._actions = actions   # keep alive until the stream has consumed it
        return self._shape_obs(obs), rew, done, term

    def step_async(self, actions):
        if not torch.is_tensor(actions):
            actions = torch.as_tensor(np.asarray(actions))
        self._pending = self.step_tensors(actions)

    def step_wait(self):
        obs, rew, done, term = self._pending
        # the episode rows are snapshotted here: the next step may overwrite them
        ep = self._ep_out.clone() if self._ep_out is not None else None
        tobs = self._term_obs.clone() if self._term_obs is not None else None   # the next step overwrites it
        infos = VecInfos(self, done.clone(), term.clone(), tobs, self.get_targets(), ep)
        return obs, rew, done.bool(), infos

    def step(self, actions):
        self.step_async(actions)
        return self.step_wait()

    # ---------------------------------------------------------------------------------------- episode metrics
    EP_FIXED = ("r", "l", "control_variation", "success_all", "settling_time_all", "success_time_frac_all")
    EP_PER_TARGET = ("avg_error", "total_error", "end_error", "rise_time", "overshoot", "success", "settling_time",
                     "success_time_frac")

    def episode_metrics(self):
        """Device tensor [N, ep_dim] of the last finished episode's metrics per env (NaN rows: none finished yet);
        columns: episode_columns()."""
        if self._ep_out is None:
            raise _capi.FwError("construct the env with metrics=True")
        return self._ep_out

    def episode_columns(self):
        cols = list(self.EP_FIXED)
        for t in self.target_names:
            cols += ["%s_%s" % (m, t) for m in self.EP_PER_TARGET]
        return cols

    def episode_info(self, row):
        """One episode row -> the entries the reference puts into `info` when an episode ends (fixed_wing.py:417-419:
        info[metric] = get_metric(metric) for every metric listed in the config) plus the Monitor-style
        info["episode"] = {"r", "l", + info_keywords} (train_rl_controller.py:153,172)."""
        nan = float("nan")
        per = {m: {} for m in self.EP_PER_TARGET}
        for k, t in enumerate(self.target_names):
            base = len(self.EP_FIXED) + k * len(self.EP_PER_TARGET)
            for j, m in enumerate(self.EP_PER_TARGET):
                v = float(row[base + j])
                if m in ("success", "settling_time", "success_time_frac") and not self.cc.goal_has_bound(t):
                    continue   # the reference's goal history only has the states with a bound (fixed_wing.py:916-931)
                per[m][t] = (v == 1.0) if m == "success" else v
        if self.cc.goal_enabled:
            per["success"]["all"] = bool(row[3] == 1.0)
            per["settling_time"]["all"] = float(row[4])
            per["success_time_frac"]["all"] = float(row[5])
        else:
            per["success"], per["settling_time"], per["success_time_frac"] = {}, {}, {}
        per["control_variation"] = {"all": float(row[2])}
        wanted = [m["name"] for m in self.cfg.get("metrics", [])]
        info = {m: per[m] for m in wanted if m in per}
        ep = {"r": float(row[0]), "l": int(row[1])}
        for kw in self.info_keywords:
            ep[kw] = per.get(kw, nan)
        info["episode"] = ep
        return info

    def close(self):
        if getattr(self, "_h", None) is not None and self._h.value:
            self._lib.fw_destroy(self._h)
            self._h = ctypes.c_void_p()

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # ---------------------------------------------------------------------------- state, counters, metrics
    def state_rows(self):
        n = self._lib.fw_state_rows(self._h)
        return [self._lib.fw_state_row_name(self._h, r).decode() for r in range(n)]

    def get_state(self):
        out = torch.empty((self._lib.fw_state_rows(self._h), self.num_envs), dtype=torch.float64, device=self.device)
        _capi.check(self._lib.fw_get_state(self._h, self._ptr(out), self._stream()))
        return out

    def set_state(self, state):
        state = state.to(self.device, torch.float64).contiguous()
        _capi.check(self._lib.fw_set_state(self._h, self._ptr(state), self._stream()))
        self._state_keepalive = state

    def get_named_state(self, names):
        rows = self.state_rows()
        st = self.get_state()
        return {n: st[rows.index(n)] for n in names}

    def get_rows(self, row0, nrows):
        """Rows [row0, row0 + nrows) of the state matrix (state_rows() names them): device float64 [nrows, N]."""
        out = torch.empty((nrows, self.num_envs), dtype=torch.float64, device=self.device)
        _capi.check(self._lib.fw_get_rows(self._h, int(row0), int(nrows), self._ptr(out), self._stream()))
        return out

    def get_targets(self):
        return self.get_rows(self._target_row0, len(self.target_names))

    def last_attempts(self):
        out = torch.empty(self.num_envs, dtype=torch.int32, device=self.device)
        _capi.check(self._lib.fw_last_attempts(self._h, self._ptr(out), self._stream()))
        return out

    def counters(self):
        c = _capi.fw_counters_t()
        _capi.check(self._lib.fw_counters(self._h, ctypes.byref(c)))
        return {k: int(getattr(c, k)) for k, _ in c._fields_}

    def reset_counters(self):
        _capi.check(self._lib.fw_reset_counters(self._h))

    def get_simulator_parameters(self, normalize=True):
        """FixedWingAircraft.get_simulator_parameters (fixed_wing.py:872-888) for every env: device tensor
        [N, n_listed_parameters] of the current (per-episode randomised) model parameters, normalised as the reference
        does ((value - original) / var).  Parameters the dynamics never read (inertia) report their nominal value:
        their draw is consumed and discarded on the device."""
        model = self.cc.cfg["simulator"].get("model", {})
        plan, slot1, _ = self.cc._rand_slots()
        st = self.get_state()
        rows = self.state_rows()
        first = rows.index("param") if "param" in rows else None
        cols = []
        for pa in model.get("parameters", []):
            name = pa["name"]
            orig = pa.get("original", None)
            if orig is None:
                orig = self.cc.params[name] if name != "ar" else self.cc.params["b"] ** 2 / self.cc.params["S_wing"]
            pid = self.cc.par_id(name) if name in self.cc.LIVE_PARAMS else -1
            if pid >= 0 and slot1[pid]:
                val = st[first + slot1[pid] - 1]
            else:
                val = torch.full((self.num_envs,), float(orig), dtype=torch.float64, device=self.device)
            if normalize:
                var = pa.get("var", model["var"])
                if model.get("var_type", "relative") == "relative":
                    if orig == 0:
                        continue
                    var = var * orig
                val = (val - orig) / var
            cols.append(val)
        if not cols:
            return torch.empty((self.num_envs, 0), dtype=torch.float64, device=self.device)
        return torch.stack(cols, dim=1)

    # ------------------------------------------------------------------------ per-env Dryden turbulence intensity
    def set_turbulence_intensity(self, levels, indices=None):
        """Pin the Dryden intensity of envs (all, or `indices`) from their next reset on (explicit or automatic; the
        running episodes keep theirs).  `levels`: a level name ("none", "light", "moderate", "severe"), a list of names
        (one per selected env), or an int array / tensor of levels 0..3, where -1 goes back to drawing from the handle's
        distribution at every reset.  Needs a mixed handle: sim_config_kw turbulence_intensity =
        {"values": [...], "probabilities": [...]}."""
        if not self.cc.turbulence_mix:
            raise _capi.FwError("set_turbulence_intensity needs per-env levels: configure turbulence_intensity as "
                                "{\"values\": [...], \"probabilities\": [...]}")
        idx = None if indices is None else torch.as_tensor(np.atleast_1d(indices), dtype=torch.long, device=self.device)
        count = self.num_envs if idx is None else len(idx)

        def code(name):
            if name not in TURB_LEVELS:
                raise ValueError("unknown turbulence level %r (levels: %s)" % (name, ", ".join(TURB_LEVELS)))
            return TURB_LEVELS.index(name)
        if isinstance(levels, str):
            lv = torch.full((count,), code(levels), dtype=torch.int32, device=self.device)
        elif isinstance(levels, (list, tuple)) and levels and all(isinstance(x, str) for x in levels):
            lv = torch.as_tensor([code(x) for x in levels], dtype=torch.int32, device=self.device)
        else:
            lv = torch.as_tensor(np.asarray(levels.cpu() if torch.is_tensor(levels) else levels), device=self.device)
            if lv.dtype.is_floating_point or lv.dtype == torch.bool:
                raise ValueError("turbulence levels must be names or integers -1..3")
            lv = lv.to(torch.int32).reshape(-1)
            if lv.numel() == 1 and count != 1:
                lv = lv.expand(count)
            if bool(((lv < -1) | (lv > 3)).any()):
                raise ValueError("turbulence levels must be in -1..3")
        if lv.numel() != count:
            raise ValueError("%d turbulence levels for %d envs" % (lv.numel(), count))
        req = self.get_rows(self.state_rows().index("turb_level_req"), 1)[0].to(torch.int32)
        if idx is None:
            req[:] = lv
        else:
            req[idx] = lv
        _capi.check(self._lib.fw_set_turbulence_levels(self._h, self._ptr(req), self._stream()))
        self._turb_req_keepalive = req

    def turbulence_levels(self):
        """Device int32 [N]: the Dryden level of every env's running episode (0 none, 1 light, 2 moderate, 3 severe).
        A handle without per-env levels reports its single intensity for every env."""
        rows = self.state_rows()
        if "turb_level" in rows:
            return self.get_rows(rows.index("turb_level"), 1)[0].to(torch.int32)
        sc = self.cc.sim_cfg
        lvl = TURB_LEVELS.index(sc.get("turbulence_intensity") or "light") if sc["turbulence"] else 0
        return torch.full((self.num_envs,), lvl, dtype=torch.int32, device=self.device)

    # ------------------------------------------------------------------------------------------- per-env aircraft
    def set_aircraft(self, values, indices=None):
        """Request the aircraft of envs (all, or `indices`) from their next reset on (explicit or automatic; the running
        episodes keep theirs).  `values`: dict name -> a scalar, an array / tensor with one value per selected env; the
        names are among the handle's aircraft_parameters, and NaN goes back to the handle's nominal value.  An env flies
        the aircraft a reference env built from a parameter file with these values would fly (include/fwgym.h
        fw_set_aircraft).  Parameters not named keep their requests."""
        names = self.cc.aircraft_parameters
        if not names:
            raise _capi.FwError("construct the env with aircraft_parameters=(...) to set aircraft per env")
        idx = None if indices is None else torch.as_tensor(np.atleast_1d(indices), dtype=torch.long, device=self.device)
        count = self.num_envs if idx is None else len(idx)
        req = self.aircraft_requests().clone()
        for name, val in dict(values).items():
            if name not in names:
                raise ValueError("%r is not an aircraft parameter of this env (aircraft_parameters: %s)"
                                 % (name, ", ".join(names)))
            v = torch.as_tensor(val.cpu() if torch.is_tensor(val) else np.asarray(val, dtype=np.float64),
                                dtype=torch.float64).to(self.device).reshape(-1)
            if v.numel() == 1 and count != 1:
                v = v.expand(count)
            if v.numel() != count:
                raise ValueError("aircraft parameter %s: %d values for %d envs" % (name, v.numel(), count))
            if idx is None:
                req[names.index(name)] = v
            else:
                req[names.index(name), idx] = v
        check_aircraft(self.cc, req)
        req = req.contiguous()
        _capi.check(self._lib.fw_set_aircraft(self._h, self._ptr(req), self._stream()))
        self._aircraft_keepalive = req

    def aircraft_requests(self):
        """Device float64 [len(aircraft_parameters), N]: the requested value of every aircraft parameter per env (NaN =
        nominal), rows in aircraft_parameters order."""
        rows = self.state_rows()
        if "aircraft_req" not in rows:
            raise _capi.FwError("construct the env with aircraft_parameters=(...)")
        return self.get_rows(rows.index("aircraft_req"), len(self.cc.aircraft_parameters))

    def aircraft(self):
        """name -> device float64 [N]: the requested aircraft of every env (NaN = nominal), as set_aircraft takes it."""
        req = self.aircraft_requests()
        return {n: req[j] for j, n in enumerate(self.cc.aircraft_parameters)}

    # ------------------------------------------------------------------------------------------ scenario banks
    def set_scenario_bank(self, state=None, target=None, turbulence_intensity=None, first=None, stride=None,
                          cycle=False, aircraft=None):
        """Attach a bank of S scenarios that the resets of this env consume in order (include/fwgym.h fw_bank_t): every
        auto-reset, and reset() without state= / target=, starts the env's next scenario - env e flies first + e, then
        + stride per episode (modulo S with `cycle`) - until the env is past the bank, after which it samples as usual.
        `state` / `target`: the names reset(state=, target=) takes, one value per scenario (NaN = sample it; a scalar
        applies to all); `turbulence_intensity`: one level per scenario (mixed handles; -1 = the env's own rule);
        `aircraft`: dict aircraft parameter -> one value per scenario (a finite value pins the scenario's aircraft like
        set_aircraft, NaN = the env's own request).
        `first` / `stride` default to 0 / num_envs; sharded ranks pass first = env_offset and stride = the total env
        count.  Allocates the result rows scenario_results() returns (cycling banks: the counters only).  Takes effect
        at the envs' next reset.  Attaching clears every env's running scenario id: an episode that is running now (from
        an earlier bank) finishes, but reports no result anywhere."""
        if not self.scenario_bank:
            raise _capi.FwError("construct the env with scenario_bank=True")
        S, st, tg, lv, air = scenario_bank.build_bank_tables(state, target, turbulence_intensity, self.target_names,
                                                             mixed=bool(self.cc.turbulence_mix), aircraft=aircraft,
                                                             aircraft_parameters=self.cc.aircraft_parameters)
        if air is not None:
            check_aircraft(self.cc, torch.as_tensor(air))
        first = 0 if first is None else int(first)
        stride = self.num_envs if stride is None else int(stride)
        scenario_bank.check_assignment(self.num_envs, S, first, stride)
        d = self.device
        keep = {"init_state": None if st is None else torch.as_tensor(st, device=d),
                "init_target": None if tg is None else torch.as_tensor(tg, device=d),
                "turb_level": None if lv is None else torch.as_tensor(lv, device=d),
                "aircraft": None if air is None else torch.as_tensor(air, device=d)}
        res = {"episodes": torch.zeros(S, dtype=torch.int32, device=d),
               "successes": torch.zeros(S, dtype=torch.int32, device=d)}
        if not cycle:
            res["term"] = torch.full((S,), -1, dtype=torch.int32, device=d)
            res["length"] = torch.full((S,), -1, dtype=torch.int32, device=d)
            res["return"] = torch.full((S,), float("nan"), dtype=torch.float64, device=d)
            if self.metrics:
                res["episode"] = torch.full((S, self.ep_dim), float("nan"), dtype=torch.float64, device=d)
        b = _capi.fw_bank_t()
        b.init_state, b.init_target, b.turb_level = (keep[k].data_ptr() if keep[k] is not None else None
                                                     for k in ("init_state", "init_target", "turb_level"))
        b.n_scenarios, b.first, b.stride, b.cycle = S, first, stride, 1 if cycle else 0
        for f, k in (("term", "term"), ("length", "length"), ("ret", "return"), ("episode", "episode"),
                     ("episodes", "episodes"), ("successes", "successes")):
            if k in res:
                setattr(b, f, res[k].data_ptr())
        _capi.check(self._lib.fw_set_bank(self._h, ctypes.byref(b), self._stream()))
        if keep["aircraft"] is not None:
            _capi.check(self._lib.fw_set_bank_aircraft(self._h, self._ptr(keep["aircraft"])))
        self._bank = (keep, res)          # the device reads these while the bank is attached
        self.n_scenarios = S
        self.config_version += 1          # the bank is a kernel parameter: captured graphs hold the old one
        return res

    def detach_scenario_bank(self):
        """Back to sampled resets (the cursors are cleared; running episodes no longer report results)."""
        _capi.check(self._lib.fw_set_bank(self._h, None, self._stream()))
        self.config_version += 1
        self._bank_detached = self._bank   # kept alive until the stream is past the last kernel that read them
        self._bank = None

    def scenario_results(self):
        """Device tensors of the attached bank, indexed by scenario id: "term" (FW_TERM_* code, -1 = not flown yet),
        "length", "return", "episode" ([S, ep_dim] metric rows, metrics=True) and the int32 counters "episodes" /
        "successes" (a cycling bank has the counters only)."""
        if self._bank is None:
            raise _capi.FwError("no scenario bank attached (set_scenario_bank)")
        return self._bank[1]

    def scenario_ids(self):
        """Device int32 [N]: the scenario each env's running episode started from, -1 when it was not from the bank."""
        rows = self.state_rows()
        if "bank_scenario" not in rows:
            raise _capi.FwError("construct the env with scenario_bank=True")
        return self.get_rows(rows.index("bank_scenario"), 1)[0].to(torch.int32)

    def kernel_variant(self):
        """Which kernel instantiations the configuration selected, e.g. "dyn=shipped env=default_turb"."""
        return self._lib.fw_kernel_variant(self._h).decode()

    def set_profiling(self, on=True):
        _capi.check(self._lib.fw_set_profiling(self._h, 1 if on else 0))

    def profile(self):
        """-> (dynamics kernel ms, env kernel ms, steps) summed since the last call (synchronises)."""
        d, e, n = ctypes.c_double(), ctypes.c_double(), ctypes.c_int64()
        _capi.check(self._lib.fw_profile(self._h, ctypes.byref(d), ctypes.byref(e), ctypes.byref(n)))
        return d.value, e.value, n.value

    METRIC_SUM_NAMES = ("episodes", "successes", "sum_return", "sum_length", "failures", "steps_term", "success_term",
                        "goal_steps")

    def metric_sums(self):
        """Local episode-metric sums (host float64 vector) — all-reduce these across ranks (parallel.py)."""
        buf = (ctypes.c_double * _capi.DEFINES["FW_N_METRIC_SUMS"])()
        _capi.check(self._lib.fw_metric_sums(self._h, buf))
        return np.array(buf[:], dtype=np.float64)

    # ------------------------------------------------------------------- SB VecEnv attribute / method plumbing
    def get_attr(self, name, indices=None):
        n = self.num_envs if indices is None else len(np.atleast_1d(indices))
        if name == "target":
            tg = self.get_targets().cpu().numpy()
            ids = range(self.num_envs) if indices is None else np.atleast_1d(indices)
            return [{t: float(tg[k, i]) for k, t in enumerate(self.target_names)} for i in ids]
        if name == "steps_count":
            sc = self.get_rows(self._steps_row, 1)[0].cpu().numpy().astype(int)
            ids = range(self.num_envs) if indices is None else np.atleast_1d(indices)
            return [int(sc[i]) for i in ids]
        if name == "simulator":
            return [SimulatorView(self)] * n
        if name == "turbulence_intensity":
            lv = self.turbulence_levels().cpu().numpy()
            ids = range(self.num_envs) if indices is None else np.atleast_1d(indices)
            return [TURB_LEVELS[int(lv[i])] for i in ids]
        return [getattr(self, name)] * n

    def set_attr(self, name, value, indices=None):
        setattr(self, name, value)

    def env_method(self, name, *args, indices=None, **kwargs):
        n = self.num_envs if indices is None else len(np.atleast_1d(indices))
        if name == "set_curriculum_level":
            self.set_curriculum_level(*args, **kwargs)
            return [None] * n
        if name == "reset":
            obs = self.reset(indices=indices, **kwargs)   # state=, target=, turbulence_noise=
            ids = range(self.num_envs) if indices is None else np.atleast_1d(indices)
            host = obs.cpu().numpy()
            return [host[i] for i in ids]
        if name == "seed":
            return [self.seed(*args, **kwargs)] * n
        raise NotImplementedError("env_method(%r) is not supported" % name)

    def set_curriculum_level(self, level):
        """fixed_wing.py:224-285; applies to every env of the batch (the reference calls it on all envs too,
        train_rl_controller.py:84,224)."""
        self.cc.set_curriculum_level(level)
        pod = self.cc.pod()
        _capi.check(self._lib.fw_set_config(self._h, ctypes.byref(pod)))
        self.config_version += 1   # the configuration is a kernel parameter: captured graphs hold the old one


def check_aircraft(cc, req):
    """Refuse aircraft requests [len(cc.aircraft_parameters), M] (NaN = nominal) that no parameter file could hold: an
    infinite value, mass, Jy, b or S_wing <= 0, or an inertia tensor with Jx Jz - Jxz^2 <= 0."""
    names = cc.aircraft_parameters
    req = req.to(torch.float64)
    if bool(torch.isinf(req).any()):
        raise ValueError("aircraft parameters must be finite (NaN = nominal)")
    nominal = cc.aircraft_nominal()
    par = dict(cc.params)

    def value(name):
        if name in names:
            r = req[names.index(name)]
            return torch.where(torch.isnan(r), torch.full_like(r, nominal[name]), r)
        return torch.full(req.shape[1:], float(par[name]), dtype=torch.float64, device=req.device)
    for name in ("mass", "Jy", "b", "S_wing"):
        if name in names and not bool((value(name) > 0).all()):
            raise ValueError("aircraft parameter %s must be > 0" % name)
    if any(n in names for n in ("Jx", "Jz", "Jxz")):
        if not bool((value("Jx") * value("Jz") - value("Jxz") ** 2 > 0).all()):
            raise ValueError("aircraft inertia must have Jx * Jz - Jxz^2 > 0")


class HostStepper:
    """Host-buffer stepping for callers whose policy lives on the CPU: actions come from host memory and observations
    / rewards / dones land in pinned host memory, every step.  Thin wrapper over the C-ABI pipeline (fw_host_open /
    fw_host_submit / fw_host_wait, include/fwgym.h): the copies run on their own CUDA streams and the device-side
    buffers are `depth`-buffered, so with `depth` submissions in flight the PCIe traffic of step t overlaps the kernels
    of step t+1 (the SubprocVecEnv reference overlaps its pipe traffic with env work the same way, one process per
    env).  submit() never blocks on the GPU; wait() blocks until that step's results are on the host.  With depth=1
    this is a plain synchronous host step."""

    def __init__(self, vec, depth=2, zero_copy=False):
        """zero_copy: the env kernel writes the results straight into mapped pinned host memory (no device -> host copy
        after the step; include/fwgym.h fw_host_open_ex)."""
        self.vec, self.depth, self.zero_copy = vec, int(depth), bool(zero_copy)
        n, od = vec.num_envs, vec.obs_dim
        _capi.check(vec._lib.fw_host_open_ex(vec._h, self.depth, 1 if zero_copy else 0))
        self._views = {}
        self.h2d_bytes = n * 3 * 4
        self.d2h_bytes = n * (od * 4 + 4 + 1 + 4)

    def submit(self, actions):
        """actions: [N, 3] float32 numpy array or CPU tensor (pinned memory makes the upload asynchronous).  Returns
        the slot to wait() on."""
        v = self.vec
        if torch.is_tensor(actions):
            if actions.dtype != torch.float32 or not actions.is_contiguous():
                actions = actions.float().contiguous()
            ptr = actions.data_ptr()
        else:
            actions = np.ascontiguousarray(actions, dtype=np.float32)
            ptr = actions.ctypes.data
        if tuple(actions.shape) != (v.num_envs, 3):
            raise ValueError("actions must have shape (%d, 3)" % v.num_envs)
        slot = ctypes.c_int()
        _capi.check(v._lib.fw_host_submit(v._h, ptr, v._stream(), ctypes.byref(slot)))
        self._keep = actions
        return slot.value

    def wait(self, slot):
        """-> (obs [N, obs_dim] float32, reward [N] float32, done [N] uint8) numpy views of the slot's pinned buffers
        (valid until the slot is submitted again); the termination codes are in self.term(slot)."""
        v = self.vec
        po, pr, pd, pt = ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p(), ctypes.c_void_p()
        _capi.check(v._lib.fw_host_wait(v._h, int(slot), ctypes.byref(po), ctypes.byref(pr), ctypes.byref(pd),
                                        ctypes.byref(pt)))
        views = self._views.get(slot)
        if views is None:
            n, od = v.num_envs, v.obs_dim
            mk = lambda p, ct, shape: np.ctypeslib.as_array(ctypes.cast(p, ctypes.POINTER(ct)), shape=shape)
            views = (mk(po, ctypes.c_float, (n, od)), mk(pr, ctypes.c_float, (n,)), mk(pd, ctypes.c_uint8, (n,)),
                     mk(pt, ctypes.c_int32, (n,)))
            self._views[slot] = views
        return views[0], views[1], views[2]

    def term(self, slot):
        return self._views[slot][3]

    def close(self):
        self._views = {}
        if self.vec._h:
            self.vec._lib.fw_host_close(self.vec._h)


class SimulatorView:
    """The slice of the PyFly object surface that callers of the reference touch (fixed_wing.py §8b): dt, params."""

    def __init__(self, env):
        self.dt = env.cc.dt
        self.params = env.cc.params
        self.state = env.cc.state
