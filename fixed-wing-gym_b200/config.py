"""Host-side configuration compiler: the reference's JSON surface -> flat POD `fw_config_t` (include/fwgym.h).

Mirrors, on the host and once per (re)configuration:
  * the config loader and recursive override of FixedWingAircraft.__init__ (fixed_wing.py:24-35) and the PyFly
    overrides it forces (fixed_wing.py:37-46);
  * observation bounds / normalisation defaults (fixed_wing.py:57-134), action scaling vectors and bounds
    (fixed_wing.py:136-191);
  * set_curriculum_level (fixed_wing.py:224-285);
  * PyFly's own config/parameter parsing (pyfly_config.json variables -> limits in radians, actuator coefficients,
    inertia Gammas) and the Dryden filter discretisation that scipy.signal.lsim performs per reset
    (scipy/signal/_ltisys.py:2254-2277), done here once.
No simulation happens here; everything per-step runs in the CUDA kernels.
"""
import copy
import json
import math
import os

import numpy as np

from . import _capi

_HERE = os.path.dirname(os.path.abspath(__file__))
DEFAULT_SIM_CONFIG = os.path.join(_HERE, "params", "pyfly_config.json")
DEFAULT_SIM_PARAMS = os.path.join(_HERE, "params", "x8_param.json")
DEFAULT_ENV_CONFIG = os.path.join(_HERE, "params", "fixed_wing_config.json")
F32_MAX = float(np.finfo(np.float32).max)

FCLASS = {"linear": 0, "exponential": 1, "quadratic": 2}
TCLASS = {"constant": 0, "linear": 1, "sinusoidal": 2, "compensate": 3}
ACT_NAMES = ["elevator", "aileron", "throttle"]
# Dryden intensities of a mixed handle, in level order (include/fwgym.h fw_sim_t.turb_mixed)
TURB_LEVELS = ("none", "light", "moderate", "severe")


class ConfigError(ValueError):
    pass


def apply_overrides(tree, overrides):
    """`config_kw` semantics of FixedWingAircraft.__init__ (fixed_wing.py:24-35): an override tree is merged into the
    parsed JSON; a dict value descends into the existing node, and so does ANY value addressed into a list (integer
    keys pick list elements, e.g. {"states": {6: {"value": "integrator"}}}); everything else replaces the leaf.  Keys
    must already exist (KeyError otherwise, like the reference: overrides cannot add entries)."""
    pending = [(tree, overrides)]
    while pending:
        node, patch = pending.pop()
        for key, val in patch.items():
            if isinstance(val, dict) or isinstance(node[key], list):
                pending.append((node[key], val))
            else:
                node[key] = val


def _set_sim_config_attrs(parent, kws):
    """PyFly's own override: recurse on dict values only."""
    for attr, val in kws.items():
        if isinstance(val, dict):
            _set_sim_config_attrs(parent[attr], val)
        else:
            parent[attr] = val


class SimVariable:
    """Limits of one PyFly Variable (value_min/max, init_min/max, constraint_min/max, wrap), radians applied."""
    LIMITS = ("value_min", "value_max", "init_min", "init_max", "constraint_min", "constraint_max", "dot_max")

    def __init__(self, spec):
        self.name = spec["name"]
        self.value_min = spec.get("value_min")
        self.value_max = spec.get("value_max")
        self.init_min = spec.get("init_min") if spec.get("init_min") is not None else self.value_min
        self.init_max = spec.get("init_max") if spec.get("init_max") is not None else self.value_max
        self.constraint_min = spec.get("constraint_min")
        self.constraint_max = spec.get("constraint_max")
        self.dot_max = spec.get("dot_max")
        if spec.get("convert_to_radians", False):
            for a in self.LIMITS:
                if getattr(self, a) is not None:
                    setattr(self, a, getattr(self, a) * (np.pi / 180))
        self.wrap = bool(spec.get("wrap", False))
        self.order = spec.get("order")
        self.tau = spec.get("tau")
        self.omega_0 = spec.get("omega_0")
        self.zeta = spec.get("zeta")
        self.disabled = bool(spec.get("disabled", False))

    @property
    def coefs(self):
        if self.order == 1:
            return [[-1 / self.tau, 0, 1 / self.tau], [0, 0, 0]]
        if self.order == 2:
            return [[0, 1, 0], [-self.omega_0 ** 2, -2 * self.zeta * self.omega_0, self.omega_0 ** 2]]
        raise ConfigError("actuator %s needs order 1 or 2" % self.name)


def dryden_transfer_functions(b, intensity, h=100.0, V_a=25.0):
    """(num, den, noise stream) of the six MIL-F-8785C shaping filters as PyFly's DrydenGustModel builds them
    (SURVEY App. D): the specification's feet units inside, W20 = 15 / 30 / 45 KNOTS, linear gusts returned in m/s
    (angular gusts are rad/s in either unit system).  An earlier recollection fed W20 as "15 * ft" and used the ft/s
    outputs as m/s, 6.4x too strong: the reference's PID then crashes 24 of 25 moderate-turbulence scenarios where the
    README reports 93 % success (oracle/pyfly_restated.py, DESIGN.md §2)."""
    ft = 3.28084
    knot_ftps = 1.6878098571
    h, b, V_a = h * ft, b * ft, V_a * ft
    if intensity is None or intensity == "light":
        W_20 = 15 * knot_ftps
    elif intensity == "moderate":
        W_20 = 30 * knot_ftps
    elif intensity == "severe":
        W_20 = 45 * knot_ftps
    else:
        raise ConfigError("Unsupported turbulence intensity %r" % (intensity,))
    L_u = h / (0.177 + 0.000823 * h) ** 1.2
    L_v, L_w = L_u, h
    sigma_w = 0.1 * W_20
    sigma_u = sigma_w / (0.177 + 0.000823 * h) ** 0.4
    sigma_v = sigma_u
    K_u = sigma_u * math.sqrt((2 * L_u) / (math.pi * V_a))
    K_v = sigma_v * math.sqrt(L_v / (math.pi * V_a))
    K_w = sigma_w * math.sqrt(L_w / (math.pi * V_a))
    T_u = L_u / V_a
    T_v1, T_v2 = math.sqrt(3.0) * L_v / V_a, L_v / V_a
    T_w1, T_w2 = math.sqrt(3.0) * L_w / V_a, L_w / V_a
    K_p = sigma_w * math.sqrt(0.8 / V_a) * ((math.pi / (4 * b)) ** (1 / 6)) / (L_w ** (1 / 3))
    K_q = K_r = 1 / V_a
    T_p = 4 * b / (math.pi * V_a)
    T_q, T_r = T_p, 3 * b / (math.pi * V_a)
    m = 1.0 / ft          # ft/s -> m/s for the three linear gust components
    return [
        ([K_u * m], [T_u, 1], 0),
        ([K_v * T_v1 * m, K_v * m], [T_v2 ** 2, 2 * T_v2, 1], 1),
        ([K_w * T_w1 * m, K_w * m], [T_w2 ** 2, 2 * T_w2, 1], 2),
        ([K_p], [T_p, 1], 3),
        ([-K_w * K_q * T_w1, -K_w * K_q, 0], [T_q * T_w2 ** 2, T_w2 ** 2 + 2 * T_q * T_w2, T_q + 2 * T_w2, 1], 1),
        ([K_v * K_r * T_v1, K_v * K_r, 0], [T_r * T_v2 ** 2, T_v2 ** 2 + 2 * T_r * T_v2, T_r + 2 * T_v2, 1], 2),
    ]


def turbulence_cdf(probabilities):
    """Level probabilities [p_none, p_light, p_moderate, p_severe] -> the fp64 cumulative table the reset draw searches
    (fw_sim_t.turb_cdf): running sums in level order, and 1 from the last level with a non-zero probability on, so a
    uniform in [0, 1) never lands past it."""
    cdf, acc = [], 0.0
    last = max(i for i, p in enumerate(probabilities) if p > 0)
    for i, p in enumerate(probabilities):
        acc += float(p)
        cdf.append(1.0 if i >= last else acc)
    return cdf


def draw_turbulence_level(cdf, u):
    """The level a reset draws for the uniform `u` (csrc/env.cuh fw_reset_env_body): the first l with u < cdf[l]."""
    return int(sum(1 for c in cdf[:-1] if u >= c))


def discretise_filter(num, den, dt):
    """The (Ad, Bd0, Bd1, C, D) that scipy.signal.lsim(interp=True) builds from a transfer function."""
    import scipy.linalg
    import scipy.signal
    A, B, C, D = scipy.signal.tf2ss(num, den)
    n, m = A.shape[0], 1
    M = np.vstack([np.hstack([A * dt, B * dt, np.zeros((n, m))]),
                   np.hstack([np.zeros((m, n + m)), np.identity(m)]),
                   np.zeros((m, n + 2 * m))])
    E = scipy.linalg.expm(M.T)
    Ad = E[:n, :n]
    Bd1 = E[n + m:, :n]
    Bd0 = E[n:n + m, :n] - Bd1
    return Ad, Bd0[0], Bd1[0], C[0], float(D[0, 0])


class CompiledConfig:
    """Holds the (mutable) parsed JSON configs, mirrors FixedWingAircraft's derived attributes and produces the POD."""

    def __init__(self, config_path=None, sim_config_path=None, sim_parameter_path=None, config_kw=None,
                 sim_config_kw=None, precision="fp64", metrics=False, scenario_bank=False, aircraft_parameters=()):
        config_path = config_path or DEFAULT_ENV_CONFIG
        with open(config_path) as f:
            self.cfg = json.load(f)
        if config_kw is not None:
            apply_overrides(self.cfg, copy.deepcopy(config_kw))
        sim_config_kw = dict(sim_config_kw or {})
        # the dict form of turbulence_intensity (per-env levels) replaces PyFly's string leaf instead of descending into it
        turb_mix = sim_config_kw.pop("turbulence_intensity") if isinstance(sim_config_kw.get("turbulence_intensity"),
                                                                         dict) else None
        sim_config_kw.update({"actuation": {"inputs": [a["name"] for a in self.cfg["action"]["states"]]}})
        sim_config_kw["turbulence_sim_length"] = self.cfg["steps_max"]
        with open(sim_config_path or DEFAULT_SIM_CONFIG) as f:
            self.sim_cfg = json.load(f)
        _set_sim_config_attrs(self.sim_cfg, copy.deepcopy(sim_config_kw))
        if turb_mix is not None:
            self.sim_cfg["turbulence_intensity"] = copy.deepcopy(turb_mix)
        with open(sim_parameter_path or DEFAULT_SIM_PARAMS) as f:
            self.params = {k: v for k, v in json.load(f).items() if not k.startswith("_")}
        self.precision = {"fp64": 0, "fp32": 1}[precision]
        self.metrics = bool(metrics)   # stream the get_metric quantities on the device (fixed_wing.py:1095-1162)
        self.scenario_bank = bool(scenario_bank)   # keep the scenario-bank rows (fw_set_bank)
        self.aircraft_parameters = tuple(aircraft_parameters or ())   # per-env aircraft rows (fw_set_aircraft)
        self.state = {v["name"]: SimVariable(v) for v in self.sim_cfg["variables"]}
        self.dt = self.sim_cfg["dt"]
        self._check_supported()
        self.steps_max = self.cfg["steps_max"]
        self.integration_window = self.cfg.get("integration_window", 0)
        self._build_spaces()
        self._rew_factors_init = copy.deepcopy(self.cfg["reward"]["factors"])
        self._curriculum_level = None
        self._target_props_init = None
        self.set_curriculum_level(1)

    # ------------------------------------------------------------------------------------------------ validation
    def _check_supported(self):
        if [a["name"] for a in self.cfg["action"]["states"]] != ACT_NAMES:
            raise ConfigError("action.states must be elevator, aileron, throttle (in this order)")
        act = self.sim_cfg["actuation"]
        if act["dynamics"] != ["elevon_left", "elevon_right", "throttle"]:
            raise ConfigError("only elevon dynamics [elevon_left, elevon_right, throttle] are supported")
        for n in ("roll", "pitch", "yaw"):
            v = self.state[n]
            if any(getattr(v, a) is not None for a in ("value_min", "value_max", "constraint_min", "constraint_max")):
                raise ConfigError("value limits / constraints on attitude state %s are not supported" % n)
        for n in ("position_n", "position_e", "position_d"):
            v = self.state[n]
            if any(getattr(v, a) is not None for a in ("value_min", "value_max", "constraint_min", "constraint_max")) or v.wrap:
                raise ConfigError("value limits / constraints on %s are not supported (position stage states are "
                                  "never formed in the integrator)" % n)
        self._rand_plan()   # raises on simulator-parameter randomisation entries the device path cannot honour
        if self.sim_cfg["turbulence"] and not self.cfg["steps_max"] > 0:
            raise ConfigError("turbulence needs steps_max > 0 (turbulence_sim_length = steps_max, fixed_wing.py:40)")
        self.turbulence_mix = self._turbulence_mix()
        self._check_aircraft()

    def _check_aircraft(self):
        names = self.aircraft_parameters
        for n in names:
            if n not in self.AIRCRAFT_PARAMS:
                raise ConfigError("aircraft_parameters: %r cannot differ per env (allowed: %s; ar is always b^2 / S_wing)"
                                  % (n, ", ".join(self.AIRCRAFT_PARAMS)))
        if len(set(names)) != len(names):
            raise ConfigError("aircraft_parameters: a name is listed twice in %r" % (names,))
        if not names:
            return
        if any(k != "states" for k in self.cfg["simulator"]):
            raise ConfigError("aircraft_parameters cannot be combined with simulator-parameter randomisation "
                              "(simulator.%s): the reference centres those draws on each aircraft's own values"
                              % next(k for k in self.cfg["simulator"] if k != "states"))
        if "b" in names and self.sim_cfg["turbulence"]:
            raise ConfigError("aircraft_parameters: a per-env wingspan b needs turbulence off (the Dryden filters are "
                              "built from b)")

    def _turbulence_mix(self):
        """sim_config_kw turbulence_intensity = {"values": [level names], "probabilities": [...]} (the reference's
        values / probabilities syntax for simulator attributes, fixed_wing.py:561-569; omitted probabilities are uniform,
        as np.random.choice) -> the probabilities of the four levels in TURB_LEVELS order; None for the string form."""
        spec = self.sim_cfg.get("turbulence_intensity")
        if not isinstance(spec, dict):
            return None
        if not self.sim_cfg["turbulence"]:
            raise ConfigError("turbulence_intensity {values, probabilities} needs turbulence: True")
        unknown = set(spec) - {"values", "probabilities"}
        if unknown or "values" not in spec:
            raise ConfigError("turbulence_intensity: expected {\"values\": [...], \"probabilities\": [...]}, got keys %s"
                              % sorted(spec))
        values = list(spec["values"])
        if not values:
            raise ConfigError("turbulence_intensity: values is empty")
        for v in values:
            if v not in TURB_LEVELS:
                raise ConfigError("turbulence_intensity: unknown level %r (levels: %s)" % (v, ", ".join(TURB_LEVELS)))
        if len(set(values)) != len(values):
            raise ConfigError("turbulence_intensity: a level is listed twice in %r" % (values,))
        probs = spec.get("probabilities")
        if probs is None:
            probs = [1.0 / len(values)] * len(values)
        probs = [float(p) for p in probs]
        if len(probs) != len(values):
            raise ConfigError("turbulence_intensity: %d values but %d probabilities" % (len(values), len(probs)))
        if any(not p >= 0 for p in probs):
            raise ConfigError("turbulence_intensity: negative probability in %r" % (probs,))
        if not abs(math.fsum(probs) - 1.0) <= 1e-12:
            raise ConfigError("turbulence_intensity: probabilities sum to %r, not 1" % math.fsum(probs))
        out = [0.0] * len(TURB_LEVELS)
        for v, p in zip(values, probs):
            out[TURB_LEVELS.index(v)] = p
        return out

    # --------------------------------------------------- fixed_wing.py:523-570 (sample_simulator_parameters) as a table
    LIVE_PARAMS = ("mass", "S_wing", "b", "c", "S_prop", "k_motor", "k_T_P", "k_Omega", "C_prop", "e", "M", "a_0", "ar",
                   "C_L_0", "C_L_alpha", "C_L_q", "C_L_delta_e", "C_D_p", "C_D_0", "C_D_alpha1", "C_D_alpha2",
                   "C_D_beta1", "C_D_beta2", "C_D_q", "C_D_delta_e", "C_m_0", "C_m_alpha", "C_m_q", "C_m_delta_e",
                   "C_m_fp", "C_Y_0", "C_Y_beta", "C_Y_p", "C_Y_r", "C_Y_delta_a", "C_Y_delta_r", "C_l_0", "C_l_beta",
                   "C_l_p", "C_l_r", "C_l_delta_a", "C_l_delta_r", "C_n_0", "C_n_beta", "C_n_p", "C_n_r",
                   "C_n_delta_a", "C_n_delta_r")
    SIM_ATTRS = ("rho", "g")     # PyFly attributes the right-hand side reads at every evaluation
    INERTIA = ("Jx", "Jy", "Jz", "Jxz")
    # what FixedWingVecEnv(aircraft_parameters=) may set per env (include/fwgym.h fw_air)
    AIRCRAFT_PARAMS = tuple(n for n in LIVE_PARAMS if n != "ar") + SIM_ATTRS + INERTIA

    def air_id(self, name):
        """aircraft parameter name -> its id (fw_air: a fw_par id, or FW_AIR_JX.. for the inertia)"""
        if name in self.INERTIA:
            return _capi.ENUMS["FW_AIR_JX"] + self.INERTIA.index(name)
        return self.par_id(name)

    def aircraft_nominal(self):
        """name -> the handle's value of every listed aircraft parameter (what a NaN request flies)"""
        return {n: float(self.sim_cfg[n] if n in self.SIM_ATTRS else self.params[n]) for n in self.aircraft_parameters}

    @staticmethod
    def par_id(name):
        """model parameter / simulator attribute name -> fw_par id (include/fwgym.h)"""
        key = "C_L_ROLL_" + name[4:].upper() if name.startswith("C_l_") else name.upper()
        return _capi.ENUMS["FW_PAR_" + key]

    def _rand_plan(self):
        """The draws FixedWingAircraft.sample_simulator_parameters makes at every reset, in its order: one entry per
        draw = dict(name, par (fw_par id or -1), dist, orig, var, clip).  Entries whose parameter the dynamics never
        read (inertia: PyFly folds it into gammas at construction) keep their draw and have par -1."""
        plan = []
        params = dict(self.params)
        params["ar"] = params["b"] ** 2 / params["S_wing"]
        for key, value in self.cfg["simulator"].items():
            if key == "states":
                continue
            if key == "model":
                dist_type = value.get("distribution", "gaussian")
                if dist_type not in ("gaussian", "uniform"):
                    raise ConfigError("Unexpected distribution type {}".format(dist_type))
                for pa in value["parameters"]:
                    name = pa["name"]
                    if name not in params:
                        raise ConfigError("simulator.model: unknown parameter %r" % name)
                    orig = pa.get("original", None)
                    if orig is None:
                        orig = params[name]
                    if orig == 0:
                        continue        # fixed_wing.py:541-542: no draw at all
                    var = pa.get("var", value["var"])
                    rel = value["var_type"] == "relative"
                    if rel:
                        var = var * abs(orig)
                    clip = pa.get("clip", value.get("clip", None)) if dist_type == "gaussian" else None
                    if clip is not None and rel:
                        clip = clip * orig        # signed, as the reference (:550)
                    plan.append(dict(name=name, par=self.par_id(name) if name in self.LIVE_PARAMS else -1,
                                     dist=0 if dist_type == "gaussian" else 1, orig=float(orig), var=float(var),
                                     clip=clip))
            else:
                if key not in self.SIM_ATTRS:
                    raise ConfigError("simulator.%s randomisation is not supported: only the model parameters and the "
                                      "simulator attributes %s reach the dynamics" % (key, ", ".join(self.SIM_ATTRS)))
                if "values" in value or isinstance(value["low"], bool):
                    raise ConfigError("simulator.%s: only low/high (uniform) ranges are supported" % key)
                plan.append(dict(name=key, par=self.par_id(key), dist=2, orig=float(value["low"]),
                                 var=float(value["high"]), clip=None))
        if len(plan) > _capi.DEFINES["FW_MAX_RAND"]:
            raise ConfigError("more than %d randomised simulator parameters" % _capi.DEFINES["FW_MAX_RAND"])
        return plan

    def _rand_slots(self):
        """-> (plan, slot1 of every fw_par id, number of per-env parameter rows).  A parameter drawn twice keeps one
        row (the last draw wins, as the reference's dict assignment); derived rows follow the drawn ones.  Aircraft
        parameters (never together with a draw) take rows in their listed order, then ar when b or S_wing is listed,
        then the derived rows, and the FW_N_INERTIA inertia rows last (inertia_slots)."""
        plan = self._rand_plan()
        slot1 = [0] * _capi.ENUMS["FW_PAR_N"]
        n = 0
        for ent in plan:
            if ent["par"] >= 0 and not slot1[ent["par"]]:
                n += 1
                slot1[ent["par"]] = n
        E = _capi.ENUMS
        for name in self.aircraft_parameters:
            if name not in self.INERTIA:
                n += 1
                slot1[self.par_id(name)] = n
        if self.aircraft_parameters and (slot1[E["FW_PAR_B"]] or slot1[E["FW_PAR_S_WING"]]):
            n += 1
            slot1[E["FW_PAR_AR"]] = n
        for derived, sources in ((E["FW_PAR_INV_MASS"], ("MASS",)), (E["FW_PAR_INV_PI_E_AR"], ("E", "AR")),
                                 (E["FW_PAR_EXP_2MA0"], ("M", "A_0"))):
            if any(slot1[E["FW_PAR_" + s_]] for s_ in sources):
                n += 1
                slot1[derived] = n
        if any(name in self.INERTIA for name in self.aircraft_parameters):
            n += _capi.DEFINES["FW_N_INERTIA"]
        return plan, slot1, n

    def inertia_slots(self):
        """slot1 of gammas[1..8], inv_Jy (fw_sim_t.inertia_slot1): the last FW_N_INERTIA parameter rows when an inertia
        entry is an aircraft parameter, else all 0."""
        k = _capi.DEFINES["FW_N_INERTIA"]
        if not any(name in self.INERTIA for name in self.aircraft_parameters):
            return [0] * k
        n = self._rand_slots()[2]
        return list(range(n - k + 1, n + 1))

    # ------------------------------------------------------------------------- fixed_wing.py:57-191 (spaces etc.)
    def _limit(self, state_name, side):
        """Bound of a simulator state for the spaces: its value limit, else its constraint, else +-float32 max."""
        st = self.state[state_name]
        for attr in ("value_" + side, "constraint_" + side):
            if getattr(st, attr) is not None:
                return getattr(st, attr)
        return F32_MAX if side == "max" else -F32_MAX

    def _observation_bounds(self, var):
        """(low, high) of one observation variable: the configured numbers (degrees converted when asked) or the state's
        limits; a relative target value spans the difference of the two."""
        rad = var.get("convert_to_radians", False)
        ends = {}
        for key, side in (("high", "max"), ("low", "min")):
            given = var.get(key, None)
            ends[key] = self._limit(var["name"], side) if given is None else (np.radians(given) if rad else given)
        low, high = ends["low"], ends["high"]
        bounded = high != F32_MAX and low != -F32_MAX
        if self.obs_norm:       # defaults of the normalisation constants are written back into the config (:101-105)
            if var.get("mean", None) is None:
                var["mean"] = high - low if bounded else 0
            if var.get("var", None) is None:
                var["var"] = (high - low) / (4 ** 2) if bounded else 1
        if var["type"] == "target" and var["value"] == "relative":
            return (low - high, high - low) if bounded else (-F32_MAX, F32_MAX)
        return low, high

    def _build_spaces(self):
        ocfg, acfg = self.cfg["observation"], self.cfg["action"]
        self.obs_norm = ocfg.get("normalize", False)
        bounds = [self._observation_bounds(var) for var in ocfg["states"]]
        row_low, row_high = [b[0] for b in bounds], [b[1] for b in bounds]
        if ocfg["length"] > 1:
            if ocfg["shape"] not in ("vector", "matrix"):
                raise ConfigError("observation.shape must be vector or matrix")
            tile = (lambda r: r * ocfg["length"]) if ocfg["shape"] == "vector" else (lambda r: [r] * ocfg["length"])
            row_low, row_high = tile(row_low), tile(row_high)
        self.observation_low = np.array(row_low, dtype=np.float64)
        self.observation_high = np.array(row_high, dtype=np.float64)

        names = [av["name"] for av in acfg["states"]]
        to_low = [self._limit(n, "min") for n in names]
        to_high = [self._limit(n, "max") for n in names]

        def space_end(av, key, fallback, unbounded):     # "max": no bound; null: the actuator's own limit; else the number
            v = av.get(key, None)
            return unbounded if v == "max" else (fallback if v is None else v)
        self.action_scale_to_low = np.array(to_low, dtype=np.float64)
        self.action_scale_to_high = np.array(to_high, dtype=np.float64)
        self.action_space_low = np.array([space_end(av, "low", lo, -F32_MAX) for av, lo in zip(acfg["states"], to_low)],
                                         dtype=np.float64)
        self.action_space_high = np.array([space_end(av, "high", hi, F32_MAX) for av, hi in zip(acfg["states"], to_high)],
                                          dtype=np.float64)
        self.scale_actions = acfg.get("scale_space", False)
        self.action_bounds_max = self.action_bounds_min = None
        mult = acfg.get("bounds_multiplier", None)
        if mult is not None:
            self.action_bounds_max = np.full(3, acfg.get("scale_high", 1)) * mult
            self.action_bounds_min = np.full(3, acfg.get("scale_low", -1)) * mult
        self.goal_enabled = self.cfg["target"]["success_streak_req"] > 0
        self._bounded_targets = {t["name"] for t in self.cfg["target"]["states"] if t.get("bound", None) is not None}

    # ------------------------------------------------------------------------------------ fixed_wing.py:224-285
    def goal_has_bound(self, target_name):
        """Is this target state part of the goal status (fixed_wing.py:916-931: only states with a bound are)?"""
        return target_name in self._bounded_targets

    def set_curriculum_level(self, level):
        """fixed_wing.py:224-285: `level` in [0, 1] shrinks every configured RANGE towards its midpoint - the init / value
        ranges of the simulator states listed under simulator.states and the target sampling ranges - and picks
        list-valued target settings by level."""
        assert 0 <= level <= 1
        self._curriculum_level = level
        for name, prop, value in self._curriculum_state_limits(level):
            setattr(self.state[name], prop, value)
        self._target_props_init = self._curriculum_targets(level)

    @staticmethod
    def _towards(mid, end, level):
        return mid - level * (mid - end)

    def _curriculum_state_limits(self, level):
        """-> [(state name, property, value)]: every property of every simulator.states entry, as the reference assigns
        them (:233-245).  A property whose name contains min / max and not "constraint" is the end of a range whose other
        end is the sibling property with the same stem; nulls pass through; degrees are converted after scaling."""
        out = []
        for entry in self.cfg["simulator"].get("states", ()):
            spec = {k: v for k, v in entry.items() if k not in ("name", "convert_to_radians")}
            to_rad = entry.get("convert_to_radians", False)
            for prop, val in spec.items():
                if val is not None:
                    if "constraint" not in prop and ("min" in prop or "max" in prop):
                        stem = prop[:-3]
                        val = self._towards((spec[stem + "max"] + spec[stem + "min"]) / 2, val, level)
                    if to_rad:
                        val = np.radians(val)
                out.append((entry["name"], prop, val))
        return out

    def _curriculum_targets(self, level):
        """-> the target properties sample_target reads (:247-265).  Per target state: low / high move towards the
        midpoint of the configured range, every other number (delta, slopes, amplitudes, periods) towards zero; bound,
        class, booleans and nulls are kept.  Other target settings: a list is indexed by round(len * level)."""
        props = {"states": {}}
        for key, val in self.cfg["target"].items():
            if key != "states":
                props[key] = val[round(len(val) * level)] if isinstance(val, list) else val
        for st in self.cfg["target"]["states"]:
            scaled = {}
            for key, val in st.items():
                if key == "name":
                    continue
                if key not in ("bound", "class") and val is not None and not isinstance(val, bool):
                    mid = (st["high"] + val) / 2 if key == "low" else ((val + st["low"]) / 2 if key == "high" else 0)
                    val = self._towards(mid, val, level)
                scaled[key] = val
            props["states"][st["name"]] = scaled
        return props

    # -------------------------------------------------------------------------------------------------- to POD
    @property
    def obs_dim(self):
        return self.cfg["observation"]["length"] * len(self.cfg["observation"]["states"])

    @property
    def obs_shape(self):
        o = self.cfg["observation"]
        n = len(o["states"])
        if o["length"] > 1 and o["shape"] == "matrix":
            return (o["length"], n)
        return (o["length"] * n,)

    def pod(self):
        c = _capi.fw_config_t()
        c.abi_version = _capi.DEFINES["FW_ABI_VERSION"]
        c.precision = self.precision
        self._fill_sim(c.sim)
        self._fill_env(c.env)
        return c

    def _fill_sim(self, s):
        P, sc = self.params, self.sim_cfg
        s.dt, s.rho, s.g = sc["dt"], sc["rho"], sc["g"]
        s.rtol, s.atol = 1e-3, 1e-6
        for k in ("mass", "S_wing", "b", "c", "S_prop", "k_motor", "k_T_P", "k_Omega", "C_prop", "e", "M", "a_0",
                  "C_L_0", "C_L_alpha", "C_L_q", "C_L_delta_e", "C_D_p", "C_D_0", "C_D_alpha1", "C_D_alpha2",
                  "C_D_beta1", "C_D_beta2", "C_D_q", "C_D_delta_e", "C_m_0", "C_m_alpha", "C_m_q", "C_m_delta_e",
                  "C_m_fp", "C_Y_0", "C_Y_beta", "C_Y_p", "C_Y_r", "C_Y_delta_a", "C_Y_delta_r", "C_l_0", "C_l_beta",
                  "C_l_p", "C_l_r", "C_l_delta_a", "C_l_delta_r", "C_n_0", "C_n_beta", "C_n_p", "C_n_r",
                  "C_n_delta_a", "C_n_delta_r"):
            setattr(s, k, float(P[k]))
        s.ar = P["b"] ** 2 / P["S_wing"]
        I = np.array([[P["Jx"], 0, -P["Jxz"]], [0, P["Jy"], 0], [-P["Jxz"], 0, P["Jz"]]])
        g0 = I[0, 0] * I[2, 2] - I[0, 2] ** 2
        gam = [g0, (np.abs(I[0, 2]) * (I[0, 0] - I[1, 1] + I[2, 2])) / g0,
               (I[2, 2] * (I[2, 2] - I[1, 1]) + I[0, 2] ** 2) / g0, I[2, 2] / g0, np.abs(I[0, 2]) / g0,
               (I[2, 2] - I[0, 0]) / I[1, 1], I[0, 2] / I[1, 1],
               ((I[0, 0] - I[1, 1]) * I[0, 0] + I[0, 2] ** 2) / g0, I[0, 0] / g0]
        for i, v in enumerate(gam):
            s.gammas[i] = float(v)
        s.Jy = float(I[1, 1])
        s.inv_Jy = 1.0 / float(I[1, 1])
        s.inv_mass = 1.0 / float(P["mass"])
        s.inv_pi_e_ar = 1.0 / (np.pi * P["e"] * s.ar)
        s.exp_2Ma0 = float(np.exp(2.0 * P["M"] * P["a_0"]))
        s.drag_model = {"induced": 0, "polynomial": 1}[sc.get("drag_model", "induced")]
        s.turbulence = 1 if sc["turbulence"] else 0
        s.max_attempts = int(sc.get("dopri5_max_attempts", 0) or 0)   # opt-in, not a PyFly key: 0 = the reference's behaviour
        s.wind_mag_min, s.wind_mag_max = sc["wind_magnitude_min"], sc["wind_magnitude_max"]
        s.wind_enabled = 1 if (sc["wind_magnitude_max"] != 0 or sc["wind_magnitude_min"] != 0
                               or sc.get("allow_wind_injection", False)) else 0
        s.turb_noise_scale = math.sqrt(math.pi / sc["dt"])
        if sc["turbulence"] and self.turbulence_mix is not None:
            self._fill_turbulence_mix(s, P, sc)
        elif sc["turbulence"]:
            length = sc.get("turbulence_sim_length", 250)
            # PyFly simulates `length` samples on t = linspace(0, length*dt, length): spacing length*dt/(length-1)
            dt_eff = float(np.diff(np.linspace(0, length * sc["dt"], length))[0]) if length > 1 else sc["dt"]
            for i, (num, den, stream) in enumerate(dryden_transfer_functions(P["b"], sc["turbulence_intensity"])):
                Ad, Bd0, Bd1, C, D = discretise_filter(num, den, dt_eff)
                f = s.filt[i]
                f.n, f.stream = Ad.shape[0], stream
                for a in range(f.n):
                    for b_ in range(f.n):
                        f.Ad[a * 3 + b_] = float(Ad[a, b_])
                    f.Bd0[a], f.Bd1[a], f.C[a] = float(Bd0[a]), float(Bd1[a]), float(C[a])
                f.D = D
        for name, var in self.state.items():
            v = s.var[_capi.sv_id(name)]
            flags = 0
            for attr, bit in (("value_min", "FW_VC_VMIN"), ("value_max", "FW_VC_VMAX"),
                              ("constraint_min", "FW_VC_CMIN"), ("constraint_max", "FW_VC_CMAX")):
                val = getattr(var, attr)
                if val is not None:
                    flags |= _capi.DEFINES[bit]
                    setattr(v, {"value_min": "vmin", "value_max": "vmax", "constraint_min": "cmin",
                                "constraint_max": "cmax"}[attr], float(val))
            v.lo = float(var.value_min) if var.value_min is not None else -math.inf
            v.hi = float(var.value_max) if var.value_max is not None else math.inf
            v.clo = float(var.constraint_min) if var.constraint_min is not None else -math.inf
            v.chi = float(var.constraint_max) if var.constraint_max is not None else math.inf
            if var.wrap:
                if name not in ("roll", "yaw", "pitch"):
                    raise ConfigError("wrap is only supported on attitude angles, not %s" % name)
                flags |= _capi.DEFINES["FW_VC_WRAP"]
            v.flags = flags
            v.init_min = float(var.init_min) if var.init_min is not None else 0.0
            v.init_max = float(var.init_max) if var.init_max is not None else 0.0
        for i, name in enumerate(sc["actuation"]["dynamics"]):
            var = self.state[name]
            co = var.coefs
            for j in range(3):
                s.act_coef[i][j] = float(co[0][j])
                s.act_coef[i][3 + j] = float(co[1][j])
            s.act_has_dot_max[i] = 1 if var.dot_max is not None else 0
            s.act_dot_max[i] = float(var.dot_max) if var.dot_max is not None else 0.0
        a = self.cfg["action"]
        s.scale_actions = 1 if self.scale_actions else 0
        s.has_scale_low = 1 if a.get("scale_low") is not None else 0
        s.has_scale_high = 1 if a.get("scale_high") is not None else 0
        s.scale_low = float(a.get("scale_low")) if a.get("scale_low") is not None else 0.0
        s.scale_high = float(a.get("scale_high")) if a.get("scale_high") is not None else 0.0
        if self.scale_actions and not (s.has_scale_low and s.has_scale_high):
            raise ConfigError("action.scale_space needs scale_low and scale_high")
        for j in range(3):
            s.act_to_low[j] = float(self.action_scale_to_low[j])
            s.act_to_high[j] = float(self.action_scale_to_high[j])
        _, slot1, _ = self._rand_slots()
        for i, v in enumerate(slot1):
            s.par_slot1[i] = v
        if self.aircraft_parameters:
            s.Jx, s.Jz, s.Jxz = float(P["Jx"]), float(P["Jz"]), float(P["Jxz"])
            for j, name in enumerate(self.aircraft_parameters):
                s.air_id[j] = self.air_id(name)
            for k, v in enumerate(self.inertia_slots()):
                s.inertia_slot1[k] = v

    @staticmethod
    def turbulence_dt(sc):
        """The sample spacing of PyFly's Dryden simulation: `length` samples on t = linspace(0, length*dt, length)."""
        length = sc.get("turbulence_sim_length", 250)
        return float(np.diff(np.linspace(0, length * sc["dt"], length))[0]) if length > 1 else sc["dt"]

    @staticmethod
    def compile_turbulence_levels(b, dt):
        """(Ad, Bd0, Bd1, C, D, stream) of the six shaping filters for light, moderate and severe.  The intensity enters
        only through the numerators, so Ad / Bd0 / Bd1 (built from the denominators) must come out bitwise equal across
        the levels: one filter state then serves every level and only the output rows C / D are per level."""
        out = {}
        for lvl in TURB_LEVELS[1:]:
            out[lvl] = [discretise_filter(num, den, dt) + (stream,)
                        for num, den, stream in dryden_transfer_functions(b, lvl)]
        ref = out[TURB_LEVELS[1]]
        for lvl in TURB_LEVELS[2:]:
            for f, (a, b_) in enumerate(zip(ref, out[lvl])):
                for k in range(3):
                    if np.asarray(a[k]).tobytes() != np.asarray(b_[k]).tobytes():
                        raise ConfigError("Dryden filter %d: the state matrices of %s and %s differ; per-env intensities "
                                          "need them equal" % (f, TURB_LEVELS[1], lvl))
        return out

    def _fill_turbulence_mix(self, s, P, sc):
        """Mixed handle: filt[] holds the shared Ad / Bd0 / Bd1 (its C / D stay zero: the kernels read turb_C / turb_D of
        the episode's level), turb_C / turb_D one row per level (level 0, none, all zero) and turb_cdf the draw table."""
        levels = self.compile_turbulence_levels(P["b"], self.turbulence_dt(sc))
        s.turb_mixed = 1
        for i, (Ad, Bd0, Bd1, _C, _D, stream) in enumerate(levels[TURB_LEVELS[1]]):
            f = s.filt[i]
            f.n, f.stream = Ad.shape[0], stream
            for a in range(f.n):
                for b_ in range(f.n):
                    f.Ad[a * 3 + b_] = float(Ad[a, b_])
                f.Bd0[a], f.Bd1[a] = float(Bd0[a]), float(Bd1[a])
        for li, lvl in enumerate(TURB_LEVELS[1:], start=1):
            for i, (_Ad, _Bd0, _Bd1, C, D, _stream) in enumerate(levels[lvl]):
                for a in range(len(C)):
                    s.turb_C[li][i][a] = float(C[a])
                s.turb_D[li][i] = D
        for li, c in enumerate(turbulence_cdf(self.turbulence_mix)):
            s.turb_cdf[li] = c

    def _fill_env(self, e):
        cfg = self.cfg
        o = cfg["observation"]
        e.steps_max = int(cfg["steps_max"])
        e.integration_window = int(self.integration_window)
        e.obs_len, e.obs_step = int(o["length"]), int(o.get("step", 1))
        e.obs_nvar = len(o["states"])
        if e.obs_nvar > _capi.DEFINES["FW_MAX_OBS_VARS"]:
            raise ConfigError("too many observation variables")
        e.obs_shape = {"vector": 0, "matrix": 1}[o["shape"]]
        e.obs_norm = 1 if self.obs_norm else 0
        noise = o.get("noise", None)
        e.obs_noise = 1 if noise is not None else 0
        if noise is not None:
            e.obs_noise_mean, e.obs_noise_std = float(noise["mean"]), float(noise["var"])   # "var" is used as a std
        tnames = list(self._target_props_init["states"].keys())
        for i, ov in enumerate(o["states"]):
            v = e.obs[i]
            v.type = {"state": 0, "target": 1, "action": 2}[ov["type"]]
            if ov["type"] == "state":
                v.ref = _capi.sv_id(ov["name"])
            elif ov["type"] == "target":
                v.ref = tnames.index(ov["name"])
                v.value_kind = {"relative": 0, "absolute": 1, "integrator": 2}[ov["value"]]
            else:
                v.ref = ACT_NAMES.index(ov["name"])
                v.window = int(ov.get("window_size", 1))
                if v.window > 9:
                    raise ConfigError("action observation window_size > 9 not supported (float32 pairwise order)")
            v.norm = 1 if ov.get("norm", True) else 0
            if self.obs_norm and v.norm:
                v.mean, v.var = float(ov["mean"]), float(ov["var"])
        if self.action_bounds_max is not None:
            e.has_bounds = 1
            for j in range(3):
                e.bounds_min[j], e.bounds_max[j] = float(self.action_bounds_min[j]), float(self.action_bounds_max[j])
        tp = self._target_props_init
        e.n_targets = len(tnames)
        if e.n_targets > _capi.DEFINES["FW_MAX_TARGETS"]:
            raise ConfigError("at most %d target states are supported" % _capi.DEFINES["FW_MAX_TARGETS"])
        e.resample_every = int(tp.get("resample_every", 0) or 0)
        e.streak_req = int(tp["success_streak_req"])
        e.streak_fraction = float(tp["success_streak_fraction"])
        e.on_success = {"none": 0, "done": 1, "new": 2}[tp["on_success"]]
        for k, name in enumerate(tnames):
            props, t = tp["states"][name], e.tgt[k]
            cls = props.get("class", "constant")
            if cls not in TCLASS:
                raise ConfigError("target class %r is not supported" % cls)
            if cls == "compensate" and name != "Va":
                raise ConfigError("target class compensate is only defined for Va (fixed_wing.py:944-976)")
            t.sv, t.cls = _capi.sv_id(name), TCLASS[cls]
            t.wrap = 1 if self.state[name].wrap else 0
            rad = bool(props.get("convert_to_radians", False))
            t.to_radians = 1 if rad else 0
            conv = (lambda x: float(np.radians(x))) if rad else float
            t.low, t.high = conv(props["low"]), conv(props["high"])
            if props.get("delta", None) is not None:
                t.has_delta, t.delta = 1, conv(props["delta"])
            if props.get("bound", None) is not None:
                t.has_bound, t.bound = 1, conv(props["bound"])
            if cls == "linear":
                t.slope_low, t.slope_high = float(props["slope_low"]), float(props["slope_high"])
            if cls == "sinusoidal":
                t.amp_low, t.amp_high = float(props["amplitude_low"]), float(props["amplitude_high"])
                t.period_low, t.period_high = float(props.get("period_low", 250)), float(props.get("period_high", 500))
        r = cfg["reward"]
        e.potential = 1 if r.get("form", "absolute") == "potential" else 0
        sf = r.get("step_fail", 0)
        e.step_fail_timesteps = 1 if sf == "timesteps" else 0
        e.step_fail_value = 0.0 if sf == "timesteps" else float(sf)
        plan, slot1, n_rows = self._rand_slots()
        e.n_rand, e.n_par_rows = len(plan), n_rows
        for j, ent in enumerate(plan):
            rd = e.rand[j]
            rd.par, rd.dist = ent["par"], ent["dist"]
            rd.slot1 = slot1[ent["par"]] if ent["par"] >= 0 else 0
            rd.orig, rd.var = ent["orig"], ent["var"]
            rd.has_clip = 1 if ent["clip"] is not None else 0
            rd.clip = float(ent["clip"]) if ent["clip"] is not None else 0.0
        e.metrics_enabled = 1 if self.metrics else 0
        e.rise_low, e.rise_high = 0.1, 0.9          # get_metric defaults (fixed_wing.py:1131)
        for m in cfg.get("metrics", []):
            if m.get("name") == "rise_time":
                e.rise_low, e.rise_high = float(m.get("low", 0.1)), float(m.get("high", 0.9))
        e.n_terms = len(r["terms"])
        seen = set()
        for i, term in enumerate(r["terms"]):
            fc = FCLASS[term["function_class"]]
            if fc in seen:
                raise ConfigError("duplicate reward term function_class")
            seen.add(fc)
            e.term_fclass[i], e.term_weight[i] = fc, float(term["weight"])
        e.n_factors = len(r["factors"])
        if e.n_factors > _capi.DEFINES["FW_MAX_FACTORS"]:
            raise ConfigError("too many reward factors")
        n_scale = 0
        for i, comp in enumerate(r["factors"]):
            F = e.fac[i]
            F.cls = {"action": 0, "state": 1, "success": 2, "step": 3, "goal": 4}[comp["class"]]
            F.fclass = FCLASS[comp["function_class"]]
            if F.fclass not in seen:
                raise ConfigError("reward factor %s uses function_class without a term" % comp.get("name"))
            if comp["class"] == "action":
                F.type = {"value": 0, "delta": 1, "bound": 2}[comp["type"]]
                if comp["type"] == "delta":
                    if comp["name"] != "action":
                        raise ConfigError("action delta reward must be named 'action' (fixed_wing.py:689)")
                    F.window = int(comp["window_size"])
                if comp["type"] == "bound" and self.action_bounds_max is None:
                    raise ConfigError("action bound reward needs action.bounds_multiplier")
            elif comp["class"] == "state":
                F.type = {"value": 0, "error": 1, "int_error": 2}[comp["type"]]
                F.ref = _capi.sv_id(comp["name"]) if comp["type"] == "value" else tnames.index(comp["name"])
            elif comp["class"] == "success":
                if comp["value"] == "timesteps":
                    F.value_timesteps = 1
                else:
                    F.value = float(comp["value"])
            elif comp["class"] == "step":
                F.value = float(comp["value"])
            elif comp["class"] == "goal":
                F.type = {"per_state": 0, "all": 1}[comp["type"]]
                F.value = float(comp["value"])
            init_scaling = self._rew_factors_init[i]["scaling"]
            if isinstance(init_scaling, list):
                # reward.randomize_scaling (fixed_wing.py:330-334): U(low, high) per reset into a per-env row
                if not r.get("randomize_scaling", False):
                    raise ConfigError("reward factor %s: scaling [low, high] needs reward.randomize_scaling" % comp.get("name"))
                n_scale += 1
                F.scale_slot1, F.scale_low, F.scale_high = n_scale, float(init_scaling[0]), float(init_scaling[1])
                F.scaling = 1.0
            else:
                F.scaling = float(comp["scaling"])
            F.shaping = 1 if comp.get("shaping", False) else 0
            if comp.get("max", None) is not None:
                F.has_max, F.max = 1, float(comp["max"])
            F.sign = float(np.sign(comp.get("sign", -1)))
        e.n_scale_rows = n_scale
        e.bank_enabled = 1 if self.scenario_bank else 0
        e.n_aircraft = len(self.aircraft_parameters)
