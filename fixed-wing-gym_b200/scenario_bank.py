"""Scenario banks (include/fwgym.h fw_bank_t): the host half - table building and validation, and a numpy mirror of
the rule by which envs take scenarios.

A bank is S scenarios of initial states and targets (NaN = sample it), optionally a Dryden level and an aircraft each.  Resets of a
handle created with scenario_bank=True consume them in order on the device: env e flies first + e, then
first + e + stride, first + e + 2 stride, ... (modulo S when cycling), and the env kernel writes each scenario's outcome
into a row of its own.
"""
import numpy as np

from . import _capi
from .config import TURB_LEVELS

N_INIT_ROWS = _capi.DEFINES["FW_N_SV"] + 3
WIND_KEYS = ("wind_n", "wind_e", "wind_d")
INT32_MAX = 2 ** 31 - 1


def state_row(name):
    """reset(state=) / bank name -> row of the init_state table (PyFly state variables, then the steady wind n, e, d)."""
    if name in WIND_KEYS:
        return _capi.DEFINES["FW_N_SV"] + WIND_KEYS.index(name)
    if name in _capi.SV_NAMES:
        return _capi.sv_id(name)
    raise ValueError("unknown state name %r (PyFly state variables, wind, wind_n / wind_e / wind_d)" % name)


def _column(val, what):
    v = np.asarray(val, dtype=np.float64)
    if v.ndim > 1:
        raise ValueError("%s: one value per scenario expected, got shape %s" % (what, v.shape))
    return v


def level_codes(levels):
    """Level names or ints (-1 = the env's own rule, 0..3 = none, light, moderate, severe) -> int32 array."""
    out = []
    for x in np.atleast_1d(np.asarray(levels, dtype=object)):
        if isinstance(x, str):
            if x not in TURB_LEVELS:
                raise ValueError("unknown turbulence level %r (levels: %s)" % (x, ", ".join(TURB_LEVELS)))
            out.append(TURB_LEVELS.index(x))
        elif isinstance(x, (bool, np.bool_)) or not float(x).is_integer() or not -1 <= int(x) <= 3:
            raise ValueError("turbulence levels must be names or integers -1..3, got %r" % (x,))
        else:
            out.append(int(x))
    return np.asarray(out, dtype=np.int32)


def build_tables(state=None, target=None, turbulence_intensity=None, target_names=(), mixed=False):
    """-> (S, init_state [N_INIT_ROWS, S] or None, init_target [FW_MAX_TARGETS, S] or None, levels [S] int32 or None):
    build_bank_tables without an aircraft column."""
    return build_bank_tables(state, target, turbulence_intensity, target_names, mixed)[:4]


def build_bank_tables(state=None, target=None, turbulence_intensity=None, target_names=(), mixed=False, aircraft=None,
                      aircraft_parameters=()):
    """-> (S, init_state [N_INIT_ROWS, S] or None, init_target [FW_MAX_TARGETS, S] or None, levels [S] int32 or None,
    aircraft [len(aircraft_parameters), S] or None).

    `state` / `target`: dicts name -> one value per scenario (a scalar applies to every scenario), with the names
    reset(state=, target=) takes; "wind" is a [3, S] (or [3]) entry.  `turbulence_intensity`: one level per scenario
    (mixed handles only).  `aircraft`: dict name -> one value per scenario of the handle's `aircraft_parameters` (NaN =
    the env's own request).  S is the length of the per-scenario entries, which must all agree."""
    cols = []          # (table, row, values)
    for name, val in dict(state or {}).items():
        if name == "wind":
            w = np.asarray(val, dtype=np.float64)
            if w.shape[:1] != (3,) or w.ndim > 2:
                raise ValueError("state 'wind' must be [3] or [3, S]")
            for k in range(3):
                cols.append(("state", state_row(WIND_KEYS[k]), w[k], "wind"))
        else:
            cols.append(("state", state_row(name), _column(val, name), name))
    target_names = list(target_names)
    for name, val in dict(target or {}).items():
        if name not in target_names:
            raise ValueError("unknown target %r (targets of this configuration: %s)" % (name, ", ".join(target_names)))
        cols.append(("target", target_names.index(name), _column(val, name), name))
    aircraft_parameters = tuple(aircraft_parameters)
    if aircraft is not None and not aircraft_parameters:
        raise ValueError("an aircraft column needs a handle with aircraft_parameters")
    for name, val in dict(aircraft or {}).items():
        if name not in aircraft_parameters:
            raise ValueError("%r is not an aircraft parameter of this env (aircraft_parameters: %s)"
                             % (name, ", ".join(aircraft_parameters)))
        cols.append(("aircraft", aircraft_parameters.index(name), _column(val, name), name))
    levels = None
    if turbulence_intensity is not None:
        if not mixed:
            raise ValueError("a per-scenario turbulence level needs per-env levels: configure turbulence_intensity as "
                             "{\"values\": [...], \"probabilities\": [...]}")
        levels = level_codes(turbulence_intensity)
    lens = {len(v) for _, _, v, _ in cols if v.ndim == 1}
    if levels is not None and levels.shape[0] != 1:
        lens.add(levels.shape[0])
    if not lens:
        raise ValueError("a scenario bank needs at least one per-scenario entry (an array over the scenarios)")
    if len(lens) != 1:
        raise ValueError("per-scenario entries of different lengths: %s" % sorted(lens))
    S = lens.pop()
    if S < 1 or S > INT32_MAX:
        raise ValueError("a bank holds 1 .. 2^31 - 1 scenarios, not %d" % S)
    init_state = init_target = air = None
    for table, row, v, _ in cols:
        if table == "state":
            if init_state is None:
                init_state = np.full((N_INIT_ROWS, S), np.nan)
            init_state[row] = v
        elif table == "aircraft":
            if air is None:
                air = np.full((len(aircraft_parameters), S), np.nan)
            air[row] = v
        else:
            if init_target is None:
                init_target = np.full((_capi.DEFINES["FW_MAX_TARGETS"], S), np.nan)
            init_target[row] = v
    if levels is not None and levels.shape[0] == 1:
        levels = np.full(S, levels[0], dtype=np.int32)
    return S, init_state, init_target, levels, air


def check_assignment(n_envs, n_scenarios, first, stride):
    """The argument rules fw_set_bank enforces, raised as ValueError before anything reaches the device."""
    if first < 0:
        raise ValueError("first must be >= 0")
    if stride < n_envs:
        raise ValueError("stride (%d) < number of envs (%d): two envs could fly one scenario" % (stride, n_envs))
    if n_scenarios < 1 or n_scenarios > INT32_MAX:
        raise ValueError("a bank holds 1 .. 2^31 - 1 scenarios")


def advance(cur, n_scenarios, stride, cycle):
    """The device's cursor step (csrc/env.cuh fw_bank_advance): + stride, modulo S when cycling, else saturating at S."""
    nx = np.asarray(cur, dtype=np.int64) + int(stride)
    return nx % n_scenarios if cycle else np.minimum(nx, n_scenarios)


def attach_cursor(n_envs, n_scenarios, first, cycle):
    """bank_next right after attaching (fw_set_bank): first + e, modulo S when cycling, else at most S."""
    c = int(first) + np.arange(n_envs, dtype=np.int64)
    return c % n_scenarios if cycle else np.minimum(c, n_scenarios)


def scenario_of(env, k, n_scenarios, first, stride, cycle):
    """Scenario of the k-th banked episode (k = 0, 1, ...) of local env `env`, -1 once the env is past the bank."""
    s = int(first) + np.asarray(env, dtype=np.int64) + np.asarray(k, dtype=np.int64) * int(stride)
    if cycle:
        return s % n_scenarios
    return np.where(s < n_scenarios, s, -1)
