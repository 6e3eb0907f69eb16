"""Per-env aircraft on the GPU (include/fwgym.h fw_set_aircraft): env e flies the aircraft a reference env built from a
parameter file with its values would fly.

The tests hold (1) a handle whose every aircraft parameter is pinned to its nominal value to the same handle with NaN
requests, bitwise; (2) the rows the reset derives (ar, 1/mass, 1/(pi e ar), gammas, 1/Jy) to what config.py compiles
from the matching parameter files; (3) variants to the CPU oracle built from variant parameter files; (4) the Philox
draws of every env to those of an unpinned handle; (5) the reset-time rule, checkpoints and sharding; (6) the bank
column to explicit requests; (7) the batched evaluation to per-file evaluations; (8) the argument errors.
"""
import ctypes
import functools
import json
import os

import numpy as np
import pytest
import torch

from bench import CONFIG_KW, SIM_KW
from oracle import harness
from oracle.env_restated import RestatedEnv
import parity_utils as pu

pytestmark = pytest.mark.gpu

SEED = 20261023
PARAMS = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "fixed-wing-gym_b200", "params")
X8 = json.load(open(os.path.join(PARAMS, "x8_param.json")))
OFF = {"turbulence": False}
SHORT = {"steps_max": 100}     # episodes end within the tests' windows, so auto-resets are covered
AIR_ROWS = ("aircraft_req",)


def bits(x):
    return x.view({torch.float32: torch.int32, torch.float64: torch.int64}.get(x.dtype, x.dtype))


def make_vec(n, names, sim_kw=None, config_kw=None, **kw):
    from fwgym_b200 import FixedWingVecEnv
    v = FixedWingVecEnv(harness.config_path(), n, config_kw=dict(CONFIG_KW if config_kw is None else config_kw),
                        sim_config_kw=dict(SIM_KW if sim_kw is None else sim_kw), seed=SEED, aircraft_parameters=names,
                        **kw)
    v.enable_f64_outputs(True)
    return v


def actions(n, steps, seed=3, scale=1.0):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return (torch.rand((steps, n, 3), generator=g, device="cuda", dtype=torch.float64) * 2 - 1) * scale


def state_bits(v, skip=AIR_ROWS):
    rows = v.state_rows()
    keep = torch.as_tensor([i for i, r in enumerate(rows) if r not in skip], device=v.device)
    return bits(v.get_state()[keep])


def variant(rs, names, scale=0.2):
    """A random airframe: every name in `names` at its nominal value times U(1 - scale, 1 + scale)."""
    P = dict(X8)
    for k in names:
        P[k] = float(X8[k] * rs.uniform(1 - scale, 1 + scale))
    while P["Jx"] * P["Jz"] - P["Jxz"] ** 2 <= 0:
        P["Jxz"] *= 0.5
    return P


def write_params(P, tmp_path, i):
    path = os.path.join(str(tmp_path), "variant%d.json" % i)
    json.dump(P, open(path, "w"))
    return path


def run_lockstep(a, b, acts):
    """Step both handles on the same actions; assert bitwise equal outputs and state (request rows aside)."""
    dones = 0
    for t in range(acts.shape[0]):
        oa = a.step_tensors(acts[t])
        ob = b.step_tensors(acts[t])
        for x, y in zip(oa, ob):
            assert torch.equal(bits(x), bits(y)), "step %d" % t
        assert torch.equal(bits(a._obs64), bits(b._obs64)) and torch.equal(bits(a._rew64), bits(b._rew64))
        dones += int(oa[2].sum())
    assert torch.equal(state_bits(a), state_bits(b))
    return dones


@pytest.mark.parametrize("precision", ["fp64", "fp32"])
def test_nominal_pin_is_bitwise_unpinned(built_lib, precision):
    from fwgym_b200.config import CompiledConfig
    names = CompiledConfig.AIRCRAFT_PARAMS            # every name: turbulence off (a per-env b needs it)
    n = 256
    a = make_vec(n, names, sim_kw=OFF, config_kw={**CONFIG_KW, **SHORT}, precision=precision)
    b = make_vec(n, names, sim_kw=OFF, config_kw={**CONFIG_KW, **SHORT}, precision=precision)
    assert a.kernel_variant().startswith("dyn=rand")
    a.set_aircraft(a.cc.aircraft_nominal())
    assert not torch.isnan(a.aircraft_requests()).any() and torch.isnan(b.aircraft_requests()).all()
    a.reset()
    b.reset()
    assert torch.equal(state_bits(a), state_bits(b))
    assert run_lockstep(a, b, actions(n, 300)) > n     # every env reset at least once on its own


def test_nominal_requests_match_the_constant_bank(built_lib):
    """NaN requests derive, on the device, exactly the constants the host compiled for the shared aircraft."""
    names = ("mass", "b", "S_wing", "e", "Jx", "Jy", "Jz", "Jxz")
    v = make_vec(8, names, sim_kw=OFF)
    v.reset()
    par = v.get_state()[[i for i, r in enumerate(v.state_rows()) if r == "param"]].cpu().numpy()
    s = v.cc.pod().sim
    from fwgym_b200 import _capi
    E = _capi.ENUMS
    row = lambda pid: par[s.par_slot1[pid] - 1]
    assert (row(E["FW_PAR_AR"]) == s.ar).all() and (row(E["FW_PAR_INV_MASS"]) == s.inv_mass).all()
    assert (row(E["FW_PAR_INV_PI_E_AR"]) == s.inv_pi_e_ar).all()
    for k in range(8):
        assert (par[s.inertia_slot1[k] - 1] == s.gammas[k + 1]).all()
    assert (par[s.inertia_slot1[8] - 1] == s.inv_Jy).all()


def test_derived_rows_match_the_host(built_lib, tmp_path):
    """256 random airframes: after a reset the derived rows are what config.py compiles from parameter files with the
    same values - bitwise where Python's ** squares b and Jxz correctly (the device multiplies; libm pow misrounds x^2
    for about one input in a thousand, then the rows that square are one ulp apart) - and exp(2 M a_0) within one ulp
    (the device exp is not correctly rounded)."""
    from fwgym_b200 import _capi
    from fwgym_b200.config import CompiledConfig
    E = _capi.ENUMS
    names = ("mass", "b", "S_wing", "e", "M", "a_0", "Jx", "Jy", "Jz", "Jxz")
    n = 256
    rs = np.random.RandomState(11)
    airframes = [variant(rs, names, 0.3) for _ in range(n)]
    v = make_vec(n, names, sim_kw=OFF)
    v.set_aircraft({k: np.array([P[k] for P in airframes]) for k in names})
    v.reset()
    par = v.get_state()[[i for i, r in enumerate(v.state_rows()) if r == "param"]].cpu().numpy()
    s = v.cc.pod().sim
    checked_exact = 0
    for e, P in enumerate(airframes):
        h = CompiledConfig(harness.config_path(), sim_parameter_path=write_params(P, tmp_path, e),
                           config_kw=CONFIG_KW, sim_config_kw=OFF).pod().sim
        got = {"ar": par[s.par_slot1[E["FW_PAR_AR"]] - 1, e], "inv_mass": par[s.par_slot1[E["FW_PAR_INV_MASS"]] - 1, e],
               "inv_pi_e_ar": par[s.par_slot1[E["FW_PAR_INV_PI_E_AR"]] - 1, e],
               "inv_Jy": par[s.inertia_slot1[8] - 1, e]}
        want = {"ar": h.ar, "inv_mass": h.inv_mass, "inv_pi_e_ar": h.inv_pi_e_ar, "inv_Jy": h.inv_Jy}
        for k in range(8):
            got["g%d" % (k + 1)] = par[s.inertia_slot1[k] - 1, e]
            want["g%d" % (k + 1)] = h.gammas[k + 1]
        exact = all(float(P[k]) ** 2 == float(P[k]) * float(P[k]) for k in ("b", "Jxz"))
        for k in want:
            if exact:
                assert got[k] == want[k], (e, k)
            else:
                np.testing.assert_array_max_ulp(np.float64(got[k]), np.float64(want[k]), maxulp=2)
        checked_exact += exact
        np.testing.assert_array_max_ulp(par[s.par_slot1[E["FW_PAR_EXP_2MA0"]] - 1, e], np.float64(h.exp_2Ma0), maxulp=1)
        for name in ("mass", "b", "S_wing", "e", "M", "a_0"):
            assert par[s.par_slot1[CompiledConfig.par_id(name)] - 1, e] == P[name]
    assert checked_exact >= n - 8


def test_oracle_parity(built_lib, tmp_path):
    """Eight variants (inertia, mass, C_prop, rho) under moderate turbulence against the restated reference env built
    from variant parameter files, across auto-resets: 1e-9 per step, done and attempt counts exact."""
    names = ("mass", "Jx", "Jy", "Jz", "Jxz", "C_prop", "rho")
    rs = np.random.RandomState(8)
    n = 8
    frames = [variant(rs, ("mass", "Jx", "Jy", "Jz", "Jxz", "C_prop")) for _ in range(n)]
    rhos = rs.uniform(1.0, 1.35, n)
    cfg = harness.config_path()
    ckw = {**CONFIG_KW, **SHORT}
    vec = make_vec(n, names, config_kw=ckw)
    vals = {k: np.array([P[k] for P in frames]) for k in names if k != "rho"}
    vals["rho"] = rhos
    vec.set_aircraft(vals)
    oracles = []
    for i, P in enumerate(frames):
        env = RestatedEnv(cfg, sim_parameter_path=write_params(P, tmp_path, i), config_kw=ckw,
                          sim_config_kw={**SIM_KW, "rho": float(rhos[i])})
        oracles.append(harness.OracleRunner(env, SEED, i))
    acts = np.random.RandomState(0).uniform(-1, 1, (260, n, 3))
    out = pu.run_parity(vec, oracles, acts)
    worst = max(max(out["obs"]), max(out["rew"]), max(out["state"]))
    assert worst < 1e-9, worst
    assert out["done_mismatch"] == 0 and out["k_mismatch"] == 0
    assert out["dones"] >= n


def test_no_draw_moves(built_lib):
    names = ("mass", "Jy", "C_prop")
    n = 64
    a, b = make_vec(n, names), make_vec(n, names)
    a.set_aircraft({"mass": 3.9, "Jy": 0.21, "C_prop": 0.95}, indices=[5])
    a.reset()
    b.reset()
    rows = a.state_rows()
    skip = {i for i, r in enumerate(rows) if r in ("param", "aircraft_req")}
    keep = torch.as_tensor([i for i in range(len(rows)) if i not in skip], device=a.device)
    sa, sb_ = bits(a.get_state()), bits(b.get_state())
    assert torch.equal(sa[keep], sb_[keep])            # env 5's initial states and targets are the same draws
    others = torch.ones(n, dtype=torch.bool, device=a.device)
    others[5] = False
    assert torch.equal(sa[:, others], sb_[:, others])
    assert not torch.equal(sa[:, 5], sb_[:, 5])
    for t, act in enumerate(actions(n, 120)):
        oa, ob = a.step_tensors(act), b.step_tensors(act)
        for x, y in zip(oa, ob):
            assert torch.equal(bits(x)[others], bits(y)[others]), t
    assert torch.equal(bits(a.get_state())[:, others], bits(b.get_state())[:, others])


def test_request_takes_effect_at_the_next_reset(built_lib):
    names = ("mass", "C_prop")
    v = make_vec(16, names, config_kw=CONFIG_KW)
    v.reset()
    rows = v.state_rows()
    p0 = rows.index("param")
    before = v.get_rows(p0, 2).clone()
    v.set_aircraft({"mass": 4.0})
    acts = actions(16, 5, scale=0.1)
    for a_ in acts:
        _, _, done, _ = v.step_tensors(a_)
        assert not bool(done.any())
    assert torch.equal(bits(v.get_rows(p0, 2)), bits(before))     # the running episodes keep their aircraft
    assert bool((v.aircraft()["mass"] == 4.0).all())
    v.reset(indices=[3])
    now = v.get_rows(p0, 2)
    assert now[0, 3].item() == 4.0 and now[1, 3].item() == X8["C_prop"]
    assert torch.equal(bits(now[:, :3]), bits(before[:, :3])) and torch.equal(bits(now[:, 4:]), bits(before[:, 4:]))


def test_requests_survive_checkpoints_and_sharding(built_lib):
    names = ("mass", "Jx", "C_prop")
    n = 64
    vals = {"mass": np.linspace(2.8, 4.2, n), "Jx": np.linspace(1.0, 1.4, n)}
    one = make_vec(n, names, config_kw={**CONFIG_KW, **SHORT})
    one.set_aircraft(vals)
    one.reset()
    acts = actions(n, 150, seed=9)
    for a_ in acts[:40]:
        one.step_tensors(a_)
    ck = one.get_state().clone()
    twin = make_vec(n, names, config_kw={**CONFIG_KW, **SHORT})
    twin.set_state(ck)
    assert torch.equal(bits(twin.aircraft_requests()), bits(one.aircraft_requests()))
    run_lockstep(one, twin, acts[40:])
    # two shards of 32 envs = one handle of 64
    full = make_vec(n, names, config_kw={**CONFIG_KW, **SHORT})
    full.set_aircraft(vals)
    full.reset()
    shards = []
    for k in range(2):
        s = make_vec(n // 2, names, config_kw={**CONFIG_KW, **SHORT}, env_offset=k * n // 2)
        s.set_aircraft({key: val[k * n // 2:(k + 1) * n // 2] for key, val in vals.items()})
        s.reset()
        shards.append(s)
    for a_ in acts:
        of = full.step_tensors(a_)
        parts = [s.step_tensors(a_[k * n // 2:(k + 1) * n // 2].contiguous()) for k, s in enumerate(shards)]
        for j in range(4):
            assert torch.equal(bits(of[j]), bits(torch.cat([p[j] for p in parts])))
    assert torch.equal(bits(full.get_state()), bits(torch.cat([s.get_state() for s in shards], dim=1)))


def test_bank_column_equals_explicit_requests(built_lib):
    """A banked aircraft column starts the same episodes as set_aircraft + a reset with the same columns; the result
    rows report each scenario's first episode."""
    names = ("mass", "Jy", "C_prop")
    n = 32
    rs = np.random.RandomState(4)
    mass = rs.uniform(2.8, 4.2, n)
    mass[::5] = np.nan                                   # those scenarios keep the env's request
    jy = rs.uniform(0.14, 0.2, n)
    state = {"roll": rs.uniform(-0.3, 0.3, n), "velocity_u": rs.uniform(18, 24, n)}
    target = {"roll": rs.uniform(-0.4, 0.4, n), "pitch": rs.uniform(-0.2, 0.2, n), "Va": rs.uniform(18, 23, n)}
    ckw = {**CONFIG_KW, **SHORT}
    a = make_vec(n, names, config_kw=ckw, scenario_bank=True)
    a.set_aircraft({"C_prop": 0.9})
    res = a.set_scenario_bank(state=state, target=target, aircraft={"mass": mass, "Jy": jy})
    a.reset()
    b = make_vec(n, names, config_kw=ckw)
    b.set_aircraft({"C_prop": 0.9, "mass": mass, "Jy": jy})
    b.reset(state=state, target=target)
    skip = ("aircraft_req", "bank_next", "bank_scenario")
    assert torch.equal(state_bits(a, skip), state_bits(b, skip))
    first_len = torch.full((n,), -1, dtype=torch.int64, device=a.device)
    first_term = torch.full((n,), -1, dtype=torch.int32, device=a.device)
    alive = torch.ones(n, dtype=torch.bool, device=a.device)
    for t, act in enumerate(actions(n, 110, seed=6)):
        oa, ob = a.step_tensors(act), b.step_tensors(act)
        for x, y in zip(oa, ob):                       # identical while every env flies its first episode
            assert torch.equal(bits(x)[alive], bits(y)[alive]), t
        fin = alive & ob[2].bool()
        first_len[fin] = t + 1
        first_term[fin] = ob[3][fin]
        alive &= ~fin
    assert not bool(alive.any())
    assert torch.equal(res["length"].long(), first_len) and torch.equal(res["term"], first_term)
    assert bool((res["episodes"] == 1).all())


def _per_file_evaluation(scen, cfg, variants, tmp_path):
    """The identify_constants way: one handle per variant, built from its own parameter file."""
    from fwgym_b200 import evaluate
    from fwgym_b200.vec_env import FixedWingVecEnv
    out = {}
    for j, var in enumerate(variants):
        P = dict(X8)
        P.update(var)
        orig = evaluate.FixedWingVecEnv
        evaluate.FixedWingVecEnv = functools.partial(FixedWingVecEnv, sim_parameter_path=write_params(P, tmp_path, j))
        try:
            out[j], vj = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1)
        finally:
            evaluate.FixedWingVecEnv = orig
        vj.close()
    return out


def test_evaluation_equals_per_file_calls(built_lib, tmp_path):
    from fwgym_b200 import evaluate
    scen = evaluate.load_test_set(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden",
                                               "test_set_wind_none.npz"))[:24]
    cfg = harness.config_path()
    variants = [{"mass": 3.0, "Jy": 0.19}, {"C_prop": 0.9, "Jx": 1.1, "Jxz": 0.8}, {}]
    ref = _per_file_evaluation(scen, cfg, variants, tmp_path)
    got, v = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, aircraft=variants)
    assert v.num_envs == 3 * len(scen)
    banked, vb = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, aircraft=variants, num_envs=20)
    for j in range(3):
        for res in (got[j], banked[j]):
            np.testing.assert_array_equal(res["lengths"], ref[j]["lengths"])
            np.testing.assert_array_equal(res["episode_rows"][:, 3], ref[j]["episode_rows"][:, 3])   # success_all
            for r1, r0 in zip(res["rewards"], ref[j]["rewards"]):
                assert pu.rel_err(r1, r0, 1e-3).max() < 1e-9
    v.close()
    vb.close()


def test_errors(built_lib):
    from fwgym_b200 import _capi
    lib = _capi.lib()
    plain = make_vec(8, ())
    assert lib.fw_aircraft_dim(plain._h) == 0
    assert lib.fw_set_aircraft(plain._h, None, None) == _capi.ENUMS["FW_ERR_ARG"]
    with pytest.raises(_capi.FwError):
        plain.set_aircraft({"mass": 3.0})
    bank = make_vec(8, (), scenario_bank=True)
    b = _capi.fw_bank_t()
    col = torch.full((1, 4), 3.0, dtype=torch.float64, device="cuda")
    b.n_scenarios, b.first, b.stride = 4, 0, 8
    assert lib.fw_set_bank(bank._h, ctypes.byref(b), None) == 0
    assert lib.fw_set_bank_aircraft(bank._h, col.data_ptr()) == _capi.ENUMS["FW_ERR_ARG"]
    air_bank = make_vec(8, ("mass",), scenario_bank=True)
    assert lib.fw_set_bank_aircraft(air_bank._h, col.data_ptr()) == _capi.ENUMS["FW_ERR_ARG"]   # no bank attached
    assert lib.fw_set_bank(air_bank._h, ctypes.byref(b), None) == 0
    assert lib.fw_set_bank_aircraft(air_bank._h, col.data_ptr()) == 0
    assert lib.fw_set_bank(air_bank._h, None, None) == 0
    with pytest.raises(ValueError, match="aircraft_parameters"):
        bank.set_scenario_bank(state={"roll": [0.0] * 4}, aircraft={"mass": [3.0] * 4})
    v = make_vec(8, ("mass", "Jx", "Jxz"))
    assert lib.fw_aircraft_dim(v._h) == 3
    with pytest.raises(ValueError, match="not an aircraft parameter"):
        v.set_aircraft({"C_prop": 1.0})
    with pytest.raises(ValueError, match="mass"):
        v.set_aircraft({"mass": -1.0})
    with pytest.raises(ValueError, match="Jx"):
        v.set_aircraft({"Jxz": 5.0})
    with pytest.raises(ValueError, match="3 values for 8 envs"):
        v.set_aircraft({"mass": [3.0, 3.1, 3.2]})
    assert bool(torch.isnan(v.aircraft_requests()).all())   # refused requests leave the rows alone
    assert lib.fw_set_aircraft(v._h, None, None) == 0
    for h in (plain, bank, air_bank, v):
        h.close()
