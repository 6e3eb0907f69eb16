"""Per-env aircraft, host side: which names may differ per env and what is refused, the parameter-row and slot layout a
list of aircraft parameters compiles to, the unchanged compilation of configurations without one, a numpy twin of
what the reset derives from an aircraft, and the request / bank / evaluation tables.  No GPU needed."""
import ctypes
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAMS = os.path.join(ROOT, "fixed-wing-gym_b200", "params")
ENV_CONFIGS = sorted(f for f in os.listdir(PARAMS) if f.startswith("fixed_wing_config"))
INERTIA_TERMS = 9


def _cc(env_config="fixed_wing_config.json", **kw):
    from fwgym_b200.config import CompiledConfig
    return CompiledConfig(os.path.join(PARAMS, env_config), **kw)


def _enums():
    from fwgym_b200 import _capi
    return _capi.ENUMS


def test_allowed_names():
    from fwgym_b200.config import CompiledConfig
    allowed = CompiledConfig.AIRCRAFT_PARAMS
    assert "ar" not in allowed and len(allowed) == len(set(allowed))
    assert set(allowed) == (set(CompiledConfig.LIVE_PARAMS) - {"ar"}) | {"rho", "g", "Jx", "Jy", "Jz", "Jxz"}
    from fwgym_b200 import _capi
    assert len(allowed) == _capi.DEFINES["FW_MAX_AIRCRAFT"]
    assert _capi.DEFINES["FW_N_INERTIA"] == INERTIA_TERMS
    assert _enums()["FW_AIR_JX"] == _enums()["FW_PAR_N"]
    cc = _cc(aircraft_parameters=allowed, sim_config_kw={"turbulence": False})   # every name at once compiles
    assert cc.pod().env.n_aircraft == len(allowed)


@pytest.mark.parametrize("names, msg", [(("ar",), "cannot differ per env"), (("Jyy",), "cannot differ per env"),
                                        (("mass", "mass"), "listed twice"), (("k",), "cannot differ per env")])
def test_bad_names(names, msg):
    from fwgym_b200.config import ConfigError
    with pytest.raises(ConfigError, match=msg):
        _cc(aircraft_parameters=names)


def test_refused_with_randomisation():
    from fwgym_b200.config import ConfigError
    with pytest.raises(ConfigError, match="randomisation"):
        _cc("fixed_wing_config_randomised.json", aircraft_parameters=("mass",))
    # a rho range alone is randomisation too (config_kw cannot add keys, so the parsed config is edited)
    cc = _cc(aircraft_parameters=("C_prop",))
    cc.cfg["simulator"]["rho"] = {"low": 1.1, "high": 1.3}
    with pytest.raises(ConfigError, match="randomisation"):
        cc._check_aircraft()


def test_refused_wingspan_under_turbulence():
    from fwgym_b200.config import ConfigError
    with pytest.raises(ConfigError, match="wingspan"):
        _cc(aircraft_parameters=("b",), sim_config_kw={"turbulence": True, "turbulence_intensity": "moderate"})
    _cc(aircraft_parameters=("S_wing", "Jx"), sim_config_kw={"turbulence": True, "turbulence_intensity": "moderate"})
    assert _cc(aircraft_parameters=("b",), sim_config_kw={"turbulence": False}).pod().env.n_aircraft == 1


def test_slots_and_rows_live_only():
    E = _enums()
    pod = _cc(aircraft_parameters=("mass", "C_prop")).pod()
    s, e = pod.sim, pod.env
    assert e.n_aircraft == 2 and e.n_rand == 0
    assert list(s.air_id)[:2] == [E["FW_PAR_MASS"], E["FW_PAR_C_PROP"]]
    slots = {i: v for i, v in enumerate(s.par_slot1) if v}
    assert slots == {E["FW_PAR_MASS"]: 1, E["FW_PAR_C_PROP"]: 2, E["FW_PAR_INV_MASS"]: 3}
    assert e.n_par_rows == 3
    assert list(s.inertia_slot1) == [0] * INERTIA_TERMS
    assert (s.Jx, s.Jz, s.Jxz) == (1.229, 0.8808, 0.9343)   # the nominal inertia (x8_param.json)


def test_slots_and_rows_with_derived_and_inertia():
    E = _enums()
    names = ("b", "Jy", "e", "M", "rho")
    pod = _cc(aircraft_parameters=names, sim_config_kw={"turbulence": False}).pod()
    s, e = pod.sim, pod.env
    assert list(s.air_id)[:5] == [E["FW_PAR_B"], E["FW_AIR_JY"], E["FW_PAR_E"], E["FW_PAR_M"], E["FW_PAR_RHO"]]
    assert all(v == 0 for v in list(s.air_id)[5:])
    slots = {i: v for i, v in enumerate(s.par_slot1) if v}
    # listed live parameters in listed order, then ar (b is listed), then the derived rows, then the inertia terms
    assert slots == {E["FW_PAR_B"]: 1, E["FW_PAR_E"]: 2, E["FW_PAR_M"]: 3, E["FW_PAR_RHO"]: 4, E["FW_PAR_AR"]: 5,
                     E["FW_PAR_INV_PI_E_AR"]: 6, E["FW_PAR_EXP_2MA0"]: 7}
    assert list(s.inertia_slot1) == list(range(8, 8 + INERTIA_TERMS))
    assert e.n_par_rows == 7 + INERTIA_TERMS


def test_no_aircraft_leaves_the_new_fields_zero():
    """Every shipped env configuration without aircraft parameters: the appended tail of fw_sim_t (from Jx on) and
    fw_env_t.n_aircraft are all zero, so those configurations compile to the bytes they compiled to before."""
    from fwgym_b200 import _capi
    S = _capi.STRUCTS["fw_sim_t"]
    sim0 = _capi.fw_config_t.sim.offset
    for cfg in ENV_CONFIGS:
        for kw in ({"turbulence": False}, {"turbulence": True, "turbulence_intensity": "moderate"}):
            pod = _cc(cfg, sim_config_kw=kw).pod()
            raw = bytes(memoryview(pod).cast("B"))
            tail = raw[sim0 + S.Jx.offset:sim0 + ctypes.sizeof(S)]
            assert tail == bytes(len(tail)), cfg
            assert pod.env.n_aircraft == 0
    assert ctypes.sizeof(S) % 32 == 24     # the congruence fwgym.cu static_asserts


def twin(P, sq=lambda x: x * x):
    """What the reset derives from an aircraft (csrc/env.cuh), in numpy float64 scalars, config.py's operation order.
    `sq` squares; the device multiplies (correctly rounded)."""
    f = np.float64
    jx, jy, jz, jxz = f(P["Jx"]), f(P["Jy"]), f(P["Jz"]), f(P["Jxz"])
    axz, xz2 = abs(jxz), sq(-jxz)
    g0 = jx * jz - xz2
    gam = [(axz * (jx - jy + jz)) / g0, (jz * (jz - jy) + xz2) / g0, jz / g0, axz / g0, (jz - jx) / jy, -jxz / jy,
           ((jx - jy) * jx + xz2) / g0, jx / g0]
    ar = sq(f(P["b"])) / f(P["S_wing"])
    return {"gammas": gam, "inv_Jy": f(1.0) / jy, "ar": ar, "inv_mass": f(1.0) / f(P["mass"]),
            "inv_pi_e_ar": f(1.0) / (f(np.pi) * f(P["e"]) * ar)}


def random_airframes(n, seed):
    base = json.load(open(os.path.join(PARAMS, "x8_param.json")))
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(n):
        P = dict(base)
        for k in ("mass", "Jx", "Jy", "Jz", "b", "S_wing", "e"):
            P[k] = float(base[k] * rng.uniform(0.7, 1.3))
        P["Jxz"] = float(base["Jxz"] * rng.uniform(0.0, 0.9))
        while P["Jx"] * P["Jz"] - P["Jxz"] ** 2 <= 0:
            P["Jxz"] *= 0.5
        out.append(P)
    return out


def compile_params(P, tmp_path, i):
    path = os.path.join(str(tmp_path), "air%d.json" % i)
    json.dump(P, open(path, "w"))
    return _cc(sim_parameter_path=path, sim_config_kw={"turbulence": False}).pod().sim


def test_numpy_twin_matches_config(tmp_path):
    """The twin with config.py's squares (Python's **, i.e. libm pow) is bitwise config.py for random airframes.  The
    device squares by a correctly rounded multiply: equal to pow wherever pow rounds x^2 correctly (every shipped
    parameter file), else one ulp apart in the rows that square."""
    n_pow_off = 0
    for i, P in enumerate(random_airframes(64, 7)):
        s = compile_params(P, tmp_path, i)
        want = {"gammas": list(s.gammas)[1:], "inv_Jy": s.inv_Jy, "ar": s.ar, "inv_mass": s.inv_mass,
                "inv_pi_e_ar": s.inv_pi_e_ar}
        host, dev = twin(P, lambda x: x ** 2), twin(P)
        exact = all(float(v) ** 2 == float(v) * float(v) for v in (P["Jxz"], P["b"]))
        n_pow_off += not exact
        for k, v in want.items():
            np.testing.assert_array_equal(np.asarray(host[k]), np.asarray(v), err_msg="%s airframe %d" % (k, i))
            if exact:
                np.testing.assert_array_equal(np.asarray(dev[k]), np.asarray(v), err_msg="%s airframe %d" % (k, i))
            else:
                np.testing.assert_array_max_ulp(np.asarray(dev[k], dtype=np.float64), np.asarray(v), maxulp=2)
    assert n_pow_off < 8


def test_shipped_parameter_files_square_exactly():
    """The nominal aircraft of every shipped parameter file compiles to the same derived values on host and device."""
    for pf in ("x8_param.json", "identified/x8_param.json", "recalled/x8_param.json"):
        P = json.load(open(os.path.join(PARAMS, pf)))
        for k in ("b", "Jxz"):
            assert float(P[k]) ** 2 == float(P[k]) * float(P[k]), (pf, k)


def test_request_validation():
    import torch
    from fwgym_b200.vec_env import check_aircraft
    cc = _cc(aircraft_parameters=("mass", "Jx", "Jxz", "S_wing"))
    nan = float("nan")
    ok = torch.tensor([[nan, 2.0], [nan, 1.3], [nan, 0.5], [nan, 0.6]], dtype=torch.float64)
    check_aircraft(cc, ok)
    for row, bad, msg in ((0, 0.0, "mass"), (0, float("inf"), "finite"), (3, -1.0, "S_wing"), (2, 5.0, "Jx \\* Jz")):
        r = ok.clone()
        r[row, 1] = bad
        with pytest.raises(ValueError, match=msg):
            check_aircraft(cc, r)
    # Jy alone: > 0, and the determinant is not its business
    cc = _cc(aircraft_parameters=("Jy",))
    check_aircraft(cc, torch.tensor([[0.3]], dtype=torch.float64))
    with pytest.raises(ValueError, match="Jy"):
        check_aircraft(cc, torch.tensor([[-0.3]], dtype=torch.float64))


def test_bank_aircraft_column():
    from fwgym_b200 import scenario_bank as sb
    names = ("mass", "C_prop")
    S, st, tg, lv, air = sb.build_bank_tables(state={"roll": [0.0, 0.1, 0.2]}, aircraft={"C_prop": [1.0, np.nan, 0.9]},
                                              target_names=["roll"], aircraft_parameters=names)
    assert S == 3 and lv is None and tg is None
    assert air.shape == (2, 3) and np.isnan(air[0]).all()
    np.testing.assert_array_equal(air[1], [1.0, np.nan, 0.9])
    # an aircraft column alone sets S
    assert sb.build_bank_tables(aircraft={"mass": [3.0, 3.1]}, aircraft_parameters=names)[0] == 2
    with pytest.raises(ValueError, match="not an aircraft parameter"):
        sb.build_bank_tables(aircraft={"rho": [1.0]}, aircraft_parameters=names)
    with pytest.raises(ValueError, match="needs a handle with aircraft_parameters"):
        sb.build_bank_tables(state={"roll": [0.0]}, aircraft={"mass": [1.0]})
    with pytest.raises(ValueError, match="different lengths"):
        sb.build_bank_tables(state={"roll": [0.0, 0.1]}, aircraft={"mass": [3.0, 3.1, 3.2]}, aircraft_parameters=names)
    # the existing four-table form is unchanged
    assert len(sb.build_tables(state={"roll": [0.0]})) == 4


def test_evaluation_columns():
    from fwgym_b200 import evaluate
    names, cols = evaluate._aircraft_columns([{"mass": 3.0}, {"C_prop": 0.9, "mass": 3.5}, {}], 2)
    assert names == ("C_prop", "mass")
    np.testing.assert_array_equal(cols["mass"], [3.0, 3.0, 3.5, 3.5, np.nan, np.nan])
    np.testing.assert_array_equal(cols["C_prop"], [np.nan, np.nan, 0.9, 0.9, np.nan, np.nan])
    assert evaluate._aircraft_columns(None, 5) == ((), None)
    with pytest.raises(ValueError, match="no parameter"):
        evaluate._aircraft_columns([{}], 2)
    with pytest.raises(ValueError, match="not both"):
        evaluate.evaluate_on_set([{}], None, turbulence_intensity=["none", "light"], aircraft=[{"mass": 3.0}])
