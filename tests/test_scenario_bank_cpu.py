"""Scenario banks, host side: building and validating the tables, the assignment rule of envs to scenarios, and the
compile-time property that selects the bank kernels.  No GPU needed."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PARAMS = os.path.join(ROOT, "fixed-wing-gym_b200", "params")
TARGETS = ["roll", "pitch", "Va"]


def sb():
    from fwgym_b200 import scenario_bank
    return scenario_bank


def test_tables_use_the_reset_name_mapping():
    from fwgym_b200 import _capi
    S = 5
    wind = np.arange(15, dtype=np.float64).reshape(3, S)
    n, st, tg, lv = sb().build_tables(state={"roll": np.linspace(-0.1, 0.1, S), "Va": 20.0, "wind": wind},
                                      target={"pitch": np.full(S, 0.05)}, target_names=TARGETS)
    assert n == S and lv is None
    assert st.shape == (_capi.DEFINES["FW_N_SV"] + 3, S) and tg.shape == (_capi.DEFINES["FW_MAX_TARGETS"], S)
    assert np.array_equal(st[_capi.sv_id("roll")], np.linspace(-0.1, 0.1, S))
    assert (st[_capi.sv_id("Va")] == 20.0).all()                      # a scalar applies to every scenario
    assert np.array_equal(st[_capi.DEFINES["FW_N_SV"]:], wind)        # wind n, e, d after the state variables
    others = [r for r in range(st.shape[0]) if r not in (_capi.sv_id("roll"), _capi.sv_id("Va"))
              and r < _capi.DEFINES["FW_N_SV"]]
    assert np.isnan(st[others]).all()                                 # NaN = sampled at the reset
    assert (tg[1] == 0.05).all() and np.isnan(tg[[0, 2]]).all()


def test_tables_without_state_or_target():
    n, st, tg, lv = sb().build_tables(target={"Va": [18.0, 19.0]}, target_names=TARGETS)
    assert n == 2 and st is None and tg is not None


@pytest.mark.parametrize("kw,match", [
    (dict(state={"rol": [0.1, 0.2]}), "unknown state"),
    (dict(target={"yaw": [0.1, 0.2]}), "unknown target"),
    (dict(state={"roll": [0.1, 0.2], "pitch": [0.1, 0.2, 0.3]}), "different lengths"),
    (dict(state={"roll": [0.1, 0.2]}, target={"Va": [18.0]}), "different lengths"),
    (dict(state={"roll": [[0.1, 0.2]]}), "one value per scenario"),
    (dict(state={"wind": [1.0, 2.0]}), "wind"),
    (dict(state={"roll": 0.1}), "at least one per-scenario"),
    (dict(state={"roll": [0.1, 0.2]}, turbulence_intensity=["light", "none"]), "per-env levels"),
])
def test_table_errors(kw, match):
    with pytest.raises(ValueError, match=match):
        sb().build_tables(target_names=TARGETS, **kw)


def test_level_column():
    n, _, _, lv = sb().build_tables(state={"roll": [0.0] * 4}, turbulence_intensity=["none", "severe", 2, -1],
                                    target_names=TARGETS, mixed=True)
    assert lv.dtype == np.int32 and list(lv) == [0, 3, 2, -1]
    for bad in (["extreme"] * 4, [4, 0, 0, 0], [0.5, 0, 0, 0]):
        with pytest.raises(ValueError):
            sb().build_tables(state={"roll": [0.0] * 4}, turbulence_intensity=bad, target_names=TARGETS, mixed=True)


def test_assignment_arguments():
    sb().check_assignment(8, 100, 0, 8)
    sb().check_assignment(8, 100, 40, 64)
    with pytest.raises(ValueError, match="stride"):
        sb().check_assignment(8, 100, 0, 7)
    with pytest.raises(ValueError, match="first"):
        sb().check_assignment(8, 100, -1, 8)


@pytest.mark.parametrize("n_envs,S,first,stride", [(8, 50, 0, 8), (8, 50, 3, 11), (5, 7, 0, 5), (16, 1000, 16, 32),
                                                    (4, 3, 0, 4), (6, 40, 45, 6)])
@pytest.mark.parametrize("cycle", [False, True])
def test_assignment_rule(n_envs, S, first, stride, cycle):
    """The closed form first + e + k stride (mod S when cycling, -1 past the bank) against the cursor the kernels keep:
    attach, then the k-th banked reset of env e takes the cursor and advances it (csrc/env.cuh fw_bank_advance)."""
    m = sb()
    cur = m.attach_cursor(n_envs, S, first, cycle)
    flown = []
    for k in range(2 * S // n_envs + 3):
        taken = np.where(cur < S, cur, -1)
        assert np.array_equal(taken, m.scenario_of(np.arange(n_envs), k, S, first, stride, cycle))
        flown += [int(x) for x in taken if x >= 0]
        cur = np.where(cur < S, m.advance(cur, S, stride, cycle), cur)
        assert (cur >= 0).all() and (cur <= S).all()
    if not cycle:
        # no scenario is flown twice; with stride == n_envs every scenario from `first` on is flown
        assert len(flown) == len(set(flown))
        if stride == n_envs:
            assert sorted(flown) == list(range(min(first, S), S))


def test_sharded_ranks_partition_the_bank():
    """Two ranks (first = env_offset, stride = total envs) fly the scenarios one rank of all envs would."""
    m = sb()
    S, N = 97, 12
    whole = {int(m.scenario_of(e, k, S, 0, N, False)) for e in range(N) for k in range(10)} - {-1}
    halves = [{int(m.scenario_of(e, k, S, off, N, False)) for e in range(N // 2) for k in range(10)} - {-1}
              for off in (0, N // 2)]
    assert not halves[0] & halves[1] and halves[0] | halves[1] == whole == set(range(S))


def test_kernel_cursor_step_matches_the_mirror():
    """The device's cursor step is the expression the mirror restates."""
    src = open(os.path.join(ROOT, "fixed-wing-gym_b200", "csrc", "env.cuh")).read()
    body = re.search(r"int32_t fw_bank_advance\(.*?\{(.*?)\n\}", src, re.S).group(1)
    assert "(int64_t)cur + b.stride" in body and "b.cycle ? nx % b.n : (nx < b.n ? nx : b.n)" in body


def test_bank_flag_compiles_into_the_config_and_shape():
    """scenario_bank=True sets fw_env_t.bank_enabled and nothing else; the bench configuration's bank twin is a
    generated shape that differs from default_turb in bank_enabled only, and shape matching compares the flag."""
    from fwgym_b200.config import CompiledConfig
    cfg = os.path.join(PARAMS, "fixed_wing_config.json")
    a = bytes(memoryview(CompiledConfig(cfg, sim_config_kw={"turbulence": True}).pod()).cast("B"))
    pb = CompiledConfig(cfg, sim_config_kw={"turbulence": True}, scenario_bank=True).pod()
    assert pb.env.bank_enabled == 1
    b = bytes(memoryview(pb).cast("B"))
    diff = [i for i in range(len(a)) if a[i] != b[i]]
    from fwgym_b200 import _capi
    off = _capi.fw_config_t.env.offset + _capi.STRUCTS["fw_env_t"].bank_enabled.offset
    assert diff == [off]
    src = open(os.path.join(ROOT, "fixed-wing-gym_b200", "csrc", "env_shapes_gen.h")).read()
    names = re.search(r"#define FW_SHAPE_LIST\(X\) (.*)", src).group(1).replace("X(", "").replace(")", "").split()
    assert "default_turb_bank" in names

    def body(kind, name):
        return set(re.search(r"constexpr fw_%s_t fw_shape_%s_%s\(\) \{(.*?)return" % (kind, kind, name), src,
                             re.S).group(1).splitlines())
    assert body("env", "default_turb_bank") - body("env", "default_turb") == {"  e.bank_enabled = 1;"}
    assert body("env", "default_turb") <= body("env", "default_turb_bank")
    assert body("sim", "default_turb_bank") == body("sim", "default_turb")
    for name in names:
        assert ("e.bank_enabled = 1;" in "".join(body("env", name))) == (name == "default_turb_bank")
    assert "a.bank_enabled != b.bank_enabled" in open(os.path.join(ROOT, "fixed-wing-gym_b200", "csrc",
                                                                    "env_shapes.h")).read()


def test_bank_struct_mirror():
    """fw_bank_t reaches Python through the header parser: pointers as void*, the sizes in order."""
    import ctypes
    from fwgym_b200 import _capi
    B = _capi.fw_bank_t
    names = [f for f, _ in B._fields_]
    assert names == ["init_state", "init_target", "turb_level", "n_scenarios", "first", "stride", "cycle", "_pad",
                     "term", "length", "ret", "episode", "episodes", "successes"]
    assert ctypes.sizeof(B) == 104 and B.n_scenarios.offset == 24 and B.term.offset == 56
