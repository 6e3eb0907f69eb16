"""Per-env Dryden intensity (mixed handles), host side: the per-level filter tables, the configuration errors, the
unchanged compilation of every existing configuration, the reset's level draw and the kernel shape a mixed
configuration selects.  No GPU needed."""
import ctypes
import hashlib
import itertools
import json
import os
import re

import numpy as np
import pytest

from oracle import philox
from turbmix_utils import RS_TURBLVL, drawn_level

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, "tests", "golden")
PARAMS = os.path.join(ROOT, "fixed-wing-gym_b200", "params")
ENV_CONFIGS = sorted(f for f in os.listdir(PARAMS) if f.startswith("fixed_wing_config"))
PARAM_FILES = [os.path.join(PARAMS, "x8_param.json"), os.path.join(PARAMS, "identified", "x8_param.json"),
               os.path.join(PARAMS, "recalled", "x8_param.json")]
SIM_CONFIGS = [os.path.join(PARAMS, "pyfly_config.json"), os.path.join(PARAMS, "identified", "pyfly_config.json")]
MIX4 = {"values": ["none", "light", "moderate", "severe"], "probabilities": [0.1, 0.2, 0.3, 0.4]}


def _cc(env_config="fixed_wing_config.json", **kw):
    from fwgym_b200.config import CompiledConfig
    return CompiledConfig(os.path.join(PARAMS, env_config), **kw)


def _shipped_b_dt():
    """Every (wing span, Dryden sample spacing) a shipped configuration combination produces."""
    from fwgym_b200.config import CompiledConfig
    out = set()
    for pf, sf, ef in itertools.product(PARAM_FILES, SIM_CONFIGS, ENV_CONFIGS):
        b = json.load(open(pf))["b"]
        sc = dict(json.load(open(sf)))
        sc["turbulence_sim_length"] = json.load(open(os.path.join(PARAMS, ef)))["steps_max"]
        out.add((b, CompiledConfig.turbulence_dt(sc)))
    return sorted(out)


@pytest.mark.parametrize("b,dt", _shipped_b_dt())
def test_filter_state_matrices_do_not_depend_on_the_level(b, dt):
    """Ad / Bd0 / Bd1 come out bitwise equal for light, moderate and severe (the intensity enters the numerators only),
    so one filter state serves every level; C scales with the intensity and D is zero."""
    from fwgym_b200.config import CompiledConfig
    lv = CompiledConfig.compile_turbulence_levels(b, dt)     # raises ConfigError when the state matrices differ
    for f in range(6):
        for k in range(3):
            assert np.asarray(lv["light"][f][k]).tobytes() == np.asarray(lv["severe"][f][k]).tobytes()
        c1, c2, c3 = (np.asarray(lv[name][f][3]) for name in ("light", "moderate", "severe"))
        nz = c1 != 0
        assert np.allclose(c2[nz] / c1[nz], 2.0, rtol=1e-12) and np.allclose(c3[nz] / c1[nz], 3.0, rtol=1e-12)
        assert all(lv[name][f][4] == 0.0 for name in ("light", "moderate", "severe"))


@pytest.mark.parametrize("sim_config", SIM_CONFIGS)
@pytest.mark.parametrize("param_file", PARAM_FILES)
def test_level_tables_equal_uniform_handles(sim_config, param_file):
    """turb_C[l] / turb_D[l] of a mixed POD are bitwise what a handle of uniform level l compiles into filt[f].C / D,
    its filt[f].Ad / Bd0 / Bd1 / n / stream are the uniform handles' (shared by every level), row 0 is zero."""
    kw = dict(sim_config_path=sim_config, sim_parameter_path=param_file)
    mixed = _cc(sim_config_kw={"turbulence": True, "turbulence_intensity": MIX4}, **kw).pod().sim
    assert mixed.turb_mixed == 1 and mixed.turbulence == 1
    assert list(mixed.turb_cdf) == [0.1, 0.1 + 0.2, 0.1 + 0.2 + 0.3, 1.0]
    assert all(mixed.turb_C[0][f][a] == 0.0 for f in range(6) for a in range(3))
    assert all(mixed.turb_D[0][f] == 0.0 for f in range(6))
    for lvl, name in enumerate(("light", "moderate", "severe"), start=1):
        uni = _cc(sim_config_kw={"turbulence": True, "turbulence_intensity": name}, **kw).pod().sim
        for f in range(6):
            U, M = uni.filt[f], mixed.filt[f]
            assert (U.n, U.stream) == (M.n, M.stream)
            assert bytes(U.Ad) == bytes(M.Ad) and bytes(U.Bd0) == bytes(M.Bd0) and bytes(U.Bd1) == bytes(M.Bd1)
            assert bytes(U.C) == bytes(mixed.turb_C[lvl][f])
            assert np.float64(U.D).tobytes() == np.float64(mixed.turb_D[lvl][f]).tobytes()


@pytest.mark.parametrize("spec,turbulence,match", [
    ({"values": ["light", "extreme"]}, True, "unknown level"),
    ({"values": ["light", "severe"], "probabilities": [1.5, -0.5]}, True, "negative"),
    ({"values": ["light", "severe"], "probabilities": [0.5, 0.4]}, True, "sum"),
    ({"values": ["light", "severe"], "probabilities": [0.5, 0.5 + 2e-12]}, True, "sum"),
    ({"values": ["light", "severe"], "probabilities": [1.0]}, True, "probabilities"),
    ({"values": ["light", "moderate", "severe"]}, False, "turbulence: True"),
    ({"values": ["light", "light"]}, True, "twice"),
    ({"levels": ["light"]}, True, "expected"),
])
def test_config_errors(spec, turbulence, match):
    from fwgym_b200.config import ConfigError
    with pytest.raises(ConfigError, match=match):
        _cc(sim_config_kw={"turbulence": turbulence, "turbulence_intensity": spec})


def test_probabilities_default_to_uniform_and_tolerate_rounding():
    s = _cc(sim_config_kw={"turbulence": True, "turbulence_intensity": {"values": ["light", "moderate", "severe"]}})
    assert s.turbulence_mix == [0.0, 1 / 3, 1 / 3, 1 / 3]
    cdf = list(s.pod().sim.turb_cdf)
    assert cdf[0] == 0.0 and cdf[1] == 1 / 3 and cdf[3] == 1.0
    # 0.1 + 0.2 + 0.7 is 1 - 1.1e-16 in fp64: accepted, and the last level with a probability is forced to 1
    s = _cc(sim_config_kw={"turbulence": True, "turbulence_intensity": {"values": ["none", "light", "moderate"],
                                                                         "probabilities": [0.1, 0.2, 0.7]}})
    assert list(s.pod().sim.turb_cdf)[2:] == [1.0, 1.0]


def test_string_intensity_compiles_as_before():
    """Every shipped env configuration, turbulence off / light / moderate / severe, fp64 / fp32: the POD is byte for byte
    what the previous ABI (10) compiled - tests/golden/pod_sha256_abi10.json holds the SHA-256 of those PODs - once the
    appended tail of fw_sim_t is taken out (and the ABI number put back), and that tail is all zero."""
    from fwgym_b200 import _capi
    want = json.load(open(os.path.join(GOLDEN, "pod_sha256_abi10.json")))
    S = _capi.STRUCTS["fw_sim_t"]
    tail0 = S.turb_mixed.offset
    sim0 = _capi.fw_config_t.sim.offset
    assert len(want) == len(ENV_CONFIGS) * 4 * 2
    for key, digest in want.items():
        cfg, ti, prec = key.split("|")
        kw = {"turbulence": False} if ti == "off" else {"turbulence": True, "turbulence_intensity": ti}
        pod = _cc(cfg, sim_config_kw=kw, precision=prec).pod()
        assert pod.sim.turb_mixed == 0
        raw = bytes(memoryview(pod).cast("B"))
        tail = raw[sim0 + tail0:sim0 + S.turb_D.offset + S.turb_D.size]
        assert tail == bytes(len(tail)), key
        # the tail starts in the old struct's end padding: the old fw_sim_t ended at the next 8-byte boundary
        old_sim_end = (tail0 + 7) // 8 * 8
        old = np.int32(10).tobytes() + raw[4:sim0 + tail0] + bytes(old_sim_end - tail0) + raw[sim0 + ctypes.sizeof(S):]
        assert hashlib.sha256(old).hexdigest() == digest, key


def _philox_np(env, tick, stream, idx, k0, k1):
    """Vectorised Philox4x32-10 (numpy uint64 arithmetic), restated independently of oracle/philox.py."""
    M0, M1, W0, W1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
    m32 = np.uint64(0xFFFFFFFF)
    c0, c1 = env.astype(np.uint64), tick.astype(np.uint64)
    c2, c3 = np.full_like(c0, stream), np.full_like(c0, idx)
    k0, k1 = k0.astype(np.uint64), k1.astype(np.uint64)
    for _ in range(10):
        p0, p1 = M0 * c0, M1 * c2
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ k0) & m32, p1 & m32, ((p0 >> np.uint64(32)) ^ c3 ^ k1) & m32, p0 & m32
        k0, k1 = (k0 + W0) & m32, (k1 + W1) & m32
    return c0, c1


def _draw_np(seeds, envs, ticks, cdf):
    w0, w1 = _philox_np(envs, ticks, RS_TURBLVL, 0, seeds & 0xFFFFFFFF, seeds >> np.uint64(32))
    u = ((w0 >> np.uint64(5)).astype(np.float64) * 67108864.0 + (w1 >> np.uint64(6)).astype(np.float64)) \
        * (1.0 / 9007199254740992.0)
    return np.searchsorted(np.asarray(cdf), u, side="right"), u


def test_level_draw_mirror_matches_numpy_restatement():
    """The CPU mirror of the reset's level draw (oracle Philox, stream 5, index 0, at the reset's tick, then the first
    level whose cumulative probability exceeds the uniform) against an independent numpy restatement on 10^5 keys."""
    from fwgym_b200.config import turbulence_cdf
    rs = np.random.RandomState(7)
    n = 100000
    seeds = rs.randint(0, 2 ** 63, n, dtype=np.int64).astype(np.uint64)
    envs = rs.randint(0, 2 ** 32, n, dtype=np.int64).astype(np.uint64)
    ticks = rs.randint(0, 2 ** 32, n, dtype=np.int64).astype(np.uint64)
    cdf = turbulence_cdf([0.1, 0.2, 0.3, 0.4])
    lv_np, u_np = _draw_np(seeds, envs, ticks, cdf)
    for i in range(n):
        key = philox.PhiloxKey(int(seeds[i]), int(envs[i]))
        assert key.uniform01(int(ticks[i]), RS_TURBLVL, 0) == u_np[i]
        assert drawn_level(int(seeds[i]), int(envs[i]), int(ticks[i]), cdf) == lv_np[i]


@pytest.mark.parametrize("probs", [[0.1, 0.2, 0.3, 0.4], [0.0, 1 / 3, 1 / 3, 1 / 3], [0.25, 0.0, 0.75, 0.0]])
def test_level_draw_frequencies(probs):
    """chi^2 of 2 x 10^5 draws (fixed seed, consecutive env ids and ticks) against the configured probabilities; levels
    with probability 0 are never drawn."""
    from scipy.stats import chisquare
    from fwgym_b200.config import turbulence_cdf
    n = 200000
    envs = np.arange(n, dtype=np.uint64) % np.uint64(4096)
    ticks = np.arange(n, dtype=np.uint64) // np.uint64(4096)
    lv, _ = _draw_np(np.full(n, 20261020, dtype=np.uint64), envs, ticks, turbulence_cdf(probs))
    counts = np.bincount(lv, minlength=4)
    p = np.asarray(probs)
    assert (counts[p == 0] == 0).all()
    assert chisquare(counts[p > 0], n * p[p > 0]).pvalue > 1e-3


def _shape_list():
    src = open(os.path.join(ROOT, "fixed-wing-gym_b200", "csrc", "env_shapes_gen.h")).read()
    return re.search(r"#define FW_SHAPE_LIST\(X\) (.*)", src).group(1).replace("X(", "").replace(")", "").split()


def _shape_sim_ints(name):
    """Integer fields of fw_shape_sim_<name>() in env_shapes_gen.h (what fw_sim_same_shape compares)."""
    src = open(os.path.join(ROOT, "fixed-wing-gym_b200", "csrc", "env_shapes_gen.h")).read()
    body = re.search(r"constexpr fw_sim_t fw_shape_sim_%s\(\) \{(.*?)return s;" % name, src, re.S).group(1)
    return dict(re.findall(r"s\.(\w+) = (-?\d+)u?;", body))


def test_mixed_config_selects_only_its_twin_shape():
    """fw_sim_same_shape compares turb_mixed: a mixed configuration matches no shape generated from a string intensity,
    and the bench configuration's mixed twin (default_turb_mixed) is generated from a mixed configuration that differs
    from default_turb in turb_mixed only; the generated file is what the generator writes now."""
    import importlib.util
    spec = importlib.util.spec_from_file_location("gen_env_shapes", os.path.join(ROOT, "scripts", "gen_env_shapes.py"))
    gen = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(gen)
    assert open(gen.OUT).read() == gen.render()
    names = _shape_list()
    assert "default_turb_mixed" in names
    for name in names:
        mixed = _shape_sim_ints(name).get("turb_mixed") == "1"
        assert mixed == (name == "default_turb_mixed"), name
    a, b = _shape_sim_ints("default_turb"), _shape_sim_ints("default_turb_mixed")
    assert {k: v for k, v in b.items() if k != "turb_mixed"} == a
    src = open(os.path.join(ROOT, "fixed-wing-gym_b200", "csrc", "env_shapes.h")).read()
    assert "a.turb_mixed != b.turb_mixed" in src
