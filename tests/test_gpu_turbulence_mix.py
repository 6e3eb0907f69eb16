"""Per-env Dryden intensity on the GPU (mixed handles: sim_config_kw turbulence_intensity = {"values", "probabilities"}).

An env's level (0 none, 1 light, 2 moderate, 3 severe) is fixed for an episode and chosen at its reset: pinned with
set_turbulence_intensity, or drawn from the handle's distribution with one uniform of Philox stream 5.  An env at level
l must compute bitwise what the same global env computes on a handle of that uniform intensity (level 0: a handle with
turbulence off), so these tests hold mixed handles (1) bitwise to four uniform handles, (2) to the CPU mirror of the
draw and to sharding, (3) to the CPU oracle rebuilt at every reset at the drawn level, (4) across a checkpoint and
(5) in the batched multi-level evaluation.
"""
import os

import numpy as np
import pytest
import torch

from bench import CONFIG_KW, SIM_KW
from oracle import harness
from oracle.cases import CASES
import parity_utils as pu
from turbmix_utils import LEVELS, drawn_level, level_cdf, level_rollout

SEED = 20261017
STEPS = 300
TOL = 1e-9
BENCH = dict(config="fixed_wing_config.json", config_kw=CONFIG_KW, sim_kw=SIM_KW)
ALL4 = {"values": list(LEVELS)}
NEW_ROWS = ("turb_level_req", "turb_level")
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def sim_kw_at(c, level):
    """The case's sim_config_kw with the intensity replaced: a level name (uniform handle; "none" = turbulence off) or
    the dict form (mixed handle)."""
    kw = dict(c["sim_kw"])
    if isinstance(level, dict):
        kw.update(turbulence=True, turbulence_intensity=level)
    elif level == "none":
        kw["turbulence"] = False
    else:
        kw.update(turbulence=True, turbulence_intensity=level)
    return kw


def make_vec(c, n, level, precision="fp64", env_offset=0):
    from fwgym_b200 import FixedWingVecEnv
    v = FixedWingVecEnv(harness.config_path(c["config"]), n, config_kw=c["config_kw"],
                        sim_config_kw=sim_kw_at(c, level), seed=SEED, precision=precision, env_offset=env_offset)
    v.enable_f64_outputs(True)
    return v


def bits(x):
    return x.view({torch.float32: torch.int32, torch.float64: torch.int64}.get(x.dtype, x.dtype))


def outputs(v):
    """Everything a step returns (after step_tensors): float32 / float64 observations and rewards, done, termination
    code and dopri5 attempts, as bit patterns."""
    return [bits(v._obs), bits(v._rew), bits(v._obs64), bits(v._rew64), v._done, v._term, v.last_attempts()]


OUT_NAMES = ("obs", "reward", "obs64", "reward64", "done", "term", "attempts")


def assert_rows_equal(got, want, mask, what):
    g, w = got[mask], want[mask]
    if not torch.equal(g, w):
        bad = torch.nonzero((g != w).reshape(g.shape[0], -1).any(1)).flatten()
        env = torch.nonzero(mask).flatten()[bad[0]]
        raise AssertionError("%s differs on %d envs, first env %d" % (what, len(bad), int(env)))


def state_without_level_rows(v):
    rows = v.state_rows()
    keep = [i for i, r in enumerate(rows) if r not in NEW_ROWS]
    return [rows[i] for i in keep], bits(v.get_state()[torch.as_tensor(keep, device=v.device)])


def actions(n, steps, seed=11, dtype=torch.float32):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return (torch.rand((steps, n, 3), generator=g, device="cuda") * 2 - 1).to(dtype)


def pinned_levels(n, pattern):
    if pattern == "mod4":
        return torch.arange(n, dtype=torch.int32, device="cuda") % 4
    g = torch.Generator(device="cuda")
    g.manual_seed(3)
    return torch.randint(0, 4, (n,), generator=g, device="cuda", dtype=torch.int32)


# ---------------------------------------------------------------------------------------------------------------------
# 1. pinned levels are bitwise the uniform handles
# ---------------------------------------------------------------------------------------------------------------------
PINNED = {
    "bench_4096_mod4": (BENCH, 4096, "fp64", "mod4"),
    "bench_4096_random": (BENCH, 4096, "fp64", "random"),
    "bench_65536_mod4": (BENCH, 65536, "fp64", "mod4"),
    "bench_65536_fp32_random": (BENCH, 65536, "fp32", "random"),
    "bench_4096_fp32_mod4": (BENCH, 4096, "fp32", "mod4"),
    "wind_mod4": (CASES["wind"], 4096, "fp64", "mod4"),
    "wind_random": (CASES["wind"], 4096, "fp64", "random"),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(PINNED))
def test_pinned_levels_equal_uniform_handles(built_lib, case):
    """A mixed handle whose envs are pinned to levels (env % 4, or a seeded random assignment) against four uniform
    handles (turbulence off, light, moderate, severe) with the same seed, N and offset, 300 steps with auto-resets on the
    same actions: every env's outputs bitwise equal to those of the handle of its level after every step, and all its
    state rows (except the two level rows) at the end."""
    c, n, prec, pattern = PINNED[case]
    lv = pinned_levels(n, pattern)
    handles = []
    try:
        mixed = make_vec(c, n, ALL4, prec)
        handles.append(mixed)
        mixed.set_turbulence_intensity(lv)
        uni = [make_vec(c, n, name, prec) for name in LEVELS]
        handles += uni
        if c is BENCH:
            assert mixed.kernel_variant().endswith("env=default_turb_mixed"), mixed.kernel_variant()
        masks = [lv == l for l in range(4)]
        for v in handles:
            v.reset()
        assert torch.equal(mixed.turbulence_levels(), lv)
        for l in range(4):
            for name, x, y in zip(OUT_NAMES[:1], outputs(mixed)[:1], outputs(uni[l])[:1]):
                assert_rows_equal(x, y, masks[l], "%s reset %s at level %s" % (case, name, LEVELS[l]))
        acts = actions(n, STEPS)
        for t in range(STEPS):
            for v in handles:
                v.step_tensors(acts[t])
            got = outputs(mixed)
            for l in range(4):
                for name, x, y in zip(OUT_NAMES, got, outputs(uni[l])):
                    assert_rows_equal(x, y, masks[l], "%s step %d %s at level %s" % (case, t, name, LEVELS[l]))
        assert torch.equal(mixed.turbulence_levels(), lv)
        rows, st = state_without_level_rows(mixed)
        for l in range(4):
            assert uni[l].state_rows() == rows
            assert_rows_equal(st.T, bits(uni[l].get_state()).T, masks[l], "%s final state at level %s" % (case, LEVELS[l]))
        assert all(v.counters()["watchdog"] == 0 for v in handles)
        ends = sum(v.counters()["resets"] for v in uni)
        print("%s: %d envs x %d steps, levels %s, %d resets on the uniform handles" %
              (case, n, STEPS, [int(m.sum()) for m in masks], ends))
    finally:
        for v in handles:
            v.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. per-reset draws
# ---------------------------------------------------------------------------------------------------------------------
PROBS = {"values": list(LEVELS), "probabilities": [0.1, 0.2, 0.3, 0.4]}


@pytest.mark.gpu
def test_drawn_levels_follow_the_mirror(built_lib):
    """Dict form: after the reset and after every step, each env's active level is the CPU mirror's draw for the tick
    of the reset that started its episode (state row episode_tick), the requested level stays -1, and every level
    occurs."""
    n, steps = 4096, STEPS
    cdf = level_cdf(PROBS["probabilities"])
    v = make_vec(BENCH, n, PROBS)
    try:
        rows = v.state_rows()
        r_tick, r_req = rows.index("episode_tick"), rows.index("turb_level_req")
        v.reset()
        acts = actions(n, steps)
        known = {}
        seen = np.zeros(4, dtype=np.int64)
        n_draws = 0
        for t in range(steps + 1):
            if t:
                v.step_tensors(acts[t - 1])
            tick = v.get_rows(r_tick, 1)[0].cpu().numpy().astype(np.int64)
            got = v.turbulence_levels().cpu().numpy()
            for e in range(n):
                key = (e, int(tick[e]))
                if key not in known:
                    known[key] = drawn_level(SEED, e, int(tick[e]), cdf)
                    seen[known[key]] += 1
                    n_draws += 1
                assert got[e] == known[key], (t, e, int(tick[e]), int(got[e]), known[key])
        assert (v.get_rows(r_req, 1)[0] == -1).all()
        assert (seen > 0).all()
        print("drawn levels: %d episode starts, level counts %s" % (n_draws, seen.tolist()))
    finally:
        v.close()


@pytest.mark.gpu
def test_one_hot_distribution_equals_pinned_handle(built_lib):
    """probabilities [0, 0, 1, 0] (every reset draws moderate) == the same mixed handle with every env pinned to
    moderate, bitwise, outputs and state, 300 steps."""
    n = 4096
    a = make_vec(BENCH, n, {"values": list(LEVELS), "probabilities": [0, 0, 1, 0]})
    b = make_vec(BENCH, n, ALL4)
    try:
        b.set_turbulence_intensity("moderate")
        a.reset(), b.reset()
        acts = actions(n, STEPS)
        every = torch.ones(n, dtype=torch.bool, device="cuda")
        for t in range(STEPS):
            a.step_tensors(acts[t]), b.step_tensors(acts[t])
            for name, x, y in zip(OUT_NAMES, outputs(a), outputs(b)):
                assert_rows_equal(x, y, every, "step %d %s" % (t, name))
        assert (a.turbulence_levels() == 2).all()
        ra, sa = state_without_level_rows(a)
        rb, sb = state_without_level_rows(b)
        assert ra == rb and torch.equal(sa, sb)
    finally:
        a.close(), b.close()


@pytest.mark.gpu
def test_drawn_levels_are_sharding_invariant(built_lib):
    """Two mixed handles with env_offset 0 and N/2 together == one N-env handle, bitwise (the draw is keyed by the
    global env id), including the level rows."""
    n = 4096
    whole = make_vec(BENCH, n, PROBS)
    halves = [make_vec(BENCH, n // 2, PROBS, env_offset=o) for o in (0, n // 2)]
    try:
        for v in [whole] + halves:
            v.reset()
        acts = actions(n, STEPS)
        every = torch.ones(n, dtype=torch.bool, device="cuda")
        for t in range(STEPS):
            whole.step_tensors(acts[t])
            halves[0].step_tensors(acts[t, :n // 2].contiguous())
            halves[1].step_tensors(acts[t, n // 2:].contiguous())
            for j, name in enumerate(OUT_NAMES):
                cat = torch.cat([outputs(h)[j] for h in halves])
                assert_rows_equal(outputs(whole)[j], cat, every, "step %d %s" % (t, name))
        st = torch.cat([bits(h.get_state()) for h in halves], dim=1)
        assert torch.equal(bits(whole.get_state()), st)
    finally:
        for v in [whole] + halves:
            v.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. oracle parity under drawn levels
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_drawn_levels_match_oracle(built_lib):
    """512 envs of the bench configuration, 250 steps, levels drawn over all four: the CPU oracle rebuilds its Dryden
    model at every reset at the level the mirror draws (tests/turbmix_utils.py).  A free-running handle and a second one
    set to the oracle's states after every step, in lockstep: done flags and attempt counts exact, active levels equal to
    the oracle's, <= 1e-9 per step on identical states, <= 1e-4 free-running (the bars of BASELINE configs[1])."""
    n, steps = 512, 250
    probs = {"values": list(LEVELS), "probabilities": [0.25, 0.25, 0.25, 0.25]}
    cdf = level_cdf(probs["probabilities"])
    acts = actions(n, steps)
    oracle_kw = dict(BENCH["sim_kw"], turbulence=True, turbulence_intensity="light")
    want = level_rollout(harness.config_path(BENCH["config"]), BENCH["config_kw"], oracle_kw, SEED, np.arange(n),
                         acts.double().cpu().numpy(), cdf)
    free, sync = make_vec(BENCH, n, probs), make_vec(BENCH, n, probs)
    try:
        rows = sync.state_rows()
        ridx = torch.as_tensor([rows.index(r) for r in pu.STATE_ROWS], device="cuda")
        worst = {"free": 0.0, "sync": 0.0}
        for v in (free, sync):
            v.reset()
            assert np.array_equal(v.turbulence_levels().cpu().numpy(), want["level"][0])
            assert pu.rel_err(v._obs64.cpu().numpy(), want["obs"][0], 1e-3).max() <= TOL
        for t in range(steps):
            for tag, v in (("free", free), ("sync", sync)):
                _, _, done, _ = v.step_tensors(acts[t])
                assert np.array_equal(done.cpu().numpy().astype(bool), want["done"][t]), (tag, t)
                assert np.array_equal(v.last_attempts().cpu().numpy(), want["k"][t]), (tag, t)
                assert np.array_equal(v.turbulence_levels().cpu().numpy(), want["level"][t + 1]), (tag, t)
                err = max(pu.rel_err(v._obs64.cpu().numpy(), want["obs"][t + 1], 1e-3).max(),
                          pu.rel_err(v._rew64.cpu().numpy(), want["rew"][t], 1e-3).max(),
                          pu.rel_err(pu.gpu_state(v), want["state"][t], 1e-3).max())
                worst[tag] = max(worst[tag], float(err))
            st = sync.get_state()
            st[ridx] = torch.as_tensor(want["state"][t].T.copy(), device="cuda")
            sync.set_state(st)
        counts = np.bincount(want["level"].ravel(), minlength=4)
        print("oracle parity under drawn levels: %d envs x %d steps, %d episode ends, level-steps %s, worst rel err per "
              "step %.2e, free-running %.2e" % (n, steps, int(want["done"].sum()), counts.tolist(), worst["sync"],
                                                worst["free"]))
        assert (counts > 0).all()
        assert worst["sync"] <= TOL and worst["free"] <= 1e-4, worst
    finally:
        free.close(), sync.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. checkpointing
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_checkpoint_keeps_levels(built_lib):
    """get_state -> set_state onto a fresh mixed handle (drawn levels, some envs pinned) continues bitwise: the requested
    and active levels travel with the state."""
    n = 4096
    a = make_vec(BENCH, n, PROBS)
    try:
        a.set_turbulence_intensity(["severe"] * 100 + ["none"] * 100, indices=np.arange(200))
        a.reset()
        acts = actions(n, 2 * 150)
        for t in range(150):
            a.step_tensors(acts[t])
        ck = a.get_state().clone()
        b = make_vec(BENCH, n, PROBS)
        try:
            b.set_state(ck)
            assert torch.equal(b.turbulence_levels(), a.turbulence_levels())
            every = torch.ones(n, dtype=torch.bool, device="cuda")
            for t in range(150, 300):
                a.step_tensors(acts[t]), b.step_tensors(acts[t])
                for name, x, y in zip(OUT_NAMES[:6], outputs(a)[:6], outputs(b)[:6]):
                    assert_rows_equal(x, y, every, "step %d %s" % (t, name))
            assert torch.equal(bits(a.get_state()), bits(b.get_state()))
            rows = b.state_rows()
            req = b.get_rows(rows.index("turb_level_req"), 1)[0]
            assert (req[:100] == 3).all() and (req[100:200] == 0).all() and (req[200:] == -1).all()
        finally:
            b.close()
    finally:
        a.close()


@pytest.mark.gpu
def test_level_api(built_lib):
    """set_turbulence_intensity / turbulence_levels / get_attr on mixed and uniform handles."""
    from fwgym_b200 import _capi
    m = make_vec(BENCH, 64, ALL4)
    u = make_vec(BENCH, 64, "moderate")
    try:
        m.set_turbulence_intensity("light")
        m.set_turbulence_intensity(["severe", "none"], indices=[3, 5])
        m.reset()
        assert m.get_attr("turbulence_intensity", indices=[0, 3, 5]) == ["light", "severe", "none"]
        m.set_turbulence_intensity(torch.full((64,), -1, dtype=torch.int32))
        with pytest.raises(ValueError):
            m.set_turbulence_intensity([4] * 64)
        with pytest.raises(_capi.FwError):
            u.set_turbulence_intensity("light")
        assert u.get_attr("turbulence_intensity", indices=[0]) == ["moderate"]
        assert int(m._lib.fw_set_turbulence_levels(u._h, None, None)) == _capi.ENUMS["FW_ERR_ARG"]
    finally:
        m.close(), u.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. the four-level evaluation as one batch
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_four_level_evaluation_equals_single_level_calls(built_lib):
    """evaluate_on_set over ["none", "light", "moderate", "severe"] (100 scenarios x 4 levels = one batch of 400 envs,
    PID controller) == four single-level calls with env_offset = j * S, bitwise: rewards, lengths, episode rows."""
    from fwgym_b200 import evaluate
    scen = evaluate.load_test_set(os.path.join(GOLDEN, "test_set_wind_none.npz"))
    cfg = harness.config_path("fixed_wing_config_examples.json")
    S = len(scen)
    res, vec = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, turbulence_intensity=list(LEVELS))
    vec.close()
    assert list(res) == list(LEVELS)
    for j, lv in enumerate(LEVELS):
        one, v1 = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, turbulence_intensity=lv,
                                           env_offset=j * S)
        v1.close()
        assert np.array_equal(res[lv]["lengths"], one["lengths"]), lv
        assert np.array_equal(res[lv]["episode_rows"].view(np.int64), one["episode_rows"].view(np.int64)), lv
        for a, b in zip(res[lv]["rewards"], one["rewards"]):
            assert np.array_equal(a.view(np.int64), b.view(np.int64)), lv
        print("%-8s mean length %.1f, success_all %.2f" % (lv, float(np.mean(one["lengths"])),
                                                            evaluate.summarise(one).get("success_all", float("nan"))))
