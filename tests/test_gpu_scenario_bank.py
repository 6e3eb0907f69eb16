"""Scenario banks on the GPU: resets that take their initial states and targets from a device table, in order, with one
result row per scenario (include/fwgym.h fw_bank_t).

A banked episode must be bitwise the episode an explicit masked fw_reset with the scenario's columns starts at the same
tick, so the tests hold (1) a bank handle to a handle without a bank whose done envs are reset by hand with the columns
the bank's cursor names, on the specialised and on the generic kernels, (2) the result rows to what the step outputs
reported, (3) the banked evaluation to the one-env-per-scenario evaluation, (4) sharded and checkpointed runs to one
uninterrupted run, and (5) the C-ABI to its argument errors.
"""
import ctypes
import os

import numpy as np
import pytest
import torch

from bench import CONFIG_KW, SIM_KW
from oracle import harness

SEED = 20261022
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
BANK_ROWS = ("bank_next", "bank_scenario")
LEVELS = ("none", "light", "moderate", "severe")


def bits(x):
    return x.view({torch.float32: torch.int32, torch.float64: torch.int64}.get(x.dtype, x.dtype))


def make_vec(n, bank=True, config="fixed_wing_config.json", config_kw=None, sim_kw=None, **kw):
    from fwgym_b200 import FixedWingVecEnv
    ckw = dict(CONFIG_KW if config_kw is None else config_kw)
    v = FixedWingVecEnv(harness.config_path(config), n, config_kw=ckw, sim_config_kw=dict(SIM_KW if sim_kw is None
                                                                                          else sim_kw),
                        seed=SEED, scenario_bank=bank, **kw)
    v.enable_f64_outputs(True)
    return v


def bank_columns(S, seed=5):
    """Per-scenario initial states / targets with NaN holes (those entries are sampled at the reset)."""
    rs = np.random.RandomState(seed)

    def col(lo, hi, holes=0.25):
        v = rs.uniform(lo, hi, S)
        v[rs.uniform(size=S) < holes] = np.nan
        return v
    state = {"roll": col(-0.3, 0.3), "pitch": col(-0.2, 0.2), "velocity_u": col(18.0, 24.0), "omega_q": col(-0.1, 0.1)}
    target = {"roll": col(-0.5, 0.5), "Va": col(17.0, 23.0)}
    return state, target


def state_without_bank_rows(v):
    rows = v.state_rows()
    keep = torch.as_tensor([i for i, r in enumerate(rows) if r not in BANK_ROWS], device=v.device)
    return bits(v.get_state()[keep])


def actions(n, steps, seed=3):
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    return torch.rand((steps, n, 3), generator=g, device="cuda", dtype=torch.float32) * 2 - 1


# ---------------------------------------------------------------------------------------------------------------------
# 1. banked resets == explicit masked resets with the scenario's columns
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("generic", [False, True], ids=["default_turb_bank", "generic_bank"])
def test_banked_resets_equal_explicit_resets(built_lib, monkeypatch, generic):
    """Bench configuration (Dryden gusts, observation noise), steps_max 40, 150 steps: every env flies >= 3 episodes, the
    bank (3 N scenarios) runs out on the way, so the last episodes fall back to sampling.  Handle B (same seed, no bank,
    auto_reset off) resets its done envs after every step with the columns A's cursor gave them; obs / reward / done /
    termination code, A's terminal observations and the whole state (minus the bank rows) must be bitwise equal."""
    if generic:
        monkeypatch.setenv("FWGYM_FORCE_GENERIC", "1")
    N, S, T = 256, 768, 150
    ckw = dict(CONFIG_KW, steps_max=40)
    A = make_vec(N, config_kw=ckw, keep_terminal_obs=True)
    B = make_vec(N, bank=False, config_kw=ckw, auto_reset=False)
    assert A.kernel_variant().endswith("env=" + ("generic_bank" if generic else "default_turb_bank"))
    assert B.kernel_variant().endswith("env=" + ("generic" if generic else "default_turb"))
    state, target = bank_columns(S)
    A.set_scenario_bank(state=state, target=target)
    st_tab, tg_tab = A._bank[0]["init_state"], A._bank[0]["init_target"]

    def columns(ids):
        fly = (ids >= 0).unsqueeze(0)
        idx = ids.clamp(min=0).long()
        return (torch.where(fly, st_tab[:, idx], torch.full_like(st_tab[:, idx], float("nan"))).contiguous(),
                torch.where(fly, tg_tab[:, idx], torch.full_like(tg_tab[:, idx], float("nan"))).contiguous())

    A.reset()
    ids = A.scenario_ids()
    assert torch.equal(ids.cpu(), torch.arange(N, dtype=torch.int32))
    s0, t0 = columns(ids)
    B._lib.fw_reset(B._h, None, B._ptr(s0), B._ptr(t0), None, 0, B._ptr(B._obs), B._ptr(B._obs64), B._stream())
    assert torch.equal(bits(A._obs64), bits(B._obs64))
    episodes = torch.zeros(N, dtype=torch.long, device="cuda")
    acts = actions(N, T)
    for t in range(T):
        A.step_tensors(acts[t])
        B.step_tensors(acts[t])
        done = A._done.bool()
        assert torch.equal(A._done, B._done) and torch.equal(A._term, B._term), t
        assert torch.equal(bits(A._rew64), bits(B._rew64)) and torch.equal(bits(A._rew), bits(B._rew)), t
        assert torch.equal(bits(A._term_obs[done]), bits(B._obs[done])), t      # B has not reset yet
        episodes += done.long()
        if done.any():
            si, ti = columns(A.scenario_ids())
            mask = done.to(torch.uint8)
            B._lib.fw_reset(B._h, B._ptr(mask), B._ptr(si), B._ptr(ti), None, 0, B._ptr(B._obs), B._ptr(B._obs64),
                            B._stream())
            B._keep = (mask, si, ti)
        assert torch.equal(bits(A._obs), bits(B._obs)) and torch.equal(bits(A._obs64), bits(B._obs64)), t
        assert torch.equal(state_without_bank_rows(A), state_without_bank_rows(B)), t
    assert int(episodes.min()) >= 3
    res = A.scenario_results()
    flown = res["episodes"].cpu().numpy()
    assert flown.max() == 1 and flown.sum() == S          # every scenario once, then the envs sampled
    assert (A.get_named_state(["bank_next"])["bank_next"] == S).all()
    A.close()
    B.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. result rows
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_result_rows_match_step_outputs(built_lib):
    """Metrics on (generic bank kernels): for every banked episode, the scenario's term / length / return / metric row
    equal the step's termination code and the env's episode row, bitwise; each scenario is flown once."""
    N, S = 64, 200
    A = make_vec(N, config_kw=dict(CONFIG_KW, steps_max=30), metrics=True)
    assert A.kernel_variant().endswith("env=generic_bank")
    state, target = bank_columns(S, seed=9)
    res = A.set_scenario_bank(state=state, target=target)
    A.reset()
    seen = {}
    acts = actions(N, 160, seed=4)
    for t in range(160):
        ids = A.scenario_ids().long()
        A.step_tensors(acts[t])
        done = A._done.bool() & (ids >= 0)
        if done.any():
            sc = ids[done]
            ep = A.episode_metrics()[done]
            assert torch.equal(res["term"][sc], A._term[done])
            assert torch.equal(res["length"][sc].double(), ep[:, 1])
            assert torch.equal(bits(res["return"][sc]), bits(ep[:, 0]))
            assert torch.equal(bits(res["episode"][sc]), bits(ep))
            for s in sc.cpu().numpy():
                assert s not in seen
                seen[int(s)] = t
    assert sorted(seen) == list(range(S))
    assert (res["episodes"] == 1).all()
    assert torch.equal(res["successes"].bool(), res["episode"][:, 3] == 1.0)
    A.close()


@pytest.mark.gpu
def test_writes_stop_at_S_and_detach_restores_sampling(built_lib):
    """Raw C-ABI with guard regions behind every result buffer: nothing is written at or beyond S (a bank replaced by a
    smaller one while its episodes run).  A handle whose bank was detached before its reset flies bitwise like a handle
    that never had one."""
    from fwgym_b200 import _capi
    N, S, G = 32, 40, 64
    A = make_vec(N, config_kw=dict(CONFIG_KW, steps_max=20), metrics=True)
    d = A.device
    big_state, big_target = bank_columns(4 * S)
    A.set_scenario_bank(state=big_state, target=big_target, first=S)     # episodes with ids S .. 2S - 1 and beyond
    A.reset()
    term = torch.full((S + G,), -7, dtype=torch.int32, device=d)
    length = torch.full((S + G,), -7, dtype=torch.int32, device=d)
    ret = torch.full((S + G,), -7.0, dtype=torch.float64, device=d)
    epi = torch.full((S + G, A.ep_dim), -7.0, dtype=torch.float64, device=d)
    cnt = torch.zeros(2, S + G, dtype=torch.int32, device=d)
    b = _capi.fw_bank_t()
    b.n_scenarios, b.first, b.stride = S, 0, N
    b.term, b.length, b.ret, b.episode = term.data_ptr(), length.data_ptr(), ret.data_ptr(), epi.data_ptr()
    b.episodes, b.successes = cnt[0].data_ptr(), cnt[1].data_ptr()
    _capi.check(A._lib.fw_set_bank(A._h, ctypes.byref(b), A._stream()))
    # (attaching clears bank_scenario, so force the running episodes' ids back to S .. S + N - 1 through the state)
    st = A.get_state()
    st[A.state_rows().index("bank_scenario")] = torch.arange(S, S + N, dtype=torch.float64, device=d)
    A.set_state(st)
    for t, a in enumerate(actions(N, 80, seed=6)):
        A.step_tensors(a)
    torch.cuda.synchronize()
    assert (term[S:] == -7).all() and (length[S:] == -7).all() and (ret[S:] == -7.0).all() and (epi[S:] == -7.0).all()
    assert (cnt[:, S:] == 0).all()
    assert (cnt[0, :S] == 1).all() and (length[:S] > 0).all()          # the new bank was flown from 0
    A.close()
    # detach
    A = make_vec(N)
    C = make_vec(N, bank=False)
    A.set_scenario_bank(state=big_state, target=big_target)
    A.detach_scenario_bank()
    A.reset()
    C.reset()
    assert (A.scenario_ids() == -1).all()
    for a in actions(N, 60, seed=7):
        A.step_tensors(a)
        C.step_tensors(a)
        assert torch.equal(bits(A._obs64), bits(C._obs64)) and torch.equal(A._done, C._done)
    assert torch.equal(state_without_bank_rows(A), state_without_bank_rows(C))
    A.close()
    C.close()


@pytest.mark.gpu
def test_cycling_bank_and_level_column(built_lib):
    """A cycling bank of 7 scenarios on 16 envs (mixed handle): every episode start is from the bank, the counters add up
    to the banked episodes that ended, and every banked episode flies at its scenario's level (-1: the env's own rule,
    here pinned at 'light')."""
    N, S = 16, 7
    v = make_vec(N, config_kw=dict(CONFIG_KW, steps_max=15), sim_kw={"turbulence": True,
                                                                      "turbulence_intensity": {"values": list(LEVELS)}})
    v.set_turbulence_intensity("light")
    lv = np.array([0, 3, -1, 2, 1, 3, 0], dtype=np.int32)
    res = v.set_scenario_bank(state={"roll": np.linspace(-0.2, 0.2, S)}, turbulence_intensity=lv, stride=N + 3,
                              cycle=True)
    assert set(res) == {"episodes", "successes"}
    v.reset()
    ended = 0
    for a in actions(N, 60, seed=8):
        ids = v.scenario_ids().long()
        assert (ids >= 0).all()
        levels = v.turbulence_levels().long()
        want = torch.as_tensor(lv, device=v.device).long()[ids]
        assert torch.equal(levels, torch.where(want >= 0, want, torch.ones_like(want)))
        v.step_tensors(a)
        ended += int(v._done.sum())
    assert int(res["episodes"].sum()) == ended
    v.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3. banked evaluation
# ---------------------------------------------------------------------------------------------------------------------
def completed_test_set():
    """test_set_wind_none with every initial state entry filled in from one reset of a 100-env handle (so that nothing is
    sampled and a scenario starts the same on whichever env flies it)."""
    from fwgym_b200 import FixedWingVecEnv, evaluate
    scen = evaluate.load_test_set(os.path.join(GOLDEN, "test_set_wind_none.npz"))
    cfg = harness.config_path("fixed_wing_config_examples.json")
    v = FixedWingVecEnv(cfg, len(scen), config_kw=dict(evaluate.EVAL_CONFIG_KW, action={"scale_space": False}),
                        sim_config_kw={"turbulence": False}, seed=1)
    state, target = evaluate._scenario_columns(scen, 1)
    v.reset(state=state, target=target)
    names = ["roll", "pitch", "yaw", "omega_p", "omega_q", "omega_r", "position_n", "position_e", "position_d",
             "velocity_u", "velocity_v", "velocity_w", "elevon_left", "elevon_right", "throttle"]
    st = {k: x.cpu().numpy() for k, x in v.get_named_state(names).items()}
    v.close()
    out = []
    for i, s in enumerate(scen):
        d = {k: float(st[k][i]) for k in names}
        if "wind" in s["state"]:
            d["wind"] = s["state"]["wind"]
        out.append({"state": d, "target": dict(s["target"])})
    return out, cfg


def assert_same_outcomes(got, want, first_ids):
    assert np.array_equal(got["lengths"], want["lengths"])
    g, w = got["episode_rows"], want["episode_rows"]
    assert np.array_equal(g[:, 1:].view(np.int64), w[:, 1:].view(np.int64))      # every metric column
    for i in first_ids:                                                           # the env's first scenario
        assert g[i, 0].tobytes() == w[i, 0].tobytes()
        assert np.array_equal(got["rewards"][i].view(np.int64), want["rewards"][i].view(np.int64))


@pytest.mark.gpu
def test_banked_evaluation_equals_one_env_per_scenario(built_lib):
    """PID, turbulence off: 100 scenarios on 32 envs == 100 envs, bitwise in lengths and every metric column (returns and
    reward traces for each env's first scenario; a later scenario flies on an env that carries the reference's state
    from its earlier episodes, which test_banked_scenarios_against_the_oracle holds to the CPU oracle).  Four levels on
    32 envs: the 'none' block equals its single-level call likewise, and every scenario flies at its level."""
    from fwgym_b200 import evaluate
    scen, cfg = completed_test_set()
    one, v1 = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1)
    v1.close()
    banked, vb = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, num_envs=32)
    assert vb.num_envs == 32 and vb.kernel_variant().endswith("env=generic_bank")
    vb.close()
    assert_same_outcomes(banked, one, range(32))
    by_level, v4 = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1, num_envs=32,
                                            turbulence_intensity=list(LEVELS), keep_rewards=False)
    v4.close()
    assert list(by_level) == list(LEVELS) and by_level["none"]["rewards"] is None
    g, w = by_level["none"], one
    assert np.array_equal(g["lengths"], w["lengths"])
    assert np.array_equal(g["episode_rows"][:, 1:].view(np.int64), w["episode_rows"][:, 1:].view(np.int64))
    assert all((by_level[lv]["lengths"] > 0).all() for lv in LEVELS)
    # the same banked four-level run, stepped here: the Dryden level of every running episode is its scenario's
    S, N = len(scen), 32
    kw, sim_kw = evaluate._eval_kw(None, "pid", list(LEVELS), None)
    v = evaluate.FixedWingVecEnv(cfg, N, config_kw=kw, sim_config_kw=sim_kw, seed=1, metrics=True,
                                 scenario_bank=True)
    state, target = evaluate._scenario_columns(scen, len(LEVELS))
    res = v.set_scenario_bank(state=state, target=target,
                              turbulence_intensity=[lv for lv in LEVELS for _ in range(S)])
    v.reset()
    pid = evaluate.DevicePID(v)
    new = torch.ones(N, dtype=torch.bool, device=v.device)
    flown = torch.full((len(LEVELS) * S,), -1, dtype=torch.long, device=v.device)
    for _ in range(20000):
        ids = v.scenario_ids().long()
        on = ids >= 0
        lvl = v.turbulence_levels().long()
        assert torch.equal(lvl[on], ids[on] // S)
        flown[ids[on]] = lvl[on]
        _, _, done, _ = v.step_tensors(pid(new))
        new = done.bool()
        if bool((res["length"] >= 0).all()):
            break
    assert torch.equal(flown, torch.arange(len(LEVELS) * S, device=v.device) // S)
    v.close()


# ---------------------------------------------------------------------------------------------------------------------
# 3b. banked scenarios against the CPU oracle, oracle envs reused across episodes
# ---------------------------------------------------------------------------------------------------------------------
def _examples_oracle_case():
    """The evaluation setting of the examples configuration (PID, physical actions, turbulence off) with a short
    episode cap, a streak of 20 steps that the PID reaches (on_success done), and an integrator observation, whose
    value at a reset reads the previous episode's error history (fixed_wing.py:317 before :318)."""
    from fwgym_b200 import evaluate
    kw = dict(evaluate.EVAL_CONFIG_KW, action={"scale_space": False}, steps_max=150, integration_window=10,
              observation={"states": {6: {"value": "integrator"}}})
    kw["target"] = dict(kw["target"], success_streak_req=20)
    return dict(config="fixed_wing_config_examples.json", config_kw=kw, controller="pid", steps=450)


def _zoo_oracle_case():
    """Every reward class, including the success reward the goal-achieved latch (fixed_wing.py:51,382) pays only on the
    first success of an env object, under random actions."""
    from oracle.cases import CASES
    kw = dict(CASES["reward_zoo"]["config_kw"], steps_max=40)
    return dict(config="fixed_wing_config_zoo.json", config_kw=kw, controller="random", steps=130)


@pytest.mark.gpu
@pytest.mark.parametrize("case", ["examples", "zoo"])
def test_banked_scenarios_against_the_oracle(built_lib, case):
    """64 envs fly test-set scenarios through a bank (3 N of them, so the last episodes fall back to sampling) next to
    64 CPU oracle envs that are reused across episodes and reset, when an episode ends, with the scenario the cursor rule
    names for that env.  Every step: observations, rewards and the 27 state values within 1e-9, done and dopri5 attempt
    counts exact; the scenario ids the device reports are the rule's.  Some banked episodes must start on an env whose
    goal-achieved latch an earlier episode set."""
    import parity_utils as pu
    from fwgym_b200 import evaluate, scenario_bank
    c = _examples_oracle_case() if case == "examples" else _zoo_oracle_case()
    N, TOL, seed = 64, 1e-9, 7
    scen_all = evaluate.load_test_set(os.path.join(GOLDEN, "test_set_wind_none.npz"))
    S = 3 * N
    scen = [scen_all[i % len(scen_all)] for i in range(S)]
    cfg = harness.config_path(c["config"])
    sim_kw = {"turbulence": False}
    from fwgym_b200 import FixedWingVecEnv
    v = FixedWingVecEnv(cfg, N, config_kw=c["config_kw"], sim_config_kw=sim_kw, seed=seed, scenario_bank=True)
    v.enable_f64_outputs(True)
    state, target = evaluate._scenario_columns(scen, 1)
    v.set_scenario_bank(state=state, target=target)
    orcs = [harness.OracleRunner(harness.make_env("restated", cfg, c["config_kw"], sim_kw), seed, e, auto_reset=False)
            for e in range(N)]
    k = np.zeros(N, dtype=np.int64)                     # banked episodes started per env

    def start(e):
        sid = int(scenario_bank.scenario_of(e, k[e], S, 0, N, False))
        k[e] += 1
        if sid < 0:
            return sid, orcs[e].reset()
        return sid, orcs[e].reset(state=dict(scen[sid]["state"]), target=dict(scen[sid]["target"]))

    v.reset()
    first = [start(e) for e in range(N)]
    assert np.array_equal(v.scenario_ids().cpu().numpy(), [f[0] for f in first])
    obs_o = np.stack([np.asarray(f[1], dtype=np.float64).ravel() for f in first])
    assert pu.rel_err(v._obs64.cpu().numpy(), obs_o, 1e-3).max() <= TOL
    pid = evaluate.DevicePID(v) if c["controller"] == "pid" else None
    rs = np.random.RandomState(3)
    new = torch.ones(N, dtype=torch.bool, device=v.device)
    flags_row = v.state_rows().index("flags")
    latched_starts, episodes = 0, np.zeros(N, dtype=np.int64)
    for t in range(c["steps"]):
        if pid is not None:
            a = pid(new).clone()
        else:
            a = torch.as_tensor(rs.uniform(-1.2, 1.2, (N, 3)), device=v.device)
        ah = a.cpu().numpy()
        v.step_tensors(a)
        res = [o.step(ah[e]) for e, o in enumerate(orcs)]
        done_o = np.array([r[2] for r in res])
        done_g = v._done.cpu().numpy().astype(bool)
        assert np.array_equal(done_g, done_o), t
        assert np.array_equal(v.last_attempts().cpu().numpy(), [o.attempts_last() for o in orcs]), t
        assert pu.rel_err(v._rew64.cpu().numpy(), np.array([r[1] for r in res]), 1e-3).max() <= TOL, t
        obs_o = np.stack([np.asarray(r[0], dtype=np.float64).ravel() for r in res])
        ids = v.scenario_ids().cpu().numpy()
        flags = v.get_rows(flags_row, 1)[0].cpu().numpy().astype(np.int64)
        for e in np.nonzero(done_o)[0]:
            sid, ob = start(e)
            assert ids[e] == sid, (t, e)
            obs_o[e] = np.asarray(ob, dtype=np.float64).ravel()
            episodes[e] += 1
            if sid >= 0 and flags[e] & 1:
                latched_starts += 1
        assert pu.rel_err(v._obs64.cpu().numpy(), obs_o, 1e-3).max() <= TOL, t
        assert pu.rel_err(pu.gpu_state(v), np.stack([o.ode_state() for o in orcs]), 1e-3).max() <= TOL, t
        new = v._done.bool()
    assert episodes.min() >= 2 and episodes.mean() >= 3, episodes
    assert latched_starts > 0
    print("%s: %d episodes, %d banked starts on latched envs" % (case, int(episodes.sum()), latched_starts))
    v.close()


# ---------------------------------------------------------------------------------------------------------------------
# 4. sharding and checkpoints
# ---------------------------------------------------------------------------------------------------------------------
def run_bank(vecs, S, steps, acts, firsts, stride, snapshot_at=None):
    state, target = bank_columns(S, seed=13)
    res = [v.set_scenario_bank(state=state, target=target, first=f, stride=stride) for v, f in zip(vecs, firsts)]
    for v in vecs:
        v.reset()
    snap = None
    for t in range(steps):
        if t == snapshot_at:
            snap = ([v.get_state().clone() for v in vecs], [{k: x.clone() for k, x in r.items()} for r in res])
        off = 0
        for v in vecs:
            v.step_tensors(acts[t][off:off + v.num_envs].contiguous())
            off += v.num_envs
    return res, snap


def merged(results):
    """Result rows of several handles that share one bank: counters add up, each outcome row comes from the handle that
    flew the scenario."""
    out = {}
    for k in results[0]:
        x = torch.stack([r[k] for r in results])
        if k in ("episodes", "successes"):
            out[k] = x.sum(0)
        else:
            flew = torch.stack([r["length"] >= 0 for r in results]).long().argmax(0)
            out[k] = x[flew, torch.arange(x.shape[1], device=x.device)]
    return out


@pytest.mark.gpu
def test_sharded_and_checkpointed_runs_give_the_same_results(built_lib):
    N, S, T = 64, 160, 120
    ckw = dict(CONFIG_KW, steps_max=25)
    acts = actions(N, T, seed=12)
    whole = make_vec(N, config_kw=ckw, metrics=True)
    (rw,), snap = run_bank([whole], S, T, acts, [0], N, snapshot_at=50)
    halves = [make_vec(N // 2, config_kw=ckw, metrics=True, env_offset=o) for o in (0, N // 2)]
    rh, _ = run_bank(halves, S, T, acts, [0, N // 2], N)
    m = merged(rh)
    assert (rw["length"] >= 0).sum() > N
    for k in rw:
        assert torch.equal(bits(rw[k]), bits(m[k])), k
    # checkpoint: a new handle attaches the bank, takes the results so far and the state, and runs on
    resumed = make_vec(N, config_kw=ckw, metrics=True)
    state, target = bank_columns(S, seed=13)
    rr = resumed.set_scenario_bank(state=state, target=target)
    for k, x in snap[1][0].items():
        rr[k].copy_(x)
    resumed.set_state(snap[0][0])
    for t in range(50, T):
        resumed.step_tensors(acts[t])
    for k in rw:
        assert torch.equal(bits(rw[k]), bits(rr[k])), k
    for v in [whole, resumed] + halves:
        v.close()


# ---------------------------------------------------------------------------------------------------------------------
# 5. C-ABI errors
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_c_abi_errors(built_lib):
    from fwgym_b200 import _capi
    ARG = _capi.ENUMS["FW_ERR_ARG"]
    plain = make_vec(8, bank=False)
    nomet = make_vec(8)
    met = make_vec(8, metrics=True)
    buf = torch.zeros(64, dtype=torch.float64, device="cuda")
    lev = torch.zeros(16, dtype=torch.int32, device="cuda")

    def call(v, **fields):
        b = _capi.fw_bank_t()
        b.n_scenarios, b.first, b.stride = 16, 0, 8
        for k, x in fields.items():
            setattr(b, k, x)
        return v._lib.fw_set_bank(v._h, ctypes.byref(b), v._stream())
    assert call(plain) == ARG
    assert plain._lib.fw_set_bank(plain._h, None, plain._stream()) == ARG
    assert call(nomet) == 0 and call(met, episode=buf.data_ptr()) == 0
    assert call(nomet, stride=7) == ARG
    assert call(nomet, n_scenarios=0) == ARG
    assert call(nomet, n_scenarios=2 ** 31) == ARG
    assert call(nomet, first=-1) == ARG
    assert call(nomet, episode=buf.data_ptr()) == ARG
    for f in ("term", "length", "ret", "episode"):
        assert call(met, cycle=1, **{f: buf.data_ptr()}) == ARG, f
    assert call(met, cycle=1, episodes=lev.data_ptr(), successes=lev.data_ptr()) == 0
    assert call(nomet, turb_level=lev.data_ptr()) == ARG
    with pytest.raises(ValueError):
        nomet.set_scenario_bank(state={"roll": [0.0] * 4}, stride=7)
    for v in (plain, nomet, met):
        v.close()
