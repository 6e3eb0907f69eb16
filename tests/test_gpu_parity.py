"""GPU parity tests proper: the CUDA path (through the C-ABI / VecEnv) against (a) the committed golden fixtures
generated from the UNMODIFIED reference env file, (b) the live CPU oracle on the same seeded inputs.

Tolerances (BASELINE.json north_star): bit-exact for integer / indexing state (done flags, dopri5 attempt counts,
termination codes, step counters); floating point <= 1e-9 relative per step in fp64 (observations, rewards and the
27 simulator state values, relative to max(|ref|, 1e-3)); <= 1e-4 relative over a 100-step turbulence-off rollout.
"""
import os

import numpy as np
import pytest
import torch

from oracle import harness
from oracle.cases import CASES
from oracle.make_golden import SEED
import parity_utils as pu

pytestmark = pytest.mark.gpu
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
TOL = 1e-9


def make_vec(c, n=None, seed=SEED, sim_config_kw=None, **kw):
    from fwgym_b200 import FixedWingVecEnv
    return FixedWingVecEnv(harness.config_path(c["config"]), n or c["n"], config_kw=c["config_kw"],
                           sim_config_kw=sim_config_kw or c["sim_kw"], seed=seed, keep_terminal_obs=True, **kw)


@pytest.mark.parametrize("name", sorted(CASES))
def test_golden_fixture(built_lib, name):
    """CUDA vs fixtures produced by the reference's own fixed_wing.py (oracle/make_golden.py)."""
    c = CASES[name]
    g = np.load(os.path.join(GOLDEN, "case_%s.npz" % name))
    vec = make_vec(c)
    vec.enable_f64_outputs(True)
    vec.reset()
    assert pu.rel_err(vec._obs64.cpu().numpy(), g["obs"][0], 1e-3).max() <= TOL
    worst = dict(obs=0.0, rew=0.0, state=0.0, term_obs=0.0)
    for t, a in enumerate(g["actions"]):
        _, _, done, _ = vec.step_tensors(torch.as_tensor(a, dtype=torch.float64, device=vec.device))
        done = done.cpu().numpy().astype(bool)
        assert np.array_equal(done, g["done"][t]), "done flags differ at step %d" % t
        k = vec.last_attempts().cpu().numpy()   # every env, incl. the step that ended an episode (failing attempt counted)
        assert np.array_equal(k, g["k"][t]), "dopri5 attempt counts differ at step %d" % t
        worst["obs"] = max(worst["obs"], pu.rel_err(vec._obs64.cpu().numpy(), g["obs"][t + 1], 1e-3).max())
        worst["rew"] = max(worst["rew"], pu.rel_err(vec._rew64.cpu().numpy(), g["rew"][t], 1e-3).max())
        worst["state"] = max(worst["state"], pu.rel_err(pu.gpu_state(vec), g["state"][t], 1e-3).max())
        if done.any():
            tobs = vec._term_obs.cpu().numpy()[done]
            worst["term_obs"] = max(worst["term_obs"], pu.rel_err(tobs, g["term_obs"][t][done], 1e-3).max())
    assert worst["obs"] <= TOL and worst["rew"] <= TOL and worst["state"] <= TOL, worst
    assert worst["term_obs"] <= 1e-6, worst   # terminal observations are float32 on the device
    vec.close()


@pytest.mark.parametrize("name", ["default", "turb_noise", "examples", "failure", "cnn"])
def test_generic_kernel_instantiation(built_lib, name, monkeypatch):
    """The dynamics kernel has two instantiations (dynamics.cuh): FwSpecShipped covers the shipped configurations and
    FwSpecGeneric everything else (any variable clipped / constrained, steady wind, polynomial drag).  The env / reset
    kernels have one instantiation per shipped configuration SHAPE plus the table-walking generic one
    (env_shapes.h).  These cases normally run on the specialised kernels; force the generic ones and hold them
    to the same fixtures."""
    monkeypatch.setenv("FWGYM_FORCE_GENERIC", "1")
    vec = make_vec(CASES[name])
    assert vec.kernel_variant() == "dyn=generic env=generic"
    vec.close()
    test_golden_fixture(built_lib, name)


def test_kernel_variant_selection(built_lib):
    """The host picks the specialised instantiations exactly for the configurations whose structure they were
    generated from; numbers (noise level, constraint values, curriculum level) do not change the choice."""
    want = {"default": "dyn=shipped env=default", "turb_noise": "dyn=shipped env=default_turb",
            "examples": "dyn=shipped env=examples_turb", "failure": "dyn=shipped env=default",
            "dev_history": "generic", "success_new": "generic", "wind": "dyn=generic env=generic",
            "param_rand": "dyn=rand env=generic", "cnn": "env=cnn_turb"}
    for name, v in want.items():
        vec = make_vec(CASES[name])
        assert vec.kernel_variant().endswith(v), (name, vec.kernel_variant())
        if name == "default":
            vec.set_curriculum_level(0.5)
            assert vec.kernel_variant().endswith(v)
        vec.close()


def test_live_oracle_64_envs(built_lib):
    """BASELINE configs[1] at an oracle-sized N: per-step parity on identical states, actions and seeds."""
    c = CASES["default"]
    n, steps = 64, 12
    vec = make_vec(c, n=n, seed=5)
    orc = pu.make_oracles(n, harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 5)
    acts = np.random.RandomState(3).uniform(-1, 1, (steps, n, 3))
    out = pu.run_parity(vec, orc, acts)
    assert out["done_mismatch"] == 0 and out["k_mismatch"] == 0
    assert max(out["obs"]) <= TOL and max(out["rew"]) <= TOL and max(out["state"]) <= TOL, out


def test_on_success_override_stays_on_specialised_kernels(built_lib):
    """`target.on_success` is a runtime number in every instantiation (the evaluation harness overrides it on the
    examples configuration, evaluate_controller.py:68-76): the examples shape is kept, the 100-step success streak ends
    the episode exactly when the oracle's does, and the steps after the auto-reset still match."""
    c = dict(config="fixed_wing_config_examples.json", n=4, sim_kw={"turbulence": False},
             config_kw={"target": {"on_success": "done", "states": {0: {"bound": 150}, 1: {"bound": 80}, 2: {"bound": 25}}}})
    n, steps = 4, 108
    vec = make_vec(c, n=n, seed=5)
    assert vec.kernel_variant().endswith("env=examples"), vec.kernel_variant()
    orc = pu.make_oracles(n, harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 5)
    acts = np.random.RandomState(3).uniform(-0.3, 0.3, (steps, n, 3))
    out = pu.run_parity(vec, orc, acts)
    assert out["dones"] == n and out["done_mismatch"] == 0 and out["k_mismatch"] == 0
    assert max(out["obs"]) <= TOL and max(out["rew"]) <= TOL and max(out["state"]) <= TOL, out
    vec.close()


@pytest.mark.parametrize("n", [33, 197])
def test_ragged_env_counts(built_lib, n):
    """Env counts that fill neither a warp (32), an init block (64) nor an env chunk (128): the partial last warp /
    block / chunk is stepped, counted and handed over like a full one (turbulence + noise on, so every kernel's tail
    lanes run the full path), and the row stride padding never leaks into results."""
    c = CASES["turb_noise"]
    steps = 6
    vec = make_vec(c, n=n, seed=9)
    orc = pu.make_oracles(n, harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 9)
    acts = np.random.RandomState(n).uniform(-1, 1, (steps, n, 3))
    out = pu.run_parity(vec, orc, acts)
    assert out["done_mismatch"] == 0 and out["k_mismatch"] == 0
    # free-running (device and oracle each continue from their OWN state), under turbulence: observations / rewards hold
    # the per-step bar; a raw simulator state near a zero crossing of one sensitive aircraft showed 1.7e-9 for one step
    # (absolute 1.7e-12, env 3 of 197 - not in the ragged part; scripts/gpu_debug_ragged.py), hence the rollout bar there
    assert max(out["obs"]) <= TOL and max(out["rew"]) <= TOL and max(out["state"]) <= 1e-7, out
    ctr = vec.counters()
    assert ctr["env_steps"] == n * steps and ctr["watchdog"] == 0
    vec.close()


def test_capi_argument_errors(built_lib):
    """The boundary refuses bad calls with a status and a message instead of launching anything: null buffers, a slot that
    was never submitted, a row range outside the state, an ABI version the library was not built for."""
    import ctypes
    from fwgym_b200 import _capi
    lib = _capi.lib()
    vec = make_vec(CASES["default"], n=8)
    vec.reset()
    h, null = vec._h, ctypes.c_void_p(0)
    before = vec.get_state().clone()
    # fw_step without actions / without any observation buffer
    rc = lib.fw_step(h, null, 0, vec._ptr(vec._obs), vec._ptr(vec._rew), vec._ptr(vec._done), vec._ptr(vec._term),
                     null, null, null, 1, vec._stream())
    assert rc == -1 and b"fw_step" in lib.fw_last_error()
    acts = torch.zeros((8, 3), dtype=torch.float64, device=vec.device)
    rc = lib.fw_step(h, vec._ptr(acts), 1, null, vec._ptr(vec._rew), vec._ptr(vec._done), vec._ptr(vec._term),
                     null, null, null, 1, vec._stream())
    assert rc == -1 and b"observation" in lib.fw_last_error()
    # host pipeline: waiting on a slot that was never submitted, submitting without fw_host_open
    slot = ctypes.c_int(0)
    hact = torch.zeros((8, 3), dtype=torch.float32).pin_memory()
    assert lib.fw_host_submit(h, ctypes.c_void_p(hact.data_ptr()), vec._stream(), ctypes.byref(slot)) == -1
    pp = [ctypes.c_void_p() for _ in range(4)]
    assert lib.fw_host_wait(h, 3, *[ctypes.byref(x) for x in pp]) == -1
    # row export outside the state
    buf = torch.zeros(16, dtype=torch.float64, device=vec.device)
    assert lib.fw_get_rows(h, 10 ** 6, 1, vec._ptr(buf), vec._stream()) == -1
    # a configuration of another ABI version
    pod = vec.cc.pod()
    pod.abi_version += 1
    out = ctypes.c_void_p()
    assert lib.fw_create(ctypes.byref(pod), 8, 0, vec.device.index or 0, ctypes.byref(out)) == -5
    assert lib.fw_set_config(h, ctypes.byref(pod)) == -5
    # nothing above touched the state, and the handle still steps
    torch.cuda.synchronize()
    assert torch.equal(before, vec.get_state())
    vec.step_tensors(acts)
    assert vec.counters()["env_steps"] == 8
    with pytest.raises(_capi.FwError):
        _capi.check(lib.fw_host_wait(h, 3, *[ctypes.byref(x) for x in pp]))
    vec.close()


def test_config1_4096_envs_100_steps(built_lib):
    """BASELINE configs[1] at its STATED size (SURVEY §8d.2): 4096 envs, fp64 dopri5, turbulence off, 100 steps against
    the CPU oracle stepped on every host core (identical actions and Philox streams).  Two device envs:
      * FREE-RUNNING for all 100 steps: done flags, termination reasons and per-env dopri5 attempt counts bit-exact at
        every step — including the step an episode fails in — and states / observations / rewards within the north
        star's 100-step budget of 1e-4 (measured: < 1e-6; a tumbling aircraft amplifies 1e-16 rounding differences);
      * PER-STEP parity on identical states: the 27 simulator state values are overwritten with the oracle's after every
        step, so each step starts from the oracle's state; states / observations / rewards <= 1e-9 relative per step."""
    from fwgym_b200.vec_env import term_name
    c = CASES["default"]
    n, steps, seed = 4096, 100, 41
    acts = np.random.RandomState(11).uniform(-1, 1, (steps, n, 3))
    want = pu.oracle_rollout_parallel(harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], seed, acts)
    free, sync = make_vec(c, n=n, seed=seed), make_vec(c, n=n, seed=seed)
    rows = sync.state_rows()
    ridx = torch.as_tensor([rows.index(r) for r in pu.STATE_ROWS], device=sync.device)
    for v in (free, sync):
        v.enable_f64_outputs(True)
        v.reset()
        assert pu.rel_err(v._obs64.cpu().numpy(), want["obs"][0], 1e-3).max() <= TOL
    worst = {"free": dict(obs=0.0, rew=0.0, state=0.0), "sync": dict(obs=0.0, rew=0.0, state=0.0)}
    n_done = n_fail = 0
    for t in range(steps):
        at = torch.as_tensor(acts[t], dtype=torch.float64, device=sync.device)
        for tag, v in (("free", free), ("sync", sync)):
            _, _, done, term = v.step_tensors(at)
            done = done.cpu().numpy().astype(bool)
            assert np.array_equal(done, want["done"][t]), "%s: done flags differ at step %d" % (tag, t)
            assert np.array_equal(v.last_attempts().cpu().numpy(), want["k"][t]), "%s: attempt counts differ at step %d" % (tag, t)
            tc = term.cpu().numpy()
            for i in np.nonzero(done)[0]:
                assert term_name(int(tc[i])) == want["term"][t][i], (tag, t, i, tc[i], want["term"][t][i])
            w = worst[tag]
            w["obs"] = max(w["obs"], pu.rel_err(v._obs64.cpu().numpy(), want["obs"][t + 1], 1e-3).max())
            w["rew"] = max(w["rew"], pu.rel_err(v._rew64.cpu().numpy(), want["rew"][t], 1e-3).max())
            es = pu.rel_err(pu.gpu_state(v), want["state"][t], 1e-3)
            if es.max() > w["state"]:
                i, j = np.unravel_index(np.argmax(es), es.shape)
                w["state"], w["where"] = es.max(), (t, int(i), pu.STATE_ROWS[j], float(want["state"][t][i, j]),
                                                   float(pu.gpu_state(v)[i, j] - want["state"][t][i, j]), int(want["k"][t][i]))
        n_done += int(done.sum())
        n_fail += int((tc[done] >= 16).sum())
        st = sync.get_state()
        st[ridx] = torch.as_tensor(want["state"][t].T.copy(), device=sync.device)
        sync.set_state(st)
    print("configs[1] 4096 x 100: %d episodes ended (%d constraint failures), %d dopri5 attempts; worst rel err "
          "free-running %r, per-step on identical states %r" % (n_done, n_fail, int(want["k"].sum()), worst["free"], worst["sync"]))
    assert max(worst["sync"][q] for q in ("obs", "rew", "state")) <= TOL, worst
    assert max(worst["free"][q] for q in ("obs", "rew", "state")) <= 1e-4, worst
    free.close(), sync.close()


def test_rollout_100_steps(built_lib):
    """<= 1e-4 relative over a 100-step turbulence-off rollout."""
    c = CASES["default"]
    n = 8
    vec = make_vec(c, n=n, seed=9)
    orc = pu.make_oracles(n, harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 9)
    acts = np.random.RandomState(4).uniform(-1, 1, (100, n, 3))
    out = pu.run_parity(vec, orc, acts)
    assert out["done_mismatch"] == 0
    assert out["state"][-1] <= 1e-4 and max(out["obs"]) <= 1e-4, (out["state"][-1], max(out["obs"]))


def test_scenario_injection(built_lib):
    """reset(state=, target=) with the reference's test-set scenarios (evaluate_controller.py:119)."""
    ts = np.load(os.path.join(GOLDEN, "test_set_wind_none.npz"))
    skeys, tkeys = list(ts["state_keys"]), list(ts["target_keys"])
    n = 8
    c = dict(config="fixed_wing_config_examples.json", config_kw={"action": {"scale_space": False}},
             sim_kw={"turbulence": False, "turbulence_intensity": "none"})
    vec = make_vec(c, n=n, seed=1)
    vec.enable_f64_outputs(True)
    state = {k: ts["state"][:n, i] for i, k in enumerate(skeys)}
    target = {k: ts["target"][:n, i] for i, k in enumerate(tkeys)}
    vec.reset(state=state, target=target)
    orc = pu.make_oracles(n, harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 1)
    obs_o = np.stack([o.reset(state={k: float(state[k][i]) for k in skeys}, target={k: float(target[k][i]) for k in tkeys})
                      for i, o in enumerate(orc)])
    assert pu.rel_err(vec._obs64.cpu().numpy(), obs_o, 1e-3).max() <= TOL
    acts = np.random.RandomState(8).uniform(-0.4, 0.4, (10, n, 3))
    acts[:, :, 2] = np.abs(acts[:, :, 2])
    for a in acts:
        vec.step_tensors(torch.as_tensor(a, dtype=torch.float64, device=vec.device))
        res = [o.step(a[i]) for i, o in enumerate(orc)]
        assert pu.rel_err(vec._obs64.cpu().numpy(), np.stack([r[0] for r in res]), 1e-3).max() <= TOL
        assert pu.rel_err(vec._rew64.cpu().numpy(), np.array([r[1] for r in res]), 1e-3).max() <= TOL


def test_overlapped_env_kernel_is_bitwise_identical(built_lib, monkeypatch):
    """The env kernel normally runs as a programmatic dependent of the attempt kernel (its blocks start while the
    attempt kernel's tail is still running and wait on per-chunk completion counters).  Serialised launches
    (FWGYM_OVERLAP=0) must give bitwise identical states, and no block may ever have given up waiting."""
    c = CASES["turb_noise"]
    n = 4096 + 77      # several chunks per SM and a ragged last chunk
    acts = torch.rand((12, n, 3), dtype=torch.float64, device="cuda") * 2 - 1
    states = []
    for overlap in ("1", "0"):
        monkeypatch.setenv("FWGYM_OVERLAP", overlap)
        vec = make_vec(c, n=n, seed=33)
        vec.reset()
        for a in acts:
            vec.step_tensors(a)
        states.append(vec.get_state().cpu().numpy())
        assert vec.counters()["watchdog"] == 0
        vec.close()
    assert np.array_equal(states[0], states[1], equal_nan=True)


@pytest.mark.parametrize("zero_copy", [False, True])
def test_host_buffer_pipeline_matches_device_step(built_lib, zero_copy):
    """fw_host_submit / fw_host_wait (HostStepper): host actions in, host results out, two submissions in flight -
    the same numbers as stepping on device tensors, ragged env count, pageable and pinned action buffers; with a
    device -> host copy per step and with the env kernel writing straight into mapped pinned memory (zero_copy: the
    observations leave through a shared-memory tile), incl. envs that finish and are reset in the step."""
    from fwgym_b200 import HostStepper
    c = dict(CASES["turb_noise"])
    c["config_kw"] = dict(c["config_kw"], steps_max=6)
    n, steps = 1000, 9
    acts = (torch.rand((steps, n, 3)) * 2 - 1)
    ref = make_vec(c, n=n, seed=17)
    ref.reset()
    want = []
    for a in acts:
        o, r, d, t = ref.step_tensors(a.cuda())
        want.append((o.cpu().numpy().copy(), r.cpu().numpy().copy(), d.cpu().numpy().copy(), t.cpu().numpy().copy()))
    ref.close()
    vec = make_vec(c, n=n, seed=17)
    vec.reset()
    hs = HostStepper(vec, depth=2, zero_copy=zero_copy)
    pinned = acts.pin_memory()
    pending, got = [], []
    for i in range(steps):
        pending.append(hs.submit(pinned[i] if i % 2 else acts[i].numpy()))
        if len(pending) == 2:
            s = pending.pop(0)
            o, r, d = hs.wait(s)
            got.append((o.copy(), r.copy(), d.copy(), hs.term(s).copy()))
    while pending:
        s = pending.pop(0)
        o, r, d = hs.wait(s)
        got.append((o.copy(), r.copy(), d.copy(), hs.term(s).copy()))
    with pytest.raises(Exception):
        hs.wait(0)          # nothing in flight in that slot
    for w, g in zip(want, got):
        for x, y in zip(w, g):
            assert np.array_equal(x.reshape(y.shape), y, equal_nan=True)
    hs.close()
    vec.close()


def test_simulator_parameters_are_randomised_per_episode(built_lib):
    """SURVEY §8f row 4 (fixed_wing.py:523-570, :872-888): every env draws its own model parameters at every reset;
    the clipped gaussian keeps them inside the configured window, parameters change across episodes, and the derived
    rows (1/mass ...) follow.  The step-level numbers are pinned by the param_rand golden fixtures."""
    c = CASES["param_rand"]
    vec = make_vec(c, n=512, seed=3)
    vec.reset()
    p0 = vec.get_simulator_parameters(normalize=False).cpu().numpy()
    names = [pa["name"] for pa in vec.cc.cfg["simulator"]["model"]["parameters"]]
    mass, clalpha = p0[:, names.index("mass")], p0[:, names.index("C_L_alpha")]
    assert mass.std() > 0.05 and abs(mass.mean() - 3.364) < 0.1
    assert mass.min() >= 3.364 * 0.75 - 1e-12 and mass.max() <= 3.364 * 1.25 + 1e-12          # clip 0.25 relative
    assert clalpha.std() > 1.5 * mass.std()                                                    # var 0.2 vs 0.1
    # negative original with a relative clip: np.clip(v, orig - clip*orig, orig + clip*orig) has min > max -> constant
    cmq = p0[:, names.index("C_m_q")]
    assert np.allclose(cmq, -1.3047 * 1.25, rtol=0, atol=1e-12)
    assert np.all(p0[:, names.index("Jx")] == 1.229)                                           # never reaches the dynamics
    st, rows = vec.get_state().cpu().numpy(), vec.state_rows()
    prm = st[rows.index("param"):rows.index("param") + rows.count("param")]
    _, slot1, _ = vec.cc._rand_slots()
    inv_mass = prm[slot1[vec.cc.par_id("mass")] - 1] * prm[slot1[_enum("FW_PAR_INV_MASS")] - 1]
    assert np.allclose(inv_mass, 1.0, atol=1e-15)
    acts = torch.zeros((vec.num_envs, 3), dtype=torch.float64, device=vec.device)
    for _ in range(c["config_kw"]["steps_max"]):
        vec.step_tensors(acts)                      # every env ends its episode (steps_max) and is reset
    p1 = vec.get_simulator_parameters(normalize=False).cpu().numpy()
    assert (p1[:, names.index("mass")] != mass).mean() > 0.99
    pn = vec.get_simulator_parameters(normalize=True).cpu().numpy()
    assert pn.shape[1] == len(names) - 1            # C_D_q has a zero original: skipped, as in the reference
    vec.close()


def _enum(name):
    from fwgym_b200 import _capi
    return _capi.ENUMS[name]


def test_sharding_invariance(built_lib):
    """RNG is keyed by the GLOBAL env id: one handle of 32 envs == two handles of 16 with offsets 0 and 16, bitwise."""
    c = CASES["turb_noise"]
    acts = torch.rand((15, 32, 3), dtype=torch.float64, device="cuda") * 2 - 1
    whole = make_vec(c, n=32, seed=21)
    a, b = make_vec(c, n=16, seed=21, env_offset=0), make_vec(c, n=16, seed=21, env_offset=16)
    ow = whole.reset().clone()
    oa, ob = a.reset().clone(), b.reset().clone()
    assert torch.equal(ow, torch.cat([oa, ob]))
    for t in range(15):
        ow, rw, dw, _ = whole.step_tensors(acts[t])
        oa, ra, da, _ = a.step_tensors(acts[t, :16].contiguous())
        ob, rb, db, _ = b.step_tensors(acts[t, 16:].contiguous())
        assert torch.equal(ow, torch.cat([oa, ob])) and torch.equal(rw, torch.cat([ra, rb]))
    assert torch.equal(whole.get_state(), torch.cat([a.get_state(), b.get_state()], dim=1))


def test_fp32_mode_reported(built_lib):
    """Opt-in fp32 dynamics (stated separately from the fp64 parity bar): state error vs the fp64 oracle after 20
    steps is printed and only sanity-bounded (< 0.1 relative); integer state (done flags) still matches."""
    c = CASES["default"]
    n = 8
    vec = make_vec(c, n=n, seed=5, precision="fp32")
    orc = pu.make_oracles(n, harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 5)
    acts = np.random.RandomState(3).uniform(-1, 1, (20, n, 3))
    out = pu.run_parity(vec, orc, acts)
    print("fp32 mode: max rel state err over 20 steps %.3e, obs %.3e" % (max(out["state"]), max(out["obs"])))
    assert out["done_mismatch"] == 0
    assert max(out["state"]) < 0.1   # fp32 adaptive stepping decorrelates quickly; reported, not a parity claim


def test_fp32_mode_feature_config_integer_state(built_lib):
    """BASELINE configs[4] (SURVEY §8d.5) under precision="fp32": the dev configuration with a 5-row matrix observation,
    integrator targets, integration window and target resampling.  fp32 dopri5 decorrelates the floating-point state
    from the fp64 oracle (reported, stated separately from the parity bar), but the INTEGER / indexing state must not
    move: done flags and termination codes against the reference-file fixture, and step counters, target-step counters,
    history lengths and the resample schedule against the fp64 run, bit-exact at every step."""
    c = CASES["dev_history"]
    g = np.load(os.path.join(GOLDEN, "case_dev_history.npz"))
    v32, v64 = make_vec(c, precision="fp32"), make_vec(c)
    assert v32.kernel_variant() == v64.kernel_variant()
    rows = v64.state_rows()
    ints = [rows.index(r) for r in ("steps_count", "steps_for_target", "hist_len", "rng_tick", "episode_tick")]
    v32.enable_f64_outputs(True)
    v32.reset(), v64.reset()
    worst_state = worst_obs = 0.0
    resamples = 0
    for t, a in enumerate(g["actions"]):
        at = torch.as_tensor(a, dtype=torch.float64, device=v32.device)
        _, _, d32, t32 = v32.step_tensors(at)
        _, _, d64, t64 = v64.step_tensors(at)
        assert np.array_equal(d32.cpu().numpy().astype(bool), g["done"][t]), "fp32 done flags differ at step %d" % t
        assert torch.equal(t32, t64) and torch.equal(d32, d64)
        s32, s64 = v32.get_state(), v64.get_state()
        assert torch.equal(s32[ints], s64[ints]), "integer state differs at step %d" % t
        resamples += int((s64[rows.index("steps_for_target")] == 0).sum())
        worst_state = max(worst_state, pu.rel_err(pu.gpu_state(v32), g["state"][t], 1e-3).max())
        worst_obs = max(worst_obs, pu.rel_err(v32._obs64.cpu().numpy(), g["obs"][t + 1], 1e-3).max())
    assert resamples > 0 and g["done"].sum() > 0
    print("fp32 mode on the config-5 feature set: integer state bit-exact over %d steps (%d episode ends, %d target "
          "resamples); max rel error vs the fp64 fixture: state %.3e, observation %.3e"
          % (len(g["actions"]), int(g["done"].sum()), resamples, worst_state, worst_obs))
    assert worst_state < 0.1
    v32.close(), v64.close()


def test_seed_then_reset_reproduces_episodes(built_lib):
    """FixedWingAircraft.seed reseeds the env's generator and the simulator (fixed_wing.py:214-222): on a LIVE env,
    seed(s) + reset() must replay the same episodes (the per-env draw counters restart with the key)."""
    c = CASES["turb_noise"]
    vec = make_vec(c, n=64, seed=5)
    acts = torch.rand((8, 64, 3), dtype=torch.float64, device=vec.device) * 2 - 1
    runs = []
    for rep in range(2):
        vec.seed(123)
        obs = [vec.reset().clone()]
        for a in acts:
            obs.append(vec.step_tensors(a)[0].clone())
        runs.append(torch.stack(obs))
    assert torch.equal(runs[0], runs[1])
    vec.seed(124)
    assert not torch.equal(vec.reset(), runs[0][0])
    vec.close()


def test_watchdog_error_is_sticky(built_lib):
    """An env-kernel block that gives up waiting for its aircraft must not pass silently: nothing is committed for
    its envs, and fw_step / fw_counters / the host pipeline fail until a full reset re-arms the step queue."""
    from fwgym_b200 import _capi
    c = CASES["default"]
    vec = make_vec(c, n=300, seed=2)
    vec.reset()
    acts = torch.zeros((300, 3), dtype=torch.float64, device=vec.device)
    vec.step_tensors(acts)
    before = vec.get_state().clone()
    _capi.check(vec._lib.fw_debug_watchdog(vec._h, 64, 1))       # block 0 of the next step waits for a 129th aircraft
    obs, rew, done, term = vec.step_tensors(acts)                 # enqueues; the error surfaces at the next call
    torch.cuda.synchronize()
    assert torch.isnan(obs[:128]).all() and torch.isnan(rew[:128]).all() and (term[:128] == -1).all()
    assert torch.isfinite(obs[128:]).all()                        # the other blocks stepped normally
    with pytest.raises(_capi.FwError, match="gave up waiting"):
        vec.step_tensors(acts)
    with pytest.raises(_capi.FwError, match="gave up waiting"):
        vec.counters()
    with pytest.raises(_capi.FwError):
        vec.reset(indices=[0])                                    # a partial reset does not recover
    _capi.check(vec._lib.fw_debug_watchdog(vec._h, 0, 0))
    rows = vec.state_rows()
    after = vec.get_state()
    assert torch.equal(after[:, :128], before[:, :128])           # nothing was committed for the starved chunk
    assert (after[rows.index("steps_count"), 128:] == before[rows.index("steps_count"), 128:] + 1).all()
    vec.reset()                                                   # full reset: flag cleared, queue re-armed
    for _ in range(3):
        obs, rew, done, term = vec.step_tensors(acts)
    assert torch.isfinite(obs).all() and vec.counters()["watchdog"] >= 1
    vec.close()


def test_injected_turbulence_noise(built_lib):
    """reset(turbulence_noise=...) (fixed_wing.py:287,308 -> PyFly.reset): the caller's [4, T] standard-normal samples
    drive the Dryden filters of the episode instead of the env's own stream; compared with the CPU oracle given the
    same arrays, per env, incl. the wrap-around past T and the return to the Philox stream after an auto-reset."""
    c = dict(CASES["turb_noise"])
    c["config_kw"] = dict(c["config_kw"], steps_max=25)
    n, T = 4, 12
    noise = np.random.RandomState(7).standard_normal((n, 4, T))
    vec = make_vec(c, n=n, seed=9)
    vec.enable_f64_outputs(True)
    vec.reset(turbulence_noise=noise)
    orc = pu.make_oracles(n, harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 9)
    obs_o = np.stack([np.asarray(o.reset(turbulence_noise=noise[i]), dtype=np.float64).ravel() for i, o in enumerate(orc)])
    assert pu.rel_err(vec._obs64.cpu().numpy(), obs_o, 1e-3).max() <= TOL
    acts = np.random.RandomState(8).uniform(-1, 1, (40, n, 3))
    dones = 0
    for a in acts:
        _, _, done, _ = vec.step_tensors(torch.as_tensor(a, dtype=torch.float64, device=vec.device))
        res = [o.step(a[i]) for i, o in enumerate(orc)]
        assert np.array_equal(done.cpu().numpy().astype(bool), np.array([r[2] for r in res]))
        dones += int(done.sum())
        assert pu.rel_err(vec._obs64.cpu().numpy(), np.stack([np.ravel(r[0]) for r in res]), 1e-3).max() <= TOL
        assert pu.rel_err(pu.gpu_state(vec), np.stack([o.ode_state() for o in orc]), 1e-3).max() <= TOL
    assert dones >= n          # every env went through an auto-reset and back to its own stream
    # the single-env facade forwards the keyword like the reference
    from fwgym_b200 import FixedWingAircraft
    env = FixedWingAircraft(harness.config_path(c["config"]), config_kw=c["config_kw"], sim_config_kw=c["sim_kw"])
    env.seed(9)
    o1 = env.reset(turbulence_noise=noise[0])
    assert pu.rel_err(o1, obs_o[0], 1e-3).max() <= TOL
    env.close()
    vec.close()


def test_numeric_failure_and_attempt_cap(built_lib):
    """Hardening beyond the reference: (a) a simulator state that leaves the representable range (the dev configuration
    has no body-rate constraints; under random actions its rates grow without bound) ends the episode with termination
    "numeric" instead of spinning in dopri5 (scipy's loop never returns on a NaN step size) or feeding NaNs back;
    (b) sim_config_kw dopri5_max_attempts caps the attempts of one env step the same way (off by default)."""
    from fwgym_b200 import FixedWingVecEnv
    from fwgym_b200.vec_env import term_name
    cfg = harness.config_path("fixed_wing_config_dev.json")
    vec = FixedWingVecEnv(cfg, 64, sim_config_kw={"turbulence": False}, seed=3)
    vec.reset()
    st, rows = vec.get_state(), vec.state_rows()
    for k in ("omega_p", "omega_q", "omega_r"):
        st[rows.index(k), :8] = 1e153   # where unconstrained rates end up after ~100 random-action steps: products overflow
    vec.set_state(st)
    acts = torch.zeros((64, 3), dtype=torch.float64, device=vec.device)
    ended = torch.zeros(64, dtype=torch.bool, device=vec.device)
    for _ in range(3):     # step sizes of 1e-17 s: the hang guard (or a non-finite value) ends these episodes
        obs, rew, done, term = vec.step_tensors(acts)
        assert all(term_name(int(t)) == "numeric" for t in term[:8][done[:8].bool()])
        assert not done[8:].any() and torch.isfinite(obs[8:]).all()  # the others fly on
        assert torch.isfinite(obs[:8][done[:8].bool()]).all()         # a finished env is reset on the spot
        assert int(vec.last_attempts().max()) <= 20000
        ended |= done.bool()
    assert ended[:8].all()
    for _ in range(5):
        obs, rew, done, term = vec.step_tensors(acts)
    assert torch.isfinite(obs).all() and torch.isfinite(vec.get_state()[:27]).all()
    vec.close()
    c = CASES["default"]
    vec = make_vec(c, n=2048, seed=12, sim_config_kw={"turbulence": False, "dopri5_max_attempts": 4})
    vec.reset()
    g = torch.Generator(device="cuda"); g.manual_seed(2)
    n_numeric = 0
    for t in range(10):
        a = torch.rand((2048, 3), generator=g, device="cuda", dtype=torch.float64) * 2 - 1
        _, _, done, term = vec.step_tensors(a)
        k = vec.last_attempts()
        assert int(k.max()) <= 4
        numeric = term == 3
        assert (k[numeric] == 4).all() and done[numeric.bool()].all()
        n_numeric += int(numeric.sum())
    assert n_numeric > 0
    vec.close()


def test_single_env_facade(built_lib):
    """FixedWingAircraft facade (N=1): reference constructor / reset / step signatures and 4-tuple."""
    from fwgym_b200 import FixedWingAircraft
    env = FixedWingAircraft(harness.config_path(), sim_config_kw={"turbulence": False})
    env.seed(3)
    obs = env.reset()
    assert obs.shape == (14,) and obs.dtype == np.float64
    orc = pu.make_oracles(1, harness.config_path(), None, {"turbulence": False}, 3)[0]
    orc.auto_reset = False
    o0 = orc.reset()
    assert pu.rel_err(obs, o0, 1e-3).max() <= TOL
    for t in range(5):
        a = np.array([0.1 * t, -0.2, 0.5])
        obs, rew, done, info = env.step(a)
        o, r, d, i = orc.step(a)
        assert pu.rel_err(obs, o, 1e-3).max() <= TOL and abs(rew - r) <= TOL and done == d
        assert set(info["target"]) == {"roll", "pitch", "Va"}
    env.close()


@pytest.mark.parametrize("name", ["failure", "success_done", "norm_step2", "dev_history"])
def test_episode_metrics_golden(built_lib, name):
    """SURVEY §8f row 1: the device's streaming episode metrics against FixedWingAircraft.get_metric of the unmodified
    reference file (fixtures: oracle/make_golden_metrics.py), at every episode end of the case.  Integer-valued
    columns (length, success, settling_time, rise_time) exact, floats <= 1e-9 relative, NaN where the reference has
    nan / no entry."""
    c = CASES[name]
    g = np.load(os.path.join(GOLDEN, "case_%s.npz" % name))
    rows = np.load(os.path.join(GOLDEN, "metrics_%s.npz" % name))["rows"]
    want = {(int(r[0]), int(r[1])): r[2:] for r in rows}
    from fwgym_b200 import FixedWingVecEnv
    vec = FixedWingVecEnv(harness.config_path(c["config"]), c["n"], config_kw=c["config_kw"], sim_config_kw=c["sim_kw"],
                          seed=SEED, metrics=True)
    cols = vec.episode_columns()
    exact = [j for j, n in enumerate(cols) if n == "l" or n.split("_")[0] in ("success", "settling", "rise")
             and "frac" not in n]
    vec.reset()
    seen = 0
    for t, a in enumerate(g["actions"]):
        _, _, done, _ = vec.step_tensors(torch.as_tensor(a, dtype=torch.float64, device=vec.device))
        done = done.cpu().numpy().astype(bool)
        assert np.array_equal(done, g["done"][t])
        ep = vec.episode_metrics().cpu().numpy()
        for i in np.nonzero(done)[0]:
            got, ref = ep[i], want[(t, int(i))]
            assert np.array_equal(np.isnan(got), np.isnan(ref)), (name, t, i, cols, got, ref)
            ok = ~np.isnan(ref)
            assert np.array_equal(got[exact][ok[exact]], ref[exact][ok[exact]]), (t, i, got[exact], ref[exact])
            fin = ok & np.isfinite(ref)
            assert np.array_equal(np.isinf(got), np.isinf(ref))
            assert (np.abs(got[fin] - ref[fin]) <= TOL * np.maximum(np.abs(ref[fin]), 1e-3)).all(), \
                (t, i, [(cols[j], got[j], ref[j]) for j in np.nonzero(fin)[0] if abs(got[j] - ref[j]) > TOL * max(abs(ref[j]), 1e-3)])
            seen += 1
    assert seen == len(want)
    vec.close()


def test_episode_info_dicts(built_lib):
    """infos[i] of a finished env carries what the reference puts there (fixed_wing.py:417-419) + Monitor's episode."""
    c = CASES["norm_step2"]
    from fwgym_b200 import FixedWingVecEnv
    vec = FixedWingVecEnv(harness.config_path(c["config"]), c["n"], config_kw=c["config_kw"], sim_config_kw=c["sim_kw"],
                          seed=SEED, metrics=True, info_keywords=("success", "control_variation"))
    vec.reset()
    g = np.load(os.path.join(GOLDEN, "case_%s.npz" % "norm_step2"))
    for t, a in enumerate(g["actions"]):
        obs, rew, done, infos = vec.step(torch.as_tensor(a, dtype=torch.float64, device=vec.device))
        if done.any():
            i = int(torch.nonzero(done)[0])
            info = infos[i]
            assert set(info["success"]) == {"roll", "pitch", "Va", "all"}
            assert info["episode"]["l"] == 30 and "control_variation" in info["episode"]
            assert info["termination"] == "steps" and "rise_time" in info and "all" in info["control_variation"]
            break
    else:
        raise AssertionError("no episode finished")
    vec.close()


def test_pid_evaluation_harness(built_lib):
    """SURVEY §8f row 2: batched scenario replay under the device PID controller against (a) the CPU oracle driven by
    the restated pyfly PIDController on the same scenarios (<= 1e-9 on every reward until the episode ends, equal
    lengths) and (b) the reference's published PID trace examples/evaluations/eval_res_PID_none.npy — the gap to (b)
    is REPORTED, not asserted: it measures the recalled aircraft constants (DESIGN.md §2), not the kernels."""
    from fwgym_b200 import evaluate
    from oracle.pyfly_restated import PIDController
    scen = evaluate.load_test_set(os.path.join(GOLDEN, "test_set_wind_none.npz"))
    cfg = harness.config_path("fixed_wing_config_examples.json")
    res, vec = evaluate.evaluate_on_set(scen, cfg, controller="pid", seed=1)
    gold = np.load(os.path.join(GOLDEN, "eval_res_PID_none_rewards.npz"))
    # (a) CPU oracle on the first scenarios
    kw = dict(evaluate.EVAL_CONFIG_KW)
    kw["action"] = {"scale_space": False}
    for i in range(3):
        env = harness.make_env("restated", cfg, kw, {"turbulence": False, "turbulence_intensity": "none"})
        obs = env.reset(state=dict(scen[i]["state"]), target=dict(scen[i]["target"]))
        pid = PIDController(env.simulator.dt)
        pid.set_reference(env.target["roll"], env.target["pitch"], env.target["Va"])
        rews, done = [], False
        while not done:
            obs, r, done, info = env.step(pid.get_action(obs[0], obs[1], obs[2], obs[3:6]))
            pid.set_reference(info["target"]["roll"], info["target"]["pitch"], info["target"]["Va"])
            rews.append(r)
        assert len(rews) == res["lengths"][i]
        assert pu.rel_err(res["rewards"][i], np.array(rews), 1e-3).max() <= TOL
    # (b) published trace: report
    off = np.concatenate([[0], np.cumsum(gold["lengths"])])
    gaps = [np.abs(res["rewards"][i][:min(len(res["rewards"][i]), gold["lengths"][i])] -
                   gold["rewards"][off[i]:off[i] + min(len(res["rewards"][i]), gold["lengths"][i])]).max()
            for i in range(len(scen))]
    same_len = int((res["lengths"] == gold["lengths"]).sum())
    s = evaluate.summarise(res)
    print("PID on test_set_wind_none (100 scenarios): success_all %.2f, mean length %.1f (published %.1f); max |reward "
          "gap| to the published trace: median %.3g, worst %.3g; %d/100 episode lengths equal"
          % (s.get("success_all", float("nan")), res["lengths"].mean(), gold["lengths"].mean(), np.median(gaps),
             np.max(gaps), same_len))
    assert np.isfinite(gaps).all()
    vec.close()


def test_pretrained_mlp_controller_evaluation(built_lib):
    """SURVEY §8f row 3 (policy-in-the-loop sanity run): the reference's shipped PPO2 MlpPolicy
    (examples/models/mlp_controller, weights + VecNormalize statistics extracted into tests/golden/mlp_controller.npz)
    flies the 100 scenarios of test_set_wind_none on the device.  (a) Parity: the CPU oracle under a numpy twin of the
    policy gives the same rewards (<= 1e-7: the policy's float64 matmuls sum in a different order on the two sides)
    and episode lengths.  (b) The published evaluation of this controller (eval_res_RL_MLP_none.npy: 100 % success,
    mean episode 270 steps) is compared and REPORTED — like the PID trace it measures the recalled aircraft
    constants (DESIGN.md §2), not the kernels.  Measured: 95 / 100 scenarios succeed (99 / 95 / 98 % roll / pitch / Va)
    with the calibrated thrust constant; with the recalled one it was 36 / 100, which is how the error was found
    (oracle/calibrate_thrust.py)."""
    from fwgym_b200 import evaluate
    par = dict(np.load(os.path.join(GOLDEN, "mlp_controller.npz")))
    scen = evaluate.load_test_set(os.path.join(GOLDEN, "test_set_wind_none.npz"))
    cfg = harness.config_path("fixed_wing_config_examples.json")
    res, vec = evaluate.evaluate_on_set(scen, cfg, controller=par, seed=1)
    W = [(par["pi_fc0_w"].astype(np.float64), par["pi_fc0_b"].astype(np.float64)),
         (par["pi_fc1_w"].astype(np.float64), par["pi_fc1_b"].astype(np.float64)),
         (par["pi_w"].astype(np.float64), par["pi_b"].astype(np.float64))]
    std = np.sqrt(par["obs_var"] + 1e-8)

    def policy(obs, raw):
        o = np.asarray(obs, dtype=np.float64).reshape(-1)
        x = o if raw else np.clip((o - par["obs_mean"]) / std, -10, 10)
        x = np.tanh(x @ W[0][0] + W[0][1])
        x = np.tanh(x @ W[1][0] + W[1][1])
        return np.clip(x @ W[2][0] + W[2][1], vec.action_space.low.astype(np.float64),
                       vec.action_space.high.astype(np.float64))

    for i in range(2):
        env = harness.make_env("restated", cfg, dict(evaluate.EVAL_CONFIG_KW),
                               {"turbulence": False, "turbulence_intensity": "none"})
        obs = env.reset(state=dict(scen[i]["state"]), target=dict(scen[i]["target"]))
        rews, done, raw = [], False, True
        while not done:
            obs, r, done, info = env.step(policy(obs, raw))
            raw = False
            rews.append(r)
        assert len(rews) == res["lengths"][i]
        assert pu.rel_err(res["rewards"][i], np.array(rews), 1e-3).max() <= 1e-7
    s = evaluate.summarise(res)
    ret_std = float(np.sqrt(par["ret_var"] + 1e-8))
    off = np.concatenate([[0], np.cumsum(par["pub_lengths"])])
    gaps = []
    for i in range(len(scen)):
        m = int(min(len(res["rewards"][i]), par["pub_lengths"][i]))
        ours = np.clip(res["rewards"][i][:m] / ret_std, -10, 10)       # VecNormalize(training=False) reward scaling
        gaps.append(np.abs(ours - par["pub_rewards"][off[i]:off[i] + m]).max())
    print("shipped MLP controller on test_set_wind_none (100 scenarios): success roll/pitch/Va/all %.2f/%.2f/%.2f/%.2f "
          "(published %.2f/%.2f/%.2f/%.2f), mean length %.1f (published %.1f), settling_time_all %.1f (published %.1f), "
          "control_variation %.3f (published %.3f); max |normalised reward gap|: median %.3g, worst %.3g"
          % (s.get("success_roll", np.nan), s.get("success_pitch", np.nan), s.get("success_Va", np.nan),
             s.get("success_all", np.nan), par["pub_success_roll"].mean(), par["pub_success_pitch"].mean(),
             par["pub_success_Va"].mean(), par["pub_success_all"].mean(), res["lengths"].mean(),
             par["pub_lengths"].mean(), s.get("settling_time_all", np.nan), np.nanmean(par["pub_settling_time_all"]),
             s.get("control_variation_all", np.nan), np.nanmean(par["pub_control_variation_all"]),
             np.median(gaps), np.max(gaps)))
    assert np.isfinite(gaps).all()
    assert s.get("success_all", 0.0) >= 0.85    # a policy trained on true PyFly flies the restated aircraft
    vec.close()
