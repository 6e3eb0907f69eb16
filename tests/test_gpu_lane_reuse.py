"""Lane reuse in the persistent attempt kernel (DESIGN.md §4.2, csrc/fwgym.cu fw_attempt_kernel).

A lane whose aircraft finished its env step parks the result and adopts the next waiting aircraft (priority list, then
natural order), reloading everything the aircraft's step depends on.  Below ~38 k envs (fp64: 8 resident warps per SM on
148 SMs) a lane takes one aircraft per launch; at the bench's 65 536 envs ~40 % of them are adopted by a lane that
already flew one.  These tests force heavy reuse with the switches fw_create reads (FWGYM_ATTEMPT_WARPS_PER_SM: one warp
per SM; FWGYM_LONG_DIV: priority-list threshold; fw_debug_set_order: adoption order of the natural queue) and hold it
(1) bitwise to runs with other lane assignments and (2, 3) to the CPU oracle on sampled envs at full size.  Per-env
results do not depend on N (the RNG is keyed by the global env id), so the oracle runs only the sampled envs.
"""
import time

import numpy as np
import pytest
import torch

from bench import CONFIG_KW, SIM_KW
from oracle import harness
from oracle.cases import CASES
import parity_utils as pu

TOL = 1e-9
SEED = 20261017
BENCH = dict(config="fixed_wing_config.json", config_kw=CONFIG_KW, sim_kw=SIM_KW)
SWITCHES = ("FWGYM_ATTEMPT_WARPS_PER_SM", "FWGYM_LONG_DIV")
ONE_WARP_PER_SM = {"FWGYM_ATTEMPT_WARPS_PER_SM": 1}
TERM_NUMERIC = 3


def make_vec(c, n, monkeypatch, precision="fp64", **switches):
    """A handle of case `c` created under the kernel switches `switches` (fw_create reads them); they are cleared
    again before the next handle is made."""
    from fwgym_b200 import FixedWingVecEnv
    for k in SWITCHES:
        monkeypatch.delenv(k, raising=False)
    for k, v in switches.items():
        monkeypatch.setenv(k, str(v))
    try:
        v = FixedWingVecEnv(harness.config_path(c["config"]), n, config_kw=c["config_kw"], sim_config_kw=c["sim_kw"],
                            seed=SEED, precision=precision)
    finally:
        for k in SWITCHES:
            monkeypatch.delenv(k, raising=False)
    return v


class Order:
    """Adoption order of a handle's natural queue: "identity", "reversed" or a fresh "random" permutation before every
    step.  fw_debug_set_order does not check its argument, so it only ever gets a device int32 permutation of exactly
    N elements, kept referenced while the handle steps and unset before the handle is closed."""

    def __init__(self, vec, kind, gen):
        self.vec, self.kind, self.gen, self.keep = vec, kind, gen, []
        if kind == "reversed":
            self._set(torch.arange(vec.num_envs - 1, -1, -1, dtype=torch.int32, device=vec.device))

    def _set(self, perm):
        from fwgym_b200 import _capi
        assert perm.dtype == torch.int32 and perm.is_cuda and tuple(perm.shape) == (self.vec.num_envs,)
        self.keep = [perm] + self.keep[:1]          # this step's and the previous step's array
        _capi.check(self.vec._lib.fw_debug_set_order(self.vec._h, self.vec._ptr(perm)))

    def before_step(self):
        if self.kind == "random":
            self._set(torch.randperm(self.vec.num_envs, generator=self.gen, dtype=torch.int32, device=self.vec.device))

    def close(self):
        from fwgym_b200 import _capi
        torch.cuda.synchronize()
        _capi.check(self.vec._lib.fw_debug_set_order(self.vec._h, None))
        self.keep = []
        self.vec.close()


def bits(x):
    """Integer view for bitwise comparison: NaN payloads and -0.0 count."""
    return x.view({torch.float32: torch.int32, torch.float64: torch.int64}.get(x.dtype, x.dtype))


def first_difference(what, x, y, rows=None):
    """Where two outputs differ: the first env (and, for the state matrix, the rows that differ)."""
    ne = bits(x) != bits(y)
    if rows is not None:
        bad_rows = [rows[r] for r in torch.nonzero(ne.any(1)).flatten().tolist()]
        env = int(torch.nonzero(ne.any(0))[0])
        return "%s differs in %d envs (first %d), rows %s" % (what, int(ne.any(0).sum()), env, bad_rows)
    ne = ne.reshape(len(ne), -1).any(1)
    return "%s differs in %d envs (first %d)" % (what, int(ne.sum()), int(torch.nonzero(ne)[0]))


# ---------------------------------------------------------------------------------------------------------------------
# 1. lane-assignment invariance, bitwise
# ---------------------------------------------------------------------------------------------------------------------
VARIANTS = {
    "bench": (BENCH, 65536, "fp64"),
    "bench_ragged": (BENCH, 65491, "fp64"),
    "bench_fp32": (BENCH, 65536, "fp32"),           # default fp32 grid: 16 warps per SM = 75 776 lanes, no reuse in A
    "wind": (CASES["wind"], 65536, "fp64"),          # FwSpecGeneric: steady wind reloaded on adoption
    "param_rand_uniform": (CASES["param_rand_uniform"], 65536, "fp64"),   # FwSpecRand: parameter cache refilled
}
INVARIANCE_STEPS = 230      # the post-reset transient + 200 steps of the stationary episode mix
SAME_COUNTERS = ("env_steps", "attempts", "accepted", "failures", "resets", "rhs_evals")


@pytest.mark.gpu
@pytest.mark.parametrize("variant", list(VARIANTS))
def test_lane_assignment_invariance(built_lib, variant, monkeypatch):
    """Four handles, same seed, same actions, different lane assignment: A default grid and priority list, identity
    order; B default, a fresh random order every step; C one warp per SM with every aircraft whose first step is
    below dt on the priority list; D one warp per SM, empty priority list, reversed order.  After every step B, C and
    D equal A bitwise in the float32 outputs, the attempt counts and the whole state matrix."""
    c, n, precision = VARIANTS[variant]
    lanes = 32 * torch.cuda.get_device_properties(0).multi_processor_count   # one warp per SM
    assert n >= 4 * lanes, "C and D must reuse lanes: %d envs on %d lanes" % (n, lanes)
    gen = torch.Generator(device="cuda")
    gen.manual_seed(7)
    setups = (("A", {}, "identity"), ("B", {}, "random"),
              ("C", dict(ONE_WARP_PER_SM, FWGYM_LONG_DIV=1), "identity"),
              ("D", dict(ONE_WARP_PER_SM, FWGYM_LONG_DIV=0), "reversed"))
    handles = []
    try:
        for name, sw, kind in setups:
            v = make_vec(c, n, monkeypatch, precision=precision, **sw)
            handles.append((name, Order(v, kind, gen)))
        rows = handles[0][1].vec.state_rows()
        obs0 = [o.vec.reset().clone() for _, o in handles]
        for (name, _), x in zip(handles[1:], obs0[1:]):
            assert torch.equal(bits(obs0[0]), bits(x)), first_difference("%s: reset observation" % name, obs0[0], x)
        act_gen = torch.Generator(device="cuda")
        act_gen.manual_seed(3)
        ends = 0
        for t in range(INVARIANCE_STEPS):
            a = torch.rand((n, 3), generator=act_gen, device="cuda") * 2 - 1      # float32: the bench's input path
            outs = []
            for _, o in handles:
                o.before_step()
                obs, rew, done, term = o.vec.step_tensors(a)
                outs.append((obs, rew, done, term, o.vec.last_attempts(), o.vec.get_state()))
            ends += int(outs[0][2].sum())
            for (name, _), out in zip(handles[1:], outs[1:]):
                for what, x, y in zip(("observation", "reward", "done", "termination", "attempts"), outs[0], out):
                    assert torch.equal(bits(x), bits(y)), first_difference("%s step %d: %s" % (name, t, what), x, y)
                assert torch.equal(bits(outs[0][5]), bits(out[5])), \
                    first_difference("%s step %d: state" % (name, t), outs[0][5], out[5], rows)
        ctr = [o.vec.counters() for _, o in handles]
        for (name, _), cn in zip(handles, ctr):
            assert cn["watchdog"] == 0, (name, cn)
            assert all(cn[k] == ctr[0][k] for k in SAME_COUNTERS), (name, cn, ctr[0])
        print("lane invariance %s (%s): N=%d, one warp per SM = %d lanes (%.1f aircraft per lane per step in C, D); "
              "%d steps compared bitwise, %d episode ends, %d dopri5 attempts, %d failures; warp passes A/B/C/D %s"
              % (variant, precision, n, lanes, n / lanes, INVARIANCE_STEPS, ends, ctr[0]["attempts"],
                 ctr[0]["failures"], [cn["warp_max_attempts"] for cn in ctr]))
    finally:
        for _, o in handles:
            o.close()


# ---------------------------------------------------------------------------------------------------------------------
# 2. / 3. sampled oracle parity under reuse
# ---------------------------------------------------------------------------------------------------------------------
def compose_sample(parts, n, size, rng):
    """Union of the named id lists (first occurrence kept), filled up to `size` with random envs."""
    ids, seen, counts = [], set(), {}
    for name, lst in parts:
        new = [int(i) for i in dict.fromkeys(int(i) for i in lst) if i not in seen]   # a list may repeat an id too
        seen.update(new)
        ids += new
        counts[name] = len(new)
    fill = [int(i) for i in rng.permutation(n) if int(i) not in seen][:max(0, size - len(ids))]
    counts["random"] = len(fill)
    return np.array(ids + fill, dtype=np.int64), counts


def bench_sample(done, term, k, n, size=512, rng=None):
    """Envs where a full-size run goes wrong first: warp and block boundaries, the last env, a spread; the aligned
    32-env group with the most episode ends in one step (a full-warp cooperative reset with many resetting lanes); the
    envs with the most attempts and the most episode ends; numeric terminations; random envs for the rest."""
    groups = done[:, :n // 32 * 32].reshape(len(done), -1, 32).sum(-1)
    t, g = np.unravel_index(np.argmax(groups), groups.shape)
    numeric = np.nonzero((done & (term == TERM_NUMERIC)).any(0))[0][:32]
    parts = [("boundaries", [0, 1, 31, 32, 127, 128, n - 1] + list(range(0, n, 1024))),
             ("warp group %d (%d ends at step %d)" % (g, groups[t, g], t), range(32 * g, 32 * g + 32)),
             ("most attempts", np.argsort(-k.sum(0), kind="stable")[:64]),
             ("most episode ends", np.argsort(-done.sum(0), kind="stable")[:64]),
             ("numeric", numeric)]
    return compose_sample(parts, n, size, rng)


def reuse_sample(done, term, k, n, size=128, rng=None):
    return compose_sample([("most episode ends", np.argsort(-done.sum(0), kind="stable")[:size // 2])], n, size, rng)


def sampled_oracle_parity(c, n, steps, monkeypatch, choose, switches, random_order, label):
    """Pass A (device, free-running) records every env and step and picks the sample; the oracle steps only the
    sampled global ids; passes B (free-running, must equal A bitwise on every env) and C (the sampled columns' 27
    simulator values overwritten with the oracle's after every step) step in lockstep on the same float32 actions.
    Bars as BASELINE configs[1] (tests/test_gpu_parity.py::test_config1_4096_envs_100_steps), on every sampled env and
    step: done flags, termination names and attempt counts exact in both; <= 1e-9 per step on identical states (C),
    <= 1e-4 free-running (B)."""
    from fwgym_b200.vec_env import term_name
    act_gen = torch.Generator(device="cuda")
    act_gen.manual_seed(11)
    acts = torch.rand((steps, n, 3), generator=act_gen, device="cuda") * 2 - 1      # float32: the bench's input path
    order_gen = torch.Generator(device="cuda")
    order_gen.manual_seed(5)

    def open_handle():
        v = make_vec(c, n, monkeypatch, **switches)
        v.enable_f64_outputs(True)
        return Order(v, "random" if random_order else "identity", order_gen)

    # ---- pass A: the record (kept on the device: obs / reward for the bitwise check of pass B)
    oa = open_handle()
    try:
        obs0 = oa.vec.reset().clone()
        rec = {k: [] for k in ("obs", "rew", "done", "term", "k")}
        for t in range(steps):
            oa.before_step()
            obs, rew, done, term = oa.vec.step_tensors(acts[t])
            for key, x in zip(rec, (obs, rew, done, term, oa.vec.last_attempts())):
                rec[key].append(x.clone())
        state_a = oa.vec.get_state()
    finally:
        oa.close()
    rec = {key: torch.stack(x) for key, x in rec.items()}
    done_h, term_h, k_h = (rec[key].cpu().numpy() for key in ("done", "term", "k"))
    ids, counts = choose(done_h.astype(bool), term_h, k_h, n, rng=np.random.RandomState(17))
    assert len(ids) == len(set(ids.tolist())) and ids.min() >= 0 and ids.max() < n
    # ---- the oracle on the sampled global ids only
    t0 = time.perf_counter()
    want = pu.oracle_rollout_ids(harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], SEED, ids,
                                 acts[:, torch.as_tensor(ids, device="cuda")].double().cpu().numpy())
    t_oracle = time.perf_counter() - t0
    # ---- passes B (free-running) and C (per step on the oracle's states), lockstep
    sidx = torch.as_tensor(ids, device="cuda")
    ob = oc = None
    try:
        ob, oc = open_handle(), open_handle()
        rows = oc.vec.state_rows()
        ridx = torch.as_tensor([rows.index(r) for r in pu.STATE_ROWS], device="cuda")
        for o in (ob, oc):
            x = o.vec.reset()
            assert torch.equal(bits(x), bits(obs0)), first_difference("%s reset observation" % label, obs0, x)
            assert pu.rel_err(o.vec._obs64[sidx].cpu().numpy(), want["obs"][0], 1e-3).max() <= TOL
        worst = {tag: dict(obs=(0.0,), rew=(0.0,), state=(0.0,)) for tag in ("free", "sync")}

        def track(tag, what, err, t, names):
            if err.max() > worst[tag][what][0]:
                i, j = np.unravel_index(np.argmax(err), err.shape) if err.ndim == 2 else (int(np.argmax(err)), None)
                worst[tag][what] = (float(err.max()), "step %d env %d%s" % (t, ids[i], "" if j is None else " " + names[j]))

        for t in range(steps):
            for tag, o in (("free", ob), ("sync", oc)):
                o.before_step()
                obs, rew, done, term = o.vec.step_tensors(acts[t])
                k = o.vec.last_attempts()
                if tag == "free":
                    for what, x, y in zip(("observation", "reward", "done", "termination", "attempts"),
                                          (obs, rew, done, term, k), (rec[key][t] for key in rec)):
                        assert torch.equal(bits(x), bits(y)), \
                            first_difference("%s step %d, free-running vs pass A: %s" % (label, t, what), y, x)
                d = done[sidx].cpu().numpy().astype(bool)
                assert np.array_equal(d, want["done"][t]), \
                    "%s %s: done flags differ at step %d, envs %s" % (label, tag, t, ids[d != want["done"][t]])
                kk = k[sidx].cpu().numpy()
                assert np.array_equal(kk, want["k"][t]), \
                    "%s %s: attempt counts differ at step %d, envs %s" % (label, tag, t, ids[kk != want["k"][t]])
                tc = term[sidx].cpu().numpy()
                for i in np.nonzero(d)[0]:
                    assert term_name(int(tc[i])) == want["term"][t][i], (label, tag, t, ids[i], tc[i], want["term"][t][i])
                track(tag, "obs", pu.rel_err(o.vec._obs64[sidx].cpu().numpy(), want["obs"][t + 1], 1e-3), t,
                      ["obs[%d]" % j for j in range(want["obs"].shape[2])])
                track(tag, "rew", pu.rel_err(o.vec._rew64[sidx].cpu().numpy(), want["rew"][t], 1e-3), t, None)
                st = o.vec.get_state()[ridx][:, sidx].T.cpu().numpy()
                track(tag, "state", pu.rel_err(st, want["state"][t], 1e-3), t, pu.STATE_ROWS)
            st = oc.vec.get_state()
            st[ridx.unsqueeze(1), sidx.unsqueeze(0)] = torch.as_tensor(want["state"][t].T.copy(), device="cuda")
            oc.vec.set_state(st)
        state_b = ob.vec.get_state()
        assert torch.equal(bits(state_b), bits(state_a)), \
            first_difference("%s final state, free-running vs pass A" % label, state_a, state_b, rows)
    finally:
        for o in (ob, oc):
            if o is not None:
                o.close()
    n_done = int(want["done"].sum())
    n_numeric = int(sum(term_name(TERM_NUMERIC) == s for s in want["term"].ravel()))
    print("%s: N=%d, %d steps; sample of %d envs %s; in it %d episode ends, %d numeric terminations, %d dopri5 attempts "
          "(oracle: %d env-steps in %.1f s); worst rel err per step on identical states %r, free-running %r"
          % (label, n, steps, len(ids), counts, n_done, n_numeric, int(want["k"].sum()), len(ids) * steps, t_oracle,
             worst["sync"], worst["free"]))
    assert max(w[0] for w in worst["sync"].values()) <= TOL, worst
    assert max(w[0] for w in worst["free"].values()) <= 1e-4, worst


@pytest.mark.gpu
def test_bench_workload_sampled_oracle(built_lib, monkeypatch):
    """The bench workload at its full size (65 536 envs, default grid: ~40 % of the aircraft of a step are adopted by
    a lane that already flew one), 250 steps from reset, against the oracle on 512 sampled envs."""
    sampled_oracle_parity(BENCH, 65536, 250, monkeypatch, bench_sample, {}, False, "bench workload, full size")


REUSE_CASES = ("wind", "param_rand_uniform")


@pytest.mark.gpu
@pytest.mark.parametrize("case", REUSE_CASES)
def test_reuse_heavy_sampled_oracle(built_lib, case, monkeypatch):
    """The FwSpecGeneric (steady wind) and FwSpecRand instantiations with ~3.5 aircraft
    per lane per step: 16 384 envs on one warp per SM, every aircraft whose first step is below dt on the priority
    list, a random adoption order every step; 60 steps against the oracle on 128 sampled envs."""
    switches = dict(ONE_WARP_PER_SM, FWGYM_LONG_DIV=1)
    sampled_oracle_parity(CASES[case], 16384, 60, monkeypatch, reuse_sample, switches, True, "reuse-heavy %s" % case)


def test_bench_sample_is_distinct_and_complete():
    """The full-size sample: exactly 512 distinct ids in range, every listed boundary env, the whole busiest warp
    group and every numeric termination in it (the boundary list itself repeats env 0)."""
    rng = np.random.RandomState(0)
    T, n = 250, 65536
    done = rng.rand(T, n) < 0.005
    done[40, 32 * 77:32 * 78] = True
    term = np.where(done, rng.choice([1, TERM_NUMERIC, 16], size=(T, n), p=[0.9, 0.02, 0.08]), 0)
    k = rng.randint(1, 9, (T, n))
    ids, counts = bench_sample(done, term, k, n, rng=np.random.RandomState(17))
    assert len(ids) == 512 == len(set(ids.tolist())) and ids.min() >= 0 and ids.max() < n
    assert sum(counts.values()) == 512
    assert {0, 1, 31, 32, 127, 128, n - 1, 1024, n - 1024} <= set(ids.tolist())
    assert set(range(32 * 77, 32 * 78)) <= set(ids.tolist())
    numeric = np.nonzero((done & (term == TERM_NUMERIC)).any(0))[0][:32]
    assert set(numeric.tolist()) <= set(ids.tolist())


# ---------------------------------------------------------------------------------------------------------------------
# 4. the oracle over an explicit id list (CPU)
# ---------------------------------------------------------------------------------------------------------------------
def test_oracle_rollout_ids_matches_contiguous_rollout():
    """oracle_rollout_ids on non-contiguous, unordered global ids gives exactly the arrays of those envs in a
    contiguous oracle_rollout_parallel run (the streams are keyed by the global env id, not by position)."""
    c = CASES["default"]
    args = (harness.config_path(c["config"]), c["config_kw"], c["sim_kw"], 41)
    acts = np.random.RandomState(5).uniform(-1, 1, (10, 8, 3))
    whole = pu.oracle_rollout_parallel(*args, acts, procs=2)
    ids = np.array([6, 1, 4, 7])
    part = pu.oracle_rollout_ids(*args, ids, acts[:, ids], procs=3)
    assert set(part) == set(whole)
    for key in whole:
        assert np.array_equal(part[key], whole[key][:, ids]), key
    assert part["state"].shape == (10, 4, 27)
