"""Full-size (BASELINE.json sizes) checks through size-independent properties: determinism, counter identities,
unit quaternions, checkpoint round trip, actuator/airspeed bounds."""
import numpy as np
import pytest
import torch

from oracle import harness

pytestmark = pytest.mark.gpu
N = 65536
CONFIG_KW = {"observation": {"noise": {"mean": 0, "var": 0.1}}}
SIM_KW = {"turbulence": True, "turbulence_intensity": "moderate"}


def make(n=N, seed=3, **kw):
    from fwgym_b200 import FixedWingVecEnv
    return FixedWingVecEnv(harness.config_path(), n, config_kw=CONFIG_KW, sim_config_kw=SIM_KW, seed=seed, **kw)


def test_determinism_and_invariants(built_lib):
    acts = torch.rand((12, N, 3), device="cuda") * 2 - 1
    runs = []
    for rep in range(2):
        v = make()
        v.reset()
        for t in range(12):
            obs, rew, done, term = v.step_tensors(acts[t])
        runs.append((obs.clone(), rew.clone(), v.get_state().clone(), v.counters()))
        rows = v.state_rows()
        v.close()
    assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1])
    assert torch.equal(runs[0][2], runs[1][2])
    st, ctr = runs[0][2], runs[0][3]
    q = st[:4]
    assert torch.allclose((q * q).sum(0), torch.ones(N, dtype=torch.float64, device="cuda"), atol=1e-12)
    assert ctr["env_steps"] == 12 * N
    assert ctr["rhs_evals"] == 2 * ctr["env_steps"] + 6 * ctr["attempts"]
    assert ctr["attempts"] >= ctr["accepted"] >= ctr["env_steps"] - ctr["failures"]
    el, er, th = (st[rows.index(k)] for k in ("elevon_left", "elevon_right", "throttle"))
    lo, hi = np.radians(-30) - 1e-12, np.radians(35) + 1e-12
    assert el.min() >= lo and el.max() <= hi and er.min() >= lo and er.max() <= hi
    assert th.min() >= 0 and th.max() <= 1
    assert torch.isfinite(runs[0][0]).all() and torch.isfinite(runs[0][1]).all()
    steps = st[rows.index("steps_count")]
    assert steps.max() <= 12


def test_checkpoint_roundtrip(built_lib):
    """get_state / set_state: a restored handle continues bit-identically (checkpoint/resume, SURVEY §5)."""
    n = 4096
    acts = torch.rand((10, n, 3), device="cuda") * 2 - 1
    a = make(n=n, seed=8)
    a.reset()
    for t in range(5):
        a.step_tensors(acts[t])
    snap = a.get_state().clone()
    b = make(n=n, seed=8)
    b.set_state(snap)
    for t in range(5, 10):
        oa, ra, da, _ = a.step_tensors(acts[t])
        ob, rb, db, _ = b.step_tensors(acts[t])
        assert torch.equal(oa, ob) and torch.equal(ra, rb) and torch.equal(da, db)


def test_vecenv_surface(built_lib):
    """SB-style VecEnv duck typing used by the reference's scripts (train_rl_controller.py:223-225)."""
    v = make(n=256, keep_terminal_obs=True)
    obs = v.reset()
    assert obs.shape == (256, 14) and obs.dtype == torch.float32
    assert v.observation_space.shape == (14,) and v.action_space.shape == (3,)
    o, r, d, infos = v.step(np.zeros((256, 3), dtype=np.float32))
    assert o.shape == (256, 14) and r.shape == (256,) and d.dtype == torch.bool and len(infos) == 256
    assert set(infos[0]["target"]) == {"roll", "pitch", "Va"}
    v.env_method("set_curriculum_level", 0.25)
    v.reset()
    tg = v.get_attr("target")
    assert all(abs(t["roll"]) <= np.radians(15) + 1e-9 for t in tg)   # +-60 deg scaled by 0.25
    assert v.get_attr("steps_count")[0] == 0


@pytest.mark.parametrize("graph", [False, True])
def test_ppo_loop_runs(built_lib, graph):
    """SURVEY §8f row 3 (BASELINE configs[3] at a small size): PPO2-default loop with the device VecNormalize and a
    torch MLP policy steps the batched env, updates without NaNs and reports the time split - eagerly and with the
    rollout (policy + env kernels incl. the programmatic dependent launch + GAE) captured into a CUDA graph."""
    from fwgym_b200 import FixedWingVecEnv, ppo
    env = FixedWingVecEnv(harness.config_path("fixed_wing_config_examples.json"), 2048, seed=4)
    env.env_method("set_curriculum_level", 0.25)
    model, norm, stats = ppo.train(env, total_env_steps=2048 * 32 * 3, n_steps=32, cuda_graph=graph)
    assert stats["iterations"] == 3 and stats["env_steps"] == 2048 * 32 * 3
    assert env.counters()["env_steps"] == 2048 * 32 * 3 and env.counters()["watchdog"] == 0
    assert all(np.isfinite(h["loss"]) for h in stats["history"])
    assert abs(sum(stats["time_fraction"].values()) - 1.0) < 1e-9
    assert all(torch.isfinite(p).all() for p in model.parameters())
    assert float(norm.obs_rms.count) > 2048 * 32
    print("PPO smoke (cuda_graph=%s): %.3g env-steps/s inside training; time split %s"
          % (graph, stats["env_steps_per_s"], {k: round(v, 3) for k, v in stats["time_fraction"].items()}))
    env.close()


def test_bench_dump_outputs_repeat(built_lib, tmp_path):
    """bench.py --dump-outputs: the last timed step's obs / reward / done / term, the same in two runs with the same
    arguments, and every timed pass runs --steps steps."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    dumps = []
    for rep in range(2):
        out_dir = tmp_path / str(rep)
        out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--steps", "3", "--warmup", "2",
                              "--envs-per-gpu", "512", "--burn-in", "20", "--no-cpu-baseline",
                              "--dump-outputs", str(out_dir)], capture_output=True, text=True, timeout=600, cwd=root)
        assert out.returncode == 0, out.stderr[-2000:]
        line = json.loads(out.stdout)
        assert line["steps"] == 3 and line["e2e"]["steps"] == 3
        dumps.append({k: np.load(out_dir / (k + ".npy")) for k in ("obs", "reward", "done", "term")})
    d = dumps[0]
    assert d["obs"].shape == (512, 14) and d["obs"].dtype == np.float32 and d["reward"].shape == (512,)
    assert set(np.unique(d["done"])) <= {0.0, 1.0} and np.isfinite(d["obs"]).all()
    for k in d:
        assert np.array_equal(d[k], dumps[1][k]), k


def test_vecnormalize_and_gae_on_device(built_lib):
    """DeviceVecNormalize / compute_gae on cuda:0 against the numpy twins of stable-baselines' VecNormalize and PPO2's
    GAE (tests/test_ppo_cpu.py holds the oracle and runs the same check on the CPU)."""
    import test_ppo_cpu
    test_ppo_cpu.check_vecnormalize_and_gae("cuda:0")
