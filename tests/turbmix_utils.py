"""Test infrastructure for per-env Dryden intensities (mixed handles): the CPU mirror of the level a reset draws, and an
oracle runner that rebuilds its Dryden model at every reset at that level."""
import numpy as np

from oracle import harness, philox
from oracle.pyfly_restated import DrydenGustModel

RS_TURBLVL = 5                       # csrc/philox.cuh FW_RS_TURBLVL
LEVELS = ("none", "light", "moderate", "severe")


def level_cdf(probabilities):
    from fwgym_b200.config import turbulence_cdf
    return turbulence_cdf(probabilities)


def drawn_level(seed, genv, tick, cdf):
    """The level the reset of global env `genv` at rng tick `tick` draws (one uniform of stream FW_RS_TURBLVL, index 0,
    then the first level whose cumulative probability exceeds it)."""
    from fwgym_b200.config import draw_turbulence_level
    return draw_turbulence_level(cdf, philox.PhiloxKey(seed, genv).uniform01(tick, RS_TURBLVL, 0))


class LevelOracleRunner(harness.OracleRunner):
    """OracleRunner whose episodes fly at the level the device draws for them: at each reset the mirror draws the level
    for the reset's tick and the simulator's Dryden model is swapped for one of that intensity (level 0: turbulence off,
    no noise).  `pinned`: a fixed level instead of the draw."""

    def __init__(self, env, seed, env_id, cdf, pinned=None):
        super().__init__(env, seed, env_id)
        self.seed_, self.cdf, self.pinned = seed, cdf, pinned
        self.levels = []
        sim = env.simulator
        self._models = {}
        self._dt, self._b = sim.wind.dryden.dt, sim.params["b"]

    def _model(self, lvl):
        if lvl not in self._models:
            self._models[lvl] = DrydenGustModel(self._dt, self._b, intensity=LEVELS[lvl])
        return self._models[lvl]

    def reset(self, state=None, target=None, turbulence_noise=None):
        lvl = self.pinned if self.pinned is not None else drawn_level(self.seed_, self.key.env, self.tick, self.cdf)
        wind = self.env.simulator.wind
        wind.turbulence = self.turbulence = lvl != 0
        if lvl:
            wind.dryden = self._model(lvl)
        self.levels.append(lvl)
        return super().reset(state, target, turbulence_noise)


def level_rollout_slice(args):
    """Worker (own process): free-running rollout of LevelOracleRunners with global ids `env_ids` on `actions`
    [T, n, 3] -> dict of per-step arrays as tests/parity_utils.oracle_rollout_slice, plus `level` [T + 1, n]: the level of
    each env's running episode after the reset and after every step."""
    config, config_kw, sim_kw, seed, env_ids, actions, cdf = args
    orcs = [LevelOracleRunner(harness.make_env("restated", config, config_kw, sim_kw), seed, int(g), cdf)
            for g in env_ids]
    obs = [np.stack([np.asarray(o.reset(), dtype=np.float64).ravel() for o in orcs])]
    lvl = [[o.levels[-1] for o in orcs]]
    rew, done, k, state = [], [], [], []
    for t in range(actions.shape[0]):
        res = [o.step(actions[t, i]) for i, o in enumerate(orcs)]
        obs.append(np.stack([np.asarray(r[0], dtype=np.float64).ravel() for r in res]))
        rew.append([float(r[1]) for r in res])
        done.append([bool(r[2]) for r in res])
        k.append([o.attempts_last() for o in orcs])
        state.append(np.stack([o.ode_state() for o in orcs]))
        lvl.append([o.levels[-1] for o in orcs])
    return dict(obs=np.array(obs), rew=np.array(rew), done=np.array(done), k=np.array(k), state=np.array(state),
                level=np.array(lvl))


def level_rollout(config, config_kw, sim_kw, seed, env_ids, actions, cdf, procs=None):
    """level_rollout_slice over spawned worker processes (the caller holds a CUDA context), in the order of env_ids."""
    import multiprocessing as mp
    import os
    env_ids = np.asarray(env_ids, dtype=np.int64)
    n = len(env_ids)
    procs = min(procs or os.cpu_count() or 1, n)
    bounds = np.linspace(0, n, procs + 1).astype(int)
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    old = os.environ.get("PYTHONPATH", "")
    os.environ["PYTHONPATH"] = os.pathsep.join([root, os.path.join(root, "tests")] + ([old] if old else []))
    try:
        with mp.get_context("spawn").Pool(procs) as pool:
            parts = pool.map(level_rollout_slice,
                             [(config, config_kw, sim_kw, seed, env_ids[lo:hi], actions[:, lo:hi], cdf)
                              for lo, hi in zip(bounds[:-1], bounds[1:]) if hi > lo], chunksize=1)
    finally:
        os.environ["PYTHONPATH"] = old
    return {key: np.concatenate([p[key] for p in parts], axis=1) for key in parts[0]}
