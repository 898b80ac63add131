"""The C oracle of WorldBuilderEnv (SURVEY.md section 8f rank 3) against golden vectors produced by the reference itself
(tests/golden/builder_golden.npz) and, in the build container, the live reference.  Integer dynamics: EXACT."""

import numpy as np
import pytest

from oracle import golden_files, ref_loader, replay
from oracle.c_oracle import BuilderOracle

CASES = ["random_g10", "random_hi_ids", "farmer_g10", "spam_g10", "farmer_g4"]


@pytest.fixture(scope="module")
def bgold():
    return golden_files.load("builder")


def meta(g, name):
    n_envs, n_steps, seed, base, G = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, G=G)


@pytest.mark.parametrize("name", CASES)
def test_c_oracle_matches_golden_exactly(bgold, name):
    g, m = bgold, meta(bgold, name)
    orc = BuilderOracle(m["n_envs"], m["G"], seed=m["seed"], env_id_base=m["base"])
    orc.reset()
    assert (orc.grid == 0).all() and orc.resources[0].tolist() == [25, 20, 10, 3] and orc.capacity[0, 0] == 10
    wins = 0
    for t in range(m["n_steps"]):
        orc.step(g[f"{name}/action"][:, t].astype(np.int64))
        assert np.array_equal(orc.reward, g[f"{name}/reward"][:, t]), t
        assert np.array_equal(orc.terminated, g[f"{name}/terminated"][:, t]) and not orc.truncated.any()
        assert np.array_equal(orc.grid, g[f"{name}/grid"][:, t]) and np.array_equal(orc.resources, g[f"{name}/resources"][:, t])
        assert np.array_equal(orc.capacity[:, 0], g[f"{name}/capacity"][:, t])
        assert np.array_equal(orc.win_steps[:, 0], g[f"{name}/win_steps"][:, t])
        st = orc.state()
        assert np.array_equal(st["steps"], g[f"{name}/steps"][:, t]) and np.array_equal(st["building_counts"], g[f"{name}/counts"][:, t])
        assert np.array_equal(st["rng_counter"], g[f"{name}/rng_counter"][:, t])
        wins += int(g[f"{name}/won"][:, t].sum())
    s = orc.stats()
    assert s["n_episodes"] == int(g[f"{name}/terminated"].sum()) and s["wins"] == wins


def test_reference_facts(bgold):
    g = bgold
    assert g["farmer_g10/won"].sum() >= 1                                         # +100 win episodes exist
    won = g["farmer_g10/won"] == 1
    assert (g["farmer_g10/reward"][won] == 100).all()
    lost = (g["random_g10/terminated"] == 1) & (g["random_g10/won"] == 0)
    assert lost.sum() > 10 and (g["random_g10/reward"][lost] == -100).all()      # starvation -> -100
    assert (g["farmer_g4/grid"] > 0).sum(axis=(2, 3)).max() == 16                 # the 4x4 board fills up completely


def test_invalid_action_and_modes():
    orc = BuilderOracle(3, seed=1)
    orc.reset()
    orc.step(np.array([9, -1, 0]))
    assert orc.invalid == 2 and orc.state()["steps"].tolist() == [0, 0, 1]
    dis = BuilderOracle(4, seed=2, autoreset="disabled")
    dis.reset()
    for t in range(40):
        dis.step(np.full(4, 4))       # houses only: starves, then keeps reporting the dead state (no auto-reset)
    assert dis.terminated.all() and (dis.reward == -100).all() and (dis.resources[:, 3] == 0).all()


@pytest.mark.skipif(not ref_loader.reference_available(),
                    reason="needs the original project's sources (BENG_REFERENCE_ROOT=<its checkout>)")
def test_c_oracle_matches_live_reference():
    env_mod, gl = ref_loader.load_builder()
    real_np = gl.np
    n, T, seed = 4, 600, 71
    rng = np.random.default_rng(9)
    orc = BuilderOracle(n, seed=seed)
    orc.reset()
    try:
        envs = []
        for e in range(n):
            rr = replay.ReplayRandom(seed, e)
            gl.np = replay.NumpyWithReplayRandint(rr)
            env = env_mod.WorldBuilderEnv()
            env.reset()
            envs.append((env, rr))
        for t in range(T):
            acts = rng.choice(5, size=n, p=[0.35, 0.2, 0.15, 0.15, 0.15])
            orc.step(acts)
            for e, (env, rr) in enumerate(envs):
                gl.np = replay.NumpyWithReplayRandint(rr)
                obs, r, term, trunc, info = env.step(int(acts[e]))
                if term:
                    obs, info = env.reset()
                assert r == orc.reward[e] and term == bool(orc.terminated[e])
                assert np.array_equal(obs["grid"], orc.grid[e]) and np.array_equal(obs["resources"], orc.resources[e])
    finally:
        gl.np = real_np
