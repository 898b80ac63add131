"""The float64 C oracle of SmartClimateEnv (SURVEY.md section 8f rank 3) against golden vectors produced by the
reference itself (tests/golden/climate_golden.npz) and, in the build container, the live reference.  EXACT: the
oracle evaluates the reference's float64 expressions in the same order on the same libm."""
import logging

import numpy as np
import pytest

from oracle import golden_files, ref_loader, replay
from oracle.c_oracle import ClimateOracle

CASES = ["random_default", "random_hi_ids", "thermostat", "extremes", "small_office"]


@pytest.fixture(scope="module")
def kgold():
    return golden_files.load("climate")


def meta(g, name):
    n_envs, n_steps, seed, base, max_occ, minutes = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, max_occupancy=max_occ, episode_minutes=minutes)


@pytest.mark.parametrize("name", CASES)
def test_c_oracle_matches_golden_exactly(kgold, name):
    g, m = kgold, meta(kgold, name)
    orc = ClimateOracle(m["n_envs"], m["max_occupancy"], m["episode_minutes"], seed=m["seed"], env_id_base=m["base"])
    assert np.array_equal(orc.reset(), g[f"{name}/reset_obs"])
    for t in range(m["n_steps"]):
        obs, rew, term, trunc = orc.step(g[f"{name}/ac_temp"][:, t], g[f"{name}/lights"][:, t])
        assert np.array_equal(orc.reward64, g[f"{name}/reward"][:, t]), t
        assert np.array_equal(term, g[f"{name}/terminated"][:, t]) and not trunc.any()
        assert np.array_equal(obs, g[f"{name}/obs"][:, t]), t
        for k, arr in (("comfort", orc.comfort), ("ac_penalty", orc.ac_penalty), ("light_penalty", orc.light_penalty)):
            assert np.array_equal(arr, g[f"{name}/{k}"][:, t]), (k, t)
        st = orc.state()
        for k, gk in (("room_temp", "room_temp"), ("num_people", "num_people"), ("energy_usage", "energy_usage"),
                      ("comfort_time", "comfort_time"), ("current_step", "step"), ("rng_counter", "rng_counter")):
            assert np.array_equal(st[k].astype(np.float64), g[f"{name}/{gk}"][:, t].astype(np.float64)), (k, t)
    assert orc.stats()["n_episodes"] == int(g[f"{name}/terminated"].sum())


def test_reference_facts(kgold):
    g = kgold
    term = g["random_default/terminated"]
    assert term.sum() == 6 and (g["random_default/step"][term == 1] == 0).all()   # 1440-step limit -> terminated -> reset
    assert g["random_default/reset_obs"].shape == (3, 9)
    assert (g["random_default/obs"][:, :, 4] >= 16).all() and (g["random_default/obs"][:, :, 4] <= 32).all()  # ac clipped
    assert g["random_default/room_temp"].max() == 50.0                              # clamp reached
    assert g["small_office/num_people"].max() <= 3


@pytest.mark.skipif(not ref_loader.reference_available(),
                    reason="needs the original project's sources (BENG_REFERENCE_ROOT=<its checkout>)")
def test_c_oracle_matches_live_reference():
    mod = ref_loader.load_climate()
    n, T, seed = 3, 1600, 44
    rng = np.random.default_rng(1)
    orc = ClimateOracle(n, seed=seed)
    orc.reset()
    envs = []
    for e in range(n):
        env = mod.SmartClimateEnv(log_level=logging.ERROR)
        env.rng = replay.ReplayGenerator(seed, e)
        obs, _ = env.reset()
        assert np.array_equal(obs, orc.obs[e])
        envs.append(env)
    for t in range(T):
        ac = (rng.random(n) * 24 + 12).astype(np.float32)
        lights = rng.integers(0, 2, (n, 4)).astype(np.int8)
        orc.step(ac, lights)
        for e, env in enumerate(envs):
            obs, r, term, trunc, info = env.step({"ac_temp": ac[e:e + 1], "lights": lights[e]})
            if term:
                obs, _ = env.reset()
            assert r == orc.reward64[e] and term == bool(orc.terminated[e]) and np.array_equal(obs, orc.obs[e])
