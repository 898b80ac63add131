"""GPU parity tests for smartclimate (SURVEY.md section 8f rank 3): CUDA path (through the C ABI) against the float64
CPU oracle and the golden vectors recorded from the reference.

Tolerances: float32 observations and float64 state/rewards are compared at rtol 1e-5 / atol 1e-6 and rtol 1e-9 (the only
source of difference is CUDA's log/cos vs glibc's in the Box-Muller normal draw); integer fields (people, step, comfort
time, RNG counter, terminated) are exact."""

import numpy as np
import pytest
import torch

from oracle import golden_files

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
RTOL, ATOL, RTOL64 = 1e-5, 1e-6, 1e-9
CASES = ["random_default", "random_hi_ids", "thermostat", "extremes", "small_office"]


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    assert torch.cuda.is_available()
    p._lib.load()
    return p


@pytest.fixture(scope="module")
def kgold():
    return golden_files.load("climate")


def np_(t):
    return t.cpu().numpy()


def meta(g, name):
    n_envs, n_steps, seed, base, max_occ, minutes = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, max_occupancy=max_occ, episode_minutes=minutes)


@pytest.mark.parametrize("name", CASES)
def test_golden_replay(pkg, kgold, name):
    g, m = kgold, meta(kgold, name)
    env = pkg.BatchedSmartClimateEnv(m["n_envs"], m["max_occupancy"], episode_minutes=m["episode_minutes"], device=DEV,
                                     seed=m["seed"], env_id_base=m["base"])
    obs, info = env.reset()
    assert obs.shape == (m["n_envs"], 9) and info == {}
    np.testing.assert_allclose(np_(obs), g[f"{name}/reset_obs"], rtol=RTOL, atol=ATOL)
    ac = torch.from_numpy(g[f"{name}/ac_temp"]).to(DEV)
    li = torch.from_numpy(g[f"{name}/lights"]).to(DEV)
    for t in range(m["n_steps"]):
        obs, rew, term, trunc, info = env.step({"ac_temp": ac[:, t].contiguous(), "lights": li[:, t].contiguous()})
        assert np.array_equal(np_(term).astype(np.uint8), g[f"{name}/terminated"][:, t]) and not np_(trunc).any()
        np.testing.assert_allclose(np_(obs), g[f"{name}/obs"][:, t], rtol=RTOL, atol=ATOL, err_msg=f"obs, step {t}")
        np.testing.assert_allclose(np_(info["reward64"]), g[f"{name}/reward"][:, t], rtol=RTOL64, atol=1e-9)
        np.testing.assert_allclose(np_(rew), g[f"{name}/reward"][:, t].astype(np.float32), rtol=RTOL, atol=ATOL)
        for k in ("comfort", "ac_penalty", "light_penalty"):
            np.testing.assert_allclose(np_(info[k]), g[f"{name}/{k}"][:, t], rtol=RTOL64, atol=1e-9)
        assert np.array_equal(np_(env.num_people), g[f"{name}/num_people"][:, t])
        assert np.array_equal(np_(env.current_step), g[f"{name}/step"][:, t])
        assert np.array_equal(np_(env.comfort_time), g[f"{name}/comfort_time"][:, t])
        assert np.array_equal(np_(env.rng_counter), g[f"{name}/rng_counter"][:, t].astype(np.int64))
        np.testing.assert_allclose(np_(env.room_temp), g[f"{name}/room_temp"][:, t], rtol=RTOL64)
        np.testing.assert_allclose(np_(env.energy_usage), g[f"{name}/energy_usage"][:, t], rtol=RTOL64)
    assert env.episode_stats()["n_episodes"] == int(g[f"{name}/terminated"].sum())


@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
def test_random_rollout_vs_oracle(pkg, mode):
    from oracle.c_oracle import ClimateOracle

    n, seed, base, T = 10007, 5, 900, 330
    env = pkg.BatchedSmartClimateEnv(n, episode_minutes=300, device=DEV, seed=seed, env_id_base=base, autoreset_mode=mode)
    orc = ClimateOracle(n, episode_minutes=300, seed=seed, env_id_base=base, autoreset=mode)
    np.testing.assert_allclose(np_(env.reset()[0]), orc.reset(), rtol=RTOL, atol=ATOL)
    gen = torch.Generator(device=DEV).manual_seed(2)
    for t in range(T):
        ac = torch.rand(n, device=DEV, generator=gen) * 24 + 12
        li = torch.randint(0, 2, (n, 4), device=DEV, generator=gen).to(torch.int8)
        env.step({"ac_temp": ac, "lights": li})
        orc.step(np_(ac), np_(li))
        assert np.array_equal(np_(env.terminated).astype(np.uint8), orc.terminated), t
        np.testing.assert_allclose(np_(env.obs), orc.obs, rtol=RTOL, atol=ATOL, err_msg=f"obs, step {t}")
        np.testing.assert_allclose(np_(env.reward64), orc.reward64, rtol=RTOL64, atol=1e-9)
        if t % 30 == 0 or t >= 298:
            st = orc.state()
            assert np.array_equal(np_(env.num_people), st["num_people"]) and np.array_equal(np_(env.current_step), st["current_step"])
            assert np.array_equal(np_(env.rng_counter), st["rng_counter"].astype(np.int64))
            np.testing.assert_allclose(np_(env.total_reward), st["total_reward"], rtol=RTOL64, atol=1e-7)
    if mode != "disabled":
        s, o = env.episode_stats(), orc.stats()
        assert s["n_episodes"] == o["n_episodes"] == n
        np.testing.assert_allclose([s["sum_return"], s["sum_length"]], [o["sum_return"], o["sum_length"]], rtol=1e-9)


def test_million_env_batch_host_path_and_state_dict(pkg):
    from oracle.c_oracle import ClimateOracle

    n, seed = 1 << 20, 0
    env = pkg.BatchedSmartClimateEnv(n, device=DEV, seed=seed)
    orc = ClimateOracle(n, seed=seed)
    np.testing.assert_allclose(np_(env.reset()[0]), orc.reset(), rtol=RTOL, atol=ATOL)
    gen = torch.Generator(device=DEV).manual_seed(0)
    for t in range(6):
        ac = torch.rand(n, device=DEV, generator=gen) * 24 + 12
        li = torch.randint(0, 2, (n, 4), device=DEV, generator=gen).to(torch.int8)
        obs, rew, term, trunc, info = env.step({"ac_temp": ac.view(n, 1), "lights": li})
        orc.step(np_(ac), np_(li))
        np.testing.assert_allclose(np_(obs), orc.obs, rtol=RTOL, atol=ATOL)
        assert bool((obs[:, 4] >= 16).all() and (obs[:, 4] <= 32).all() and (obs[:, 0] >= 10).all() and (obs[:, 0] <= 50).all())
    small = pkg.BatchedSmartClimateEnv(3000, device=DEV, seed=4)
    twin = pkg.BatchedSmartClimateEnv(3000, device=DEV, seed=4)
    small.reset(), twin.reset()
    rng = np.random.default_rng(0)
    for t in range(20):
        act = {"ac_temp": (rng.random((3000, 1)) * 20 + 14).astype(np.float32), "lights": rng.integers(0, 2, (3000, 4)).astype(np.int8)}
        obs, rew, term, trunc, _ = small.step_host(act)
        twin.step(act)
        assert isinstance(obs, np.ndarray) and np.array_equal(obs, np_(twin.obs)) and np.array_equal(rew, np_(twin.reward))
    clone = pkg.BatchedSmartClimateEnv(3000, device=DEV, seed=99)
    clone.load_state_dict(small.state_dict())
    small.step(act), clone.step(act)
    assert torch.equal(small.obs, clone.obs)


def test_single_env_facade_and_truncation_flag(pkg, kgold):
    g, name = kgold, "thermostat"
    m = meta(g, name)
    env = pkg.SmartClimateEnv(device=DEV, seed=m["seed"], env_id=m["base"])
    obs, info = env.reset()
    assert obs.shape == (9,) and obs.dtype == np.float32 and info == {}
    assert set(env.action_space.keys()) == {"ac_temp", "lights"}
    for t in range(50):
        a = {"ac_temp": np.array([g[f"{name}/ac_temp"][0, t]], np.float32), "lights": g[f"{name}/lights"][0, t]}
        obs, r, term, trunc, info = env.step(a)
        assert isinstance(r, float) and term is False and trunc is False
        np.testing.assert_allclose(r, g[f"{name}/reward"][0, t], rtol=RTOL64, atol=1e-9)
        np.testing.assert_allclose(obs, g[f"{name}/obs"][0, t], rtol=RTOL, atol=ATOL)
        assert set(info) == {"comfort", "ac_penalty", "light_penalty", "comfort_time", "energy_usage", "step"}
        assert info["step"] == t + 1 and info["comfort_time"] == g[f"{name}/comfort_time"][0, t]
    on = pkg.BatchedSmartClimateEnv(512, episode_minutes=5, device=DEV, seed=1, time_limit_truncation=True)
    on.reset()
    for t in range(12):
        _, _, term, trunc, _ = on.step({"ac_temp": torch.full((512,), 22.0, device=DEV), "lights": torch.zeros((512, 4), dtype=torch.int8, device=DEV)})
        assert torch.equal(term, trunc) and bool(term.all()) == ((t + 1) % 5 == 0)
