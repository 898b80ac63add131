"""GPU parity tests for world_builder_env (SURVEY.md section 8f rank 3): CUDA path (through the C ABI) against the CPU
oracle and the golden vectors recorded from the reference.  Integer dynamics: EXACT (array equality everywhere)."""

import numpy as np
import pytest
import torch

from oracle import golden_files

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
CASES = ["random_g10", "random_hi_ids", "farmer_g10", "spam_g10", "farmer_g4"]


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    assert torch.cuda.is_available()
    p._lib.load()
    return p


@pytest.fixture(scope="module")
def bgold():
    return golden_files.load("builder")


def np_(t):
    return t.cpu().numpy()


def meta(g, name):
    n_envs, n_steps, seed, base, G = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, G=G)


@pytest.mark.parametrize("name", CASES)
def test_golden_replay(pkg, bgold, name):
    g, m = bgold, meta(bgold, name)
    env = pkg.BatchedWorldBuilderEnv(m["n_envs"], m["G"], device=DEV, seed=m["seed"], env_id_base=m["base"])
    obs, info = env.reset()
    assert set(obs) == {"grid", "resources", "population_capacity", "win_steps"} and not bool(obs["grid"].any())
    assert np_(obs["resources"])[0].tolist() == [25, 20, 10, 3] and np_(obs["population_capacity"])[0, 0] == 10
    acts = torch.from_numpy(g[f"{name}/action"].astype(np.int64)).to(DEV)
    wins = 0
    for t in range(m["n_steps"]):
        obs, rew, term, trunc, info = env.step(acts[:, t].contiguous())
        assert np.array_equal(np_(rew), g[f"{name}/reward"][:, t]), t
        assert np.array_equal(np_(term).astype(np.uint8), g[f"{name}/terminated"][:, t]) and not np_(trunc).any()
        assert np.array_equal(np_(obs["grid"]), g[f"{name}/grid"][:, t]), t
        assert np.array_equal(np_(obs["resources"]), g[f"{name}/resources"][:, t])
        assert np.array_equal(np_(obs["population_capacity"])[:, 0], g[f"{name}/capacity"][:, t])
        assert np.array_equal(np_(obs["win_steps"])[:, 0], g[f"{name}/win_steps"][:, t])
        assert np.array_equal(np_(env.steps), g[f"{name}/steps"][:, t])
        assert np.array_equal(np_(env.building_counts), g[f"{name}/counts"][:, t])
        assert np.array_equal(np_(env.rng_counter), g[f"{name}/rng_counter"][:, t].astype(np.int64))
        wins += int(g[f"{name}/won"][:, t].sum())
    s = env.episode_stats()
    assert s["n_episodes"] == int(g[f"{name}/terminated"].sum()) and s["wins"] == wins


@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("n,G", [(10007, 10), (333, 4), (130, 15)])
def test_random_rollout_vs_oracle(pkg, mode, n, G):
    from oracle.c_oracle import BuilderOracle

    seed, base, T = 23, 400, 150
    env = pkg.BatchedWorldBuilderEnv(n, G, flatten_obs=(G == 10), device=DEV, seed=seed, env_id_base=base, autoreset_mode=mode)
    orc = BuilderOracle(n, G, seed=seed, env_id_base=base, autoreset=mode)
    env.reset(), orc.reset()
    gen = torch.Generator(device=DEV).manual_seed(1)
    probs = torch.tensor([0.35, 0.2, 0.15, 0.15, 0.15], device=DEV)
    for t in range(T):
        a = torch.multinomial(probs, n, replacement=True, generator=gen)
        obs, rew, term, trunc, info = env.step(a)
        orc.step(np_(a))
        assert np.array_equal(np_(rew), orc.reward) and np.array_equal(np_(term).astype(np.uint8), orc.terminated), t
        assert np.array_equal(np_(env.grid), orc.grid) and np.array_equal(np_(env.resources), orc.resources), t
        assert np.array_equal(np_(env.win_steps), orc.win_steps) and np.array_equal(np_(env.population_capacity), orc.capacity)
        if G == 10:
            assert obs is env.flat_obs and np.array_equal(np_(obs), orc.flat_obs()), t
        if t % 25 == 0:
            st = orc.state()
            assert np.array_equal(np_(env.steps), st["steps"]) and np.array_equal(np_(env.building_counts), st["building_counts"])
            assert np.array_equal(np_(env.rng_counter), st["rng_counter"].astype(np.int64))
    if mode != "disabled":
        assert env.episode_stats() == orc.stats()


def test_million_env_batch_and_invariants(pkg):
    from oracle.c_oracle import BuilderOracle

    n, seed = 1 << 20, 0
    env = pkg.BatchedWorldBuilderEnv(n, device=DEV, seed=seed)
    orc = BuilderOracle(n, seed=seed)
    env.reset(), orc.reset()
    lib = pkg._lib.load()
    a = torch.zeros(n, dtype=torch.int64, device=DEV)
    for t in range(12):
        lib.beng_fill_random_actions(a.data_ptr(), n, 1, 5, t, 0, seed, torch.cuda.current_stream().cuda_stream)
        obs, rew, term, trunc, info = env.step(a)
        orc.step(np_(a))
        assert np.array_equal(np_(rew), orc.reward) and np.array_equal(np_(obs["resources"]), orc.resources), t
        if t % 4 == 3:
            assert np.array_equal(np_(obs["grid"]), orc.grid)
        # invariant: the number of buildings on the grid equals the sum of the building counts
        assert torch.equal((obs["grid"] > 0).sum(dim=(1, 2)).int(), env.building_counts.sum(dim=1).int())
    assert env.episode_stats() == orc.stats()


def test_host_path_invalid_actions_facade(pkg, bgold):
    n, seed = 2000, 3
    a_env = pkg.BatchedWorldBuilderEnv(n, device=DEV, seed=seed, debug_checks=True)
    b_env = pkg.BatchedWorldBuilderEnv(n, device=DEV, seed=seed)
    a_env.reset(), b_env.reset()
    rng = np.random.default_rng(0)
    for t in range(30):
        act = rng.integers(0, 5, n)
        obs, rew, term, trunc, _ = a_env.step_host(act)
        b_env.step(torch.from_numpy(act).to(DEV))
        assert isinstance(obs["grid"], np.ndarray) and np.array_equal(obs["grid"], np_(b_env.grid))
        assert np.array_equal(rew, np_(b_env.reward)) and np.array_equal(obs["resources"], np_(b_env.resources))
    with pytest.raises(ValueError, match="Invalid action"):
        a_env.step(torch.full((n,), 7, dtype=torch.int64, device=DEV))
    clone = pkg.BatchedWorldBuilderEnv(n, device=DEV, seed=99)
    clone.load_state_dict(b_env.state_dict())
    act = torch.from_numpy(rng.integers(0, 5, n)).to(DEV)
    b_env.step(act), clone.step(act)
    assert torch.equal(b_env.grid, clone.grid) and torch.equal(b_env.reward, clone.reward)
    # single-env façade against the golden farmer trajectory
    g, name = bgold, "farmer_g10"
    m = meta(g, name)
    env = pkg.WorldBuilderEnv(device=DEV, seed=m["seed"], env_id=m["base"])
    obs, info = env.reset()
    assert info["population"] == 3 and info["resources"] == {"food": 25, "wood": 20, "stone": 10}
    for t in range(40):
        obs, r, term, trunc, info = env.step(int(g[f"{name}/action"][0, t]))
        assert isinstance(r, int) and r == g[f"{name}/reward"][0, t] and trunc is False
        if term:
            break
        assert np.array_equal(obs["grid"], g[f"{name}/grid"][0, t]) and info["steps"] == t + 1
        assert list(info["building_counts"].values()) == g[f"{name}/counts"][0, t].tolist()
    with pytest.raises(ValueError):
        env.step(5)
