"""GPU parity tests for traffic_management_env: the CUDA path (through the C ABI) against the CPU oracle and the
golden vectors recorded from the reference.  Integer dynamics and float64-of-integer reward/observation: EXACT
(observations compared bit for bit via array equality / crc32; float64 rewards compared with ==)."""
import zlib

import numpy as np
import pytest
import torch

from oracle import golden_files

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
CASES = ["random_default", "random_hi_ids", "all_zero", "all_ns", "all_ew", "alternate", "custom_grid"]


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    assert torch.cuda.is_available()
    p._lib.load()
    return p


@pytest.fixture(scope="module")
def tgold():
    return golden_files.load("traffic")


def np_(t):
    return t.cpu().numpy()


def crc_rows(obs):
    return np.array([zlib.crc32(o.tobytes()) for o in obs], dtype=np.uint32)


def meta(g, name):
    n_envs, n_steps, seed, base, snap, rows, cols, ni, maxv = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, snap=snap, grid=(rows, cols), ni=ni,
                max_vehicles=maxv, spawn_rate=float(g[f"{name}/spawn_rate"]))


def assert_state(env, st, t):
    assert np.array_equal(np_(env.current_timestep), st["timestep"]), t
    assert np.array_equal(np_(env.timestep), st["timestep"]), t  # info["timestep"], written by the kernel itself
    assert np.array_equal(np_(env.num_vehicles), st["num_vehicles"]), t
    assert np.array_equal(np_(env.rng_counter), st["rng_counter"].astype(np.int64)), t
    assert np.array_equal(np_(env.light_phase), st["phase"]) and np.array_equal(np_(env.vehicles_passed), st["passed"])
    assert np.array_equal(np_(env.queue_lengths), st["qlen"]), t
    if "timer" in st:
        assert np.array_equal(np_(env.light_timer), st["timer"]) and np.array_equal(np_(env.total_waiting_time), st["waiting"])
        assert np.array_equal(np_(env.queue_waiting_sums), st["qwait"]) and np.array_equal(np_(env.total_reward), st["total_reward"])


@pytest.mark.parametrize("name", CASES)
def test_golden_replay(pkg, tgold, name):
    g, m = tgold, meta(tgold, name)
    env = pkg.BatchedTrafficManagementEnv(m["n_envs"], m["grid"], m["ni"], m["max_vehicles"], m["spawn_rate"],
                                          device=DEV, seed=m["seed"], env_id_base=m["base"])
    obs, info = env.reset()
    assert obs.shape == (m["n_envs"], min(m["ni"], m["grid"][0] * m["grid"][1]) * 14 + 4)
    assert np.array_equal(np_(obs), g[f"{name}/reset_obs"])
    acts = torch.from_numpy(g[f"{name}/action"].astype(np.int64)).to(DEV)
    for t in range(m["n_steps"]):
        obs, rew, term, trunc, info = env.step(acts[:, t].contiguous())
        assert np.array_equal(np_(info["reward64"]), g[f"{name}/reward"][:, t]), t
        assert np.array_equal(np_(rew), g[f"{name}/reward"][:, t].astype(np.float32))
        assert np.array_equal(np_(term).astype(np.uint8), g[f"{name}/terminated"][:, t]) and not np_(trunc).any()
        assert np.array_equal(crc_rows(np_(obs)), g[f"{name}/obs_crc"][:, t]), t
        assert_state(env, {k: g[f"{name}/{k}"][:, t] for k in ("timestep", "num_vehicles", "rng_counter", "phase",
                                                               "passed", "qlen")}, t)
        if t % m["snap"] == 0:
            assert np.array_equal(np_(obs), g[f"{name}/snap_obs"][:, t // m["snap"]])
    assert env.episode_stats()["n_episodes"] == int(g[f"{name}/terminated"].sum())


@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("n,kw", [(4099, {}), (1000, dict(grid_size=(3, 4), num_intersections=7, max_vehicles=20, spawn_rate=0.6)),
                                  (257, dict(grid_size=(2, 2), num_intersections=9, max_vehicles=200, spawn_rate=1.0))])
def test_random_rollout_vs_oracle(pkg, mode, n, kw):
    """Crosses the 1000-step limit; ragged env counts; non-default grids (generic-NI kernel); all auto-reset modes."""
    from oracle.c_oracle import TrafficOracle

    seed, base, T = 13, 700, 1010
    env = pkg.BatchedTrafficManagementEnv(n, device=DEV, seed=seed, env_id_base=base, autoreset_mode=mode, **kw)
    orc = TrafficOracle(n, kw.get("grid_size", (5, 5)), kw.get("num_intersections", 9), kw.get("max_vehicles", 50),
                        kw.get("spawn_rate", 0.3), seed=seed, env_id_base=base, autoreset=mode)
    assert np.array_equal(np_(env.reset()[0]), orc.reset())
    ni = env.num_intersections
    lib = pkg._lib.load()
    actions = torch.zeros((n, ni), dtype=torch.int64, device=DEV)
    for t in range(T):
        lib.beng_fill_random_actions(actions.data_ptr(), n, ni, 3, t, base, seed, torch.cuda.current_stream().cuda_stream)
        env.step(actions)
        orc.step(np_(actions))
        assert np.array_equal(np_(env.reward64), orc.reward64), t
        assert np.array_equal(np_(env.terminated).astype(np.uint8), orc.terminated), t
        if t % 25 == 0 or t >= 997:
            assert np.array_equal(np_(env.obs), orc.obs), t
            assert_state(env, orc.state(), t)
    if mode != "disabled":
        s, o = env.episode_stats(), orc.stats()
        assert s["n_episodes"] == o["n_episodes"] == n
        np.testing.assert_allclose([s["sum_return"], s["sum_length"]], [o["sum_return"], o["sum_length"]], rtol=1e-12)


def test_full_size_batch_vs_oracle(pkg):
    """BASELINE config: 65,536 envs per GPU: 120 steps against the oracle, exact."""
    from oracle.c_oracle import TrafficOracle

    n, seed, T = 65536, 0, 120
    env = pkg.BatchedTrafficManagementEnv(n, device=DEV, seed=seed)
    orc = TrafficOracle(n, seed=seed)
    assert np.array_equal(np_(env.reset()[0]), orc.reset())
    lib = pkg._lib.load()
    actions = torch.zeros((n, 9), dtype=torch.int64, device=DEV)
    for t in range(T):
        lib.beng_fill_random_actions(actions.data_ptr(), n, 9, 3, t, 0, seed, torch.cuda.current_stream().cuda_stream)
        obs, rew, term, trunc, info = env.step(actions)
        orc.step(np_(actions), want_obs=(t % 20 == 19))
        assert np.array_equal(np_(info["reward64"]), orc.reward64), t
        if t % 20 == 19:
            assert np.array_equal(np_(obs), orc.obs), t
        # invariants: one-hot phases, capped features, vehicle count bounded by max_vehicles
        assert bool((obs[:, :36].view(n, 9, 4).sum(-1) == 1).all())
        assert bool((obs[:, 36:72] <= 20).all()) and bool((obs[:, 72:108] <= 100).all())
        assert bool((info["num_vehicles"] <= 50).all())
    assert_state(env, orc.state(), T)


def test_sharding_host_path_masked_reset_state_dict(pkg):
    from custom_gymnasium_environments_b200.dist import shard_range

    n, T, seed = 3000, 80, 4
    from oracle.c_oracle import TrafficOracle

    whole = pkg.BatchedTrafficManagementEnv(n, device=DEV, seed=seed)
    host = pkg.BatchedTrafficManagementEnv(n, device=DEV, seed=seed)
    orc = TrafficOracle(n, seed=seed)
    orc.reset()
    shards = []
    for r in range(3):
        s, c = shard_range(n, r, 3)
        shards.append((s, c, pkg.BatchedTrafficManagementEnv(c, device=DEV, seed=seed, env_id_base=s)))
    whole.reset(), host.reset()
    for _, _, e in shards:
        e.reset()
    gen = torch.Generator(device=DEV).manual_seed(0)
    for t in range(T):
        a = torch.randint(0, 3, (n, 9), device=DEV, generator=gen)
        whole.step(a)
        orc.step(np_(a), want_obs=False)
        obs, rew, term, trunc, _ = host.step_host(np_(a))
        assert isinstance(obs, np.ndarray) and np.array_equal(obs, np_(whole.obs)) and np.array_equal(rew, np_(whole.reward))
        for s, c, e in shards:
            e.step(a[s:s + c].contiguous())
            assert torch.equal(e.obs, whole.obs[s:s + c]) and torch.equal(e.reward64, whole.reward64[s:s + c])
    mask = torch.zeros(n, dtype=torch.bool, device=DEV)
    mask[::2] = True
    obs_after, _ = whole.reset(options={"reset_mask": mask})
    # the masked reset against the oracle's: selected envs are fresh (every state word, observation of a fresh env),
    # the others untouched, and both continue identically
    assert np.array_equal(np_(obs_after), orc.reset(np_(mask)))
    assert_state(whole, orc.state(), "masked reset")
    a = torch.randint(0, 3, (n, 9), device=DEV, generator=gen)
    whole.step(a)
    orc.step(np_(a))
    assert np.array_equal(np_(whole.obs), orc.obs) and np.array_equal(np_(whole.reward64), orc.reward64)
    assert_state(whole, orc.state(), "step after masked reset")
    assert bool((whole.current_timestep[::2] == 1).all()) and bool((whole.current_timestep[1::2] == T + 1).all())
    assert bool((whole.num_vehicles[::2] <= 1).all()) and bool((whole.num_vehicles[1::2] > 1).any())
    clone = pkg.BatchedTrafficManagementEnv(n, device=DEV, seed=77)
    clone.load_state_dict(whole.state_dict())
    a = torch.randint(0, 3, (n, 9), device=DEV, generator=gen)
    whole.step(a), clone.step(a)
    assert torch.equal(whole.obs, clone.obs) and torch.equal(whole.reward64, clone.reward64)


def test_single_env_facade(pkg, tgold):
    g, name = tgold, "random_default"
    m = meta(g, name)
    env = pkg.TrafficManagementEnv(device=DEV, seed=m["seed"], env_id=m["base"])
    obs, info = env.reset()
    assert obs.shape == (130,) and obs.dtype == np.float32 and info["timestep"] == 0 and info["num_vehicles"] == 0
    assert env.action_space.nvec.tolist() == [3] * 9 and env.observation_space.shape == (130,)
    for t in range(60):
        obs, r, term, trunc, info = env.step(g[f"{name}/action"][0, t])
        assert isinstance(r, float) and r == g[f"{name}/reward"][0, t] and term is False and trunc is False
        assert zlib.crc32(obs.tobytes()) == g[f"{name}/obs_crc"][0, t]
        assert set(info) == {"timestep", "num_vehicles", "total_reward", "metrics", "intersection_states"}
        assert info["timestep"] == t + 1 and info["num_vehicles"] == g[f"{name}/num_vehicles"][0, t]
        assert info["total_reward"] == g[f"{name}/total_reward"][0, t]
        st = info["intersection_states"]
        assert len(st) == 9 and st[0]["light_phase"] in ("NS_GREEN", "NS_YELLOW", "EW_GREEN", "EW_YELLOW")
        assert [s["vehicles_passed"] for s in st] == g[f"{name}/passed"][0, t].tolist()
        assert set(info["metrics"]) == {"total_vehicles_passed", "total_waiting_time", "average_waiting_time",
                                        "total_queue_length", "average_queue_length", "throughput"}


def test_infos_are_views_the_kernel_writes(pkg):
    """The infos dict is made of tensors the kernel writes in place (a masked `info["timestep"]` used to cost an extra
    elementwise launch per step inside the timed region; tests/test_single_launch_gpu.py counts the launches)."""
    n = 4096
    env = pkg.BatchedTrafficManagementEnv(n, device=DEV, seed=5, autoreset_mode="next_step", max_timesteps=7)
    env.reset()
    actions = torch.randint(0, 3, (n, env.num_intersections), device=DEV)
    lib = pkg._lib.load()
    for t in range(20):
        before = lib.beng_launch_count()
        _, _, _, _, infos = env.step(actions)
        assert lib.beng_launch_count() - before == 1
        assert infos["timestep"].data_ptr() == env.timestep.data_ptr()
        assert torch.equal(infos["timestep"], env.current_timestep.to(torch.int32))
        assert torch.equal(infos["num_vehicles"], env.num_vehicles)

