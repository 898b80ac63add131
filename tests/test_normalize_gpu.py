"""VecNormalize on the B200: parity with the float64 oracle (oracle/vecnormalize.py) over long rollouts of every float
env, accuracy of the batch moments, bit-identical raw env outputs, determinism and CUDA-graph capture, freezing,
clipping, masked resets, checkpoints, launch counts and refusals."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.vecnormalize import VecNormalizeOracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KINDS = ("crypto_discrete", "crypto_continuous", "traffic", "climate", "builder")


def make_env(kind, n, mode="same_step", seed=5):
    import custom_gymnasium_environments_b200 as pkg

    if kind.startswith("crypto"):  # short episodes: many dones in 200 steps
        return pkg.BatchedCryptoTradingEnv(n, None, kind.split("_")[1], device=DEV, seed=seed, autoreset_mode=mode,
                                           max_steps=37)
    if kind == "traffic":
        return pkg.BatchedTrafficManagementEnv(n, device=DEV, seed=seed, autoreset_mode=mode, max_timesteps=41)
    if kind == "climate":
        return pkg.BatchedSmartClimateEnv(n, episode_minutes=43, device=DEV, seed=seed, autoreset_mode=mode)
    if kind == "builder":
        return pkg.BatchedWorldBuilderEnv(n, flatten_obs=True, device=DEV, seed=seed, autoreset_mode=mode)
    if kind == "snake":
        return pkg.BatchedSnakeEnv(n, device=DEV, seed=seed, autoreset_mode=mode, max_steps=45)
    raise ValueError(kind)


def make_actions(kind, env, g):
    n = env.num_envs
    if kind == "crypto_discrete":
        return torch.randint(0, 5, (n,), device=DEV, generator=g)
    if kind == "crypto_continuous":
        return torch.rand((n, 2), device=DEV, generator=g) * 2 - 1
    if kind == "traffic":
        return torch.randint(0, 3, (n, env.num_intersections), device=DEV, generator=g)
    if kind == "climate":
        return {"ac_temp": torch.rand(n, device=DEV, generator=g) * 16 + 16,
                "lights": torch.randint(0, 2, (n, 4), device=DEV, generator=g).to(torch.int8)}
    if kind == "builder":
        return torch.randint(0, 5, (n,), device=DEV, generator=g)
    if kind == "snake":
        return torch.randint(0, 4, (n,), device=DEV, generator=g)
    raise ValueError(kind)


def raw_obs(env):
    flat = getattr(env, "flat_obs", None)
    return flat if flat is not None else env.obs


def assert_f32_close(dev, ref, what):
    """Within one float32 ulp or 1e-6 absolute."""
    dev, ref = np.asarray(dev, np.float32), np.asarray(ref, np.float32)
    diff = np.abs(dev.astype(np.float64) - ref.astype(np.float64))
    ok = (diff <= 1e-6) | (diff <= np.spacing(np.abs(ref)).astype(np.float64))
    assert ok.all(), f"{what}: {int((~ok).sum())} of {ok.size} differ, max {diff.max()}"


def assert_stats_close(w, orc, what):
    cpu = lambda t: t.cpu().numpy()  # noqa: E731
    if w.norm_obs:
        np.testing.assert_allclose(cpu(w.obs_rms.mean), orc.obs_rms.mean, rtol=1e-10, atol=1e-12, err_msg=what)
        np.testing.assert_allclose(cpu(w.obs_rms.var), orc.obs_rms.var, rtol=1e-10, atol=1e-12, err_msg=what)
        assert float(w.obs_rms.count) == orc.obs_rms.count, what
    if w.norm_reward:
        np.testing.assert_allclose(float(w.ret_rms.mean), orc.ret_rms.mean, rtol=1e-10, atol=1e-12, err_msg=what)
        np.testing.assert_allclose(float(w.ret_rms.var), orc.ret_rms.var, rtol=1e-10, err_msg=what)
        assert float(w.ret_rms.count) == orc.ret_rms.count, what
        np.testing.assert_allclose(cpu(w.returns), orc.returns, rtol=1e-10, atol=1e-12, err_msg=what)


def run_parity(kind, n, steps, mode, seed=5):
    from custom_gymnasium_environments_b200 import VecNormalize

    env = make_env(kind, n, mode, seed)
    w = VecNormalize(env)
    orc = VecNormalizeOracle(n, w.dim)
    obs, _ = w.reset()
    assert_f32_close(obs.cpu().numpy(), orc.reset(raw_obs(env).cpu().numpy()), f"{kind} reset obs")
    assert_stats_close(w, orc, f"{kind} after reset")
    g = torch.Generator(device=DEV).manual_seed(seed)
    dones = 0
    for t in range(steps):
        obs, rew, term, trunc, _ = w.step(make_actions(kind, env, g))
        term_np, trunc_np = term.cpu().numpy(), trunc.cpu().numpy()
        dones += int((term_np | trunc_np).sum())
        o_obs, o_rew = orc.step(raw_obs(env).cpu().numpy(), env.reward.cpu().numpy(), term_np, trunc_np)
        assert_f32_close(obs.cpu().numpy(), o_obs, f"{kind} {mode} obs, step {t}")
        assert_f32_close(rew.cpu().numpy(), o_rew, f"{kind} {mode} reward, step {t}")
        assert_stats_close(w, orc, f"{kind} {mode} step {t}")
    return dones


@pytest.mark.parametrize("mode", ["same_step", "next_step"])
@pytest.mark.parametrize("kind", KINDS)
def test_parity_with_oracle(kind, mode):
    dones = run_parity(kind, 2053, 200, mode)
    assert dones > (0 if kind == "builder" else 2053), f"{kind}: only {dones} episodes ended in 200 steps"


@pytest.mark.parametrize("kind,n,steps", [("climate", 1 << 20, 4), ("crypto_discrete", 262144, 3)])
def test_parity_large_batch(kind, n, steps):
    run_parity(kind, n, steps, "same_step")


def test_large_offset_columns_through_the_c_abi():
    """Batch moments stay float64-accurate for columns far from zero (a plain sum of squares loses them)."""
    from custom_gymnasium_environments_b200 import _lib as L

    lib = L.load()
    n, dim = 100003, 4
    rng = np.random.default_rng(1)
    noise = rng.standard_normal((n, dim))
    x = np.stack([1e6 + noise[:, 0], 1e3 + 1e-3 * noise[:, 1], 1e-3 * noise[:, 2], -7.0 + 2.0 * noise[:, 3]],
                 axis=1).astype(np.float32)
    obs = torch.from_numpy(x).to(DEV)
    out = torch.empty_like(obs)
    # count 0: the merge then leaves exactly the batch's moments in the record, to compare with np.mean / np.var
    rms = torch.zeros(2 * dim + 1, dtype=torch.float64, device=DEV)
    ws = torch.zeros(lib.beng_normalize_workspace_bytes(n, dim), dtype=torch.uint8, device=DEV)
    p = L.NormalizeParams(1e9, 10.0, 1e-8, 0.99, L.NORM_OBS | L.NORM_UPDATE, 0)
    io = L.NormalizeIO(obs.data_ptr(), None, None, None, None, rms.data_ptr(), None, ws.data_ptr(), out.data_ptr(), None)
    assert lib.beng_normalize(C.byref(p), C.byref(io), n, dim, torch.cuda.current_stream().cuda_stream) == 0
    torch.cuda.synchronize()
    r, x64 = rms.cpu().numpy(), x.astype(np.float64)
    mean, var = x64.mean(0), x64.var(0)
    np.testing.assert_allclose(r[:dim], mean, rtol=1e-12, atol=1e-15)
    np.testing.assert_allclose(r[dim:2 * dim], var, rtol=1e-9)
    assert r[-1] == n
    assert int(ws[:4].view(torch.int32)[0]) == 0  # the arrival counter rewound itself
    expected = np.clip((x64 - mean) / np.sqrt(var + 1e-8), -1e9, 1e9).astype(np.float32)
    assert_f32_close(out.cpu().numpy(), expected, "normalized large-offset columns")


def test_wrapped_env_outputs_are_unchanged():
    from custom_gymnasium_environments_b200 import VecNormalize

    n = 1024
    env, twin = make_env("crypto_discrete", n), make_env("crypto_discrete", n)
    w = VecNormalize(env)
    w.reset(), twin.reset()
    g = torch.Generator(device=DEV).manual_seed(2)
    for t in range(60):
        a = make_actions("crypto_discrete", env, g)
        _, _, term, trunc, info = w.step(a)
        _, _, t_term, t_trunc, t_info = twin.step(a)
        assert torch.equal(env.obs, twin.obs) and torch.equal(env.reward, twin.reward), t
        assert torch.equal(term, t_term) and torch.equal(trunc, t_trunc), t
        assert torch.equal(info["episode"]["r"], t_info["episode"]["r"]), t
        assert torch.equal(info["episode"]["l"], t_info["episode"]["l"]), t
        assert torch.equal(info["cash"], t_info["cash"]) and torch.equal(info["reward64"], t_info["reward64"]), t
    sd, t_sd = env.state_dict(), twin.state_dict()
    assert sd.keys() == t_sd.keys()
    for k in sd:
        if k == "stats":
            continue
        assert (torch.equal(sd[k], t_sd[k]) if isinstance(sd[k], torch.Tensor) else sd[k] == t_sd[k]), k
    # The crypto kernel adds its float64 episode statistics {n_episodes, sum_return, sum_length, sum_final_value} with
    # atomics in warp-scheduling order, so two unwrapped twins already differ in the last bits of the two money sums;
    # the counts are whole numbers and exact.
    s, ts = sd["stats"].cpu().numpy(), t_sd["stats"].cpu().numpy()
    assert s[0] > 0 and s[0] == ts[0] and s[2] == ts[2]
    np.testing.assert_allclose(s[[1, 3]], ts[[1, 3]], rtol=1e-12)


def rollout_state(kind, n, steps, seed=3):
    from custom_gymnasium_environments_b200 import VecNormalize

    env = make_env(kind, n)
    w = VecNormalize(env)
    w.reset()
    g = torch.Generator(device=DEV).manual_seed(seed)
    for _ in range(steps):
        obs, rew, *_ = w.step(make_actions(kind, env, g))
    return [t.clone() for t in (w.obs_rms.data, w.ret_rms.data, w.returns, obs, rew)]


@pytest.mark.parametrize("kind,n", [("crypto_continuous", 20000), ("climate", 300000)])
def test_two_runs_are_bit_identical(kind, n):
    a, b = rollout_state(kind, n, 25), rollout_state(kind, n, 25)
    for x, y in zip(a, b):
        assert torch.equal(x, y)


def assert_same_wrappers(a, b, what):
    for name in ("obs", "reward", "returns"):
        assert torch.equal(getattr(a, name), getattr(b, name)), f"{what}: {name}"
    assert torch.equal(a.obs_rms.data, b.obs_rms.data) and torch.equal(a.ret_rms.data, b.ret_rms.data), what
    assert torch.equal(a.env.obs, b.env.obs) and torch.equal(a.env.terminated, b.env.terminated), what


@pytest.mark.parametrize("k", [1, 3, 7])
def test_graph_replay_equals_eager_steps(k):
    from custom_gymnasium_environments_b200 import VecNormalize

    n, kind = 3000, "crypto_discrete"
    a, b = VecNormalize(make_env(kind, n)), VecNormalize(make_env(kind, n))
    a.reset(), b.reset()
    act = torch.zeros(n, dtype=torch.int64, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(4)
    act.copy_(make_actions(kind, a.env, g))
    a.step(act), b.step(act)  # warm-up (one eager step each)
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for _ in range(k):
            a.step(act)
    for r in range(4):
        act.copy_(make_actions(kind, a.env, g))
        graph.replay()
        for _ in range(k):
            b.step(act)
        torch.cuda.synchronize()
        assert_same_wrappers(a, b, f"replay {r}")
        act.copy_(make_actions(kind, a.env, g))  # eager steps between replays
        a.step(act), b.step(act)
        torch.cuda.synchronize()
        assert_same_wrappers(a, b, f"eager after replay {r}")


def test_frozen_statistics_still_normalize():
    from custom_gymnasium_environments_b200 import VecNormalize

    n, kind = 4096, "traffic"
    w = VecNormalize(make_env(kind, n))
    w.reset()
    g = torch.Generator(device=DEV).manual_seed(6)
    for _ in range(30):
        w.step(make_actions(kind, w.env, g))
    w.training = False
    obs_rms, ret_rms, returns = w.obs_rms.data.clone(), w.ret_rms.data.clone(), w.returns.clone()
    finished = 0
    for _ in range(20):
        obs, rew, term, trunc, _ = w.step(make_actions(kind, w.env, g))
        returns[term | trunc] = 0.0  # finished envs' returns are zeroed also when frozen
        finished += int((term | trunc).sum())
        assert torch.equal(w.obs_rms.data, obs_rms) and torch.equal(w.ret_rms.data, ret_rms)
        assert torch.equal(w.returns, returns)
        mean, var = obs_rms[:w.dim].cpu().numpy(), obs_rms[w.dim:2 * w.dim].cpu().numpy()
        raw = w.env.obs.cpu().numpy().astype(np.float64)
        assert_f32_close(obs.cpu().numpy(), np.clip((raw - mean) / np.sqrt(var + 1e-8), -10, 10), "frozen obs")
        rref = w.env.reward.cpu().numpy().astype(np.float64) / np.sqrt(float(ret_rms[1]) + 1e-8)
        assert_f32_close(rew.cpu().numpy(), np.clip(rref, -10, 10), "frozen reward")
    assert finished > 0


def test_clip_bounds_hold():
    from custom_gymnasium_environments_b200 import VecNormalize

    n, kind = 4096, "crypto_discrete"
    w = VecNormalize(make_env(kind, n), clip_obs=0.5, clip_reward=0.05)
    w.reset()
    g = torch.Generator(device=DEV).manual_seed(7)
    for _ in range(40):
        obs, rew, *_ = w.step(make_actions(kind, w.env, g))
        # clipped in float64, then rounded to float32: the bound that holds is the float32 value of the clip
        assert float(obs.abs().max()) <= np.float32(0.5) and float(rew.abs().max()) <= np.float32(0.05)
    assert bool((obs.abs() == 0.5).any()) and bool((rew.abs() == np.float32(0.05)).any())


def test_masked_reset_zeroes_selected_returns_and_keeps_obs_rms():
    from custom_gymnasium_environments_b200 import VecNormalize

    n, kind = 5000, "climate"
    w = VecNormalize(make_env(kind, n, mode="disabled"))
    w.reset()
    g = torch.Generator(device=DEV).manual_seed(8)
    for _ in range(10):
        w.step(make_actions(kind, w.env, g))
    mask = torch.arange(n, device=DEV) % 3 == 0
    rms, returns = w.obs_rms.data.clone(), w.returns.clone()
    assert bool((returns[mask] != 0).any())
    obs, _ = w.reset(options={"reset_mask": mask})
    assert torch.equal(w.obs_rms.data, rms)
    assert bool((w.returns[mask] == 0).all()) and torch.equal(w.returns[~mask], returns[~mask])
    mean, var = rms[:w.dim].cpu().numpy(), rms[w.dim:2 * w.dim].cpu().numpy()
    raw = w.env.obs.cpu().numpy().astype(np.float64)
    assert_f32_close(obs.cpu().numpy(), np.clip((raw - mean) / np.sqrt(var + 1e-8), -10, 10), "masked reset obs")
    # a full reset counts the batch and zeroes every return
    w.reset()
    assert float(w.obs_rms.count) == float(rms[-1]) + n and bool((w.returns == 0).all())


def test_checkpoint_continues_bit_identically():
    from custom_gymnasium_environments_b200 import VecNormalize

    n, kind = 3000, "crypto_discrete"
    a = VecNormalize(make_env(kind, n), gamma=0.95, clip_obs=5.0)
    a.reset()
    g = torch.Generator(device=DEV).manual_seed(9)
    for _ in range(15):
        a.step(make_actions(kind, a.env, g))
    sd = a.state_dict()
    b = VecNormalize(make_env(kind, n, seed=123))
    b.load_state_dict(sd)
    assert b.gamma == 0.95 and b.clip_obs == 5.0
    for t in range(15):
        act = make_actions(kind, a.env, g)
        oa, ra, *_ = a.step(act)
        ob, rb, *_ = b.step(act)
        assert torch.equal(oa, ob) and torch.equal(ra, rb), t
        assert_same_wrappers(a, b, f"step {t} after the checkpoint")


@pytest.mark.parametrize("kind,norm_obs,training,added", [
    ("crypto_discrete", True, True, 2), ("crypto_discrete", True, False, 1), ("snake", False, True, 2),
    ("snake", False, False, 1), ("builder", True, True, 2)])
def test_launches_per_step(kind, norm_obs, training, added):
    from custom_gymnasium_environments_b200 import VecNormalize, _lib

    lib = _lib.load()
    env = make_env(kind, 2048)
    w = VecNormalize(env, norm_obs=norm_obs, training=training)
    w.reset()
    g = torch.Generator(device=DEV).manual_seed(10)
    acts = [make_actions(kind, env, g) for _ in range(3)]
    twin = make_env(kind, 2048)
    twin.reset()
    before = lib.beng_launch_count()
    twin.step(acts[0])
    env_launches = lib.beng_launch_count() - before
    before = lib.beng_launch_count()
    for a in acts:
        w.step(a)
    assert lib.beng_launch_count() - before == 3 * (env_launches + added)


def test_refusals_and_reward_only_snake():
    from custom_gymnasium_environments_b200 import BatchedWorldBuilderEnv, VecNormalize

    with pytest.raises(ValueError, match="norm_obs"):
        VecNormalize(make_env("snake", 64))
    with pytest.raises(ValueError, match="norm_obs"):
        VecNormalize(BatchedWorldBuilderEnv(64, device=DEV))
    n = 2053
    env = make_env("snake", n)
    w = VecNormalize(env, norm_obs=False)
    orc = VecNormalizeOracle(n, norm_obs=False)
    obs, _ = w.reset()
    assert obs is env.obs and obs.dtype == torch.int8
    orc.reset(None)
    g = torch.Generator(device=DEV).manual_seed(11)
    for t in range(120):
        obs, rew, term, trunc, _ = w.step(make_actions("snake", env, g))
        assert obs.dtype == torch.int8
        _, o_rew = orc.step(None, env.reward.cpu().numpy(), term.cpu().numpy(), trunc.cpu().numpy())
        assert_f32_close(rew.cpu().numpy(), o_rew, f"snake reward, step {t}")
        assert_stats_close(w, orc, f"snake step {t}")
    with pytest.raises(ValueError, match="out_obs"):
        w.step(make_actions("snake", env, g), out_obs=torch.empty(n, 1, device=DEV))


def test_out_obs_receives_the_normalized_observation():
    from custom_gymnasium_environments_b200 import VecNormalize

    n, kind = 2048, "climate"
    a, b = VecNormalize(make_env(kind, n)), VecNormalize(make_env(kind, n))
    a.reset(), b.reset()
    buf = torch.full((4, n, a.dim), float("nan"), device=DEV)
    g = torch.Generator(device=DEV).manual_seed(12)
    for t in range(4):
        act = make_actions(kind, a.env, g)
        oa, *_ = a.step(act, out_obs=buf[t])
        ob, *_ = b.step(act)
        assert oa.data_ptr() == buf[t].data_ptr() and torch.equal(buf[t], ob)
    with pytest.raises(ValueError, match="out_obs"):
        a.step(act, out_obs=torch.empty(n, a.dim + 1, device=DEV))
