"""GPU parity tests for crypto_trading_env: the CUDA path (through the C ABI) against the float64 CPU oracle
and the golden vectors recorded from the reference.

Tolerances (BASELINE.json north_star: "float envs must match within a stated rtol of 1e-5 per step"):
  observations / float32 rewards : rtol 1e-5, atol 1e-6  (atol for features that cross zero: MACD, Bollinger offset)
  float64 state (cash, holdings, prices, psychology, rewards, portfolio value): rtol 1e-9 free-running over
      thousands of steps -- the only differences are the last-ulp results of CUDA's log/cos vs glibc's
  integer fields (terminated, step, regime, trade kind, RNG counter): exact
"""
import numpy as np
import pytest
import torch

from oracle import golden_files

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
RTOL, ATOL = 1e-5, 1e-6
RTOL64 = 1e-9
CASES = ["discrete_random", "discrete_hi_ids", "discrete_buyer", "discrete_seller", "discrete_hold",
         "continuous_random", "custom_config"]


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    assert torch.cuda.is_available()
    p._lib.load()
    return p


@pytest.fixture(scope="module")
def cgold():
    return golden_files.load("crypto")


def np_(t):
    return t.cpu().numpy()


def close_obs(a, b, what=""):
    np.testing.assert_allclose(a, b, rtol=RTOL, atol=ATOL, err_msg=what)


def meta(g, name):
    n_envs, n_steps, seed, base, snap, cont = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, snap=snap, cont=bool(cont))


def make_env(pkg, g, name, m, **kw):
    cfg = pkg.TradingConfig()
    if name == "custom_config":
        c = g["custom_cfg"]
        cfg = pkg.TradingConfig(initial_balance=c[0], trading_fee_rate=c[1], slippage_rate=c[2], min_price=c[3],
                                max_price=c[4], volatility_base=c[5], market_psychology_factor=c[6])
    return pkg.BatchedCryptoTradingEnv(m["n_envs"], cfg, "continuous" if m["cont"] else "discrete", device=DEV,
                                       seed=m["seed"], env_id_base=m["base"], **kw)


def assert_state(env, ref, t):
    """ref: dict of numpy arrays with the oracle/golden state after the step."""
    for k, dev in (("cash", env.cash), ("holdings", env.holdings), ("psychology", env.market_psychology),
                   ("trend_strength", env.trend_strength)):
        np.testing.assert_allclose(np_(dev), ref[k], rtol=RTOL64, atol=1e-12, err_msg=f"{k} at step {t}")
    assert np.array_equal(np_(env.market_regime), ref["regime"].astype(np.int64)), f"regime at {t}"
    assert np.array_equal(np_(env.current_step), ref["step"].astype(np.int64)), f"step at {t}"
    assert np.array_equal(np_(env.rng_counter), ref["rng_counter"].astype(np.int64)), f"rng counter at {t}"


@pytest.mark.parametrize("name", CASES)
def test_golden_replay(pkg, cgold, name):
    g, m = cgold, meta(cgold, name)
    env = make_env(pkg, g, name, m)
    obs, info = env.reset()
    assert obs.shape == (m["n_envs"], 261) and obs.dtype == torch.float32 and info == {}
    close_obs(np_(obs), g[f"{name}/reset_obs"], "reset obs")
    act = g[f"{name}/action"]
    dt = torch.float32 if m["cont"] else torch.int64
    acts = torch.from_numpy(act.astype(np.float32 if m["cont"] else np.int64)).to(DEV, dt)
    for t in range(m["n_steps"]):
        obs, rew, term, trunc, info = env.step(acts[:, t].contiguous())
        assert np.array_equal(np_(term).astype(np.uint8), g[f"{name}/terminated"][:, t]), t
        assert not np_(trunc).any()
        assert np.array_equal(np_(info["trade_kind"]), g[f"{name}/trade_kind"][:, t]), t
        np.testing.assert_allclose(np_(info["reward64"]), g[f"{name}/reward"][:, t], rtol=RTOL64, atol=1e-9)
        np.testing.assert_allclose(np_(rew), g[f"{name}/reward"][:, t].astype(np.float32), rtol=RTOL, atol=ATOL)
        np.testing.assert_allclose(np_(info["portfolio_value"]), g[f"{name}/portfolio_value"][:, t], rtol=RTOL64)
        np.testing.assert_allclose(np_(info["current_price"]), g[f"{name}/current_price"][:, t], rtol=RTOL64)
        if t % 5 == 0 or t == m["n_steps"] - 1:
            assert_state(env, {k: g[f"{name}/{k}"][:, t] for k in ("cash", "holdings", "psychology",
                                                                   "trend_strength", "regime", "step",
                                                                   "rng_counter")}, t)
        close_obs(np_(obs)[:, 250:], g[f"{name}/obs_tail"][:, t], f"indicator features at step {t}")
        if t % m["snap"] == 0:
            close_obs(np_(obs), g[f"{name}/snap_obs"][:, t // m["snap"]], f"full obs at step {t}")
    assert env.episode_stats()["n_episodes"] == int(g[f"{name}/terminated"].sum())


@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("n,action_type", [(4099, "discrete"), (1000, "continuous")])
def test_random_rollout_vs_oracle(pkg, mode, n, action_type):
    """Crosses the 1000-step limit (so auto-reset, the non-reset market simulator and the window rotation at a
    reset are all exercised), ragged env counts, both action types, all three auto-reset modes."""
    from oracle.c_oracle import CryptoOracle

    seed, base, T = 21, 500, 1012
    env = pkg.BatchedCryptoTradingEnv(n, None, action_type, device=DEV, seed=seed, env_id_base=base,
                                      autoreset_mode=mode)
    orc = CryptoOracle(n, seed=seed, env_id_base=base, autoreset=mode, action_type=action_type)
    close_obs(np_(env.reset()[0]), orc.reset(), "reset")
    gen = torch.Generator(device=DEV).manual_seed(3)
    for t in range(T):
        if action_type == "discrete":
            a = torch.randint(0, 5, (n,), device=DEV, generator=gen)
        else:
            a = torch.rand((n, 2), device=DEV, generator=gen) * 2.6 - 1.3
        env.step(a)
        orc.step(np_(a))
        assert np.array_equal(np_(env.terminated).astype(np.uint8), orc.terminated), t
        if t % 40 == 0 or t >= 995:
            close_obs(np_(env.obs), orc.obs, f"obs at step {t}")
            np.testing.assert_allclose(np_(env.reward64), orc.reward64, rtol=RTOL64, atol=1e-9)
            st = orc.state()
            assert_state(env, st, t)
    if mode != "disabled":
        s, o = env.episode_stats(), orc.stats()
        assert s["n_episodes"] == o["n_episodes"] >= n
        np.testing.assert_allclose([s["sum_return"], s["sum_length"], s["sum_final_value"]],
                                   [o["sum_return"], o["sum_length"], o["sum_final_value"]], rtol=1e-9)


@pytest.mark.parametrize("mode", ["same_step", "next_step"])
def test_sparse_autoresets_match_oracle(pkg, mode):
    """Episodes that end on DIFFERENT steps: a few envs per warp reset in a step, which is the path where the whole warp
    rebuilds one env's 50-candle window together (csrc/crypto.cu::coop_warmup_window; a batch whose episodes all end on
    the same step takes the one-lane-per-env path instead).  The phases are staggered with masked resets; every step is
    compared, including the regime changes that shift the draw positions inside a warm-up (RNG counter exact)."""
    from oracle.c_oracle import CryptoOracle

    n, seed, limit = 4001, 17, 37
    env = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=seed, autoreset_mode=mode, max_steps=limit)
    orc = CryptoOracle(n, seed=seed, autoreset=mode, max_steps=limit)
    close_obs(np_(env.reset()[0]), orc.reset(), "reset")
    gen = torch.Generator(device=DEV).manual_seed(5)
    idx = torch.arange(n, device=DEV)
    for t in range(limit - 1):  # stagger: env i restarts its episode after (i % limit) steps
        a = torch.randint(0, 5, (n,), device=DEV, generator=gen)
        env.step(a), orc.step(np_(a), want_obs=False)
        mask = (idx % limit) == t
        env.reset(options={"reset_mask": mask})
        orc.reset(np_(mask))
    resets_per_step = []
    for t in range(150):
        a = torch.randint(0, 5, (n,), device=DEV, generator=gen)
        env.step(a), orc.step(np_(a))
        assert np.array_equal(np_(env.terminated).astype(np.uint8), orc.terminated), t
        resets_per_step.append(int(orc.terminated.sum()))
        close_obs(np_(env.obs), orc.obs, f"obs at step {t}")
        np.testing.assert_allclose(np_(env.reward64), orc.reward64, rtol=RTOL64, atol=1e-9)
        assert_state(env, orc.state(), t)
    assert 0 < max(resets_per_step) < n // 8, "the resets were meant to be sparse"
    s, o = env.episode_stats(), orc.stats()
    assert s["n_episodes"] == o["n_episodes"] > n


def test_teacher_forced_per_step_error(pkg):
    """Re-sync the oracle from the device state before every step: bounds the PER-STEP error independently of
    any accumulated drift (SURVEY.md section 7, 'compare with teacher forcing')."""
    from oracle.c_oracle import CryptoOracle

    n, seed, T = 2048, 8, 120
    env = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=seed)
    orc = CryptoOracle(n, seed=seed)
    env.reset(), orc.reset()
    gen = torch.Generator(device=DEV).manual_seed(1)
    worst = 0.0
    for t in range(T):
        orc.set_state({"cash": np_(env.cash), "holdings": np_(env.holdings),
                       "trend_strength": np_(env.trend_strength), "psychology": np_(env.market_psychology),
                       "regime": np_(env.market_regime), "step": np_(env.current_step),
                       "rng_counter": np_(env.rng_counter), "candles": np_(env.price_history())})
        a = torch.randint(0, 5, (n,), device=DEV, generator=gen)
        env.step(a)
        orc.step(np_(a))
        d, o = np_(env.obs).astype(np.float64), orc.obs.astype(np.float64)
        worst = max(worst, float(np.max(np.abs(d - o) / (ATOL + RTOL * np.abs(o)))))
        np.testing.assert_allclose(np_(env.reward64), orc.reward64, rtol=1e-12, atol=1e-9)
        np.testing.assert_allclose(np_(env.cash), orc.state()["cash"], rtol=1e-14)
    assert worst < 1.0, worst


def test_full_size_batch_vs_oracle(pkg):
    """BASELINE config: 262,144 envs per GPU, discrete actions: 25 steps against the oracle + invariants."""
    from oracle.c_oracle import CryptoOracle

    n, seed, T = 262144, 0, 25
    env = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=seed)
    orc = CryptoOracle(n, seed=seed)
    close_obs(np_(env.reset()[0]), orc.reset(), "reset")
    lib = pkg._lib.load()
    actions = torch.zeros(n, dtype=torch.int64, device=DEV)
    for t in range(T):
        lib.beng_fill_random_actions(actions.data_ptr(), n, 1, 5, t, 0, seed, torch.cuda.current_stream().cuda_stream)
        obs, rew, term, trunc, info = env.step(actions)
        orc.step(np_(actions), want_obs=(t % 8 == 7))
        assert np.array_equal(np_(info["trade_kind"]), orc.trade_kind)
        np.testing.assert_allclose(np_(info["reward64"]), orc.reward64, rtol=RTOL64, atol=1e-9)
        if t % 8 == 7:
            close_obs(np_(obs), orc.obs, f"obs at step {t}")
        # invariants of the encoding: newest close normalises to 1, high >= close >= low, RSI and psychology in [0, 1]
        o = obs.view(n, -1)
        newest = o[:, 245:250]
        assert bool(((newest[:, 3] - 1.0).abs() < 1e-6).all())
        assert bool((newest[:, 1] >= newest[:, 3] - 1e-6).all()) and bool((newest[:, 2] <= newest[:, 3] + 1e-6).all())
        assert bool(((o[:, 253] >= 0) & (o[:, 253] <= 1) & (o[:, 260] >= 0) & (o[:, 260] <= 1)).all())
        assert bool((rew <= 1e-3).all())  # the reward is never positive (SURVEY.md section 3.3)
    assert_state(env, orc.state(), T)


def test_trajectories_do_not_depend_on_sharding(pkg):
    from custom_gymnasium_environments_b200.dist import shard_range

    n, T, seed = 3000, 60, 4
    whole = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=seed)
    shards = []
    for r in range(3):
        s, c = shard_range(n, r, 3)
        shards.append((s, c, pkg.BatchedCryptoTradingEnv(c, None, "discrete", device=DEV, seed=seed, env_id_base=s)))
    whole.reset()
    for _, _, e in shards:
        e.reset()
    gen = torch.Generator(device=DEV).manual_seed(0)
    for t in range(T):
        a = torch.randint(0, 5, (n,), device=DEV, generator=gen)
        whole.step(a)
        for s, c, e in shards:
            e.step(a[s:s + c].contiguous())
            assert torch.equal(e.obs, whole.obs[s:s + c]) and torch.equal(e.reward64, whole.reward64[s:s + c])


def test_host_path_masked_reset_and_state_dict(pkg):
    n, seed = 1500, 6
    a = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=seed)
    b = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=seed)
    a.reset(), b.reset()
    rng = np.random.default_rng(0)
    for t in range(60):  # crosses a full rotation of the 50-slot ring
        act = rng.integers(0, 5, n)
        obs, rew, term, trunc, _ = a.step_host(act)
        b.step(torch.from_numpy(act).to(DEV))
        assert isinstance(obs, np.ndarray) and obs.dtype == np.float32
        assert np.array_equal(obs, np_(b.obs)) and np.array_equal(rew, np_(b.reward)) and np.array_equal(term, np_(b.terminated))
    # masked reset: selected envs restart from 50000-ish prices with fresh cash, others keep their window
    before = a.price_history().clone()
    mask = torch.zeros(n, dtype=torch.bool, device=DEV)
    mask[::3] = True
    a.reset(options={"reset_mask": mask})
    after = a.price_history()
    assert torch.equal(after[1::3], before[1::3]) and not torch.equal(after[::3], before[::3])
    assert bool((a.cash[::3] == 10000.0).all()) and bool((a.current_step[::3] == 0).all())
    assert bool((a.current_step[1::3] == 60).all())
    # state_dict round trip
    clone = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=999)
    clone.load_state_dict(a.state_dict())
    act = torch.from_numpy(rng.integers(0, 5, n)).to(DEV)
    a.step(act), clone.step(act)
    assert torch.equal(a.obs, clone.obs) and torch.equal(a.reward64, clone.reward64)
    # re-keying reproduces the constructor stream (incl. a fresh market simulator)
    a.reset(seed=seed)
    fresh = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV, seed=seed)
    fresh.reset()
    assert torch.equal(a.obs, fresh.obs)


def test_single_env_facade(pkg, cgold):
    """CryptoTradingEnv (gym.Env surface): shapes, info keys, hold reward == -1.0 exactly, golden trajectory."""
    g, name = cgold, "discrete_buyer"
    m = meta(g, name)
    env = pkg.CryptoTradingEnv(action_type="discrete", device=DEV, seed=m["seed"], env_id=m["base"])
    obs, info = env.reset()
    assert obs.shape == (261,) and obs.dtype == np.float32 and info == {}
    close_obs(obs, g[f"{name}/reset_obs"][0])
    for t in range(40):
        a = int(g[f"{name}/action"][0, t])
        obs, r, term, trunc, info = env.step(a)
        assert isinstance(r, float) and trunc is False and isinstance(term, bool)
        np.testing.assert_allclose(r, g[f"{name}/reward"][0, t], rtol=RTOL64, atol=1e-9)
        assert set(info) == {"portfolio_value", "cash", "holdings", "current_price", "market_regime",
                             "market_psychology", "trade_info"}
        kind = int(g[f"{name}/trade_kind"][0, t])
        assert (info["trade_info"] is None) == (kind == 0)
        if kind:
            ti = info["trade_info"]
            assert ti["action"] == ("buy" if kind == 1 else "sell") and ti["fee"] > 0 and ti["slippage"] > 0
        if a == 0:
            assert r == -1.0
    env2 = pkg.CryptoTradingEnv(device=DEV)  # continuous is the reference default
    env2.reset()
    obs, r, *_ = env2.step(np.array([0.5, -0.2], dtype=np.float32))
    assert obs.shape == (261,) and r < 0
