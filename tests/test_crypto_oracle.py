"""The float64 C oracle of CryptoTradingEnv against golden vectors produced by the reference itself
(tests/golden/crypto_golden.npz, oracle/gen_golden_crypto.py) and, in the build container, the live reference.
The oracle reproduces the reference's float64 operation order (incl. NumPy's pairwise sums), so the comparison
is EXACT here; the rtol of 1e-5 is only needed between the oracle and the CUDA path (tests/test_crypto_gpu.py)."""
import os

import numpy as np
import pytest

from oracle import golden_files, ref_loader, replay
from oracle.c_oracle import CRYPTO_DEFAULT_CFG, CryptoOracle

CASES = ["discrete_random", "discrete_hi_ids", "discrete_buyer", "discrete_seller", "discrete_hold",
         "continuous_random", "custom_config"]


@pytest.fixture(scope="module")
def cgold():
    return golden_files.load("crypto")


def meta(g, name):
    n_envs, n_steps, seed, base, snap, cont = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, snap=snap, cont=bool(cont))


def make_oracle(g, name, m, autoreset="same_step"):
    cfg = tuple(g["custom_cfg"]) if name == "custom_config" else CRYPTO_DEFAULT_CFG
    return CryptoOracle(m["n_envs"], seed=m["seed"], env_id_base=m["base"], autoreset=autoreset,
                        action_type="continuous" if m["cont"] else "discrete", cfg=cfg)


@pytest.mark.parametrize("name", CASES)
def test_c_oracle_matches_golden_exactly(cgold, name):
    g, m = cgold, meta(cgold, name)
    orc = make_oracle(g, name, m)
    assert np.array_equal(orc.reset(), g[f"{name}/reset_obs"])
    act = g[f"{name}/action"]
    for t in range(m["n_steps"]):
        a = act[:, t].astype(np.float32) if m["cont"] else act[:, t].astype(np.int64)
        obs, rew, term, trunc = orc.step(a)
        assert np.array_equal(orc.reward64, g[f"{name}/reward"][:, t]), t
        assert np.array_equal(term, g[f"{name}/terminated"][:, t]) and not trunc.any()
        assert np.array_equal(orc.portfolio_value, g[f"{name}/portfolio_value"][:, t])
        assert np.array_equal(orc.current_price, g[f"{name}/current_price"][:, t])
        assert np.array_equal(orc.trade_kind, g[f"{name}/trade_kind"][:, t])
        st = orc.state()
        for k in ("cash", "holdings", "psychology", "trend_strength", "regime", "step", "rng_counter"):
            assert np.array_equal(st[k].astype(np.float64), g[f"{name}/{k}"][:, t].astype(np.float64)), (k, t)
        assert np.array_equal(obs[:, 250:], g[f"{name}/obs_tail"][:, t]), t
        if t % m["snap"] == 0:
            assert np.array_equal(obs, g[f"{name}/snap_obs"][:, t // m["snap"]])
    assert orc.stats()["n_episodes"] == int(g[f"{name}/terminated"].sum())


def test_reference_facts(cgold):
    """SURVEY.md section 0 facts 5, 7, 8 as pinned by the reference's own outputs."""
    g = cgold
    assert g["discrete_random/reset_obs"].shape[1] == 261                       # 261, not the declared 260
    hold = g["discrete_hold/reward"][:, :49]
    assert (hold == -1.0).all()                                                 # hold reward is exactly -1.0
    assert (g["discrete_hold/reward"][:, 50] == -1.0).all()                     # action 7: no branch matches -> hold
    term = g["discrete_random/terminated"]
    steps = g["discrete_random/step"]
    assert term.sum() >= 12 and (steps[term == 1] == 0).all()                   # time limit -> terminated, then reset
    # the market simulator is NOT reset: psychology right after a reset differs from the constructor's 0.5 path
    psy_after = g["discrete_random/psychology"][term == 1]
    assert np.abs(psy_after - 0.5).max() > 0.05


def test_next_step_and_disabled_modes(cgold):
    g, name = cgold, "discrete_random"
    m = meta(g, name)
    act = g[f"{name}/action"].astype(np.int64)
    dis = make_oracle(g, name, m, "disabled")
    nxt = make_oracle(g, name, m, "next_step")
    same = make_oracle(g, name, m, "same_step")
    for o in (dis, nxt, same):
        o.reset()
    T = 1003
    first_term = int(np.nonzero(g[f"{name}/terminated"].any(axis=0))[0][0])     # an env hits 10x balance early
    only_limit = np.nonzero(g[f"{name}/terminated"][:, :999].sum(axis=1) == 0)[0]  # envs that only hit the time limit
    assert first_term < 999 and len(only_limit) >= 3
    for t in range(T):
        for o in (dis, nxt, same):
            o.step(act[:, t])
        if t < first_term:
            assert np.array_equal(dis.obs, same.obs) and np.array_equal(nxt.obs, same.obs)
    # disabled: keeps stepping past the limit, terminated stays set (crypto_trading_env.py:382-386)
    assert (dis.state()["step"] == T).all() and dis.terminated.all()
    # next_step: the step after the terminal one resets (reward 0) instead of trading
    assert (nxt.state()["step"][only_limit] == 2).all() and (same.state()["step"][only_limit] == 3).all()


@pytest.mark.skipif(not ref_loader.reference_available(),
                    reason="needs the original project's sources (BENG_REFERENCE_ROOT=<its checkout>)")
def test_c_oracle_matches_live_reference():
    mod = ref_loader.load_crypto()
    real_np = mod.np
    n, T, seed = 3, 1100, 77
    rng = np.random.default_rng(5)
    tape = rng.integers(0, 5, (n, T))
    orc = CryptoOracle(n, seed=seed)
    orc.reset()
    try:
        for e in range(n):
            rr = replay.ReplayRandom(seed, e)
            mod.random, mod.np = rr, replay.NumpyWithReplayNormal(rr)
            env = mod.CryptoTradingEnv(action_type="discrete")
            obs, _ = env.reset()
            assert np.array_equal(obs, orc.obs[e])
            one = CryptoOracle(1, seed=seed, env_id_base=e)
            one.reset()
            for t in range(T):
                obs, r, term, trunc, info = env.step(int(tape[e, t]))
                one.step(tape[e, t:t + 1])
                if term:
                    obs, _ = env.reset()
                assert r == one.reward64[0] and term == bool(one.terminated[0])
                assert np.array_equal(obs, one.obs[0])
                assert info["portfolio_value"] == one.portfolio_value[0]
    finally:
        mod.np = real_np


def macd_weight_vectors(hist=50):
    """The two constant vectors of csrc/crypto.cu::make_macd_weights, restated in numpy: run the reference's recurrences
    (`_ema`, crypto_trading_env.py:108-119; the EMA-of-MACD-history of `macd`, :94-100) on the coefficient vectors of the
    closes instead of on the closes.  -> (wm, wg) with MACD line = wm . closes, signal line = wg . closes."""
    mf, ms, mg = 2.0 / 13.0, 2.0 / 27.0, 2.0 / 10.0
    wf, ws, sg = np.zeros(hist), np.zeros(hist), np.zeros(hist)
    wf[0] = ws[0] = 1.0
    for t in range(1, hist):
        wf[:t] *= 1.0 - mf
        ws[:t] *= 1.0 - ms
        wf[t], ws[t] = mf, ms
        if t == 25:
            sg = wf - ws
        elif t > 25:
            sg = (wf - ws) * mg + sg * (1.0 - mg)
    return wf - ws, sg


def test_macd_is_a_pair_of_dot_products():
    """What the CUDA step kernel relies on (DESIGN.md section 7): an EMA seeded with prices[0] is linear in the window, so
    MACD line and signal line are dot products of the 50 closes with constant weights that sum to zero -- taken with
    (close - newest close), as the kernel does.  Checked against the oracle's serial float64 recurrences (features 254..256
    = macd / range, signal / range, histogram / range) far inside the 1e-5 observation tolerance."""
    wm, wg = macd_weight_vectors()
    assert abs(wm.sum()) < 1e-15 and abs(wg.sum()) < 1e-15
    n = 512
    orc = CryptoOracle(n, seed=5)
    orc.reset()
    rng = np.random.default_rng(0)
    worst = 0.0
    for t in range(120):
        obs, *_ = orc.step(rng.integers(0, 5, n))
        closes = orc.state(with_candles=True)["candles"][:, :, 3]          # (n, 50) float64, oldest first
        d = closes - closes[:, -1:]
        span = closes.max(axis=1) - closes.min(axis=1)
        ok = span > 0
        feats = np.stack([d @ wm, d @ wg, d @ wm - d @ wg], axis=1)[ok] / span[ok, None]
        ref = obs[ok, 254:257].astype(np.float64)
        worst = max(worst, float(np.max(np.abs(feats - ref) / (1e-6 + 1e-5 * np.abs(ref)))))
    assert worst < 0.05, worst  # (the float32 rounding of the oracle's observation is the only difference)


def test_staged_reference_copies_are_byte_identical():
    """oracle/make_ref.py: the files bench.py's CPU arm and the live-reference tests run on the GPU box are byte-for-byte
    the reference's (sha256 manifest; compared with /root/reference itself when it is present)."""
    from oracle import make_ref

    if not make_ref.source_available() and not os.path.exists(os.path.join(make_ref.DEST, "MANIFEST.json")):
        pytest.skip("neither /root/reference nor oracle/_ref is present")
    if make_ref.source_available():
        make_ref.stage(verbose=False)
    assert make_ref.check()
