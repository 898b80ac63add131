"""The 11 indicator features of the crypto observation (obs[250:261]) where the kernel leaves the reference's operation
order (csrc/crypto.cu, compose_unit / finish_unit): constant price windows at non-round prices, injected windows whose
error can be bounded feature by feature, realistic price floors, the covariance of the whole step under a power-of-two
rescaling of every price, and the price domain the kernel accepts.

n = 333 covers full 32-env units, a partial unit and the ragged tail of the tile store."""
import ctypes as C

import numpy as np
import pytest
import torch

from oracle.c_oracle import CryptoOracle
from test_crypto_features import CLOSES, numpy_features

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
RTOL, ATOL = 1e-5, 1e-6  # tests/test_crypto_gpu.py
N = 333
U = 2.0 ** -24  # float32 unit roundoff
FEAT = slice(253, 260)  # RSI, MACD x 3, Bollinger x 3


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    assert torch.cuda.is_available()
    p._lib.load()
    return p


def np_(t):
    return t.cpu().numpy()


def cfg_tuple(c):
    return (c.initial_balance, c.trading_fee_rate, c.slippage_rate, c.min_price, c.max_price, c.volatility_base,
            c.market_psychology_factor)


def close_obs(a, b, what=""):
    np.testing.assert_allclose(a, b, rtol=RTOL, atol=ATOL, err_msg=what)


def assert_features_equal(dev, orc, what):
    bad = np.nonzero((dev[:, FEAT] != orc[:, FEAT]).any(1))[0]
    assert bad.size == 0, (f"{what}: features 253..259 differ in {bad.size} envs, first env {bad[0]}: "
                           f"device {dev[bad[0], FEAT]} oracle {orc[bad[0], FEAT]}")


# ---------------------------------------------------------------------------------------------------------------- B1
@pytest.mark.parametrize("c", CLOSES)
def test_pinned_windows_match_oracle(pkg, c):
    """min_price == max_price == c: every window is 20 (50) copies of c, so features 253..259 depend on c alone and must
    be bit-identical.  Staggered episodes of 37 steps send the constant windows through the TMA path, the re-read path
    of units with an in-step reset, and the warp-cooperative rebuild of a window."""
    limit, seed = 37, 19
    cfg = pkg.TradingConfig(min_price=c, max_price=c)
    env = pkg.BatchedCryptoTradingEnv(N, cfg, "discrete", device=DEV, seed=seed, autoreset_mode="same_step",
                                      max_steps=limit)
    orc = CryptoOracle(N, seed=seed, cfg=cfg_tuple(cfg), max_steps=limit)
    dev, ref = np_(env.reset()[0]), orc.reset()
    assert_features_equal(dev, ref, f"c={c} reset")
    assert np.array_equal(ref[:, FEAT], np.tile(numpy_features(np.full(50, c)), (N, 1)))
    close_obs(dev, ref, f"c={c} reset")
    gen = torch.Generator(device=DEV).manual_seed(2)
    idx = torch.arange(N, device=DEV)
    for t in range(limit - 1):  # stagger: env i restarts its episode after (i % limit) steps
        a = torch.randint(0, 5, (N,), device=DEV, generator=gen)
        env.step(a), orc.step(np_(a), want_obs=False)
        mask = (idx % limit) == t
        env.reset(options={"reset_mask": mask})
        orc.reset(np_(mask))
    for t in range(60):
        a = torch.randint(0, 5, (N,), device=DEV, generator=gen)
        env.step(a), orc.step(np_(a))
        assert np.array_equal(np_(env.terminated).astype(np.uint8), orc.terminated), t
        dev = np_(env.obs)
        assert_features_equal(dev, orc.obs, f"c={c} step {t}")
        close_obs(dev, orc.obs, f"c={c} step {t}")
    assert orc.stats()["n_episodes"] > N


# ---------------------------------------------------------------------------------------------------------------- B2
@pytest.mark.parametrize("volatility", [0.02, 0.05])
def test_realistic_floors_match_oracle(pkg, volatility):
    """Non-round price bounds: prices pin at the floor 45000.7 (and the ceiling 99999.99) for many steps."""
    n, seed, T = 2000, 13, 250
    cfg = pkg.TradingConfig(min_price=45000.7, max_price=99999.99, volatility_base=volatility)
    env = pkg.BatchedCryptoTradingEnv(n, cfg, "discrete", device=DEV, seed=seed)
    orc = CryptoOracle(n, seed=seed, cfg=cfg_tuple(cfg))
    close_obs(np_(env.reset()[0]), orc.reset(), "reset")
    gen = torch.Generator(device=DEV).manual_seed(4)
    constant = 0
    for t in range(T):
        a = torch.randint(0, 5, (n,), device=DEV, generator=gen)
        env.step(a), orc.step(np_(a))
        assert np.array_equal(np_(env.terminated).astype(np.uint8), orc.terminated), t
        close_obs(np_(env.obs), orc.obs, f"obs at step {t}")
        last20 = orc.state(with_candles=True)["candles"][:, -20:, 3]
        constant += int((last20 == last20[:, -1:]).all(1).sum())
    assert constant >= 500, f"only {constant} env-steps had a constant 20-close window"


# ---------------------------------------------------------------------------------------------------------------- B3
# Per-feature error bounds of one teacher-forced step, device against oracle, |dev - orc| <= bound.  u = 2^-24.
B_CLOSE = 2 * U     # close / cur: both sides round a quotient known to ~4e-15 to float32: <= 1 ulp apart
B_PORT = 2 * U      # cash / ib, holdings * cur / ib, value / ib, psychology: one float32 rounding each side (1/ib: 1e-16)
B_OHLV = 4 * U      # o/h/l/v: float32 storage of this step's candle (u) + float32 1/cur (u) + product (u) + oracle's cast (u)
B_RSI = 7 * U       # two float32 casts (2u) + __fdividef (2 ulp = 4u) + oracle's cast (u); the float64 sums are identical
B_RSI_ABS = 2.0 ** -50  # the oracle's 100 - 100 / (1 + rs) cancels when rs is small: a few float64 ulps of 100, / 100
B_MACD = 9 * U      # float32 pm (u) + range from float32 max/min of float32 differences (3u) + __fdividef (4u) + cast (u)
B_BAND = 16 * U     # sd: float32 variance (u) + rsqrtf (4u) + product (u); two float32 casts (2u) + __fdividef (4u) + cast (u)
B_PCT = 8 * U       # (cur - sma) / sma: two float32 casts (2u) + __fdividef (4u) + oracle's cast (u)
# The reference's own float64 recurrences run on absolute prices: its EMAs and its pairwise mean carry an absolute error
# of C * 2^-52 * close (the three EMAs: <= 3.7 measured against exact rational arithmetic on these window families; the
# pairwise mean of 20 closes: <= ~2.6 from its 19 roundings), while the kernel takes the same sums on differences to the
# newest close, nearly exactly.  Divided by the close range (MACD) or the band width (Bollinger), that is
# C * 2^-52 * close / range of the feature: it is why a window whose spread is 1e-12 of the price cannot be held to an
# ulp bound.  C = 32 leaves a factor of ~8 over both.
C_COND = 32.0


def families(c, rng):
    """-> list of (name, final 50 closes oldest first, newest == c)."""
    eps = 1e-3
    up = c * (1 + eps)
    fam = []
    w = np.full(50, up)
    w[-1] = c
    fam.append(("outlier: newest", w))
    w = np.full(50, c)
    w[30] = up
    fam.append(("outlier: oldest of the last 20", w))
    w = np.full(50, c)
    w[0] = up
    fam.append(("outlier: slot 0 only", w))
    j = np.arange(50)
    fam.append(("rising", c * (1 - eps * (49 - j))))
    fam.append(("falling", c * (1 + eps * (49 - j))))
    d = np.ldexp(1.0, int(np.floor(np.log2(c))) - 8)  # exact: c and c + d are both doubles, d a power of two
    fam.append(("zig-zag", np.where((49 - j) % 2 == 0, c, c + d)))
    fam.append(("constant", np.full(50, c)))
    for s in (1e-2, 1e-5, 1e-8, 1e-12):
        w = c * (1 + s * rng.uniform(-1, 1, 50))
        w[-1] = c
        fam.append((f"spread {s:g}", w))
    for f in fam:
        f[1][-1] = c
    return fam


def inject(env, windows, rng):
    """Write pre-step windows (n, 50) of closes into the ring, open/high/low/volume as float32."""
    sd = env.state_dict()
    head = int(sd["window_head"])
    order = [(head + 1 + k) % 50 for k in range(50)]
    n = windows.shape[0]
    close = sd["close"].clone()
    ohlv = sd["ohlv"].clone()
    w = torch.from_numpy(windows.T.copy()).to(DEV)  # (50, n)
    close[order, :n] = w
    ohlv[order, :n, 0] = (w * torch.from_numpy(rng.uniform(0.99, 1.01, (50, n))).to(DEV)).float()
    ohlv[order, :n, 1] = (w * torch.from_numpy(rng.uniform(1.0, 1.02, (50, n))).to(DEV)).float()
    ohlv[order, :n, 2] = (w * torch.from_numpy(rng.uniform(0.98, 1.0, (50, n))).to(DEV)).float()
    ohlv[order, :n, 3] = torch.from_numpy(rng.uniform(0.5, 2.0, (50, n))).to(DEV).float()
    sd["close"], sd["ohlv"] = close, ohlv
    env.load_state_dict(sd)


def bounds(orc_obs, final):
    """(n, 261) bound on |dev - orc| for one step, from the oracle's observation and the final windows (n, 50)."""
    o = np.abs(orc_obs.astype(np.float64))
    b = np.empty_like(o)
    cur = final[:, -1]
    rng50 = final.max(1) - final.min(1)
    last20 = final[:, -20:]
    width = 4 * last20.std(1)
    cond_macd = np.where(rng50 > 0, C_COND * 2.0 ** -52 * cur / np.where(rng50 > 0, rng50, 1), 0)[:, None]
    cond_band = np.where(width > 0, C_COND * 2.0 ** -52 * cur / np.where(width > 0, width, 1), 0)
    cols = np.arange(250)
    b[:, cols] = B_OHLV * o[:, cols]
    b[:, cols[3::5]] = B_CLOSE * o[:, cols[3::5]]
    b[:, [250, 251, 252, 260]] = B_PORT * o[:, [250, 251, 252, 260]]
    b[:, 253] = B_RSI * o[:, 253] + B_RSI_ABS
    b[:, 254:257] = B_MACD * o[:, 254:257] + cond_macd
    b[:, 257] = B_BAND * np.maximum(o[:, 257], 1.0) + cond_band
    b[:, 258] = (B_BAND + cond_band) * o[:, 258]
    b[:, 259] = B_PCT * o[:, 259] + C_COND * 2.0 ** -52
    return b


GROUPS = {"close": np.arange(3, 250, 5), "open/high/low/volume": np.setdiff1d(np.arange(250), np.arange(3, 250, 5)),
          "portfolio + psychology": np.array([250, 251, 252, 260]), "rsi": np.array([253]),
          "macd": np.array([254, 255, 256]), "band position": np.array([257]), "band width": np.array([258]),
          "close vs sma": np.array([259])}


@pytest.mark.parametrize("c", [45000.7, 1000.0, 0.01])
def test_injected_windows_one_step_error_bounds(pkg, c):
    """Windows written into the ring, one teacher-forced step with the bounds pinned to the newest close (so the step's
    new candle is c): every feature within the bound derived for it above."""
    seed = 23
    rng = np.random.default_rng(int(c * 100) % 1000)
    fam = families(c, rng)
    final = np.stack([fam[i % len(fam)][1] for i in range(N)])
    names = [fam[i % len(fam)][0] for i in range(N)]
    pre = np.concatenate([final[:, :1], final[:, :-1]], axis=1)  # the step drops the oldest and appends c
    cfg = pkg.TradingConfig(min_price=c, max_price=c)
    env = pkg.BatchedCryptoTradingEnv(N, cfg, "discrete", device=DEV, seed=seed)
    orc = CryptoOracle(N, seed=seed, cfg=cfg_tuple(cfg))
    env.reset()
    gen = torch.Generator(device=DEV).manual_seed(6)
    worst = {g: 0.0 for g in GROUPS}
    for rep in range(3):  # three draws of actions and open/high/low/volume per window
        inject(env, pre, rng)
        orc.set_state({"cash": np_(env.cash), "holdings": np_(env.holdings),
                       "trend_strength": np_(env.trend_strength), "psychology": np_(env.market_psychology),
                       "regime": np_(env.market_regime), "step": np_(env.current_step),
                       "rng_counter": np_(env.rng_counter), "candles": np_(env.price_history())})
        a = torch.randint(0, 5, (N,), device=DEV, generator=gen)
        env.step(a), orc.step(np_(a))
        assert np.array_equal(np_(env.price_history())[:, :, 3], final)
        dev, ref = np_(env.obs).astype(np.float64), orc.obs.astype(np.float64)
        err = np.abs(dev - ref)
        bnd = bounds(orc.obs, final)
        for g, cols in GROUPS.items():
            r = err[:, cols] / np.where(bnd[:, cols] > 0, bnd[:, cols], np.inf)
            r[(err[:, cols] > 0) & (bnd[:, cols] == 0)] = np.inf
            worst[g] = max(worst[g], float(r.max()))
        over = np.argwhere(err > bnd)
        assert over.size == 0, (f"c={c}: {len(over)} values over the bound; first: env {over[0][0]} ({names[over[0][0]]}), "
                                f"feature {over[0][1]}: device {dev[tuple(over[0])]!r} oracle {ref[tuple(over[0])]!r} "
                                f"bound {bnd[tuple(over[0])]!r}")
    print(f"\nc={c}: worst error / bound per group: " + ", ".join(f"{g} {v:.3g}" for g, v in worst.items()))
    # the families pin the indicators where they are known exactly
    obs = np_(env.obs)
    for name, want in (("rising", 1.0), ("falling", 0.0), ("zig-zag", 0.5)):
        rows = [i for i in range(N) if names[i] == name]
        assert np.all(obs[rows, 253] == want), name


# ---------------------------------------------------------------------------------------------------------------- B4
# Default bounds 100 .. 100000 scaled by 2^k stay inside [2^-100, 2^100] for -106 <= k <= 83.
SCALES = [-106, -100, -90, -75, -60, -40, -20, -1, 1, 20, 40, 50, 55, 60, 70, 83]


def test_scale_covariance_on_device(pkg):
    """Every price (window, bounds) times 2^k and the holdings times 2^-k: the device step is the same computation on
    scaled values (tests/test_crypto_features.py shows the oracle is), so features 0..3 of each candle and the 11
    indicator features are bit-identical, the volume column scales by exactly 2^-k, and the money does not change.
    This also holds the hardware approximations behind __fdividef and rsqrtf to not depending on the exponent."""
    seed = 29
    base = pkg.BatchedCryptoTradingEnv(N, None, "discrete", device=DEV, seed=seed, autoreset_mode="disabled")
    base.reset()
    gen = torch.Generator(device=DEV).manual_seed(8)
    for _ in range(60):
        base.step(torch.randint(0, 5, (N,), device=DEV, generator=gen))
    sd = base.state_dict()
    tape = [torch.randint(0, 5, (N,), device=DEV, generator=gen) for _ in range(20)]
    vol = np.arange(4, 250, 5)
    other = np.setdiff1d(np.arange(261), vol)

    def run(k):
        cfg = pkg.TradingConfig(min_price=100.0 * 2.0 ** k, max_price=100000.0 * 2.0 ** k)
        env = pkg.BatchedCryptoTradingEnv(N, cfg, "discrete", device=DEV, seed=seed, autoreset_mode="disabled")
        s = {key: (v.clone() if torch.is_tensor(v) else v) for key, v in sd.items()}
        s["close"] *= 2.0 ** k
        s["ohlv"][..., :3] *= 2.0 ** k
        s["scal"][1] *= 2.0 ** -k
        env.load_state_dict(s)
        out = []
        for a in tape:
            obs, _, term, _, info = env.step(a)
            out.append(dict(obs=np_(obs).copy(), term=np_(term).copy(), reward64=np_(info["reward64"]).copy(),
                            value=np_(info["portfolio_value"]).copy(), price=np_(info["current_price"]).copy(),
                            trade=np_(info["trade_kind"]).copy(), cash=np_(env.cash).copy(),
                            ctr=np_(env.rng_counter).copy(), close=np_(env.price_history())[:, :, 3].copy()))
        return out

    ref = run(0)
    kinds = np.stack([r["trade"] for r in ref])
    assert (kinds == 1).sum() > 100 and (kinds == 2).sum() > 100, "the tape must trade both ways"
    failures = []
    for k in SCALES:
        got = run(k)
        for t, (g, r) in enumerate(zip(got, ref)):
            bad = []
            for key in ("term", "reward64", "value", "trade", "cash", "ctr"):
                if not np.array_equal(g[key], r[key]):
                    bad.append(key)
            if not np.array_equal(g["price"], r["price"] * 2.0 ** k):
                bad.append("current_price")
            if not np.array_equal(g["close"], r["close"] * 2.0 ** k):
                bad.append("close")
            cols = other[np.nonzero((g["obs"][:, other] != r["obs"][:, other]).any(0))[0]]
            if cols.size:
                bad.append(f"obs features {cols.tolist()}")
            want_vol = (r["obs"][:, vol].astype(np.float64) * 2.0 ** -k).astype(np.float32)
            if not np.array_equal(g["obs"][:, vol], want_vol):
                bad.append("volume column")
            if bad:
                failures.append(f"k={k} step {t}: {', '.join(bad)}")
                break  # the first failing step of each k
    assert not failures, "\n".join(failures)


# ---------------------------------------------------------------------------------------------------------------- B5
REJECTED = [(float("nan"), 1e5), (100.0, float("nan")), (100.0, float("inf")), (-float("inf"), 1e5),
            (float("inf"), float("inf")), (0.0, 1e5), (-5.0, 1e5), (200.0, 100.0), (2.0 ** -101, 1.0),
            (1.0, 2.0 ** 101), (1e-31, 1e5), (100.0, 1e31)]


@pytest.mark.parametrize("lo,hi", REJECTED)
def test_price_bounds_outside_domain_are_rejected(pkg, lo, hi):
    env = pkg.BatchedCryptoTradingEnv(40, pkg.TradingConfig(min_price=lo, max_price=hi), "discrete", device=DEV)
    with pytest.raises(RuntimeError, match="BENG_ERR_UNSUPPORTED"):
        env.reset()
    stream = torch.cuda.current_stream().cuda_stream
    unsupported = -2  # BENG_ERR_UNSUPPORTED, include/beng.h
    assert env.lib.beng_crypto_reset(C.byref(env.params), C.byref(env._state), C.byref(env._io), None, 40, 1,
                                     stream) == unsupported
    assert env.lib.beng_crypto_step(C.byref(env.params), C.byref(env._state), env._actions.data_ptr(),
                                    C.byref(env._io), 40, stream) == unsupported


@pytest.mark.parametrize("lo,hi", [(2.0 ** -100, 2.0 ** -100), (2.0 ** 100, 2.0 ** 100), (2.0 ** -100, 2.0 ** 100)])
def test_price_domain_edges_are_accepted(pkg, lo, hi):
    cfg = pkg.TradingConfig(min_price=lo, max_price=hi)
    env = pkg.BatchedCryptoTradingEnv(40, cfg, "discrete", device=DEV, seed=1)
    orc = CryptoOracle(40, seed=1, cfg=cfg_tuple(cfg))
    close_obs(np_(env.reset()[0]), orc.reset(), "reset")
    for t in range(3):
        a = torch.full((40,), t % 5, dtype=torch.int64, device=DEV)
        env.step(a), orc.step(np_(a))
        assert np.isfinite(np_(env.obs)).all()
        close_obs(np_(env.obs), orc.obs, f"step {t}")
