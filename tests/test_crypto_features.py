"""The C oracle's indicator features (obs[253:260]) on constant price windows against NumPy's own arithmetic, and the
oracle's covariance under a power-of-two rescaling of every price (tests/test_crypto_features_gpu.py relies on both).

Prices pin at min_price / max_price often.  A window of 20 identical closes c then goes through np.mean / np.std of
np.full(20, c), and NumPy's pairwise sum of 20 copies of c is exact only for some c (100.0, 30000.0): for most others
(1000.1, 45000.7) sma != c, std > 0 and the Bollinger position (feature 257) is 0.25 or 0.75, not 0.5."""
import numpy as np
import pytest

from oracle.c_oracle import CRYPTO_DEFAULT_CFG, CryptoOracle
from oracle.crypto_port import _bollinger, _macd, _rsi

ROUND_CLOSES = [100.0, 1000.0, 30000.0, 100000.0]
ODD_CLOSES = [0.01, 1000.1, 45000.7, 99999.99]
RANDOM_CLOSES = [float(c) for c in np.random.default_rng(7).uniform(1.0, 1e5, 24)]
CLOSES = ROUND_CLOSES + ODD_CLOSES + RANDOM_CLOSES


def pinned_cfg(c):
    cfg = list(CRYPTO_DEFAULT_CFG)
    cfg[3] = cfg[4] = c  # min_price == max_price == c: every close of every window is c
    return tuple(cfg)


def numpy_features(closes):
    """obs[253:260] as the reference computes them (crypto_trading_env.py:45-119, :536-554), float32."""
    cur = closes[-1]
    line, sig, hist = _macd(closes)
    span = max(closes) - min(closes)
    up, mid, lo = _bollinger(closes)
    out = [_rsi(closes) / 100.0]
    out += [line / span, sig / span, hist / span] if span > 0 else [0.0, 0.0, 0.0]
    out += [(cur - lo) / (up - lo) if up > lo else 0.5, (up - lo) / mid if mid > 0 else 0.0,
            (cur - mid) / mid if mid > 0 else 0.0]
    return np.array(out, dtype=np.float32)


def test_closes_cover_both_cases():
    """The list holds closes whose 20-copy sum is exact (band position 0.5) and closes where it is not."""
    pos = [numpy_features(np.full(50, c))[4] for c in CLOSES]
    assert {0.5, 0.25, 0.75} <= set(pos)
    assert all(numpy_features(np.full(50, c))[4] == 0.5 for c in ROUND_CLOSES)
    assert numpy_features(np.full(50, 1000.1))[4] == 0.75


@pytest.mark.parametrize("c", CLOSES)
def test_constant_window_features_equal_numpy(c):
    n = 4
    orc = CryptoOracle(n, seed=11, cfg=pinned_cfg(c))
    want = numpy_features(np.full(50, c))
    obs = orc.reset()
    assert np.array_equal(orc.state(with_candles=True)["candles"][:, :, 3], np.full((n, 50), c))
    assert np.array_equal(obs[:, 253:260], np.tile(want, (n, 1))), (c, obs[0, 253:260], want)
    rng = np.random.default_rng(1)
    for t in range(5):
        orc.step(rng.integers(0, 5, n))
        assert np.array_equal(orc.obs[:, 253:260], np.tile(want, (n, 1))), (c, t)


def test_constant_window_closed_form():
    """csrc/crypto.cu::bollinger_constant computes features 257..259 of a constant window from t = c - sma alone:
    std == |t| exactly, so the band position is 0.75 / 0.25 / 0.5 for t > 0 / t < 0 / t == 0, the width 4|t| / sma and
    the offset t / sma.  NumPy itself, over closes across the whole price domain [2^-100, 2^100] and next to powers of
    two, where the pairwise sum crosses a binade."""
    rng = np.random.default_rng(11)
    p2 = np.exp2(np.round(rng.uniform(-99, 99, 1500)))
    cs = np.concatenate([rng.uniform(1.0, 1e5, 3000), np.exp2(rng.uniform(-100, 100, 3000)), p2,
                         np.nextafter(p2, 0), np.nextafter(p2, np.inf), [2.0 ** -100, 2.0 ** 100]])
    for c in cs:
        w = np.full(20, c)
        sma = np.mean(w)
        up, mid, lo = _bollinger(w)
        s = c * 16.0
        for _ in range(4):
            s = s + c
        t = c - s / 20.0
        assert mid == sma and np.std(w) == abs(t) and up == sma + 2 * abs(t) and lo == sma - 2 * abs(t), c
        assert numpy_features(np.full(50, c))[4:].tolist() == [np.float32(0.75 if t > 0 else 0.25 if t < 0 else 0.5),
                                                               np.float32(4 * abs(t / sma)), np.float32(t / sma)], c


# ---------------------------------------------------------------------------------------------------------------
# Scale covariance.  Multiplying every price (candles, bounds) by 2^k and the holdings by 2^-k changes no rounding in
# the oracle: the price walk multiplies the price by (1 + pct), which does not depend on the price; a buy adds
# net / (price + slippage) to the holdings and a sell receives amount * (price - slippage), so the holdings scale by
# 2^-k and the cash does not change; every indicator is a ratio of two price-scaled quantities.  Only the volume
# column of the observation (volume / price) scales, by 2^-k.  A reset would break it (the warm-up starts at 50000.0
# whatever the bounds), so the episodes run with auto-reset disabled.

SCALES = [1, -1, 20, -20, 60, -60, 90, -90]
VOLUME_COLS = np.arange(4, 250, 5)
OTHER_COLS = np.setdiff1d(np.arange(261), VOLUME_COLS)


def scaled_cfg(cfg, k):
    c = list(cfg)
    c[3], c[4] = c[3] * 2.0 ** k, c[4] * 2.0 ** k
    return tuple(c)


def scaled_state(st, k):
    s = {key: v.copy() for key, v in st.items()}
    s["holdings"] = s["holdings"] * 2.0 ** -k
    s["candles"][:, :, :4] *= 2.0 ** k  # open, high, low, close; not the volume
    return s


def run(orc, tape):
    out = []
    for a in tape:
        orc.step(a)
        st = orc.state()
        out.append(dict(obs=orc.obs.copy(), reward64=orc.reward64.copy(), term=orc.terminated.copy(),
                        trade=orc.trade_kind.copy(), price=orc.current_price.copy(), value=orc.portfolio_value.copy(),
                        cash=st["cash"], holdings=st["holdings"], ctr=st["rng_counter"]))
    return out


def test_oracle_scale_covariance():
    n, seed = 256, 5
    base = CryptoOracle(n, seed=seed, autoreset="disabled")
    base.reset()
    rng = np.random.default_rng(3)
    for _ in range(60):
        base.step(rng.integers(0, 5, n))
    st = base.state(with_candles=True)
    tape = [rng.integers(0, 5, n) for _ in range(20)]  # buys and sells of both sizes, holds
    ref = run(base, tape)
    kinds = np.stack([r["trade"] for r in ref])
    assert (kinds == 1).sum() > 100 and (kinds == 2).sum() > 100, "the tape must trade both ways"
    for k in SCALES:
        orc = CryptoOracle(n, seed=seed, autoreset="disabled", cfg=scaled_cfg(CRYPTO_DEFAULT_CFG, k))
        orc.set_state(scaled_state(st, k))
        got = run(orc, tape)
        for t, (g, r) in enumerate(zip(got, ref)):
            where = f"k={k} step {t}"
            for key in ("reward64", "term", "trade", "value", "cash", "ctr"):
                assert np.array_equal(g[key], r[key]), f"{key}, {where}"
            assert np.array_equal(g["holdings"], r["holdings"] * 2.0 ** -k), where
            assert np.array_equal(g["price"], r["price"] * 2.0 ** k), where
            assert np.array_equal(g["obs"][:, OTHER_COLS], r["obs"][:, OTHER_COLS]), where
            want_vol = (r["obs"][:, VOLUME_COLS].astype(np.float64) * 2.0 ** -k).astype(np.float32)
            assert np.array_equal(g["obs"][:, VOLUME_COLS], want_vol), where
