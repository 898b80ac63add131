"""Generate tests/golden/crypto_golden.npz by running the UNMODIFIED reference CryptoTradingEnv.

Build container only (needs /root/reference):   python -m oracle.gen_golden_crypto

The reference's module-level `random` and its `np.random.normal` (crypto_trading_env.py:13,148) are rebound
to ReplayRandom(seed, env_id) -- the engine's counter-based stream -- and the env is driven with a recorded
action tape in the reference's own caller loop (`if terminated: env.reset()` == SAME_STEP auto-reset).
Everything recorded is the reference's output.

Cases: discrete random tape crossing the 1000-step limit twice; discrete buy-heavy / sell-heavy / hold tapes;
continuous actions (passed as Python floats so that all arithmetic stays float64 -- SURVEY.md fact 8: with
float32 arrays NumPy 2 silently demotes `cash` to float32, which is a reference artefact, not the spec);
a custom TradingConfig.
"""
from __future__ import annotations

import os

import numpy as np

from . import golden_files, philox, ref_loader, replay

SNAP_EVERY = 23

# name, n_envs, n_steps, seed, env_id_base, action mode
CASES = [
    ("discrete_random", 6, 2100, 0, 0, "random"),
    ("discrete_hi_ids", 3, 400, 0xABCDEF012345, (1 << 34) + 9, "random"),
    ("discrete_buyer", 3, 600, 1, 10, "buyer"),
    ("discrete_seller", 3, 600, 2, 20, "churn"),
    ("discrete_hold", 2, 300, 3, 30, "hold"),
    ("continuous_random", 4, 700, 4, 40, "continuous"),
    ("custom_config", 3, 500, 5, 50, "random"),
]
CUSTOM_CFG = dict(initial_balance=2500.0, trading_fee_rate=0.002, slippage_rate=0.001, min_price=30000.0,
                  max_price=70000.0, volatility_base=0.05, market_psychology_factor=0.3)
REGIME_CODE = {"bull_run": 0, "bear_market": 1, "sideways": 2, "crash": 3, "recovery": 4}


def run_case(mod, name, n_envs, n_steps, seed, base, mode):
    cont = mode == "continuous"
    rec = {k: np.zeros((n_envs, n_steps), dt) for k, dt in [
        ("reward", np.float64), ("terminated", np.uint8), ("portfolio_value", np.float64), ("cash", np.float64),
        ("holdings", np.float64), ("current_price", np.float64), ("psychology", np.float64),
        ("trend_strength", np.float64), ("regime", np.int8), ("trade_kind", np.uint8), ("step", np.int32),
        ("rng_counter", np.uint32)]}
    rec["action"] = np.zeros((n_envs, n_steps, 2), np.float32) if cont else np.zeros((n_envs, n_steps), np.int8)
    rec["obs_tail"] = np.zeros((n_envs, n_steps, 11), np.float32)   # features 250..260 after every step
    snap_steps = np.arange(0, n_steps, SNAP_EVERY)
    snaps = np.zeros((n_envs, len(snap_steps), 261), np.float32)
    reset_obs = np.zeros((n_envs, 261), np.float32)
    tape = philox.action_tape(seed, base + np.arange(n_envs, dtype=np.uint64), 0, n_steps, 5)
    crng = np.random.default_rng(seed + 99)
    for e in range(n_envs):
        rr = replay.ReplayRandom(seed, base + e)
        mod.random = rr
        mod.np = replay.NumpyWithReplayNormal(rr)
        cfg = mod.TradingConfig(**CUSTOM_CFG) if name == "custom_config" else None
        env = mod.CryptoTradingEnv(config=cfg, action_type="continuous" if cont else "discrete")
        obs, info = env.reset()
        assert obs.shape == (261,) and info == {}
        reset_obs[e] = obs
        for t in range(n_steps):
            if cont:
                a32 = (crng.random(2) * 2.4 - 1.2).astype(np.float32)   # beyond [-1, 1] on purpose (clip path)
                act = [float(a32[0]), float(a32[1])]
                rec["action"][e, t] = a32
            else:
                a = {"random": int(tape[e, t]), "buyer": (2, 1, 2, 0, 3)[t % 5] if t % 97 else 4,
                     "churn": (2, 4, 4, 3, 1, 4)[t % 6], "hold": 0 if t % 50 else 7}[mode]
                act = a
                rec["action"][e, t] = a
            obs, r, term, trunc, info = env.step(act)
            assert trunc is False
            rec["reward"][e, t] = r
            rec["terminated"][e, t] = term
            rec["portfolio_value"][e, t] = info["portfolio_value"]
            rec["current_price"][e, t] = info["current_price"]
            ti = info["trade_info"]
            rec["trade_kind"][e, t] = 0 if ti is None else (1 if ti["action"] == "buy" else 2)
            if term:
                obs, _ = env.reset()
            rec["cash"][e, t] = env.cash
            rec["holdings"][e, t] = env.holdings
            rec["psychology"][e, t] = env.market_sim.market_psychology
            rec["trend_strength"][e, t] = env.market_sim.trend_strength
            rec["regime"][e, t] = REGIME_CODE[env.market_sim.current_regime.value]
            rec["step"][e, t] = env.current_step
            rec["rng_counter"][e, t] = rr.counter
            rec["obs_tail"][e, t] = obs[250:]
            if t % SNAP_EVERY == 0:
                snaps[e, t // SNAP_EVERY] = obs
    out = {f"{name}/{k}": v for k, v in rec.items()}
    out[f"{name}/snap_obs"] = snaps
    out[f"{name}/reset_obs"] = reset_obs
    out[f"{name}/meta"] = np.array([n_envs, n_steps, seed, base, SNAP_EVERY, int(cont)], dtype=np.uint64)
    return out


def main():
    assert ref_loader.reference_available(), "needs /root/reference (build container only)"
    mod = ref_loader.load_crypto()
    real_np = mod.np
    blob = {}
    try:
        for case in CASES:
            blob.update(run_case(mod, *case))
            n = case[0]
            print(n, "episodes", int(blob[f"{n}/terminated"].sum()), "trades", int((blob[f"{n}/trade_kind"] > 0).sum()),
                  "regimes seen", sorted(set(blob[f"{n}/regime"].ravel().tolist())))
    finally:
        mod.np = real_np
    blob["cases"] = np.array([c[0] for c in CASES])
    blob["custom_cfg"] = np.array([CUSTOM_CFG[k] for k in ("initial_balance", "trading_fee_rate", "slippage_rate",
                                                           "min_price", "max_price", "volatility_base",
                                                           "market_psychology_factor")])
    for path in golden_files.save("crypto", blob):
        print("wrote", os.path.relpath(path), os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
