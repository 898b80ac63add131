"""crypto_trading_env on the B200 engine.

  BatchedCryptoTradingEnv   gymnasium.vector.VectorEnv-compatible; N envs stepped by ONE CUDA kernel
                            (csrc/crypto.cu) through the C ABI (include/beng.h).
  CryptoTradingEnv          the reference's single-instance gym.Env surface
                            (crypto_trading_env/crypto_trading_env.py:224-561), a 1-env view of the same engine.
  TradingConfig             same fields/defaults as the reference dataclass (crypto_trading_env.py:28-38).

Reference quirks kept on purpose (SURVEY.md section 0): the observation has 261 elements although the reference
DECLARES a (260,) space (:285-286 vs :534-559); the time limit is reported as `terminated` (:382-388); the
MarketSimulator (regime, trend strength, psychology) is NOT reset by reset() (:257, :301-340); the reward is the
portfolio change valued at the OLD price, minus 1.0 when no trade executed (:440-445).
Money/price arithmetic is float64 on the device exactly as in the reference; observations are float32.
"""
from __future__ import annotations

import ctypes as C
from dataclasses import asdict, dataclass

import numpy as np
import torch

from . import _lib
from .spaces import Box, Discrete, batch_space
from .vector import _EnvBase, AUTORESET_MODES, LazyInfos as _LazyInfos, _BatchedEnv, as_device_actions, host_source, stream_ptr

HISTORY = 50
OBS_DIM = 261
REGIME_NAMES = ("bull_run", "bear_market", "sideways", "crash", "recovery")  # MarketRegime values, :20-25
CRYPTO_STAT_NAMES = ("n_episodes", "sum_return", "sum_length", "sum_final_value")


@dataclass
class TradingConfig:
    """Configuration for the trading environment (crypto_trading_env.py:28-38)."""
    initial_balance: float = 10000.0
    trading_fee_rate: float = 0.001
    slippage_rate: float = 0.0005
    history_length: int = 50
    min_price: float = 100.0
    max_price: float = 100000.0
    volatility_base: float = 0.02
    market_psychology_factor: float = 0.1


class BatchedCryptoTradingEnv(_BatchedEnv):
    """N independent CryptoTradingEnv instances; state resident in HBM as [field][env] arrays."""

    metadata = {"render_modes": [], "render_fps": 30, "autoreset_mode": "same_step"}
    _reset_fn = "beng_crypto_reset"
    _state_tensors = ("_scal", "_meta", "_ep_return", "_close", "_ohlv")
    _stat_names = CRYPTO_STAT_NAMES
    _host_names = ("_actions", "obs", "reward", "terminated", "truncated")

    def __init__(self, num_envs: int, config: TradingConfig | None = None, action_type: str = "continuous",
                 render_mode=None, *, device="cuda", seed: int = 0, env_id_base: int = 0,
                 autoreset_mode="same_step", max_steps: int = 1000, info_outputs: bool = True,
                 time_limit_truncation: bool = False):
        super().__init__(num_envs, device, autoreset_mode, render_mode)
        n = self.num_envs
        self.config = config or TradingConfig()
        if self.config.history_length != HISTORY:
            raise ValueError("history_length is fixed at 50 in the CUDA engine")
        if action_type not in ("continuous", "discrete"):
            raise ValueError("action_type must be 'continuous' or 'discrete'")
        self.action_type = action_type
        self.max_steps = int(max_steps)

        # the reference declares (260,) but returns 261 values; the spaces here describe what is returned
        self.single_observation_space = Box(-np.inf, np.inf, (OBS_DIM,), np.float32)
        if action_type == "continuous":
            self.single_action_space = Box(-1.0, 1.0, (2,), np.float32)       # :290-293
        else:
            self.single_action_space = Discrete(5)                             # :296
        self.observation_space = batch_space(self.single_observation_space, n)
        self.action_space = batch_space(self.single_action_space, n)

        c = self.config
        self.params = _lib.CryptoParams(c.initial_balance, c.trading_fee_rate, c.slippage_rate, c.min_price,
                                        c.max_price, c.volatility_base, c.market_psychology_factor, self.max_steps,
                                        AUTORESET_MODES[self.autoreset_mode], int(action_type == "continuous"),
                                        0, int(bool(time_limit_truncation)), 0, int(seed), int(env_id_base))
        dev = self.device
        with torch.cuda.device(dev):
            z = lambda *shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
            # state
            self._scal = z(4, n, dt=torch.float64)       # cash, holdings, trend_strength, psychology
            self._meta = z(2, n, dt=torch.int32)         # step | regime<<16 | flags<<24 ; rng counter
            self._ep_return = z(n, dt=torch.float64)
            pitch = int(self.lib.beng_crypto_window_pitch(n))   # rows padded to whole 32-env units (TMA boxes)
            self._close = z(HISTORY, pitch, dt=torch.float64)
            self._ohlv = z(HISTORY, pitch, 4, dt=torch.float32)   # open, high, low, volume: one 16-byte record per env
            # outputs
            self.obs = z(n, OBS_DIM, dt=torch.float32)
            self.reward = z(n, dt=torch.float32)
            self.terminated = z(n, dt=torch.bool)
            self.truncated = z(n, dt=torch.bool)
            self.reward64 = z(n, dt=torch.float64) if info_outputs else None
            self.portfolio_value = z(n, dt=torch.float64) if info_outputs else None
            self.current_price = z(n, dt=torch.float64) if info_outputs else None
            self.trade_kind = z(n, dt=torch.uint8) if info_outputs else None
            self.ep_return = z(n, dt=torch.float64)
            self.ep_length = z(n, dt=torch.int32)
            self.stats = z(4, dt=torch.float64)
            # {window head, arrivals}: the slot of the newest candle, advanced by the step kernel itself, so that a
            # step's arguments never change (a CUDA graph can capture it) and no host state moves per step
            self._head = z(2, dt=torch.int32)
            self._actions = z(n, 2, dt=torch.float32) if action_type == "continuous" else z(n, dt=torch.int64)
        self._state = _lib.CryptoState(self._scal.data_ptr(), self._meta.data_ptr(), self._ep_return.data_ptr(),
                                       self._close.data_ptr(), self._ohlv.data_ptr())
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        self._io = _lib.CryptoIO(self.obs.data_ptr(), self.reward.data_ptr(), self.terminated.data_ptr(),
                                 self.truncated.data_ptr(), ptr(self.reward64), ptr(self.portfolio_value),
                                 ptr(self.current_price), ptr(self.trade_kind), self.ep_return.data_ptr(),
                                 self.ep_length.data_ptr(), self.stats.data_ptr(), self._head.data_ptr())
        self._info_cache = None

    # ------------------------------------------------------------------ state views
    @property
    def cash(self):
        return self._scal[0]

    @property
    def holdings(self):
        return self._scal[1]

    @property
    def trend_strength(self):
        return self._scal[2]

    @property
    def market_psychology(self):
        return self._scal[3]

    @property
    def current_step(self):
        return self._meta[0] & 0xFFFF

    @property
    def market_regime(self):
        """Regime codes (index into REGIME_NAMES)."""
        return (self._meta[0] >> 16) & 0xFF

    @property
    def rng_counter(self):
        return self._meta[1].to(torch.int64) & 0xFFFFFFFF

    def price_history(self) -> torch.Tensor:
        """(n, 50, 5) float64 window, oldest first: open, high, low, close, volume (open/high/low/volume are
        kept in float32 on the device)."""
        order = (self._head[0].long() + 1 + torch.arange(HISTORY, device=self.device)) % HISTORY
        n = self.num_envs
        close = self._close[order][:, :n]                # (50, n)
        ohlv = self._ohlv[order][:, :n].to(torch.float64)  # (50, n, 4)
        cand = torch.stack([ohlv[..., 0], ohlv[..., 1], ohlv[..., 2], close, ohlv[..., 3]], dim=-1)  # (50, n, 5)
        return cand.permute(1, 0, 2).contiguous()

    def _infos(self):
        if self._info_cache is None:  # all entries are views of persistent buffers: build once
            info = _LazyInfos({"cash": self.cash, "holdings": self.holdings,
                               "market_psychology": self.market_psychology,
                               "episode": {"r": self.ep_return, "l": self.ep_length}, "_episode": self.terminated})
            info.lazy["market_regime"] = lambda: self.market_regime  # decoded from the packed state on access
            if self.portfolio_value is not None:
                info.update(portfolio_value=self.portfolio_value, current_price=self.current_price,
                            trade_kind=self.trade_kind, reward64=self.reward64)
            self._info_cache = info
        return self._info_cache

    # ------------------------------------------------------------------ VectorEnv API
    # reset(): CryptoTradingEnv.reset (:301-340).  `seed` also re-creates the market simulators (the reference seeds
    # both global RNGs, :305-307).

    def step(self, actions):
        """One step of every env (:342-398) -> (obs, rewards, terminations, truncations, infos).
        Discrete: int64 (n,) with 0=hold 1=buy 5% 2=buy 20% 3=sell 5% 4=sell 20% (anything else holds, like the
        reference).  Continuous: float32 (n, 2) = [buy, sell], clipped to [0, 1] x 10 % caps (:408-422).

        One kernel launch with the same arguments every call and no host state that changes per step (the window head
        lives on the device), so a loop of step() calls with device-resident actions can be captured once with
        torch.cuda.graph and replayed, interleaved with eager steps as needed."""
        self._require_reset()
        act = as_device_actions(actions, self._actions)
        self._call("beng_crypto_step", C.byref(self.params), C.byref(self._state), act.data_ptr(), C.byref(self._io),
                   self.num_envs, stream_ptr(self.device))
        return self.obs, self.reward, self.terminated, self.truncated, self._infos()

    def step_host(self, actions, *, copy_obs: bool = True, sync: bool = True):
        """step() for callers holding HOST arrays (numpy in, numpy out) through `beng_crypto_step_host`."""
        self._require_reset()
        h = self._host_buffers()
        src = self._host_src = host_source(actions, h["_actions"])
        self._call("beng_crypto_step_host", C.byref(self.params), C.byref(self._state), self._actions.data_ptr(),
                   C.byref(self._io), self.num_envs, src.data_ptr(), h["obs"].data_ptr() if copy_obs else None,
                   h["reward"].data_ptr(), h["terminated"].data_ptr(), h["truncated"].data_ptr(),
                   stream_ptr(self.device))
        if sync:
            self._sync()
        obs = h["obs"].numpy() if copy_obs else self.obs
        return obs, h["reward"].numpy(), h["terminated"].numpy(), h["truncated"].numpy(), {}

    # ------------------------------------------------------------------ extras
    def state_dict(self) -> dict:
        return dict(super().state_dict(), window_head=int(self._head[0].item()), config=asdict(self.config))

    def load_state_dict(self, sd: dict):
        head = int(sd["window_head"])
        if not 0 <= head < HISTORY:
            raise ValueError(f"window_head must be in 0..{HISTORY - 1}, got {head}")
        super().load_state_dict(sd)
        self._head.copy_(torch.tensor([head, 0], dtype=torch.int32))


class CryptoTradingEnv(_EnvBase):
    """Single-instance gym.Env surface of the reference (crypto_trading_env.py:224-561) on the CUDA engine: a
    1-env BatchedCryptoTradingEnv with auto-reset disabled; numpy observations, Python floats, the reference's
    info keys (trade_info is rebuilt on the host from the cash/holdings deltas)."""

    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 30}

    def __init__(self, config: TradingConfig | None = None, action_type: str = "continuous", render_mode=None, *,
                 device="cuda", seed: int = 0, env_id: int = 0):
        self.config = config or TradingConfig()
        self.action_type = action_type
        self.render_mode = render_mode
        self.max_steps = 1000
        self._vec = BatchedCryptoTradingEnv(1, self.config, action_type, device=device, seed=seed,
                                            env_id_base=env_id, autoreset_mode="disabled", max_steps=self.max_steps)
        self.observation_space = self._vec.single_observation_space
        self.action_space = self._vec.single_action_space

    cash = property(lambda self: float(self._vec.cash.item()))
    holdings = property(lambda self: float(self._vec.holdings.item()))
    current_step = property(lambda self: int(self._vec.current_step.item()))

    def reset(self, seed=None, options=None):
        obs, _ = self._vec.reset(seed=seed)
        return obs[0].cpu().numpy().copy(), {}

    def step(self, action):
        v = self._vec
        cash0, hold0, price0 = self.cash, self.holdings, float(v._close[v._head[0].long(), 0].item())
        if self.action_type == "continuous":
            act = np.asarray(action, dtype=np.float32).reshape(1, 2)
        else:
            act = np.asarray([int(action)], dtype=np.int64)
        obs, rew, term, trunc, info = v.step(act)
        kind = int(info["trade_kind"].item())
        trade_info = None
        if kind:
            c = self.config
            if kind == 1:
                amount, crypto_amount = cash0 - self.cash, self.holdings - hold0
                fee = amount * c.trading_fee_rate
                price = (amount - fee) / crypto_amount
                trade_info = {"action": "buy", "amount": amount, "crypto_amount": crypto_amount, "price": price,
                              "fee": fee, "slippage": price - price0}
            else:
                net_cash, crypto_amount = self.cash - cash0, hold0 - self.holdings
                received = net_cash / (1.0 - c.trading_fee_rate)
                price = received / crypto_amount
                trade_info = {"action": "sell", "amount": net_cash, "crypto_amount": crypto_amount, "price": price,
                              "fee": received * c.trading_fee_rate, "slippage": price0 - price}
        out_info = {"portfolio_value": float(info["portfolio_value"].item()), "cash": self.cash,
                    "holdings": self.holdings, "current_price": float(info["current_price"].item()),
                    "market_regime": REGIME_NAMES[int(info["market_regime"].item())],
                    "market_psychology": float(info["market_psychology"].item()), "trade_info": trade_info}
        return (obs[0].cpu().numpy().copy(), float(info["reward64"].item()), bool(term.item()), False, out_info)

    def render(self):
        return None

    def close(self):
        self._vec.close()
