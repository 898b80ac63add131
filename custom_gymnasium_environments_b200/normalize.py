"""Running normalization of observations and rewards for the batched envs (Stable-Baselines3 `VecNormalize` semantics),
computed on the device by libbeng's `beng_normalize` (csrc/normalize.cu).

    env = VecNormalize(BatchedCryptoTradingEnv(262_144, action_type="discrete"))
    obs, infos = env.reset()
    obs, reward, terminated, truncated, infos = env.step(actions)   # normalized obs and reward

A training step adds two kernel launches to the env's own (a moments pass and an apply pass), a frozen step
(`training = False`) one.  All per-step state lives on the device, so a loop of step() calls with device-resident
actions can be captured in one CUDA graph and replayed.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .spaces import Box
from .vector import stream_ptr


class RunningMeanStd:
    """SB3's RunningMeanStd as one float64 device tensor `data` = mean, var, count; `mean`, `var` and `count` are views
    of it (mean 0, var 1, count 1e-4 at construction)."""

    def __init__(self, shape: tuple, device):
        self.shape = tuple(shape)
        k = int(np.prod(self.shape))
        self.data = torch.zeros(2 * k + 1, dtype=torch.float64, device=device)
        self.data[k:2 * k] = 1.0
        self.data[2 * k] = 1e-4

    @property
    def mean(self) -> torch.Tensor:
        k = (self.data.numel() - 1) // 2
        return self.data[:k].view(self.shape)

    @property
    def var(self) -> torch.Tensor:
        k = (self.data.numel() - 1) // 2
        return self.data[k:2 * k].view(self.shape)

    @property
    def count(self) -> torch.Tensor:
        return self.data[-1]


class VecNormalize:
    """VectorEnv-compatible wrapper that normalizes the observations and rewards of a batched env with running
    statistics, like Stable-Baselines3's `VecNormalize`:

    - step(): in training, update `obs_rms` with the batch's observations, return
      clip((obs - mean) / sqrt(var + epsilon), +-clip_obs) (float64 arithmetic, float32 result); in training, update the
      discounted returns (returns = returns * gamma + reward) and `ret_rms` with them, return
      clip(reward / sqrt(ret_rms.var + epsilon), +-clip_reward); then zero the returns of finished envs (also when not
      training).
    - reset(): zero the returns and, in training, update `obs_rms` with the reset observations.  A masked reset
      (options={"reset_mask": m}) zeroes the returns of the selected envs only and does NOT update `obs_rms`: the rows
      that were not reset have already been counted by the step that produced them.
    - terminated, truncated and infos pass through untouched (infos["episode"] keeps the raw episode returns); the raw
      observation and reward stay available as `env.obs` / `env.reward`.

    norm_obs=True needs a float32 (num_envs, dim) observation: crypto, traffic, climate and builder with
    flatten_obs=True.  norm_obs=False, norm_reward=True works with every env.  Statistics are per process (each rank
    keeps its own, as in SB3)."""

    def __init__(self, env, norm_obs: bool = True, norm_reward: bool = True, clip_obs: float = 10.0,
                 clip_reward: float = 10.0, gamma: float = 0.99, epsilon: float = 1e-8, training: bool = True):
        space = env.single_observation_space
        if norm_obs and not (isinstance(space, Box) and len(space.shape) == 1 and space.dtype == np.float32):
            raise ValueError("norm_obs=True needs a float32 Box observation of shape (dim,) per env; got "
                             f"{space!r} (use norm_obs=False to normalize only the rewards)")
        self.env = env
        self.lib = _lib.load()
        self.device = env.device
        self.num_envs = env.num_envs
        self.norm_obs, self.norm_reward = bool(norm_obs), bool(norm_reward)
        self.clip_obs, self.clip_reward = float(clip_obs), float(clip_reward)
        self.gamma, self.epsilon = float(gamma), float(epsilon)
        self.training = bool(training)
        n = self.num_envs
        self.dim = int(space.shape[0]) if self.norm_obs else 1
        dev = self.device
        with torch.cuda.device(dev):
            self.obs_rms = RunningMeanStd((self.dim,) if self.norm_obs else (), dev)
            self.ret_rms = RunningMeanStd((), dev)
            self.returns = torch.zeros(n, dtype=torch.float64, device=dev)
            self.obs = torch.zeros(n, self.dim, dtype=torch.float32, device=dev) if self.norm_obs else None
            self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
            ws = int(self.lib.beng_normalize_workspace_bytes(n, self.dim))
            self._workspace = torch.zeros(max(ws, 16), dtype=torch.uint8, device=dev)

    # ------------------------------------------------------------------ VectorEnv surface
    single_observation_space = property(lambda self: self.env.single_observation_space)
    single_action_space = property(lambda self: self.env.single_action_space)
    observation_space = property(lambda self: self.env.observation_space)
    action_space = property(lambda self: self.env.action_space)
    metadata = property(lambda self: self.env.metadata)

    def __getattr__(self, name):
        if name == "env":  # not set yet (during construction)
            raise AttributeError(name)
        return getattr(self.env, name)

    def _normalize(self, obs, reward, terminated, truncated, flags: int, obs_out, update: bool):
        """beng_normalize on the current stream: flags = _lib.NORM_OBS / NORM_REWARD, plus NORM_UPDATE when `update`."""
        if update:
            flags |= _lib.NORM_UPDATE
        if flags & _lib.NORM_OBS:
            if obs.dtype != torch.float32 or obs.shape != (self.num_envs, self.dim) or not obs.is_contiguous():
                raise ValueError(f"the env returned a {tuple(obs.shape)} {obs.dtype} observation; "
                                 f"expected contiguous float32 ({self.num_envs}, {self.dim})")
        ptr = lambda t: None if t is None else t.data_ptr()  # noqa: E731
        params = _lib.NormalizeParams(self.clip_obs, self.clip_reward, self.epsilon, self.gamma, flags, 0)
        io = _lib.NormalizeIO(ptr(obs), ptr(reward), ptr(terminated), ptr(truncated), self.returns.data_ptr(),
                              self.obs_rms.data.data_ptr(), self.ret_rms.data.data_ptr(), self._workspace.data_ptr(),
                              ptr(obs_out), self.reward.data_ptr() if reward is not None else None)
        with torch.cuda.device(self.device):
            rc = self.lib.beng_normalize(C.byref(params), C.byref(io), self.num_envs, self.dim,
                                         stream_ptr(self.device))
        _lib.check(rc, "beng_normalize")

    def reset(self, *, seed=None, options=None):
        """Reset the env -> (normalized obs, infos); see the class docstring for the masked-reset rule."""
        obs, infos = self.env.reset(seed=seed, options=options)
        mask = None if not options else options.get("reset_mask")
        if mask is None:
            self.returns.zero_()
        else:
            self.returns.masked_fill_(torch.as_tensor(mask, device=self.device).reshape(self.num_envs).bool(), 0.0)
        if not self.norm_obs:
            return obs, infos
        # a masked reset normalizes without counting the rows again
        self._normalize(obs, None, None, None, _lib.NORM_OBS, self.obs, self.training and mask is None)
        return self.obs, infos

    def step(self, actions, out_obs: torch.Tensor | None = None):
        """Step the env and normalize -> (obs, reward, terminated, truncated, infos).  `out_obs`: optional contiguous
        float32 (num_envs, dim) CUDA tensor (e.g. a rollout-buffer slot) that receives the normalized observations
        instead of `self.obs`; needs norm_obs=True."""
        if out_obs is not None:
            if not self.norm_obs:
                raise ValueError("out_obs needs norm_obs=True")
            if out_obs.shape != (self.num_envs, self.dim) or out_obs.dtype != torch.float32 \
                    or not out_obs.is_contiguous() or out_obs.device != self.device:
                raise ValueError(f"out_obs must be a contiguous float32 CUDA tensor of shape ({self.num_envs}, {self.dim})")
        obs, reward, terminated, truncated, infos = self.env.step(actions)
        flags = (_lib.NORM_OBS if self.norm_obs else 0) | (_lib.NORM_REWARD if self.norm_reward else 0)
        if flags:
            out = (self.obs if out_obs is None else out_obs) if self.norm_obs else None
            self._normalize(obs if self.norm_obs else None, reward if self.norm_reward else None, terminated,
                            truncated, flags, out, self.training)
        if self.norm_obs:
            obs = out
        return obs, self.reward if self.norm_reward else reward, terminated, truncated, infos

    def close(self, **kwargs):
        self.env.close(**kwargs)

    # ------------------------------------------------------------------ checkpoints
    def _options(self) -> dict:
        return dict(norm_obs=self.norm_obs, norm_reward=self.norm_reward, clip_obs=self.clip_obs,
                    clip_reward=self.clip_reward, gamma=self.gamma, epsilon=self.epsilon, training=self.training)

    def state_dict(self) -> dict:
        """Statistics, discounted returns, options and the wrapped env's state dict."""
        return {"obs_rms": self.obs_rms.data.clone(), "ret_rms": self.ret_rms.data.clone(),
                "returns": self.returns.clone(), "options": self._options(), "env": self.env.state_dict()}

    def load_state_dict(self, sd: dict):
        opts = sd["options"]
        if bool(opts["norm_obs"]) != self.norm_obs or (self.norm_obs and sd["obs_rms"].numel() != self.obs_rms.data.numel()):
            raise ValueError("the state dict was saved with another observation normalization")
        self.obs_rms.data.copy_(sd["obs_rms"])
        self.ret_rms.data.copy_(sd["ret_rms"])
        self.returns.copy_(sd["returns"])
        self.norm_reward, self.training = bool(opts["norm_reward"]), bool(opts["training"])
        self.clip_obs, self.clip_reward = float(opts["clip_obs"]), float(opts["clip_reward"])
        self.gamma, self.epsilon = float(opts["gamma"]), float(opts["epsilon"])
        self.env.load_state_dict(sd["env"])
