"""float64 NumPy restatement of Stable-Baselines3's VecNormalize semantics, the reference the tests hold
custom_gymnasium_environments_b200.VecNormalize to.  Test-only: the product never imports it.

It is fed the raw batches the wrapped env produced (observation, reward, terminated, truncated) and returns what the
wrapper must return for them.
"""
from __future__ import annotations

import numpy as np


class RunningMeanStd:
    """mean 0, var 1, count 1e-4; update() merges a batch of rows with Chan's parallel update."""

    def __init__(self, shape=()):
        self.mean = np.zeros(shape, np.float64)
        self.var = np.ones(shape, np.float64)
        self.count = 1e-4

    def update(self, x):
        x = np.asarray(x, np.float64)
        self.update_from_moments(np.mean(x, axis=0), np.var(x, axis=0), x.shape[0])

    def update_from_moments(self, b_mean, b_var, n):
        delta = b_mean - self.mean
        tot = self.count + n
        self.mean = self.mean + delta * n / tot
        m2 = self.var * self.count + b_var * n + np.square(delta) * self.count * n / tot
        self.var = m2 / tot
        self.count = tot


class VecNormalizeOracle:
    def __init__(self, num_envs, obs_dim=None, norm_obs=True, norm_reward=True, clip_obs=10.0, clip_reward=10.0,
                 gamma=0.99, epsilon=1e-8, training=True):
        self.norm_obs, self.norm_reward = norm_obs, norm_reward
        self.clip_obs, self.clip_reward, self.gamma, self.epsilon = clip_obs, clip_reward, gamma, epsilon
        self.training = training
        self.obs_rms = RunningMeanStd((obs_dim,) if norm_obs else ())
        self.ret_rms = RunningMeanStd(())
        self.returns = np.zeros(num_envs, np.float64)

    def normalize_obs(self, obs):
        if not self.norm_obs:
            return obs
        x = (np.asarray(obs, np.float64) - self.obs_rms.mean) / np.sqrt(self.obs_rms.var + self.epsilon)
        return np.clip(x, -self.clip_obs, self.clip_obs).astype(np.float32)

    def normalize_reward(self, reward):
        if not self.norm_reward:
            return reward
        x = np.asarray(reward, np.float64) / np.sqrt(self.ret_rms.var + self.epsilon)
        return np.clip(x, -self.clip_reward, self.clip_reward).astype(np.float32)

    def step(self, obs, reward, terminated, truncated):
        """-> (normalized obs, normalized reward)."""
        if self.training and self.norm_obs:
            self.obs_rms.update(obs)
        out_obs = self.normalize_obs(obs)
        if self.training and self.norm_reward:
            self.returns = self.returns * self.gamma + np.asarray(reward, np.float64)
            self.ret_rms.update(self.returns)
        out_rew = self.normalize_reward(reward)
        self.returns[np.asarray(terminated, bool) | np.asarray(truncated, bool)] = 0.0
        return out_obs, out_rew

    def reset(self, obs, mask=None):
        """-> normalized obs.  A masked reset zeroes the selected returns and does not update obs_rms."""
        if mask is None:
            self.returns[:] = 0.0
            if self.training and self.norm_obs:
                self.obs_rms.update(obs)
        else:
            self.returns[np.asarray(mask, bool)] = 0.0
        return self.normalize_obs(obs)
