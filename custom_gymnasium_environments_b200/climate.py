"""smartclimate on the B200 engine (SURVEY.md section 8f rank 3).

  BatchedSmartClimateEnv   gymnasium.vector.VectorEnv-compatible; N envs stepped by ONE CUDA kernel
                           (csrc/climate.cu) through the C ABI (include/beng.h).
  SmartClimateEnv          the reference's single-instance gym.Env surface
                           (smartclimate_rl-main/smartclimate/env.py:10-128), a 1-env view of the same engine.

The reference's Dict action {'ac_temp': Box(16, 32, (1,)), 'lights': MultiBinary(4)} (env.py:37-41) is kept: batched
actions are {'ac_temp': float32 (n, 1) or (n,), 'lights': int8 (n, 4)}.  The 1440-minute limit is reported as
`terminated` (env.py:107); arithmetic is float64 on the device like the reference's Python floats.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .spaces import Box, Dict, MultiBinary, batch_space
from .vector import _EnvBase, AUTORESET_MODES, _BatchedEnv, as_device_actions, host_source, stream_ptr

OBS_DIM = 9
CLIMATE_STAT_NAMES = ("n_episodes", "sum_return", "sum_length")


def _shaped(x, shape):
    """An action component (tensor, array or list) reshaped to `shape`."""
    return x.reshape(shape) if isinstance(x, torch.Tensor) else np.reshape(x, shape)


class BatchedSmartClimateEnv(_BatchedEnv):
    """N independent SmartClimateEnv instances; state resident in HBM as [field][env] arrays."""

    metadata = {"render_modes": [], "render_fps": 10, "autoreset_mode": "same_step"}
    _reset_fn = "beng_climate_reset"
    _state_tensors = ("_f64", "_i32")
    _stat_names = CLIMATE_STAT_NAMES
    _host_names = ("_ac", "_lights", "obs", "reward", "terminated", "truncated")

    def __init__(self, num_envs: int, max_occupancy: int = 8, comfort_temp_range=(20.0, 24.0),
                 episode_minutes: int = 1440, *, device="cuda", seed: int = 0, env_id_base: int = 0,
                 autoreset_mode="same_step", time_limit_truncation: bool = False, render_mode=None):
        super().__init__(num_envs, device, autoreset_mode, render_mode)
        n = self.num_envs
        self.max_occupancy = int(max_occupancy)
        self.comfort_temp_range = tuple(comfort_temp_range)  # kept for API parity; unused by the reference's dynamics
        self.episode_minutes = int(episode_minutes)

        self.single_action_space = Dict({"ac_temp": Box(16.0, 32.0, (1,), np.float32), "lights": MultiBinary(4)})
        self.single_observation_space = Box(
            np.array([0.0, 0, 0.0, 10.0, 16.0, 0, 0, 0, 0]),
            np.array([50.0, self.max_occupancy, 23.99, 50.0, 32.0, 1, 1, 1, 1]), dtype=np.float32)   # env.py:42-46
        self.action_space = batch_space(self.single_action_space, n)
        self.observation_space = batch_space(self.single_observation_space, n)

        self.params = _lib.ClimateParams(self.max_occupancy, self.episode_minutes,
                                         AUTORESET_MODES[self.autoreset_mode], int(bool(time_limit_truncation)),
                                         int(seed), int(env_id_base))
        dev = self.device
        with torch.cuda.device(dev):
            z = lambda *shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
            self._f64 = z(5, n, dt=torch.float64)   # room_temp, outside_temp, ac_setting, total_reward, energy_usage
            self._i32 = z(4, n, dt=torch.int32)     # people|lights<<8|flags<<16 ; step ; comfort_time ; rng counter
            self.obs = z(n, OBS_DIM, dt=torch.float32)
            self.reward = z(n, dt=torch.float32)
            self.terminated = z(n, dt=torch.bool)
            self.truncated = z(n, dt=torch.bool)
            self.reward64 = z(n, dt=torch.float64)
            self.reward_terms = z(3, n, dt=torch.float64)
            self.ep_return = z(n, dt=torch.float64)
            self.ep_length = z(n, dt=torch.int32)
            self.stats = z(3, dt=torch.float64)
            self._ac = z(n, dt=torch.float32)
            self._lights = z(n, 4, dt=torch.int8)
        self._state = _lib.ClimateState(self._f64.data_ptr(), self._i32.data_ptr())
        self._io = _lib.ClimateIO(self.obs.data_ptr(), self.reward.data_ptr(), self.terminated.data_ptr(),
                                  self.truncated.data_ptr(), self.reward64.data_ptr(), self.reward_terms.data_ptr(),
                                  self.ep_return.data_ptr(), self.ep_length.data_ptr(), self.stats.data_ptr())

    # ------------------------------------------------------------------ state views
    room_temp = property(lambda self: self._f64[0])
    outside_temp = property(lambda self: self._f64[1])
    ac_setting = property(lambda self: self._f64[2])
    total_reward = property(lambda self: self._f64[3])
    energy_usage = property(lambda self: self._f64[4])
    num_people = property(lambda self: self._i32[0] & 0xFF)
    current_step = property(lambda self: self._i32[1])
    comfort_time = property(lambda self: self._i32[2])
    rng_counter = property(lambda self: self._i32[3].to(torch.int64) & 0xFFFFFFFF)

    def _infos(self):
        return {"comfort": self.reward_terms[0], "ac_penalty": self.reward_terms[1],
                "light_penalty": self.reward_terms[2], "comfort_time": self._i32[2], "energy_usage": self._f64[4],
                "step": self._i32[1], "reward64": self.reward64,
                "episode": {"r": self.ep_return, "l": self.ep_length}, "_episode": self.terminated}

    # ------------------------------------------------------------------ VectorEnv API
    # reset(): SmartClimateEnv.reset (env.py:62-70).

    def step(self, actions):
        """One step of every env (env.py:84-117).  actions = {'ac_temp': float32 (n,1)|(n,), 'lights': int8 (n,4)}."""
        self._require_reset()
        n = self.num_envs
        ac, lights = (actions["ac_temp"], actions["lights"]) if isinstance(actions, dict) else actions
        # (n,) / (n, 4) tensors, the usual case, go straight to the upload: no call or torch op per step for them
        ac = ac if isinstance(ac, torch.Tensor) and ac.ndim == 1 else _shaped(ac, (n,))
        lights = lights if isinstance(lights, torch.Tensor) and lights.ndim == 2 else _shaped(lights, (n, 4))
        ac, lights = as_device_actions(ac, self._ac), as_device_actions(lights, self._lights)
        self._call("beng_climate_step", C.byref(self.params), C.byref(self._state), ac.data_ptr(), lights.data_ptr(),
                   C.byref(self._io), self.num_envs, stream_ptr(self.device))
        return self.obs, self.reward, self.terminated, self.truncated, self._infos()

    def step_host(self, actions, *, copy_obs: bool = True, sync: bool = True):
        """step() for callers holding HOST arrays (numpy in, numpy out) through `beng_climate_step_host`."""
        self._require_reset()
        h = self._host_buffers()
        ac, lights = (actions["ac_temp"], actions["lights"]) if isinstance(actions, dict) else actions
        ac, lights = self._host_src = (host_source(ac, h["_ac"]), host_source(lights, h["_lights"]))
        self._call("beng_climate_step_host", C.byref(self.params), C.byref(self._state), self._ac.data_ptr(),
                   self._lights.data_ptr(), C.byref(self._io), self.num_envs, ac.data_ptr(), lights.data_ptr(),
                   h["obs"].data_ptr() if copy_obs else None, h["reward"].data_ptr(), h["terminated"].data_ptr(),
                   h["truncated"].data_ptr(), stream_ptr(self.device))
        if sync:
            self._sync()
        obs = h["obs"].numpy() if copy_obs else self.obs
        return obs, h["reward"].numpy(), h["terminated"].numpy(), h["truncated"].numpy(), {}


class SmartClimateEnv(_EnvBase):
    """Single-instance gym.Env surface of the reference (env.py:10-128) on the CUDA engine: a 1-env
    BatchedSmartClimateEnv with auto-reset disabled; numpy observations, Python floats, the reference's info keys."""

    metadata = {"render_modes": ["human"], "render_fps": 10}

    def __init__(self, max_occupancy: int = 8, comfort_temp_range=(20.0, 24.0), episode_minutes: int = 1440,
                 seed=None, log_level=None, *, device="cuda", env_id: int = 0, **kwargs):
        self.max_occupancy, self.comfort_temp_range, self.episode_minutes = max_occupancy, comfort_temp_range, episode_minutes
        self._vec = BatchedSmartClimateEnv(1, max_occupancy, comfort_temp_range, episode_minutes, device=device,
                                           seed=0 if seed is None else int(seed), env_id_base=env_id,
                                           autoreset_mode="disabled")
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space

    room_temp = property(lambda self: float(self._vec.room_temp.item()))
    num_people = property(lambda self: int(self._vec.num_people.item()))
    current_step = property(lambda self: int(self._vec.current_step.item()))

    def reset(self, *, seed=None, options=None):
        obs, _ = self._vec.reset(seed=seed)
        return obs[0].cpu().numpy().copy(), {}

    def step(self, action):
        act = {"ac_temp": np.asarray(action["ac_temp"], dtype=np.float32).reshape(1),
               "lights": np.asarray(action["lights"], dtype=np.int8).reshape(1, 4)}
        obs, rew, term, trunc, info = self._vec.step(act)
        out = {"comfort": float(info["comfort"].item()), "ac_penalty": float(info["ac_penalty"].item()),
               "light_penalty": float(info["light_penalty"].item()), "comfort_time": int(info["comfort_time"].item()),
               "energy_usage": float(info["energy_usage"].item()), "step": int(info["step"].item())}
        return obs[0].cpu().numpy().copy(), float(info["reward64"].item()), bool(term.item()), False, out

    def render(self, mode: str = "human"):
        return None

    def close(self):
        self._vec.close()
