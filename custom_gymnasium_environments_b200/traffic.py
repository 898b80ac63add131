"""traffic_management_env on the B200 engine.

  BatchedTrafficManagementEnv   gymnasium.vector.VectorEnv-compatible; N envs stepped by ONE CUDA kernel
                                (csrc/traffic.cu) through the C ABI (include/beng.h).
  TrafficManagementEnv          the reference's single-instance gym.Env surface
                                (traffic_management_env/environment.py:31-384), a 1-env view of the same engine.

Reference behaviour kept on purpose (SURVEY.md section 0): the 1000-step limit is `terminated`; the reward is
CUMULATIVE (it sums lifetime counters every step, environment.py:287-311); vehicles never move -- they wait in their
start intersection's queue and, once released, either leave or stay in `self.vehicles` forever, so the vehicle list
saturates at `max_vehicles` and spawning stops (fact 9).  Dynamics are integer and reproduce the reference bit for
bit; reward/observation are float64 expressions of those integers cast to float32.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .spaces import Box, MultiDiscrete, batch_space
from .vector import _EnvBase, AUTORESET_MODES, _BatchedEnv, as_device_actions, host_source, stream_ptr

# config.py:6-12,23
DEFAULT_GRID_SIZE = (5, 5)
DEFAULT_NUM_INTERSECTIONS = 9
MAX_VEHICLES = 50
DEFAULT_SPAWN_RATE = 0.3
MAX_TIMESTEPS = 1000
LIGHT_PHASES = ("NS_GREEN", "NS_YELLOW", "EW_GREEN", "EW_YELLOW")   # config.py:17
DIRECTIONS = ("NORTH", "EAST", "SOUTH", "WEST")                      # utils.py:16-21
TRAFFIC_STAT_NAMES = ("n_episodes", "sum_return", "sum_length")


class BatchedTrafficManagementEnv(_BatchedEnv):
    """N independent TrafficManagementEnv instances; state resident in HBM as [field][env] integer arrays."""

    metadata = {"render_modes": [], "render_fps": 10, "autoreset_mode": "same_step"}
    _reset_fn = "beng_traffic_reset"
    _state_tensors = ("_light", "_passed", "_waiting", "_qmeta", "_qwait", "_misc", "_total_reward")
    _stat_names = TRAFFIC_STAT_NAMES
    _host_names = ("_actions", "obs", "reward", "terminated", "truncated")

    def __init__(self, num_envs: int, grid_size=DEFAULT_GRID_SIZE, num_intersections: int = DEFAULT_NUM_INTERSECTIONS,
                 max_vehicles: int = MAX_VEHICLES, spawn_rate: float = DEFAULT_SPAWN_RATE, render_mode=None, *,
                 device="cuda", seed: int = 0, env_id_base: int = 0, autoreset_mode="same_step",
                 max_timesteps: int = MAX_TIMESTEPS, time_limit_truncation: bool = False):
        super().__init__(num_envs, device, autoreset_mode, render_mode)
        n = self.num_envs
        self.grid_size = tuple(grid_size)
        self.num_intersections = ni = min(int(num_intersections), self.grid_size[0] * self.grid_size[1])  # :82
        self.max_vehicles = int(max_vehicles)
        self.spawn_rate = float(spawn_rate)
        self.obs_dim = ni * 14 + 4                                            # environment.py:116-122

        self.single_action_space = MultiDiscrete([3] * ni)                    # :113
        self.single_observation_space = Box(0.0, np.inf, (self.obs_dim,), np.float32)   # :124-129
        self.action_space = batch_space(self.single_action_space, n)
        self.observation_space = batch_space(self.single_observation_space, n)

        self.params = _lib.TrafficParams(self.grid_size[0], self.grid_size[1], int(num_intersections),
                                         self.max_vehicles, self.spawn_rate, int(max_timesteps),
                                         AUTORESET_MODES[self.autoreset_mode], int(bool(time_limit_truncation)), 0,
                                         int(seed), int(env_id_base))
        dev = self.device
        with torch.cuda.device(dev):
            z = lambda *shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
            self._light = z(ni, n, dt=torch.int16)
            self._passed = z(ni, n, dt=torch.int32)
            self._waiting = z(ni, n, dt=torch.int32)
            self._qmeta = z(ni * 2, n, dt=torch.int32)  # rows 2i / 2i+1: queue lengths / loop-back counts, a byte per direction
            self._qwait = z(ni * 4, n, dt=torch.int32)
            self._misc = z(3, n, dt=torch.int32)
            self._total_reward = z(n, dt=torch.float64)
            self.obs = z(n, self.obs_dim, dt=torch.float32)
            self.reward = z(n, dt=torch.float32)
            self.terminated = z(n, dt=torch.bool)
            self.truncated = z(n, dt=torch.bool)
            self.reward64 = z(n, dt=torch.float64)
            self.ep_return = z(n, dt=torch.float64)
            self.ep_length = z(n, dt=torch.int32)
            self.stats = z(3, dt=torch.float64)
            self.timestep = z(n, dt=torch.int32)  # info["timestep"], written by the kernel (no per-step host-side op)
            self._actions = z(n, ni, dt=torch.int64)
        self._state = _lib.TrafficState(self._light.data_ptr(), self._passed.data_ptr(), self._waiting.data_ptr(),
                                        self._qmeta.data_ptr(), self._qwait.data_ptr(), self._misc.data_ptr(),
                                        self._total_reward.data_ptr())
        self._io = _lib.TrafficIO(self.obs.data_ptr(), self.reward.data_ptr(), self.terminated.data_ptr(),
                                  self.truncated.data_ptr(), self.reward64.data_ptr(), self.ep_return.data_ptr(),
                                  self.ep_length.data_ptr(), self.stats.data_ptr(), self.timestep.data_ptr())
        self._infos_cache = None

    # ------------------------------------------------------------------ state views (all (n, ...) tensors)
    @property
    def current_timestep(self):
        return self._misc[0] & 0xFFFF

    @property
    def num_vehicles(self):
        """len(self.vehicles) of every env."""
        return self._misc[1]

    @property
    def rng_counter(self):
        return self._misc[2].to(torch.int64) & 0xFFFFFFFF

    @property
    def total_reward(self):
        return self._total_reward

    @property
    def light_phase(self):
        """(n, ni) phase codes, index into LIGHT_PHASES."""
        return (self._light.to(torch.int32) & 0xFF).t()

    @property
    def light_timer(self):
        return ((self._light.to(torch.int32) >> 8) & 0xFF).t()

    @property
    def vehicles_passed(self):
        return self._passed.t()

    @property
    def total_waiting_time(self):
        return self._waiting.t()

    @property
    def queue_lengths(self):
        """(n, ni, 4) queue lengths, directions N, E, S, W."""
        packed = self._qmeta[0::2].t().unsqueeze(-1)  # (n, ni, 1) int32, one byte lane per direction
        return (packed >> torch.tensor([0, 8, 16, 24], device=packed.device, dtype=torch.int32)) & 0xFF

    @property
    def queue_waiting_sums(self):
        return self._qwait.t().reshape(self.num_envs, self.num_intersections, 4)

    def metrics(self) -> dict:
        """calculate_traffic_metrics (utils.py:251-267) for every env, computed on the device on demand."""
        passed = self._passed.sum(0).double()
        waiting = self._waiting.sum(0).double()
        queued = self.queue_lengths.sum((1, 2)).double()
        ni = float(self.num_intersections)
        return {"total_vehicles_passed": passed, "total_waiting_time": waiting,
                "average_waiting_time": waiting / passed.clamp(min=1), "total_queue_length": queued,
                "average_queue_length": queued / ni, "throughput": passed / ni}

    def _infos(self):
        # every value is a tensor the kernel writes in place: building the dict launches nothing
        if self._infos_cache is None:
            self._infos_cache = {"total_reward": self._total_reward, "reward64": self.reward64,
                                 "episode": {"r": self.ep_return, "l": self.ep_length}, "_episode": self.terminated,
                                 "timestep": self.timestep, "num_vehicles": self._misc[1]}
        return dict(self._infos_cache)

    # ------------------------------------------------------------------ VectorEnv API
    def _reset_result(self):
        """TrafficManagementEnv.reset (environment.py:141-166) -> (obs, infos).  reset() itself draws nothing (the
        reference seeds the global RNGs, :145-147)."""
        return self.obs, self._infos()

    def step(self, actions):
        """One step of every env (environment.py:168-203).  actions: int64 (n, ni), 0 keep / 1 NS_GREEN / 2 EW_GREEN."""
        self._require_reset()
        act = as_device_actions(actions, self._actions)
        self._call("beng_traffic_step", C.byref(self.params), C.byref(self._state), act.data_ptr(), C.byref(self._io),
                   self.num_envs, stream_ptr(self.device))
        return self.obs, self.reward, self.terminated, self.truncated, self._infos()

    def step_host(self, actions, *, copy_obs: bool = True, sync: bool = True):
        """step() for callers holding HOST arrays (numpy in, numpy out) through `beng_traffic_step_host`."""
        self._require_reset()
        h = self._host_buffers()
        src = self._host_src = host_source(actions, h["_actions"])
        self._call("beng_traffic_step_host", C.byref(self.params), C.byref(self._state), self._actions.data_ptr(),
                   C.byref(self._io), self.num_envs, src.data_ptr(), h["obs"].data_ptr() if copy_obs else None,
                   h["reward"].data_ptr(), h["terminated"].data_ptr(), h["truncated"].data_ptr(),
                   stream_ptr(self.device))
        if sync:
            self._sync()
        obs = h["obs"].numpy() if copy_obs else self.obs
        return obs, h["reward"].numpy(), h["terminated"].numpy(), h["truncated"].numpy(), {}


class TrafficManagementEnv(_EnvBase):
    """Single-instance gym.Env surface of the reference (environment.py:31-384) on the CUDA engine: a 1-env
    BatchedTrafficManagementEnv with auto-reset disabled; numpy observations, Python floats and the reference's
    info dict (timestep, num_vehicles, total_reward, metrics, intersection_states)."""

    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 10}

    def __init__(self, grid_size=DEFAULT_GRID_SIZE, num_intersections: int = DEFAULT_NUM_INTERSECTIONS,
                 max_vehicles: int = MAX_VEHICLES, spawn_rate: float = DEFAULT_SPAWN_RATE, render_mode=None, *,
                 device="cuda", seed: int = 0, env_id: int = 0):
        self._vec = BatchedTrafficManagementEnv(1, grid_size, num_intersections, max_vehicles, spawn_rate,
                                                device=device, seed=seed, env_id_base=env_id,
                                                autoreset_mode="disabled")
        self.grid_size, self.num_intersections = self._vec.grid_size, self._vec.num_intersections
        self.max_vehicles, self.spawn_rate, self.render_mode = max_vehicles, spawn_rate, render_mode
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space

    current_timestep = property(lambda self: int(self._vec.current_timestep.item()))
    total_reward = property(lambda self: float(self._vec.total_reward.item()))

    def _get_info(self):  # environment.py:365-384
        v = self._vec
        m = {k: float(t.item()) for k, t in v.metrics().items()}
        for k in ("total_vehicles_passed", "total_waiting_time", "total_queue_length"):
            m[k] = int(m[k])
        phase = v.light_phase[0].tolist()
        ql = v.queue_lengths[0].tolist()
        passed, waiting = v.vehicles_passed[0].tolist(), v.total_waiting_time[0].tolist()
        return {"timestep": self.current_timestep, "num_vehicles": int(v.num_vehicles.item()),
                "total_reward": self.total_reward, "metrics": m,
                "intersection_states": [
                    {"id": i, "light_phase": LIGHT_PHASES[phase[i]],
                     "queue_lengths": dict(zip(DIRECTIONS, ql[i])), "vehicles_passed": passed[i],
                     "total_waiting_time": waiting[i]} for i in range(self.num_intersections)]}

    def reset(self, seed=None, options=None):
        obs, _ = self._vec.reset(seed=seed)
        return obs[0].cpu().numpy().copy(), self._get_info()

    def step(self, action):
        act = np.asarray(action, dtype=np.int64).reshape(1, self.num_intersections)
        obs, rew, term, trunc, _ = self._vec.step(act)
        return (obs[0].cpu().numpy().copy(), float(self._vec.reward64.item()), bool(term.item()), False,
                self._get_info())

    def render(self):
        return None

    def close(self):
        self._vec.close()
