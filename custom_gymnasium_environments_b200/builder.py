"""world_builder_env on the B200 engine (SURVEY.md section 8f rank 3).

  BatchedWorldBuilderEnv   gymnasium.vector.VectorEnv-compatible; N envs stepped by ONE CUDA kernel
                           (csrc/builder.cu) through the C ABI (include/beng.h).
  WorldBuilderEnv          the reference's single-instance gym.Env surface
                           (world_builder_env/src/environment/world_builder_env.py:10-247), a 1-env view of the engine.

The reference's observation is a Dict {'grid' int8 (G,G), 'resources' float32 (4,), 'population_capacity' float32 (1,),
'win_steps' int32 (1,)} or, with flatten_obs=True, one float32 vector of G*G + 6 values (:71-86, :186-217); both forms are
kept.  There is no time limit: an episode ends by starvation (-100) or after 50 steps at population >= 20 (+100);
`truncated` is always False.  Integer dynamics, bit-exact against the reference.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .spaces import Box, Dict, Discrete, batch_space
from .vector import _EnvBase, AUTORESET_MODES, _BatchedEnv, as_device_actions, host_source, stream_ptr

BUILDING_NAMES = ("farm", "lumberyard", "quarry", "house")
BUILDER_STAT_NAMES = ("n_episodes", "sum_return", "sum_length", "wins")
MAX_POPULATION, WIN_STEPS = 20, 50


class BatchedWorldBuilderEnv(_BatchedEnv):
    """N independent WorldBuilderEnv instances; scalar state as [word][env] int32, the grid doubles as observation."""

    metadata = {"render_modes": [], "render_fps": 4, "autoreset_mode": "same_step"}
    _reset_fn = "beng_builder_reset"
    _state_tensors = ("_words", "grid")
    _stat_names = BUILDER_STAT_NAMES
    _host_names = ("_actions", "grid", "resources", "population_capacity", "win_steps", "reward", "terminated",
                   "_delta_dev")
    _mirror, _apply_delta_fn = "grid", "beng_builder_apply_obs_delta"

    def __init__(self, num_envs: int, grid_size: int = 10, render_mode=None, flatten_obs: bool = False, *,
                 device="cuda", seed: int = 0, env_id_base: int = 0, autoreset_mode="same_step",
                 debug_checks: bool = False):
        super().__init__(num_envs, device, autoreset_mode, render_mode)
        n = self.num_envs
        self.grid_size = G = int(grid_size)
        self.flatten_obs = bool(flatten_obs)
        self.debug_checks = bool(debug_checks)

        self.single_action_space = Discrete(5)                                            # :60
        if self.flatten_obs:
            self.single_observation_space = Box(0.0, 1000.0, (G * G + 6,), np.float32)    # :71-78
        else:
            self.single_observation_space = Dict({                                        # :80-85
                "grid": Box(0, 4, (G, G), np.int8), "resources": Box(0.0, 1000.0, (4,), np.float32),
                "population_capacity": Box(0.0, 100.0, (1,), np.float32), "win_steps": Box(0, WIN_STEPS, (1,), np.int32)})
        self.action_space = batch_space(self.single_action_space, n)
        self.observation_space = batch_space(self.single_observation_space, n)

        self.params = _lib.BuilderParams(G, AUTORESET_MODES[self.autoreset_mode], int(seed), int(env_id_base))
        dev = self.device
        with torch.cuda.device(dev):
            z = lambda *shape, dt: torch.zeros(shape, dtype=dt, device=dev)  # noqa: E731
            self._words = z(10, n, dt=torch.int32)
            self.grid = z(n, G, G, dt=torch.int8)
            self.resources = z(n, 4, dt=torch.float32)
            self.population_capacity = z(n, 1, dt=torch.float32)
            self.win_steps = z(n, 1, dt=torch.int32)
            self.flat_obs = z(n, G * G + 6, dt=torch.float32) if self.flatten_obs else None
            self.reward = z(n, dt=torch.float32)
            self.terminated = z(n, dt=torch.bool)
            self.truncated = z(n, dt=torch.bool)
            self.ep_return = z(n, dt=torch.int32)
            self.ep_length = z(n, dt=torch.int32)
            self.stats = z(4, dt=torch.int64)
            self.invalid_count = z(1, dt=torch.int32)
            self._actions = z(n, dt=torch.int64)
        self._state = _lib.BuilderState(self._words.data_ptr())
        self._io = _lib.BuilderIO(self.grid.data_ptr(), self.resources.data_ptr(), self.population_capacity.data_ptr(),
                                  self.win_steps.data_ptr(), self.flat_obs.data_ptr() if self.flatten_obs else None,
                                  self.reward.data_ptr(), self.terminated.data_ptr(), self.truncated.data_ptr(),
                                  self.ep_return.data_ptr(), self.ep_length.data_ptr(), self.stats.data_ptr(),
                                  self.invalid_count.data_ptr())

    # ------------------------------------------------------------------ state views
    food = property(lambda self: self._words[0])
    wood = property(lambda self: self._words[1])
    stone = property(lambda self: self._words[2])
    population = property(lambda self: self._words[3])
    steps = property(lambda self: self._words[6])
    reached_win_population = property(lambda self: ((self._words[7] >> 16) & 1).bool())
    rng_counter = property(lambda self: self._words[8].to(torch.int64) & 0xFFFFFFFF)

    @property
    def building_counts(self):
        """(n, 4) counts of farm, lumberyard, quarry, house."""
        c = self._words[5]
        return torch.stack([(c >> (8 * b)) & 0xFF for b in range(4)], dim=1)

    def _obs(self):
        if self.flatten_obs:
            return self.flat_obs
        return {"grid": self.grid, "resources": self.resources, "population_capacity": self.population_capacity,
                "win_steps": self.win_steps}

    def _infos(self):
        return {"steps": self._words[6], "win_steps": self.win_steps[:, 0], "population": self._words[3],
                "population_capacity": self._words[4],
                "episode": {"r": self.ep_return, "l": self.ep_length}, "_episode": self.terminated}

    # ------------------------------------------------------------------ VectorEnv API
    def _reset_result(self):
        """WorldBuilderEnv.reset (:99-123) -> (obs, infos)."""
        return self._obs(), self._infos()

    def step(self, actions):
        """One step of every env (:125-166).  actions: int64 (n,), 0 pass / 1 farm / 2 lumberyard / 3 quarry / 4 house."""
        self._require_reset()
        act = as_device_actions(actions, self._actions)
        self._mirror_valid = False
        self._call("beng_builder_step", C.byref(self.params), C.byref(self._state), act.data_ptr(), C.byref(self._io),
                   self.num_envs, stream_ptr(self.device))
        if self.debug_checks:
            n_bad = int(self.invalid_count.item())
            if n_bad:
                self.invalid_count.zero_()
                raise ValueError(f"Invalid action: {n_bad} action(s) outside Discrete(5)")  # :135-136
        return self._obs(), self.reward, self.terminated, self.truncated, self._infos()

    def step_host(self, actions, *, copy_obs: bool = True, sync: bool = True, delta_obs: bool = False):
        """step() for callers holding HOST arrays (numpy in, numpy out) through `beng_builder_step_host`.

        delta_obs=True keeps the pinned grid buffer as a mirror of the device grid and brings it up to date from one
        4-byte change record per env (`beng_builder_step_host_delta` + `beng_builder_apply_obs_delta`) instead of
        copying G*G bytes per env.  When the mirror is not current (first call, or reset()/step()/load_state_dict()/
        step_host(copy_obs=False) since the last step_host), the call copies the grid in full instead.  The returned
        obs['grid'] is read-only.  Needs sync=True and copy_obs=True.
        """
        delta = self._mirror_begin(delta_obs, sync, copy_obs)
        h = self._host_buffers()
        src = self._host_src = host_source(actions, h["_actions"])
        head = (C.byref(self.params), C.byref(self._state), self._actions.data_ptr(), C.byref(self._io),
                self.num_envs, src.data_ptr())
        results = (h["resources"].data_ptr(), h["population_capacity"].data_ptr(), h["win_steps"].data_ptr(),
                   h["reward"].data_ptr(), h["terminated"].data_ptr(), stream_ptr(self.device))
        if delta:
            self._call("beng_builder_step_host_delta", *head, self._delta_dev.data_ptr(), h["_delta_dev"].data_ptr(),
                       *results)
        else:
            self._call("beng_builder_step_host", *head, h["grid"].data_ptr() if copy_obs else None, *results)
        if sync:
            self._sync()
        obs = {"grid": self._mirror_end(delta, delta_obs, copy_obs), "resources": h["resources"].numpy(),
               "population_capacity": h["population_capacity"].numpy(), "win_steps": h["win_steps"].numpy()}
        return obs, h["reward"].numpy(), h["terminated"].numpy(), np.zeros(self.num_envs, dtype=bool), {}


class WorldBuilderEnv(_EnvBase):
    """Single-instance gym.Env surface of the reference (world_builder_env.py:10-247) on the CUDA engine: a 1-env
    BatchedWorldBuilderEnv with auto-reset disabled; numpy observations, Python numbers, the reference's info keys."""

    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 4}

    def __init__(self, grid_size: int = 10, render_mode=None, flatten_obs: bool = False, *, device="cuda",
                 seed: int = 0, env_id: int = 0):
        self.grid_size, self.render_mode, self.flatten_obs = grid_size, render_mode, flatten_obs
        self.MAX_POPULATION, self.WIN_STEPS = MAX_POPULATION, WIN_STEPS
        self._vec = BatchedWorldBuilderEnv(1, grid_size, flatten_obs=flatten_obs, device=device, seed=seed,
                                           env_id_base=env_id, autoreset_mode="disabled")
        self.action_space = self._vec.single_action_space
        self.observation_space = self._vec.single_observation_space

    def _obs(self):
        v = self._vec
        if self.flatten_obs:
            return v.flat_obs[0].cpu().numpy().copy()
        return {"grid": v.grid[0].cpu().numpy().copy(), "resources": v.resources[0].cpu().numpy().copy(),
                "population_capacity": v.population_capacity[0].cpu().numpy().copy(),
                "win_steps": v.win_steps[0].cpu().numpy().copy()}

    def _get_info(self):  # :219-231
        v = self._vec
        w = v._words[:, 0].tolist()
        return {"steps": w[6], "win_steps": w[7] & 0xFFFF, "reached_win_population": bool((w[7] >> 16) & 1),
                "resources": {"food": w[0], "wood": w[1], "stone": w[2]}, "population": w[3],
                "population_capacity": w[4],
                "building_counts": {name: (w[5] >> (8 * b)) & 0xFF for b, name in enumerate(BUILDING_NAMES)}}

    def reset(self, seed=None, options=None):
        self._vec.reset(seed=seed)
        return self._obs(), self._get_info()

    def step(self, action):
        if not self.action_space.contains(action):
            raise ValueError(f"Invalid action {action}. Action space is {self.action_space}")  # :135-136
        _, rew, term, _, _ = self._vec.step(np.array([action], dtype=np.int64))
        return self._obs(), int(rew.item()), bool(term.item()), False, self._get_info()

    def render(self):
        return None

    def close(self):
        self._vec.close()
