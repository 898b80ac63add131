"""snake_env_classic on the B200 engine.

  BatchedSnakeEnv   gymnasium.vector.VectorEnv-compatible; N envs stepped by ONE CUDA kernel
                    (csrc/snake.cu) through the C ABI (include/beng.h).
  SnakeEnvClassic   the reference's single-instance gym.Env surface
                    (snake_env_classic/snake_env.py:9-143), a 1-env view of the same engine.

Semantics follow the reference exactly (SURVEY.md section 0): the time limit is reported as
`terminated` (snake_env.py:112-119), `truncated` is always False, the death step mutates nothing
but the direction (snake_env.py:88-94), a non-eating step has reward 0.
"""
from __future__ import annotations

import ctypes as C

import numpy as np
import torch

from . import _lib
from .spaces import Box, Discrete, batch_space
from .vector import _EnvBase, AUTORESET_MODES, LazyInfos, _BatchedEnv, as_device_actions, host_source, stream_ptr

STAT_NAMES = ("n_episodes", "sum_return", "sum_length", "sum_score", "max_score")


class BatchedSnakeEnv(_BatchedEnv):
    """N independent SnakeEnvClassic instances, state resident in HBM as structure-of-arrays.

    step() returns CUDA tensors that are views of persistent buffers, valid until the next
    step()/reset() (like Gymnasium's `copy=False`).  Global env ids are
    env_id_base + [0, num_envs): the trajectory of a given global id does not depend on how
    envs are sharded over GPUs.
    """

    metadata = {"render_modes": ["rgb_array"], "render_fps": 10, "autoreset_mode": "same_step"}
    _reset_fn = "beng_snake_reset"
    _state_tensors = ("_core", "_ring")
    _stat_names = STAT_NAMES
    _host_names = ("_actions", "obs", "reward", "terminated", "truncated", "_score", "_snake_length", "_delta_dev")
    _mirror, _apply_delta_fn = "obs", "beng_snake_apply_obs_delta"

    def __init__(self, num_envs: int, grid_size: int = 20, render_mode=None, *, device="cuda", seed: int = 0,
                 env_id_base: int = 0, autoreset_mode="same_step", max_steps: int = 1000, debug_checks: bool = False,
                 materialize_info: bool = False, time_limit_truncation: bool = False):
        super().__init__(num_envs, device, autoreset_mode, render_mode)
        self.grid_size = int(grid_size)
        self.max_steps = int(max_steps)
        self.debug_checks = bool(debug_checks)
        # info["score"] / info["snake_length"] are derivable from the state record (score == length - 1).  By default
        # they are computed on access instead of being written to HBM every step (8 B per env-step);
        # materialize_info=True makes the kernel write them (the host-buffer path always does).
        self.materialize_info = bool(materialize_info)

        G, n, dev = self.grid_size, self.num_envs, self.device
        self.single_action_space = Discrete(4)                                   # snake_env.py:26
        self.single_observation_space = Box(0, 2, (G, G), np.int8)              # snake_env.py:30-32
        self.action_space = batch_space(self.single_action_space, n)
        self.observation_space = batch_space(self.single_observation_space, n)

        # time_limit_truncation=True mirrors gym.make(): the TimeLimit wrapper ALSO reports truncated=True at max_steps
        self.params = _lib.SnakeParams(G, self.max_steps, AUTORESET_MODES[self.autoreset_mode],
                                       int(bool(time_limit_truncation)), int(seed),
                                       int(env_id_base))
        with torch.cuda.device(dev):
            # state (SoA)
            self._core = torch.zeros((n, 4), dtype=torch.int32, device=dev)       # 16 B record per env
            self._ring = torch.zeros((n, G * G), dtype=torch.int16, device=dev)   # body cells (u16)
            # outputs
            self.obs = torch.zeros((n, G, G), dtype=torch.int8, device=dev)
            self.reward = torch.zeros(n, dtype=torch.float32, device=dev)
            self.terminated = torch.zeros(n, dtype=torch.bool, device=dev)
            self.truncated = torch.zeros(n, dtype=torch.bool, device=dev)
            self._score = torch.zeros(n, dtype=torch.int32, device=dev)
            self._snake_length = torch.zeros(n, dtype=torch.int32, device=dev)
            self.ep_return = torch.zeros(n, dtype=torch.float32, device=dev)
            self.ep_length = torch.zeros(n, dtype=torch.int32, device=dev)
            self.ep_score = torch.zeros(n, dtype=torch.int32, device=dev)
            # {count0, count1, parity, arrivals}: each launch counts into count[parity], zeroes the other counter and
            # flips the parity itself (beng.h), so a step's arguments never change and a CUDA graph can capture it
            self._done_counts = torch.zeros(4, dtype=torch.int32, device=dev)
            self._parity = 0  # (not used by the class; callers that drive the C functions through _make_io flip it)
            self.done_env = torch.zeros(n, dtype=torch.int32, device=dev)
            self.stats = torch.zeros(5, dtype=torch.int64, device=dev)
            self.invalid_count = torch.zeros(1, dtype=torch.int32, device=dev)
            self._actions = torch.zeros(n, dtype=torch.int64, device=dev)
            self.stats[4] = torch.iinfo(torch.int64).min
        self._state = _lib.SnakeState(self._core.data_ptr(), self._ring.data_ptr())
        self._ios = [self._make_io(self.obs)]
        self._ios_full = [self._make_io(self.obs, with_info=True)]
        self._info_fresh = True
        # True while self.obs holds the observation the last reset or step wrote, so that step() may patch it in place
        self._obs_current = False

    # ------------------------------------------------------------------ plumbing
    def _make_io(self, obs: torch.Tensor, parity: int = 0, with_info: bool | None = None) -> "_lib.SnakeIO":
        """The io block of a launch writing `obs`.  Both counter pointers name the self-managed counter block, so
        `parity` is not used: the kernels pick the counter themselves."""
        cnt = self._done_counts.data_ptr()
        info = self.materialize_info if with_info is None else with_info
        return _lib.SnakeIO(obs.data_ptr(), self.reward.data_ptr(), self.terminated.data_ptr(),
                            self.truncated.data_ptr(), self._score.data_ptr() if info else None,
                            self._snake_length.data_ptr() if info else None,
                            self.ep_return.data_ptr(), self.ep_length.data_ptr(), self.ep_score.data_ptr(),
                            cnt, self.done_env.data_ptr(), cnt,
                            self.stats.data_ptr(), self.invalid_count.data_ptr())

    def _next_io(self, full: bool = False):
        """The io block of this step (`full`: with the info outputs)."""
        self._info_fresh = full or self.materialize_info
        return (self._ios_full if full else self._ios)[0]

    @property
    def snake_length(self) -> torch.Tensor:
        """info["snake_length"] of every env (int32), from the kernel's output or derived from the state record."""
        if self._info_fresh:
            return self._snake_length
        return (self._core[:, 1] >> 16) & 0xFFFF

    @property
    def score(self) -> torch.Tensor:
        """info["score"]: always length - 1 (snake_env.py:57,102 vs :97,107)."""
        if self._info_fresh:
            return self._score
        return self.snake_length - 1

    @property
    def done_count(self) -> torch.Tensor:
        """(1,) int32: the number of envs the last step listed in `done_env`, read lazily on the device (count[parity ^ 1]
        of the counter block; no synchronisation)."""
        return self._done_counts[(self._done_counts[2:3] ^ 1).long()]

    def _infos(self):
        info = LazyInfos({"episode": {"r": self.ep_return, "l": self.ep_length, "score": self.ep_score},
                          "_episode": self.terminated})
        info.lazy["score"] = lambda: self.score
        info.lazy["snake_length"] = lambda: self.snake_length
        return info

    # ------------------------------------------------------------------ VectorEnv API
    def _reset_io(self):
        return self._ios_full[0]

    def _reset_result(self):
        """SnakeEnvClassic.reset (snake_env.py:49-65) -> (obs, infos).  (The reference ignores `seed` for food
        placement -- it draws from the global `random`, SURVEY.md section 3.1.)"""
        self._info_fresh = True
        self._obs_current = True  # the reset kernel writes every row
        return self.obs, {"score": self._score, "snake_length": self._snake_length}

    def load_state_dict(self, sd: dict):
        super().load_state_dict(sd)
        self._obs_current = False  # `obs` is not part of the state dict

    def step(self, actions, out_obs: torch.Tensor | None = None):
        """One step of every env (snake_env.py:67-119) -> (obs, rewards, terminations, truncations, infos).

        `actions`: int64 tensor/array of shape (num_envs,) with values 0..3 (CUDA int64 is zero-copy).
        `out_obs`: optional (num_envs, G, G) int8 CUDA tensor to receive the observations (e.g. a slice
        of a rollout buffer) instead of the persistent `self.obs`.

        Without `out_obs`, `self.obs` is engine state, like the world-builder's grid: while it holds the
        previous observation, the step patches only the cells that change (`beng_snake_step_inplace`) and
        reads it back for the self-collision test and the food placement.  Do not write into the returned
        tensor: clone it, or pass `out_obs=`, to keep a copy you can change.  Every `out_obs=` call
        composes full rows into that buffer.

        One kernel launch with the same arguments every call (the finished-env counters are managed on the
        device), so a loop of step() calls with device-resident actions can be captured once with
        torch.cuda.graph and replayed.  Captured steps without `out_obs` patch `self.obs` in place: replay
        them only while `self.obs` is current, i.e. not after a step(out_obs=...), step_host(copy_obs=False)
        or load_state_dict() (eager step() calls between replays are fine).  debug_checks=True reads the
        invalid-action count back, which synchronises and cannot be captured.
        """
        self._require_reset()
        act = as_device_actions(actions, self._actions)
        io, obs = self._next_io(), self.obs
        fn = "beng_snake_step_inplace" if self._obs_current else "beng_snake_step"
        if out_obs is not None:
            if out_obs.shape != self.obs.shape or out_obs.dtype != torch.int8 or not out_obs.is_contiguous() \
                    or out_obs.device != self.device:
                raise ValueError("out_obs must be a contiguous int8 CUDA tensor of shape (num_envs, G, G)")
            io, obs, fn = self._make_io(out_obs), out_obs, "beng_snake_step"
        self._mirror_valid = self._obs_current = False
        self._call(fn, C.byref(self.params), C.byref(self._state), act.data_ptr(), C.byref(io), self.num_envs,
                   stream_ptr(self.device))
        self._obs_current = obs.data_ptr() == self.obs.data_ptr()
        if self.debug_checks:
            self._raise_on_invalid()
        return obs, self.reward, self.terminated, self.truncated, self._infos()

    def _raise_on_invalid(self):
        n_bad = int(self.invalid_count.item())
        if n_bad:
            self.invalid_count.zero_()
            raise ValueError(f"Invalid action: {n_bad} action(s) outside Discrete(4)")  # snake_env.py:69-70

    # ------------------------------------------------------------------ host-buffer path (numpy in / numpy out)
    def step_host(self, actions, *, copy_obs: bool = True, sync: bool = True, delta_obs: bool = False):
        """step() for callers holding HOST arrays, like users of the reference's numpy API.

        Enqueues H2D(actions) -> kernel -> D2H(results) through `beng_snake_step_host` and (by
        default) waits; returns numpy views of pinned host buffers (valid until the next call).
        copy_obs=False leaves the observations in HBM (obs returned is the CUDA tensor).

        delta_obs=True keeps the pinned observation buffer as a mirror of the device observations
        and brings it up to date from one 4-byte change record per env (`beng_snake_step_host_delta`
        + `beng_snake_apply_obs_delta`) instead of copying G*G bytes per env.  When the mirror is
        not current (first call, or reset()/step()/load_state_dict()/step_host(copy_obs=False)
        since the last step_host), the call copies the observations in full instead.  The returned
        observation is read-only.  Needs sync=True and copy_obs=True.
        """
        delta = self._mirror_begin(delta_obs, sync, copy_obs)
        h = self._host_buffers()
        self._obs_current = False
        src = self._host_src = host_source(actions, h["_actions"])
        head = (C.byref(self.params), C.byref(self._state), self._actions.data_ptr(), C.byref(self._next_io(True)),
                self.num_envs, src.data_ptr())
        results = (h["reward"].data_ptr(), h["terminated"].data_ptr(), h["truncated"].data_ptr(),
                   h["_score"].data_ptr(), h["_snake_length"].data_ptr(), stream_ptr(self.device))
        if delta:
            self._call("beng_snake_step_host_delta", *head, self._delta_dev.data_ptr(), h["_delta_dev"].data_ptr(),
                       *results)
        else:
            self._call("beng_snake_step_host", *head, h["obs"].data_ptr() if copy_obs else None, *results)
        self._obs_current = True  # both calls compose every row of self.obs (through _ios_full)
        if sync:
            self._sync()
        obs = self._mirror_end(delta, delta_obs, copy_obs)
        if self.debug_checks:
            self._raise_on_invalid()
        infos = {"score": h["_score"].numpy(), "snake_length": h["_snake_length"].numpy()}
        return obs, h["reward"].numpy(), h["terminated"].numpy(), h["truncated"].numpy(), infos

    # ------------------------------------------------------------------ extras
    def finished_envs(self) -> torch.Tensor:
        """Local indices of the envs whose episode ended in the last step (device-side compaction)."""
        n = int(self.done_count.item())
        return self.done_env[:n]

    def export_state(self, with_body: bool = False) -> dict:
        """Unpack the SoA state into int32 tensors (tests / checkpoints)."""
        n, dev = self.num_envs, self.device
        names = ["head_r", "head_c", "food_r", "food_c", "direction", "steps", "length"]
        out = {k: torch.zeros(n, dtype=torch.int32, device=dev) for k in names}
        out["rng_counter"] = torch.zeros(n, dtype=torch.int32, device=dev)  # u32 bit pattern
        body = torch.full((n, self.grid_size ** 2), -1, dtype=torch.int32, device=dev) if with_body else None
        self._call("beng_snake_export_state", C.byref(self.params), C.byref(self._state), n,
                   *[out[k].data_ptr() for k in names], out["rng_counter"].data_ptr(),
                   body.data_ptr() if with_body else None, stream_ptr(dev))
        out["rng_counter"] = out["rng_counter"].to(torch.int64) & 0xFFFFFFFF
        if with_body:
            out["body"] = body
        return out

    def render(self):
        """rgb_array frames (num_envs, G*20, G*20, 3) from the current observation: a 3-colour LUT like
        snake_env.py:175-188 (host-side; rendering proper is out of scope)."""
        if self.render_mode != "rgb_array":
            return None
        lut = torch.tensor([[0, 0, 0], [0, 255, 0], [255, 0, 0]], dtype=torch.uint8, device=self.device)
        img = lut[self.obs.long()]
        return img.repeat_interleave(20, 1).repeat_interleave(20, 2).cpu().numpy()


class SnakeEnvClassic(_EnvBase):
    """Single-instance gym.Env surface of the reference (snake_env.py:9-143) on the CUDA engine.

    A 1-env BatchedSnakeEnv with auto-reset DISABLED, i.e. exactly the reference class: numpy
    observations, Python scalars, info dicts with the reference's keys.
    """

    metadata = {"render_modes": ["human", "rgb_array"], "render_fps": 10}

    def __init__(self, render_mode=None, grid_size: int = 20, *, device="cuda", seed: int = 0, env_id: int = 0):
        self.grid_size = grid_size
        self.render_mode = render_mode
        self.action_space = Discrete(4)
        self.observation_space = Box(0, 2, (grid_size, grid_size), np.int8)
        self.max_steps = 1000
        self._vec = BatchedSnakeEnv(1, grid_size, device=device, seed=seed, env_id_base=env_id,
                                    autoreset_mode="disabled", max_steps=self.max_steps)
        self._died = False

    @property
    def score(self) -> int:
        return int(self._vec.score.item())

    @property
    def steps(self) -> int:
        return int(self._vec.export_state()["steps"].item())

    def reset(self, seed=None, options=None):
        obs, info = self._vec.reset(seed=seed)
        return obs[0].cpu().numpy().copy(), {"score": int(info["score"].item()),
                                              "snake_length": int(info["snake_length"].item())}

    def step(self, action):
        if not self.action_space.contains(action):
            raise ValueError(f"Invalid action: {action}")  # snake_env.py:69-70
        obs, rew, term, trunc, info = self._vec.step_host(np.array([action], dtype=np.int64))
        reward = float(rew[0])
        died = reward < 0
        out_info = {"score": int(info["score"][0])}
        if not died:  # the death return carries no snake_length (snake_env.py:90,94 vs :117)
            out_info["snake_length"] = int(info["snake_length"][0])
        if reward == 0.0:
            reward = 0  # Python int 0 on a non-eating step (snake_env.py:100)
        return obs[0].copy(), reward, bool(term[0]), False, out_info

    def render(self):
        if self.render_mode == "rgb_array":
            self._vec.render_mode = "rgb_array"
            return self._vec.render()[0]
        return None

    def close(self):
        self._vec.close()
