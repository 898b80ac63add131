"""Shared host-side plumbing of the batched (VectorEnv-compatible) classes.

`gymnasium.vector.VectorEnv` is duck-typed (gymnasium is not installed in this image): the
batched classes expose num_envs, single_observation_space, single_action_space,
observation_space, action_space, metadata["autoreset_mode"], reset(seed=, options=),
step(actions), close().  When gymnasium IS importable they also subclass the real VectorEnv.
"""
from __future__ import annotations

import ctypes as C
import os

import numpy as np
import torch

from . import _lib

try:  # pragma: no cover
    from gymnasium.vector import VectorEnv as _VectorEnvBase  # type: ignore
except Exception:
    class _VectorEnvBase:  # minimal stand-in
        metadata = {}
        render_mode = None
        closed = False

        def close(self, **kwargs):
            self.closed = True

try:  # pragma: no cover
    from gymnasium import Env as _EnvBase  # type: ignore  (gym.make refuses entry points that are not gymnasium.Env)
except Exception:
    class _EnvBase:  # minimal stand-in for the single-instance facades
        metadata = {}
        render_mode = None

AUTORESET_MODES = {"disabled": 0, "next_step": 1, "same_step": 2}


def _mode_name(mode) -> str:
    name = getattr(mode, "value", mode)
    name = str(name).lower()
    if name not in AUTORESET_MODES:
        raise ValueError(f"autoreset_mode must be one of {sorted(AUTORESET_MODES)}, got {mode!r}")
    return name


def require_cuda(device) -> torch.device:
    dev = torch.device(device)
    if dev.type != "cuda":
        raise RuntimeError("the batched engine runs on CUDA devices only (there is no CPU fallback)")
    if not torch.cuda.is_available():
        raise RuntimeError("CUDA is not available: the batched engine has no CPU fallback")
    if dev.index is None:
        dev = torch.device("cuda", torch.cuda.current_device())
    return dev


def stream_ptr(device) -> int:
    return torch.cuda.current_stream(device).cuda_stream


def as_device_actions(actions, buf: torch.Tensor) -> torch.Tensor:
    """Return a contiguous tensor of `buf`'s device, dtype and shape holding `actions`: the caller's tensor itself when
    it already is one (zero-copy), otherwise `buf` after copying into it.  A tensor of another shape is reshaped; any
    other input must have exactly `buf`'s shape."""
    if isinstance(actions, torch.Tensor):
        if actions.device == buf.device and actions.dtype == buf.dtype and actions.is_contiguous() \
                and actions.shape == buf.shape and actions.data_ptr() % 16 == 0:  # (a misaligned view goes through buf)
            return actions
        buf.copy_(actions.reshape(buf.shape), non_blocking=True)
        return buf
    arr = np.asarray(actions)
    if arr.shape != tuple(buf.shape):
        raise ValueError(f"actions must have shape {tuple(buf.shape)}, got {arr.shape}")
    buf.copy_(torch.from_numpy(np.ascontiguousarray(arr)), non_blocking=False)
    return buf


def host_source(src, staging: "torch.Tensor") -> "torch.Tensor":
    """The pinned host tensor a step_host() call uploads its actions from: the caller's own tensor when it already is
    pinned, contiguous and of the staging buffer's dtype and size (no host-to-host copy inside the call), otherwise the
    env's pinned staging buffer after copying `src` (a tensor, or anything numpy accepts) into it.  The upload is
    asynchronous: with sync=False the caller must keep the tensor alive and unchanged until the stream has consumed it."""
    if not isinstance(src, torch.Tensor):
        src = torch.as_tensor(np.asarray(src))
    if src.device.type == "cpu" and src.dtype == staging.dtype and src.numel() == staging.numel() \
            and src.is_contiguous() and src.is_pinned():
        return src
    if src.data_ptr() != staging.data_ptr():
        staging.copy_(src.reshape(staging.shape))
    return staging


class _BatchedEnv(_VectorEnvBase):
    """The host-side protocol every Batched*Env shares: reset() with its seed / mask / first-call rules, the
    reset-before-step guard, libbeng calls, step_host()'s pinned host buffers, the delta-observation mirror,
    checkpoints and episode statistics.

    A subclass describes itself as data:
      _reset_fn        name of its libbeng reset function (called with `_state` and `_reset_io()`)
      _state_tensors   attributes holding its state tensors; the state_dict key is the name without its leading "_"
                       (`stats`, `seed` and `env_id_base` are added for every env)
      _stat_names      names of the entries of `stats`, for episode_stats()
      _host_names      attributes whose shape and dtype step_host()'s pinned buffers copy, keyed by the same names
      _mirror          for an env with a delta path: the observation attribute whose pinned buffer is kept as a mirror
                       of the device tensor, patched by `_apply_delta_fn` from the change records in `_delta_dev`
    and overrides _reset_io() / _reset_result() where the default (`_io`, `(obs, {})`) does not fit.
    """

    _reset_fn: str
    _state_tensors: tuple = ()
    _stat_names: tuple = ()
    _host_names: tuple = ()
    _mirror = None
    _apply_delta_fn = None

    def __init__(self, num_envs, device, autoreset_mode, render_mode):
        self.lib = _lib.load()
        self.device = require_cuda(device)
        self.num_envs = int(num_envs)
        self.render_mode = render_mode
        self.autoreset_mode = _mode_name(autoreset_mode)
        self.metadata = dict(type(self).metadata, autoreset_mode=self.autoreset_mode)
        self.closed = False
        self._host = None
        # True while the pinned mirror equals the device observations: set by a full-copy step_host(), cleared by
        # anything else that rewrites them.  step_host(delta_obs=True) patches the mirror only while it is set.
        self._mirror_valid = False
        self._needs_first_reset = True

    def _call(self, fn: str, *args):
        """libbeng's `fn(*args)` on this env's device; a non-zero return code raises RuntimeError."""
        with torch.cuda.device(self.device):
            rc = getattr(self.lib, fn)(*args)
        _lib.check(rc, fn)

    def _require_reset(self):
        if self._needs_first_reset:
            raise RuntimeError("call reset() before step()")

    def _sync(self):
        torch.cuda.current_stream(self.device).synchronize()

    # ------------------------------------------------------------------ reset
    def _reset_io(self):
        return self._io

    def _reset_result(self):
        return self.obs, {}

    def reset(self, *, seed=None, options=None):
        """Reset every env -> (obs, infos).  `seed` re-keys the counter-based stream and rewinds it.
        options={"reset_mask": bool tensor of shape (num_envs,)} resets only the selected envs; the first reset() must
        reset every env."""
        first = self._needs_first_reset
        if seed is not None:
            self.params.seed = int(seed)
            first = True
        mask = None if not options else options.get("reset_mask")
        mask_ptr = None
        if mask is not None:
            if self._needs_first_reset:
                raise RuntimeError("the first reset() must reset every env")
            mask = torch.as_tensor(mask).to(device=self.device, dtype=torch.uint8).contiguous()
            if mask.shape != (self.num_envs,):
                raise ValueError("reset_mask must have shape (num_envs,)")
            mask_ptr = mask.data_ptr()
        self._mirror_valid = False
        self._call(self._reset_fn, C.byref(self.params), C.byref(self._state), C.byref(self._reset_io()), mask_ptr,
                   self.num_envs, int(first), stream_ptr(self.device))
        self._needs_first_reset = False
        return self._reset_result()

    # ------------------------------------------------------------------ step_host() plumbing
    def _host_buffers(self) -> dict:
        """step_host()'s pinned host buffers, allocated on first use."""
        if self._host is None:
            if self._mirror is not None:
                self._delta_dev = torch.zeros(self.num_envs, dtype=torch.int32, device=self.device)  # uint32 records
            self._host = {k: torch.zeros_like(getattr(self, k), device="cpu", pin_memory=True) for k in self._host_names}
        return self._host

    def _mirror_begin(self, delta_obs: bool, sync: bool, copy_obs: bool) -> bool:
        """Argument checks of a step_host() with a `delta_obs` option -> whether this call may send change records
        instead of the observations: only while the mirror is current.  The mirror counts as stale until the call
        completes."""
        if delta_obs and not (sync and copy_obs):
            raise ValueError("step_host(delta_obs=True) needs sync=True and copy_obs=True")
        self._require_reset()
        delta = delta_obs and self._mirror_valid
        self._mirror_valid = False
        return delta

    def _mirror_end(self, delta: bool, delta_obs: bool, copy_obs: bool):
        """After the step_host() call has synchronised: patch the mirror from the change records when `delta`, and
        return the observation step_host() hands out (the mirror, read-only under delta_obs; the device tensor when
        copy_obs=False)."""
        mirror = self._host[self._mirror]
        if delta:
            self._call(self._apply_delta_fn, self._host["_delta_dev"].data_ptr(), mirror.data_ptr(), self.num_envs,
                       self.grid_size, len(os.sched_getaffinity(0)))
        self._mirror_valid = copy_obs
        if not copy_obs:
            return getattr(self, self._mirror)
        obs = mirror.numpy()
        if delta_obs:
            obs = obs.view()
            obs.flags.writeable = False  # the mirror of the next delta step
        return obs

    # ------------------------------------------------------------------ extras
    def episode_stats(self) -> dict:
        """Running episode statistics accumulated on the device since construction."""
        return dict(zip(self._stat_names, self.stats.tolist()))

    def state_dict(self) -> dict:
        sd = {name.lstrip("_"): getattr(self, name).clone() for name in self._state_tensors}
        sd.update(stats=self.stats.clone(), seed=int(self.params.seed), env_id_base=int(self.params.env_id_base))
        return sd

    def load_state_dict(self, sd: dict):
        for name in self._state_tensors + ("stats",):
            getattr(self, name).copy_(sd[name.lstrip("_")])
        self.params.seed = int(sd["seed"])
        self.params.env_id_base = int(sd["env_id_base"])
        self._mirror_valid = False
        self._needs_first_reset = False

    def render(self):
        return None  # rendering is out of scope (SURVEY.md section 2)

    def close(self, **kwargs):
        self.closed = True


class LazyInfos(dict):
    """infos dict whose derived entries are computed on access (no per-step kernels or HBM writes for values
    nobody reads).  `lazy[key]` is a zero-argument callable returning the tensor."""

    def __init__(self, *a, **k):
        super().__init__(*a, **k)
        self.lazy = {}

    def __missing__(self, key):
        if key in self.lazy:
            return self.lazy[key]()
        raise KeyError(key)

    def __contains__(self, key):
        return super().__contains__(key) or key in self.lazy

    def get(self, key, default=None):
        return self[key] if key in self else default

    def keys(self):
        return list(super().keys()) + list(self.lazy)

    def __iter__(self):
        return iter(self.keys())

    def __len__(self):
        return super().__len__() + len(self.lazy)

    def items(self):
        return [(k, self[k]) for k in self.keys()]

    def values(self):
        return [self[k] for k in self.keys()]
