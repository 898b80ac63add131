"""ctypes binding of libbeng.so -- the C ABI declared in include/beng.h.

There is NO CPU fallback: if the library is missing or a call fails, a RuntimeError is raised.
"""
from __future__ import annotations

import ctypes as C
import os

from ._build import LIB_PATH, is_stale

_lib = None


class SnakeParams(C.Structure):
    _fields_ = [("grid_size", C.c_int32), ("max_steps", C.c_int32), ("autoreset_mode", C.c_int32),
                ("time_limit_truncation", C.c_int32), ("seed", C.c_uint64), ("env_id_base", C.c_uint64)]


class SnakeState(C.Structure):
    _fields_ = [("core", C.c_void_p), ("ring", C.c_void_p)]


class SnakeIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "obs", "reward", "terminated", "truncated", "score", "snake_length", "ep_return", "ep_length", "ep_score",
        "done_count", "done_env", "done_count_next", "stats", "invalid_count")]


class CryptoParams(C.Structure):
    _fields_ = [("initial_balance", C.c_double), ("trading_fee_rate", C.c_double), ("slippage_rate", C.c_double),
                ("min_price", C.c_double), ("max_price", C.c_double), ("volatility_base", C.c_double),
                ("market_psychology_factor", C.c_double), ("max_steps", C.c_int32), ("autoreset_mode", C.c_int32),
                ("action_type", C.c_int32), ("window_head", C.c_int32), ("time_limit_truncation", C.c_int32),
                ("reserved", C.c_int32), ("seed", C.c_uint64), ("env_id_base", C.c_uint64)]


class CryptoState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("scal", "meta", "ep_return", "close", "ohlv")]


class CryptoIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in (
        "obs", "reward", "terminated", "truncated", "reward64", "portfolio_value", "current_price", "trade_kind",
        "ep_return_out", "ep_length", "stats", "window_head_dev")]


class TrafficParams(C.Structure):
    _fields_ = [("grid_rows", C.c_int32), ("grid_cols", C.c_int32), ("num_intersections", C.c_int32),
                ("max_vehicles", C.c_int32), ("spawn_rate", C.c_double), ("max_timesteps", C.c_int32),
                ("autoreset_mode", C.c_int32), ("time_limit_truncation", C.c_int32), ("reserved", C.c_int32),
                ("seed", C.c_uint64), ("env_id_base", C.c_uint64)]


class TrafficState(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("light", "passed", "waiting", "qmeta", "qwait", "misc", "total_reward")]


class TrafficIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("obs", "reward", "terminated", "truncated", "reward64", "ep_return",
                                          "ep_length", "stats", "timestep")]


class ClimateParams(C.Structure):
    _fields_ = [("max_occupancy", C.c_int32), ("episode_minutes", C.c_int32), ("autoreset_mode", C.c_int32),
                ("time_limit_truncation", C.c_int32), ("seed", C.c_uint64), ("env_id_base", C.c_uint64)]


class ClimateState(C.Structure):
    _fields_ = [("f64", C.c_void_p), ("i32", C.c_void_p)]


class ClimateIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("obs", "reward", "terminated", "truncated", "reward64", "reward_terms",
                                          "ep_return", "ep_length", "stats")]


class BuilderParams(C.Structure):
    _fields_ = [("grid_size", C.c_int32), ("autoreset_mode", C.c_int32), ("seed", C.c_uint64),
                ("env_id_base", C.c_uint64)]


class BuilderState(C.Structure):
    _fields_ = [("words", C.c_void_p)]


class BuilderIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("grid", "resources", "capacity", "win_steps", "flat_obs", "reward",
                                          "terminated", "truncated", "ep_return", "ep_length", "stats",
                                          "invalid_count")]


class NormalizeParams(C.Structure):
    _fields_ = [("clip_obs", C.c_double), ("clip_reward", C.c_double), ("epsilon", C.c_double), ("gamma", C.c_double),
                ("flags", C.c_uint32), ("reserved", C.c_int32)]


class NormalizeIO(C.Structure):
    _fields_ = [(n, C.c_void_p) for n in ("obs", "reward", "terminated", "truncated", "returns", "obs_rms", "ret_rms",
                                          "workspace", "obs_out", "reward_out")]


NORM_OBS, NORM_REWARD, NORM_UPDATE = 1, 2, 4


# name -> (restype, argtypes); also the list of symbols include/beng.h declares (tests check it).
SIGNATURES = {
    "beng_version": (C.c_int, []),
    "beng_compiled_arch": (C.c_int, []),
    "beng_launch_count": (C.c_uint64, []),
    "beng_fill_random_actions": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_int32, C.c_uint32, C.c_uint64,
                                           C.c_uint64, C.c_void_p]),
    "beng_snake_launch_config": (C.c_int, [C.c_int32, C.c_int64, C.POINTER(C.c_int32), C.POINTER(C.c_int32),
                                           C.POINTER(C.c_int32)]),
    "beng_snake_core_bytes": (C.c_size_t, [C.c_int64]),
    "beng_snake_ring_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "beng_snake_reset": (C.c_int, [C.POINTER(SnakeParams), C.POINTER(SnakeState), C.POINTER(SnakeIO), C.c_void_p,
                                   C.c_int64, C.c_int32, C.c_void_p]),
    "beng_snake_step": (C.c_int, [C.POINTER(SnakeParams), C.POINTER(SnakeState), C.c_void_p, C.POINTER(SnakeIO),
                                  C.c_int64, C.c_void_p]),
    "beng_snake_step_inplace": (C.c_int, [C.POINTER(SnakeParams), C.POINTER(SnakeState), C.c_void_p,
                                          C.POINTER(SnakeIO), C.c_int64, C.c_void_p]),
    "beng_snake_step_host": (C.c_int, [C.POINTER(SnakeParams), C.POINTER(SnakeState), C.c_void_p, C.POINTER(SnakeIO),
                                       C.c_int64] + [C.c_void_p] * 8),
    "beng_snake_step_host_delta": (C.c_int, [C.POINTER(SnakeParams), C.POINTER(SnakeState), C.c_void_p,
                                             C.POINTER(SnakeIO), C.c_int64] + [C.c_void_p] * 9),
    "beng_snake_apply_obs_delta": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32]),
    "beng_crypto_window_pitch": (C.c_int64, [C.c_int64]),
    "beng_crypto_reset": (C.c_int, [C.POINTER(CryptoParams), C.POINTER(CryptoState), C.POINTER(CryptoIO), C.c_void_p,
                                    C.c_int64, C.c_int32, C.c_void_p]),
    "beng_crypto_step": (C.c_int, [C.POINTER(CryptoParams), C.POINTER(CryptoState), C.c_void_p, C.POINTER(CryptoIO),
                                   C.c_int64, C.c_void_p]),
    "beng_crypto_step_host": (C.c_int, [C.POINTER(CryptoParams), C.POINTER(CryptoState), C.c_void_p,
                                        C.POINTER(CryptoIO), C.c_int64] + [C.c_void_p] * 6),
    "beng_traffic_reset": (C.c_int, [C.POINTER(TrafficParams), C.POINTER(TrafficState), C.POINTER(TrafficIO),
                                     C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "beng_traffic_step": (C.c_int, [C.POINTER(TrafficParams), C.POINTER(TrafficState), C.c_void_p,
                                    C.POINTER(TrafficIO), C.c_int64, C.c_void_p]),
    "beng_traffic_step_host": (C.c_int, [C.POINTER(TrafficParams), C.POINTER(TrafficState), C.c_void_p,
                                         C.POINTER(TrafficIO), C.c_int64] + [C.c_void_p] * 6),
    "beng_climate_reset": (C.c_int, [C.POINTER(ClimateParams), C.POINTER(ClimateState), C.POINTER(ClimateIO),
                                     C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "beng_climate_step": (C.c_int, [C.POINTER(ClimateParams), C.POINTER(ClimateState), C.c_void_p, C.c_void_p,
                                    C.POINTER(ClimateIO), C.c_int64, C.c_void_p]),
    "beng_climate_step_host": (C.c_int, [C.POINTER(ClimateParams), C.POINTER(ClimateState), C.c_void_p, C.c_void_p,
                                         C.POINTER(ClimateIO), C.c_int64] + [C.c_void_p] * 7),
    "beng_builder_reset": (C.c_int, [C.POINTER(BuilderParams), C.POINTER(BuilderState), C.POINTER(BuilderIO),
                                     C.c_void_p, C.c_int64, C.c_int32, C.c_void_p]),
    "beng_builder_step": (C.c_int, [C.POINTER(BuilderParams), C.POINTER(BuilderState), C.c_void_p,
                                    C.POINTER(BuilderIO), C.c_int64, C.c_void_p]),
    "beng_builder_step_host": (C.c_int, [C.POINTER(BuilderParams), C.POINTER(BuilderState), C.c_void_p,
                                         C.POINTER(BuilderIO), C.c_int64] + [C.c_void_p] * 8),
    "beng_builder_step_host_delta": (C.c_int, [C.POINTER(BuilderParams), C.POINTER(BuilderState), C.c_void_p,
                                               C.POINTER(BuilderIO), C.c_int64] + [C.c_void_p] * 9),
    "beng_builder_apply_obs_delta": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_int32, C.c_int32]),
    "beng_snake_export_state": (C.c_int, [C.POINTER(SnakeParams), C.POINTER(SnakeState), C.c_int64] +
                                [C.c_void_p] * 10),
    "beng_normalize_workspace_bytes": (C.c_size_t, [C.c_int64, C.c_int32]),
    "beng_normalize": (C.c_int, [C.POINTER(NormalizeParams), C.POINTER(NormalizeIO), C.c_int64, C.c_int32,
                                 C.c_void_p]),
}


def library_path() -> str:
    return LIB_PATH


def load():
    """Load libbeng.so (once).  Raises RuntimeError when it has not been built."""
    global _lib
    if _lib is None:
        lib_path = os.environ.get("BENG_LIB_PATH", LIB_PATH)  # A/B a different build of the same ABI (profiling only)
        if not os.path.exists(lib_path):
            raise RuntimeError(
                f"{LIB_PATH} is missing: the CUDA engine has not been built and there is no CPU fallback. "
                "Build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(or custom_gymnasium_environments_b200._build.build_library()).")
        if lib_path == LIB_PATH and is_stale() and not os.environ.get("BENG_ALLOW_STALE"):
            raise RuntimeError(
                f"{LIB_PATH} was built from different sources than the ones in csrc/ (or its .srchash is missing): "
                "rebuild with `python -c 'import __graft_entry__ as g; g.build()'` so that what runs is what the tree "
                "says (BENG_ALLOW_STALE=1 overrides).")
        lib = C.CDLL(lib_path)
        for name, (res, args) in SIGNATURES.items():
            fn = getattr(lib, name)
            fn.restype = res
            fn.argtypes = args
        _lib = lib
    return _lib


def check(rc: int, what: str):
    if rc != 0:
        kind = {-1: "BENG_ERR_BAD_ARG", -2: "BENG_ERR_UNSUPPORTED"}.get(rc, f"cudaError {rc}")
        raise RuntimeError(f"{what} failed: {kind}")
