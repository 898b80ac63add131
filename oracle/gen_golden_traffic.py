"""Generate tests/golden/traffic_golden.npz by running the UNMODIFIED reference TrafficManagementEnv.

Build container only (needs /root/reference):   python -m oracle.gen_golden_traffic

`random` is rebound in BOTH reference modules that draw (environment.py:12 and utils.py:6) to
ReplayRandom(seed, env_id); the caller loop is the reference's own (`if terminated: env.reset()`, i.e. SAME_STEP).
Everything recorded is the reference's output (observations are integer-derived, so crc32 pins them exactly).
"""
from __future__ import annotations

import os
import zlib

import numpy as np

from . import golden_files, philox, ref_loader, replay

SNAP_EVERY = 9
PHASE = {"NS_GREEN": 0, "NS_YELLOW": 1, "EW_GREEN": 2, "EW_YELLOW": 3}

# name, n_envs, n_steps, seed, env_id_base, policy, ctor kwargs
CASES = [
    ("random_default", 3, 2100, 0, 0, "random", {}),
    ("random_hi_ids", 2, 300, 0xFEDCBA987654, (1 << 35) + 3, "random", {}),
    ("all_zero", 2, 400, 1, 10, "zero", {}),
    ("all_ns", 2, 300, 2, 20, "ns", {}),
    ("all_ew", 2, 300, 3, 30, "ew", {}),
    ("alternate", 2, 400, 4, 40, "alternate", {}),
    ("custom_grid", 2, 600, 5, 50, "random",
     dict(grid_size=(3, 4), num_intersections=7, max_vehicles=20, spawn_rate=0.6)),
]


def run_case(env_mod, utils_mod, name, n_envs, n_steps, seed, base, policy, kw):
    ni = min(kw.get("num_intersections", 9), kw.get("grid_size", (5, 5))[0] * kw.get("grid_size", (5, 5))[1])
    od = ni * 14 + 4
    rec = {"action": np.zeros((n_envs, n_steps, ni), np.int8), "reward": np.zeros((n_envs, n_steps), np.float64),
           "terminated": np.zeros((n_envs, n_steps), np.uint8), "obs_crc": np.zeros((n_envs, n_steps), np.uint32),
           "num_vehicles": np.zeros((n_envs, n_steps), np.int32), "timestep": np.zeros((n_envs, n_steps), np.int32),
           "rng_counter": np.zeros((n_envs, n_steps), np.uint32), "total_reward": np.zeros((n_envs, n_steps)),
           "phase": np.zeros((n_envs, n_steps, ni), np.int8), "qlen": np.zeros((n_envs, n_steps, ni, 4), np.int16),
           "passed": np.zeros((n_envs, n_steps, ni), np.int32)}
    snaps = np.zeros((n_envs, len(range(0, n_steps, SNAP_EVERY)), od), np.float32)
    reset_obs = np.zeros((n_envs, od), np.float32)
    tape = philox.action_tape(seed, base + np.arange(n_envs, dtype=np.uint64), 0, n_steps, 3, ni)
    for e in range(n_envs):
        rr = replay.ReplayRandom(seed, base + e)
        env_mod.random = rr
        utils_mod.random = rr
        env = env_mod.TrafficManagementEnv(**kw)
        obs, info = env.reset()
        assert obs.shape == (od,) and info["timestep"] == 0
        reset_obs[e] = obs
        for t in range(n_steps):
            a = {"random": tape[e, t], "zero": np.zeros(ni, np.int64), "ns": np.ones(ni, np.int64),
                 "ew": np.full(ni, 2, np.int64),
                 "alternate": np.full(ni, 1 + (t // 7) % 2, np.int64) if t % 3 == 0 else np.zeros(ni, np.int64)}[policy]
            obs, r, term, trunc, info = env.step(a)
            assert trunc is False and info["timestep"] == env.current_timestep
            rec["action"][e, t] = a
            rec["reward"][e, t] = r
            rec["terminated"][e, t] = term
            rec["total_reward"][e, t] = info["total_reward"]
            if term:
                obs, info = env.reset()
            rec["obs_crc"][e, t] = zlib.crc32(obs.tobytes())
            rec["num_vehicles"][e, t] = len(env.vehicles)
            rec["timestep"][e, t] = env.current_timestep
            rec["rng_counter"][e, t] = rr.counter
            for i, x in enumerate(env.intersections):
                rec["phase"][e, t, i] = PHASE[x.traffic_light.current_phase]
                rec["passed"][e, t, i] = x.vehicles_passed
                for d, q in enumerate(x.vehicle_queues.values()):
                    rec["qlen"][e, t, i, d] = len(q)
            if t % SNAP_EVERY == 0:
                snaps[e, t // SNAP_EVERY] = obs
    out = {f"{name}/{k}": v for k, v in rec.items()}
    out[f"{name}/snap_obs"] = snaps
    out[f"{name}/reset_obs"] = reset_obs
    g = kw.get("grid_size", (5, 5))
    out[f"{name}/meta"] = np.array([n_envs, n_steps, seed, base, SNAP_EVERY, g[0], g[1], kw.get("num_intersections", 9),
                                    kw.get("max_vehicles", 50)], dtype=np.uint64)
    out[f"{name}/spawn_rate"] = np.array(kw.get("spawn_rate", 0.3))
    return out


def main():
    assert ref_loader.reference_available(), "needs /root/reference (build container only)"
    env_mod, utils_mod = ref_loader.load_traffic()
    blob = {}
    for case in CASES:
        blob.update(run_case(env_mod, utils_mod, *case))
        n = case[0]
        print(n, "episodes", int(blob[f"{n}/terminated"].sum()), "max vehicles", int(blob[f"{n}/num_vehicles"].max()),
              "max queue", int(blob[f"{n}/qlen"].max()), "last reward", blob[f"{n}/reward"][0, -1])
    blob["cases"] = np.array([c[0] for c in CASES])
    for path in golden_files.save("traffic", blob):
        print("wrote", os.path.relpath(path), os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
