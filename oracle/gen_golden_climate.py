"""Generate tests/golden/climate_golden.npz by running the UNMODIFIED reference SmartClimateEnv.

Build container only (needs /root/reference):   python -m oracle.gen_golden_climate

`env.rng` (a numpy Generator in the reference, smartclimate/env.py:31) is replaced by ReplayGenerator(seed, env_id)
-- the engine's counter-based stream -- right after construction; the caller loop is `if terminated: env.reset()`
(SAME_STEP auto-reset).  Everything recorded is the reference's output.
"""
from __future__ import annotations

import logging
import os

import numpy as np

from . import golden_files, ref_loader, replay


# name, n_envs, n_steps, seed, env_id_base, policy, ctor kwargs
CASES = [
    ("random_default", 3, 3100, 0, 0, "random", {}),
    ("random_hi_ids", 2, 400, 0xA1B2C3D4E5F6, (1 << 36) + 1, "random", {}),
    ("thermostat", 2, 1500, 1, 10, "thermostat", {}),
    ("extremes", 2, 600, 2, 20, "extremes", {}),
    ("small_office", 2, 700, 3, 30, "random", dict(max_occupancy=3, episode_minutes=300)),
]


def run_case(mod, name, n_envs, n_steps, seed, base, policy, kw):
    rec = {"ac_temp": np.zeros((n_envs, n_steps), np.float32), "lights": np.zeros((n_envs, n_steps, 4), np.int8),
           "reward": np.zeros((n_envs, n_steps)), "terminated": np.zeros((n_envs, n_steps), np.uint8),
           "obs": np.zeros((n_envs, n_steps, 9), np.float32), "comfort": np.zeros((n_envs, n_steps)),
           "ac_penalty": np.zeros((n_envs, n_steps)), "light_penalty": np.zeros((n_envs, n_steps)),
           "room_temp": np.zeros((n_envs, n_steps)), "num_people": np.zeros((n_envs, n_steps), np.int32),
           "energy_usage": np.zeros((n_envs, n_steps)), "comfort_time": np.zeros((n_envs, n_steps), np.int32),
           "step": np.zeros((n_envs, n_steps), np.int32), "rng_counter": np.zeros((n_envs, n_steps), np.uint32)}
    reset_obs = np.zeros((n_envs, 9), np.float32)
    arng = np.random.default_rng(seed + 7)
    for e in range(n_envs):
        env = mod.SmartClimateEnv(log_level=logging.ERROR, **kw)
        env.rng = replay.ReplayGenerator(seed, base + e)
        obs, info = env.reset()
        assert obs.shape == (9,) and obs.dtype == np.float32
        reset_obs[e] = obs
        for t in range(n_steps):
            if policy == "random":
                ac = np.float32(arng.random() * 22.0 + 13.0)      # beyond [16, 32] on purpose (clip path)
                lights = arng.integers(0, 2, 4).astype(np.int8)
            elif policy == "thermostat":
                ac = np.float32(16.0 if env.room_temp > 22 else 30.0)
                need = min(4, -(-int(env.num_people) // 2))
                lights = np.array([1] * need + [0] * (4 - need), np.int8)
            else:
                ac = np.float32((5.0, 40.0, 16.0, 32.0)[t % 4])
                lights = np.array([(t >> i) & 1 for i in range(4)], np.int8)
            obs, r, term, trunc, info = env.step({"ac_temp": np.array([ac], np.float32), "lights": lights})
            assert trunc is False
            rec["ac_temp"][e, t], rec["lights"][e, t] = ac, lights
            rec["reward"][e, t], rec["terminated"][e, t] = r, term
            rec["comfort"][e, t], rec["ac_penalty"][e, t] = info["comfort"], info["ac_penalty"]
            rec["light_penalty"][e, t] = info["light_penalty"]
            if term:
                obs, _ = env.reset()
            rec["obs"][e, t] = obs
            rec["room_temp"][e, t], rec["num_people"][e, t] = env.room_temp, env.num_people
            rec["energy_usage"][e, t], rec["comfort_time"][e, t] = env.energy_usage, env.comfort_time
            rec["step"][e, t], rec["rng_counter"][e, t] = env.current_step, env.rng.counter
    out = {f"{name}/{k}": v for k, v in rec.items()}
    out[f"{name}/reset_obs"] = reset_obs
    out[f"{name}/meta"] = np.array([n_envs, n_steps, seed, base, kw.get("max_occupancy", 8),
                                    kw.get("episode_minutes", 1440)], dtype=np.uint64)
    return out


def main():
    assert ref_loader.reference_available(), "needs /root/reference (build container only)"
    mod = ref_loader.load_climate()
    blob = {}
    for case in CASES:
        blob.update(run_case(mod, *case))
        n = case[0]
        print(n, "episodes", int(blob[f"{n}/terminated"].sum()), "room temp range",
              float(blob[f"{n}/room_temp"].min()), float(blob[f"{n}/room_temp"].max()),
              "people max", int(blob[f"{n}/num_people"].max()))
    blob["cases"] = np.array([c[0] for c in CASES])
    for path in golden_files.save("climate", blob):
        print("wrote", os.path.relpath(path), os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
