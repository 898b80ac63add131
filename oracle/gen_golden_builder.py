"""Generate tests/golden/builder_golden.npz by running the UNMODIFIED reference WorldBuilderEnv.

Build container only (needs /root/reference):   python -m oracle.gen_golden_builder

`np.random.randint` inside the reference's game_logic module (game_logic.py:137) is redirected to
ReplayRandom(seed, env_id) by rebinding that module's `np` (oracle/replay.py NumpyWithReplayRandint); the caller loop is
`if terminated: env.reset()` (SAME_STEP).  Everything recorded is the reference's output.
Policies: random; farmer (a simple winning build order, so that win episodes with +100 appear); spam (only houses:
failed builds, then starvation); a 4x4 grid that fills up (the `no empty space` branch).
"""
from __future__ import annotations

import os

import numpy as np

from . import golden_files, ref_loader, replay


# name, n_envs, n_steps, seed, env_id_base, policy, grid
CASES = [
    ("random_g10", 6, 400, 0, 0, "random", 10),
    ("random_hi_ids", 3, 200, 0x0F1E2D3C4B5A, (1 << 37) + 11, "random", 10),
    ("farmer_g10", 4, 500, 1, 10, "farmer", 10),
    ("spam_g10", 2, 120, 2, 20, "spam", 10),
    ("farmer_g4", 3, 400, 3, 30, "farmer", 4),
]


def farmer(env):
    g = env.game_logic
    food, wood, stone, pop = g.resources["food"], g.resources["wood"], g.resources["stone"], g.population
    c = g.building_counts
    if c["farm"] * 2 <= pop and wood >= 5:
        return 1
    if pop >= g.population_capacity - 1 and wood >= 10 and stone >= 5:
        return 4
    if c["lumberyard"] < 3 and stone >= 3:
        return 2
    if c["quarry"] < 3 and wood >= 5:
        return 3
    return 0


def run_case(env_mod, gl, name, n_envs, n_steps, seed, base, policy, G):
    rec = {"action": np.zeros((n_envs, n_steps), np.int8), "reward": np.zeros((n_envs, n_steps), np.float32),
           "terminated": np.zeros((n_envs, n_steps), np.uint8), "grid": np.zeros((n_envs, n_steps, G, G), np.int8),
           "resources": np.zeros((n_envs, n_steps, 4), np.float32), "capacity": np.zeros((n_envs, n_steps), np.float32),
           "win_steps": np.zeros((n_envs, n_steps), np.int32), "steps": np.zeros((n_envs, n_steps), np.int32),
           "rng_counter": np.zeros((n_envs, n_steps), np.uint32), "counts": np.zeros((n_envs, n_steps, 4), np.int32),
           "won": np.zeros((n_envs, n_steps), np.uint8)}
    arng = np.random.default_rng(seed + 5)
    for e in range(n_envs):
        rr = replay.ReplayRandom(seed, base + e)
        gl.np = replay.NumpyWithReplayRandint(rr)
        env = env_mod.WorldBuilderEnv(grid_size=G)
        obs, info = env.reset()
        assert info["population"] == 3 and obs["grid"].shape == (G, G)
        for t in range(n_steps):
            a = {"random": int(arng.integers(0, 5)), "farmer": farmer(env) if arng.random() > 0.05 else int(arng.integers(0, 5)),
                 "spam": 4}[policy]
            obs, r, term, trunc, info = env.step(a)
            assert trunc is False
            rec["action"][e, t], rec["reward"][e, t], rec["terminated"][e, t] = a, r, term
            if term:
                rec["won"][e, t] = info["population"] > 0
                obs, info = env.reset()
            rec["grid"][e, t] = obs["grid"]
            rec["resources"][e, t] = obs["resources"]
            rec["capacity"][e, t] = obs["population_capacity"][0]
            rec["win_steps"][e, t] = obs["win_steps"][0]
            rec["steps"][e, t] = info["steps"]
            rec["rng_counter"][e, t] = rr.counter
            rec["counts"][e, t] = [info["building_counts"][k] for k in ("farm", "lumberyard", "quarry", "house")]
    out = {f"{name}/{k}": v for k, v in rec.items()}
    out[f"{name}/meta"] = np.array([n_envs, n_steps, seed, base, G], dtype=np.uint64)
    return out


def main():
    assert ref_loader.reference_available(), "needs /root/reference (build container only)"
    env_mod, gl = ref_loader.load_builder()
    real_np = gl.np
    blob = {}
    try:
        for case in CASES:
            blob.update(run_case(env_mod, gl, *case))
            n = case[0]
            print(n, "episodes", int(blob[f"{n}/terminated"].sum()), "wins", int(blob[f"{n}/won"].sum()),
                  "max buildings", int((blob[f"{n}/grid"] > 0).sum(axis=(2, 3)).max()))
    finally:
        gl.np = real_np
    blob["cases"] = np.array([c[0] for c in CASES])
    for path in golden_files.save("builder", blob):
        print("wrote", os.path.relpath(path), os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
