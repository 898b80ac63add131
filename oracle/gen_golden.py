"""Generate tests/golden/snake_golden.npz by running the UNMODIFIED reference.

Run in the build container only (needs /root/reference):   python -m oracle.gen_golden

For each case the real `SnakeEnvClassic` (snake_env_classic/snake_env.py) is driven with a
recorded action tape while its module-level `random` is rebound to ReplayRandom(seed, env_id)
(the engine's counter-based stream).  The caller loop is the reference's own
(`if terminated: env.reset()`, SURVEY.md section 3.5), i.e. what the batched engine calls
SAME_STEP auto-reset.  Everything recorded is the reference's output; nothing here comes from
the oracle restatements or the CUDA path.

Policies (actions are RECORDED, so replaying the tape needs no policy):
  random  : the synthetic tape philox.action_tape(seed, env, ...)          (93 % length-1 snakes)
  greedy  : steps toward the food, avoiding walls/body when it can         (long snakes, self-collisions,
                                                                             food rejection loop)
  circle  : right, down, left, up forever                                  (never dies -> 1000-step limit)
  reverse : alternates an action with its 180-degree opposite               (reversal guard, snake_env.py:73-74)
"""
from __future__ import annotations

import os
import zlib

import numpy as np

from . import golden_files, philox, ref_loader, replay


# name, grid, n_envs, n_steps, seed, env_id_base, policy
CASES = [
    ("random_g20", 20, 32, 1200, 0, 0, "random"),
    ("random_g20_hi", 20, 8, 600, 0x1234_5678_9ABC, (1 << 33) + 5, "random"),  # 64-bit seed and env ids
    ("greedy_g20", 20, 16, 2500, 1, 100, "greedy"),
    ("greedy_g8", 8, 16, 2500, 2, 0, "greedy"),
    ("greedy_g5", 5, 8, 1500, 3, 7, "greedy"),
    ("random_g15", 15, 8, 600, 4, 0, "random"),
    ("circle_g20", 20, 4, 2100, 5, 0, "circle"),
    ("reverse_g20", 20, 4, 300, 6, 0, "reverse"),
]
SNAP_EVERY = 61  # full observation snapshots every this many steps (all steps carry a crc32)


def greedy_action(env, G):
    hr, hc = env.snake[0]
    fr, fc = env.food
    best, best_key = env.direction, None
    for a, (dr, dc) in enumerate(((-1, 0), (0, 1), (1, 0), (0, -1))):
        if abs(a - env.direction) == 2:
            continue
        nr, nc = hr + dr, hc + dc
        dead = not (0 <= nr < G and 0 <= nc < G) or (nr, nc) in env.snake
        key = (dead, abs(nr - fr) + abs(nc - fc), a)
        if best_key is None or key < best_key:
            best, best_key = a, key
    return best


def run_case(mod, name, G, n_envs, n_steps, seed, base, policy):
    rec = {k: np.zeros((n_envs, n_steps), dt) for k, dt in [
        ("action", np.int8), ("reward", np.float32), ("terminated", np.uint8), ("score", np.int32),
        ("length", np.int32), ("head_r", np.int16), ("head_c", np.int16), ("food_r", np.int16),
        ("food_c", np.int16), ("direction", np.int8), ("steps", np.int32), ("rng_counter", np.uint32),
        ("obs_crc", np.uint32), ("step_obs_crc", np.uint32), ("final_score", np.int32), ("final_steps", np.int32)]}
    snap_steps = np.arange(0, n_steps, SNAP_EVERY)
    snaps = np.zeros((n_envs, len(snap_steps), G, G), np.int8)
    reset_obs = np.zeros((n_envs, G, G), np.int8)
    reset_food = np.zeros((n_envs, 2), np.int16)
    random_tape = philox.action_tape(seed, base + np.arange(n_envs, dtype=np.uint64), 0, n_steps, 4)
    for e in range(n_envs):
        rr = replay.ReplayRandom(seed, base + e)
        mod.random = rr
        env = mod.SnakeEnvClassic(grid_size=G)
        obs, info = env.reset()
        assert info == {"score": 0, "snake_length": 1}
        reset_obs[e] = obs
        reset_food[e] = env.food
        for t in range(n_steps):
            if policy == "random":
                a = int(random_tape[e, t])
            elif policy == "greedy":
                a = greedy_action(env, G)
            elif policy == "circle":
                a = (1, 2, 3, 0)[t % 4]
            else:
                a = (1, 3, 2, 0, 1, 1)[t % 6]
            obs, r, term, trunc, info = env.step(a)
            assert trunc is False
            rec["action"][e, t] = a
            rec["reward"][e, t] = r
            rec["terminated"][e, t] = term
            rec["step_obs_crc"][e, t] = zlib.crc32(obs.tobytes())  # obs of the step itself (DISABLED view)
            rec["final_score"][e, t] = info["score"]
            rec["final_steps"][e, t] = env.steps
            if term:
                obs, info = env.reset()
            rec["score"][e, t] = env.score
            rec["length"][e, t] = len(env.snake)
            rec["head_r"][e, t], rec["head_c"][e, t] = env.snake[0]
            rec["food_r"][e, t], rec["food_c"][e, t] = env.food
            rec["direction"][e, t] = env.direction
            rec["steps"][e, t] = env.steps
            rec["rng_counter"][e, t] = rr.counter
            rec["obs_crc"][e, t] = zlib.crc32(obs.tobytes())
            if t % SNAP_EVERY == 0:
                snaps[e, t // SNAP_EVERY] = obs
    out = {f"{name}/{k}": v for k, v in rec.items()}
    out[f"{name}/snap_obs"] = snaps
    out[f"{name}/reset_obs"] = reset_obs
    out[f"{name}/reset_food"] = reset_food
    out[f"{name}/meta"] = np.array([G, n_envs, n_steps, seed, base, SNAP_EVERY], dtype=np.uint64)
    return out


def frozen_case(mod):
    """SURVEY.md section 8(c) anchor: nine step(1) succeed from reset, the tenth is a wall death that leaves
    the state untouched, and further steps keep returning (-10.0, True) (snake_env.py:88-94)."""
    rr = replay.ReplayRandom(0, 0)
    mod.random = rr
    env = mod.SnakeEnvClassic()
    env.reset()
    rows = []
    for t in range(14):
        obs, r, term, trunc, info = env.step(1 if t < 12 else 0)  # the last two turn upwards and move on
        rows.append((r, term, env.steps, env.snake[0][0], env.snake[0][1], env.direction, info["score"],
                     info.get("snake_length", -1), zlib.crc32(obs.tobytes())))
    return {"frozen/rows": np.array(rows, dtype=np.float64)}


def main():
    assert ref_loader.reference_available(), "needs /root/reference (build container only)"
    mod = ref_loader.load_snake()
    blob = {}
    for case in CASES:
        blob.update(run_case(mod, *case))
        n = case[0]
        print(n, "episodes", int(blob[f"{n}/terminated"].sum()), "max length", int(blob[f"{n}/length"].max()),
              "max final score", int(blob[f"{n}/final_score"].max()))
    blob.update(frozen_case(mod))
    blob["cases"] = np.array([c[0] for c in CASES])
    for path in golden_files.save("snake", blob):
        print("wrote", os.path.relpath(path), os.path.getsize(path), "bytes")


if __name__ == "__main__":
    main()
