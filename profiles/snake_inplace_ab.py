#!/usr/bin/env python
"""A/B of the two snake step kernels in one process, 1,048,576 envs, G = 20, SAME_STEP auto-reset, random actions.

  in_place  env.step(a)                    -> beng_snake_step_inplace (patches env.obs)
  compose   env.step(a, out_obs=env.obs)   -> beng_snake_step (composes every row into the same buffer)

Two envs with the same seed walk the same device-resident action tape (bench.py's, 256 distinct steps).  Blocks of
each variant alternate (the order swaps every block), each block timed two ways:
  back_to_back  --steps launches between two CUDA events (what bench.py times at this size)
  l2_flushed    every step on its own events, a 256 MB fill in between (untimed) evicts the previous step's lines
At the end the two envs' observations, state records and rings must be byte-equal.  Prints one JSON line, and also
writes it to --out when given.

    python profiles/snake_inplace_ab.py [--envs N] [--blocks B] [--steps K] [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (v.strip() for v in out.split(","))))
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        return {"error": repr(e)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--blocks", type=int, default=6)
    ap.add_argument("--steps", type=int, default=200, help="steps per back-to-back block")
    ap.add_argument("--flushed-steps", type=int, default=50, help="steps per L2-flushed block")
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()

    import torch

    import custom_gymnasium_environments_b200 as pkg

    if not torch.cuda.is_available():
        raise SystemExit("snake_inplace_ab.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    lib = pkg._lib.load()
    n = args.envs
    stream = torch.cuda.current_stream(dev)
    tapes = torch.empty((256, n), dtype=torch.int64, device=dev)
    for t in range(256):
        pkg._lib.check(lib.beng_fill_random_actions(tapes[t].data_ptr(), n, 1, 4, t, 0, 0, stream.cuda_stream),
                       "beng_fill_random_actions")
    envs = {name: pkg.BatchedSnakeEnv(n, 20, device=dev, seed=0) for name in ("in_place", "compose")}
    clock = {name: 0 for name in envs}

    def step(name):
        env = envs[name]
        a = tapes[clock[name] % 256]
        clock[name] += 1
        return env.step(a) if name == "in_place" else env.step(a, out_obs=env.obs)

    for env in envs.values():
        env.reset()
    for _ in range(args.warmup):
        for name in envs:
            step(name)
    torch.cuda.synchronize(dev)

    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    blocks = {name: {"back_to_back_us": [], "l2_flushed_us": []} for name in envs}
    for b in range(args.blocks):
        order = ("in_place", "compose") if b % 2 == 0 else ("compose", "in_place")
        for name in order:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.steps):
                step(name)
            e1.record(stream)
            torch.cuda.synchronize(dev)
            blocks[name]["back_to_back_us"].append(e0.elapsed_time(e1) * 1e3 / args.steps)
        for name in order:
            pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                     for _ in range(args.flushed_steps)]
            for i in range(args.flushed_steps):
                scratch.fill_(i & 0xFF)
                pairs[i][0].record(stream)
                step(name)
                pairs[i][1].record(stream)
            torch.cuda.synchronize(dev)
            blocks[name]["l2_flushed_us"].append(sum(x.elapsed_time(y) for x, y in pairs) * 1e3 / args.flushed_steps)

    a, c = envs["in_place"], envs["compose"]
    assert clock["in_place"] == clock["compose"]
    equal = {"obs": bool(torch.equal(a.obs, c.obs)), "core": bool(torch.equal(a._core, c._core)),
             "ring": bool(torch.equal(a._ring, c._ring)), "stats": bool(torch.equal(a.stats, c.stats))}

    def summary(xs):
        return {"median": statistics.median(xs), "min": min(xs), "max": max(xs), "blocks": xs}

    result = {"gpu": gpu_info(), "envs": n, "grid_size": 20, "autoreset_mode": "same_step", "warmup": args.warmup,
              "steps_per_block": args.steps, "flushed_steps_per_block": args.flushed_steps,
              "steps_taken_per_env": clock["in_place"], "outputs_equal": equal}
    for name in envs:
        result[name] = {k: summary(v) for k, v in blocks[name].items()}
    for k in ("back_to_back_us", "l2_flushed_us"):
        result[f"speedup_{k[:-3]}"] = result["compose"][k]["median"] / result["in_place"][k]["median"]
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not all(equal.values()):
        raise SystemExit(f"the two kernels disagree: {equal}")


if __name__ == "__main__":
    main()
