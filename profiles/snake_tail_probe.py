#!/usr/bin/env python
"""What the finished-env compaction and the statistics flush cost the in-place snake step (snake_patch_kernel), measured
through the C ABI, which lets a caller pass io.done_env and io.stats as NULL: 1,048,576 envs, G = 20, SAME_STEP
auto-reset, bench.py's random action tape.  One env is stepped by four variants of its io block in alternating blocks
(the order rotates every block), each block --steps back-to-back launches between two CUDA events:

  full        done_env and stats set (what BatchedSnakeEnv.step() passes)
  no_done     done_env = NULL: no per-warp atomicAdd on the finished-env counter, no list stores
  no_stats    stats = NULL: no per-warp shared-memory atomics, no closing barrier, no per-CTA global atomics
  neither     both NULL

Prints one JSON line, and also writes it to --out when given.

    python profiles/snake_tail_probe.py [--envs N] [--blocks B] [--steps K] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from snake_inplace_ab import gpu_info  # noqa: E402


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--envs", type=int, default=1 << 20)
    ap.add_argument("--blocks", type=int, default=8)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch

    import custom_gymnasium_environments_b200 as pkg

    if not torch.cuda.is_available():
        raise SystemExit("snake_tail_probe.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    lib = pkg._lib.load()
    n = args.envs
    stream = torch.cuda.current_stream(dev)
    tapes = torch.empty((256, n), dtype=torch.int64, device=dev)
    for t in range(256):
        pkg._lib.check(lib.beng_fill_random_actions(tapes[t].data_ptr(), n, 1, 4, t, 0, 0, stream.cuda_stream),
                       "beng_fill_random_actions")
    env = pkg.BatchedSnakeEnv(n, 20, device=dev, seed=0)
    env.reset()

    def io_block(parity, done, stats):
        io = env._make_io(env.obs, parity)
        if not done:
            io.done_env = None
        if not stats:
            io.stats = None
        return io

    variants = {"full": (True, True), "no_done": (False, True), "no_stats": (True, False), "neither": (False, False)}
    ios = {name: [io_block(p, *flags) for p in (0, 1)] for name, flags in variants.items()}
    clock = 0

    def step(name):
        nonlocal clock
        env._parity ^= 1
        pkg._lib.check(lib.beng_snake_step_inplace(C.byref(env.params), C.byref(env._state),
                                                   tapes[clock % 256].data_ptr(), C.byref(ios[name][env._parity]),
                                                   n, stream.cuda_stream), "beng_snake_step_inplace")
        clock += 1

    for i in range(args.warmup):
        step(list(variants)[i % len(variants)])
    torch.cuda.synchronize(dev)
    names = list(variants)
    us = {name: [] for name in names}
    for b in range(args.blocks):
        for name in names[b % len(names):] + names[:b % len(names)]:
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(stream)
            for _ in range(args.steps):
                step(name)
            e1.record(stream)
            torch.cuda.synchronize(dev)
            us[name].append(e0.elapsed_time(e1) * 1e3 / args.steps)

    result = {"gpu": gpu_info(), "envs": n, "grid_size": 20, "autoreset_mode": "same_step",
              "steps_per_block": args.steps, "blocks": args.blocks}
    full = statistics.median(us["full"])
    for name in names:
        med = statistics.median(us[name])
        result[name] = {"median_us": med, "min_us": min(us[name]), "max_us": max(us[name]), "blocks_us": us[name],
                        "saving_vs_full": 1.0 - med / full}
    line = json.dumps(result)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
