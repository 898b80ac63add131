"""End-to-end rate of step_host with the full observation copy against delta_obs=True.

    python profiles/e2e_delta_probe.py [--env snake|builder] [--blocks 6] [--out FILE]

--env snake (the default): BatchedSnakeEnv, G = 20.  --env builder: BatchedWorldBuilderEnv, G = 10, whose grid is the
part of the observation that the delta path patches.  Two envs with the same seed (same_step auto-reset) are stepped
from the same pinned host action tapes, built like bench.py's e2e tapes (beng_fill_random_actions on the device with
the env's bench.py action count, then pinned host copies), in alternating timed blocks of the full path and the delta
path within one process, after warm-up.  Every step is synchronous, as a caller of the numpy API sees it.  The delta
path's time is split into the host apply (beng_<env>_apply_obs_delta, timed around the call) and the rest (H2D
actions, kernel, D2H of records and results, stream synchronise).  At the end the two envs' host observations and
device observations must be equal.  Prints one JSON line; needs a CUDA GPU.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (pin_to_gpu_numa_node, pcie_ceiling: the same helpers as bench.py's e2e arm)

RECORD_BYTES = 4


class Snake:  # the classes themselves are the specs (never instantiated): their functions are called on the class
    probe = "snake step_host: full observation copy vs delta_obs=True"
    G, n_choices, apply = 20, 4, "beng_snake_apply_obs_delta"
    result_bytes = 4 + 1 + 1 + 4 + 4  # reward, terminated, truncated, score, snake_length per env
    steps_per_block = {1 << 20: 25, 1 << 16: 200}

    def make(pkg, n, dev):
        return pkg.BatchedSnakeEnv(n, Snake.G, device=dev, seed=0, autoreset_mode="same_step")

    def host_obs(out):
        return out[0]

    def device_obs(env):
        return env.obs


class Builder:
    probe = "world-builder step_host: full grid copy vs delta_obs=True"
    G, n_choices, apply = 10, 5, "beng_builder_apply_obs_delta"
    result_bytes = 16 + 4 + 4 + 4 + 1  # resources, population_capacity, win_steps, reward, terminated per env
    steps_per_block = {1 << 20: 100, 1 << 16: 1000}

    def make(pkg, n, dev):
        return pkg.BatchedWorldBuilderEnv(n, Builder.G, device=dev, seed=0, autoreset_mode="same_step")

    def host_obs(out):
        return out[0]["grid"]

    def device_obs(env):
        return env.grid


ENVS = {"snake": Snake, "builder": Builder}


class TimedApply:
    """Stands in for env.lib and accumulates the wall time spent in the env's apply function."""

    def __init__(self, lib, apply):
        self._lib, self._apply, self.seconds, self.calls = lib, apply, 0.0, 0

    def __getattr__(self, name):
        fn = getattr(self._lib, name)
        if name != self._apply:
            return fn

        def timed(*args):
            t0 = time.perf_counter()
            rc = fn(*args)
            self.seconds += time.perf_counter() - t0
            self.calls += 1
            return rc
        return timed


def gpu_facts(index):
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    out = subprocess.run(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                         capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return dict(zip(("gpu", "power_limit_w", "sm_clock_mhz", "sm_clock_max_mhz"), out))  # as nvidia-smi prints them


def measure(pkg, spec, n, blocks, steps_per_block, dev):
    lib, G = pkg._lib.load(), spec.G
    envs = {k: spec.make(pkg, n, dev) for k in ("full", "delta")}
    for e in envs.values():
        e.reset()
    timer = envs["delta"].lib = TimedApply(envs["delta"].lib, spec.apply)
    pool = 8
    tapes = torch.empty((pool, n), dtype=torch.int64, device=dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    for t in range(pool):
        pkg._lib.check(lib.beng_fill_random_actions(tapes[t].data_ptr(), n, 1, spec.n_choices, t, 0, 0, stream),
                       "beng_fill_random_actions")
    host_tapes = [tapes[t].cpu().pin_memory() for t in range(pool)]
    cursor = {"full": 0, "delta": 0}

    def run(kind, steps):
        env, t0 = envs[kind], time.perf_counter()
        for _ in range(steps):
            out = env.step_host(host_tapes[cursor[kind] % pool], delta_obs=(kind == "delta"))
            cursor[kind] += 1
        return time.perf_counter() - t0, out

    for kind in envs:  # warm-up; the delta env's first call seeds its mirror with a full copy
        run(kind, 3)
    secs = {"full": [], "delta": []}
    last = {}
    apply_s = 0.0
    for _ in range(blocks):
        for kind in ("full", "delta"):
            before = timer.seconds
            dt, out = run(kind, steps_per_block)
            secs[kind].append(dt)
            if kind == "delta":
                apply_s += timer.seconds - before
            last[kind] = spec.host_obs(out)
    equal = bool(np.array_equal(last["full"], last["delta"])
                 and torch.equal(spec.device_obs(envs["full"]), spec.device_obs(envs["delta"])))
    steps = blocks * steps_per_block

    def rates(kind):
        per_block = [n * steps_per_block / s for s in secs[kind]]
        total = sum(secs[kind])
        return {"env_steps_per_s": n * steps / total, "ms_per_step": 1e3 * total / steps,
                "env_steps_per_s_blocks": {"min": min(per_block), "median": statistics.median(per_block),
                                           "max": max(per_block)}}

    full, delta = rates("full"), rates("delta")
    full.update(h2d_bytes_per_step=8 * n, d2h_bytes_per_step=n * (G * G + spec.result_bytes))
    delta.update(h2d_bytes_per_step=8 * n, d2h_bytes_per_step=n * (RECORD_BYTES + spec.result_bytes),
                 apply_ms_per_step=1e3 * apply_s / steps,
                 device_ms_per_step=1e3 * (sum(secs["delta"]) - apply_s) / steps,
                 device_note="H2D actions + step kernel + D2H records/results + stream synchronise, Python included")
    ceiling = bench.pcie_ceiling(torch, dev, n * G * G)
    del envs, tapes
    torch.cuda.empty_cache()
    return {"n_envs": n, "grid_size": G, "autoreset": "same_step", "blocks": blocks, "steps_per_block": steps_per_block,
            "full": full, "delta": delta, "speedup": delta["env_steps_per_s"] / full["env_steps_per_s"],
            "pinned_copy_ceiling_gbs": {"d2h": ceiling["d2h"], "h2d": ceiling["h2d"],
                                        "bytes": int(max(1 << 20, min(n * G * G, 1 << 30)))},
            "obs_equal": equal}


def main():
    ap = argparse.ArgumentParser(description=__doc__.split("\n")[0])
    ap.add_argument("--env", choices=sorted(ENVS), default="snake")
    ap.add_argument("--blocks", type=int, default=6)
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("e2e_delta_probe.py measures the GPU path and needs a CUDA device")
    import custom_gymnasium_environments_b200 as pkg

    spec = ENVS[args.env]
    dev = torch.device("cuda:0")
    numa_bound, _ = bench.pin_to_gpu_numa_node(0)
    result = {"probe": spec.probe, "numa_bound": numa_bound, "threads": len(os.sched_getaffinity(0)), "sizes": []}
    for n, per_block in spec.steps_per_block.items():
        result["sizes"].append(measure(pkg, spec, n, args.blocks, per_block, dev))
        if n == 1 << 20:
            result.update(gpu_facts(0))  # clocks read right after the large size's timed blocks
    line = json.dumps(result)
    print(line)
    if args.out:
        with open(args.out, "w") as f:
            f.write(line + "\n")
    if not all(s["obs_equal"] for s in result["sizes"]):
        raise SystemExit("observations of the two paths differ")


if __name__ == "__main__":
    main()
