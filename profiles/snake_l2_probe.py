#!/usr/bin/env python
"""Per-env-step time of the in-place snake step (beng_snake_step_inplace, G = 20, SAME_STEP, random actions) against
the number of envs, to find where the step's L2 footprint outgrows the 126 MB L2.

For every env count (default 262,144 ... 2,097,152) one BatchedSnakeEnv is reset, stepped once (so that env.obs is
current and every timed step is the in-place one) and then stepped two ways:
  graph        K steps (distinct device-resident action tensors, K * 8 B * n >= 256 MB so the tape itself does not
               stay in L2) captured once in a CUDA graph and replayed back to back between two CUDA events: no launch
               overhead, the L2 as the previous step left it
  l2_flushed   one step at a time between its own two events, a 256 MB fill (untimed) between steps
Each figure is the median over --blocks windows; the libraries alternate window by window.

--lib NAME=PATH (repeatable) times other builds of libbeng with the same C ABI on the same env and state buffers, so
builds A/B in one process: each build's step is captured in its own graph, all of them advance the same envs, and
every build must compute the same results for the run to make sense (the tests check that; this probe does not).
Without --lib only this tree's library is timed.  Records the GPU name, power limit and SM clocks beside the numbers.

    python profiles/snake_l2_probe.py [--sizes N ...] [--lib NAME=PATH ...] [--blocks B] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
SIZES = (262144, 393216, 524288, 786432, 1048576, 2097152)


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
    ap.add_argument("--sizes", type=int, nargs="+", default=list(SIZES))
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH",
                    help="another build of libbeng.so to time on the same envs (repeatable)")
    ap.add_argument("--blocks", type=int, default=5, help="windows per build, size and mode")
    ap.add_argument("--window", type=float, default=0.25, help="seconds per back-to-back window")
    ap.add_argument("--flushed-steps", type=int, default=40, help="steps per L2-flushed window")
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch

    import custom_gymnasium_environments_b200 as pkg

    if not torch.cuda.is_available():
        raise SystemExit("snake_l2_probe.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    L = pkg._lib
    libs = {"this_tree": L.load()}
    for spec in args.lib:
        name, path = spec.split("=", 1)
        lib = C.CDLL(os.path.abspath(path))
        lib.beng_snake_step_inplace.restype, lib.beng_snake_step_inplace.argtypes = \
            L.SIGNATURES["beng_snake_step_inplace"]
        libs[name] = lib
    stream = torch.cuda.current_stream(dev)
    scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    out = {"gpu": gpu_info(), "grid_size": 20, "autoreset_mode": "same_step", "blocks": args.blocks,
           "window_s": args.window, "flushed_steps": args.flushed_steps,
           "libs": {"this_tree": "this tree's library", **dict(s.split("=", 1) for s in args.lib)}, "sizes": {}}

    for n in args.sizes:
        env = pkg.BatchedSnakeEnv(n, 20, device=dev, seed=0)
        k = max(32, math.ceil((256 << 20) / (8 * n)))
        gen = torch.Generator(device=dev).manual_seed(n)
        tape = [torch.randint(0, 4, (n,), device=dev, generator=gen) for _ in range(k)]
        env.reset()
        env.step(tape[0])
        p, st, io = C.byref(env.params), C.byref(env._state), C.byref(env._ios[0])

        def stepper(lib):
            def run(a):
                s = torch.cuda.current_stream(dev).cuda_stream  # (the capture stream inside torch.cuda.graph)
                L.check(lib.beng_snake_step_inplace(p, st, a.data_ptr(), io, n, s), "step")
            return run

        steps = {name: stepper(lib) for name, lib in libs.items()}
        graphs = {}
        for name, run in steps.items():
            for a in tape:  # warm-up outside the capture
                run(a)
            torch.cuda.synchronize(dev)
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for a in tape:
                    run(a)
            graphs[name] = g
        for g in graphs.values():
            g.replay()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        graphs["this_tree"].replay()
        e1.record(stream)
        e1.synchronize()
        reps = max(2, math.ceil(args.window / (e0.elapsed_time(e1) * 1e-3)))

        res = {name: {"graph_us": [], "l2_flushed_us": []} for name in libs}
        names = list(libs)
        clock = 0
        for b in range(args.blocks):
            order = names if b % 2 == 0 else names[::-1]
            for name in order:
                e0.record(stream)
                for _ in range(reps):
                    graphs[name].replay()
                e1.record(stream)
                e1.synchronize()
                res[name]["graph_us"].append(e0.elapsed_time(e1) * 1e3 / (reps * k))
            for name in order:
                pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))
                         for _ in range(args.flushed_steps)]
                for i in range(args.flushed_steps):
                    scratch.fill_(i & 0xFF)
                    pairs[i][0].record(stream)
                    steps[name](tape[clock % k])
                    clock += 1
                    pairs[i][1].record(stream)
                torch.cuda.synchronize(dev)
                res[name]["l2_flushed_us"].append(sum(x.elapsed_time(y) for x, y in pairs) * 1e3 / args.flushed_steps)
        row = {"steps_per_graph": k, "graph_replays_per_window": reps}
        for name, r in res.items():
            row[name] = {}
            for mode, xs in r.items():
                med = statistics.median(xs)
                row[name][mode] = {"median": round(med, 3), "min": round(min(xs), 3), "max": round(max(xs), 3),
                                   "ns_per_env_step": round(med * 1e3 / n, 4)}
        out["sizes"][str(n)] = row
        print(n, json.dumps({name: {m: v["median"] for m, v in row[name].items()} for name in libs}), flush=True)
        del graphs, env, tape
        torch.cuda.empty_cache()

    out["gpu_after"] = gpu_info()
    line = json.dumps(out)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
