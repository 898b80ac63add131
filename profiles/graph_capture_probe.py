#!/usr/bin/env python
"""Eager step() against the same steps replayed from one CUDA graph, for snake and crypto, on one GPU.

Part 1, graph vs eager (this tree's library, the classes as a user calls them, random device-resident actions):
  eager  `for a in tape: env.step(a)`, 32 steps back to back between two CUDA events
  graph  the same 32-step loop captured once with torch.cuda.graph, replayed back to back between two CUDA events
Snake (G = 20, same_step, in-place step) at 4,096 / 65,536 / 1,048,576 envs; crypto (discrete, same_step) at
4,096 / 32,768 / 262,144 envs.  Each figure is the median over --blocks windows of at least --window seconds each,
the two variants alternating window by window.

Part 2, eager A/B against another build of libbeng (--parent-lib, e.g. the parent commit's library) at the
bench.py sizes (snake 1,048,576, crypto 262,144), both libraries loaded in this process and driven through the C ABI
on the same state buffers, windows alternating:
  this tree   the device-managed contract (crypto io.window_head_dev, snake's self-managed counter block)
  other build the host-managed contract (params.window_head advanced by the host, two ping-pong counters)
so the difference is what the device-resident head / arrival counter cost per step.

Records the GPU name and power limit beside the numbers and writes one JSON file (--out).

    python profiles/graph_capture_probe.py [--parent-lib PATH] [--blocks B] [--window S] [--out FILE]
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
K = 32  # steps per captured loop


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (v.strip() for v in out.split(","))))
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        return {"error": repr(e)}


def timed(torch, fn, reps):
    """Device time of `reps` calls of fn() back to back, in seconds."""
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    e1.synchronize()
    return e0.elapsed_time(e1) * 1e-3


def alternate(torch, variants, steps_per_call, blocks, window):
    """{name: median us per step} over `blocks` windows per variant of >= `window` s, variants alternating."""
    reps = {}
    for name, fn in variants.items():  # warm-up, and the number of calls a window needs
        timed(torch, fn, 3)
        reps[name] = max(3, math.ceil(window / (timed(torch, fn, 10) / 10)))
    out = {name: [] for name in variants}
    names = list(variants)
    for b in range(blocks):
        for name in (names if b % 2 == 0 else names[::-1]):
            out[name].append(timed(torch, variants[name], reps[name]) * 1e6 / (reps[name] * steps_per_call))
    return {name: {"us_per_step": statistics.median(v), "windows_us": [round(x, 3) for x in v],
                   "steps_per_window": reps[name] * steps_per_call} for name, v in out.items()}


def make_env(pkg, kind, n, dev):
    if kind == "snake":
        env = pkg.BatchedSnakeEnv(n, 20, device=dev, seed=0)
        tape = [torch_randint(4, n, dev, t) for t in range(K)]
    else:
        env = pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=dev, seed=0)
        tape = [torch_randint(5, n, dev, t) for t in range(K)]
    env.reset()
    env.step(tape[0])  # snake: env.obs is current from here on, so every timed step is the in-place one
    return env, tape


def torch_randint(hi, n, dev, t):
    import torch

    g = torch.Generator(device=dev).manual_seed(1000 + t)
    return torch.randint(0, hi, (n,), device=dev, generator=g)


def graph_vs_eager(torch, pkg, dev, kind, n, blocks, window):
    env, tape = make_env(pkg, kind, n, dev)

    def eager():
        for a in tape:
            env.step(a)

    eager()
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        eager()
    res = alternate(torch, {"eager": eager, "graph": graph.replay}, K, blocks, window)
    res["graph_speedup"] = res["eager"]["us_per_step"] / res["graph"]["us_per_step"]
    return res


def load_other(path):
    lib = C.CDLL(path)
    from custom_gymnasium_environments_b200 import _lib

    for name in ("beng_snake_step_inplace", "beng_crypto_step"):
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = _lib.SIGNATURES[name]
    return lib


def ab_eager(torch, pkg, dev, kind, n, other, blocks, window):
    L, lib = pkg._lib, pkg._lib.load()
    env, tape = make_env(pkg, kind, n, dev)
    stream = torch.cuda.current_stream(dev).cuda_stream
    p, st = C.byref(env.params), C.byref(env._state)
    if kind == "snake":
        io_new = env._ios[0]
        counts = torch.zeros(2, dtype=torch.int32, device=dev)
        io_old = []
        for parity in (0, 1):
            io = L.SnakeIO.from_buffer_copy(io_new)
            io.done_count, io.done_count_next = counts.data_ptr() + 4 * parity, counts.data_ptr() + 4 * (1 - parity)
            io_old.append(io)

        def new():
            for a in tape:
                L.check(lib.beng_snake_step_inplace(p, st, a.data_ptr(), C.byref(io_new), n, stream), "new")

        def old():
            for t, a in enumerate(tape):
                L.check(other.beng_snake_step_inplace(p, st, a.data_ptr(), C.byref(io_old[t & 1]), n, stream), "old")
    else:
        io_new = env._io
        io_old = L.CryptoIO.from_buffer_copy(io_new)
        io_old.window_head_dev = None
        p_old = L.CryptoParams.from_buffer_copy(env.params)

        def new():
            for a in tape:
                L.check(lib.beng_crypto_step(p, st, a.data_ptr(), C.byref(io_new), n, stream), "new")

        def old():
            for a in tape:
                L.check(other.beng_crypto_step(C.byref(p_old), st, a.data_ptr(), C.byref(io_old), n, stream), "old")
                p_old.window_head = (p_old.window_head + 1) % 50

    res = alternate(torch, {"this_tree": new, "other_build": old}, K, blocks, window)
    res["delta_us"] = res["this_tree"]["us_per_step"] - res["other_build"]["us_per_step"]
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--parent-lib", default=None, help="libbeng.so of another build for the eager A/B (part 2)")
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--window", type=float, default=0.5, help="seconds per timed window")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "graph_capture_probe_b200.json"))
    args = ap.parse_args()

    import torch

    import custom_gymnasium_environments_b200 as pkg

    if not torch.cuda.is_available():
        raise SystemExit("graph_capture_probe.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    out = {"gpu": gpu_info(), "device_name": torch.cuda.get_device_name(dev), "steps_per_graph": K,
           "window_s": args.window, "blocks": args.blocks, "graph_vs_eager": {}, "eager_ab": {}}
    for kind, sizes in (("snake", (4096, 65536, 1 << 20)), ("crypto", (4096, 32768, 262144))):
        for n in sizes:
            out["graph_vs_eager"][f"{kind}_{n}"] = r = graph_vs_eager(torch, pkg, dev, kind, n, args.blocks, args.window)
            print(kind, n, {k: (v["us_per_step"] if isinstance(v, dict) else v) for k, v in r.items()}, flush=True)
    if args.parent_lib:
        out["eager_ab"]["other_build"] = os.path.basename(os.path.dirname(os.path.abspath(args.parent_lib)))
        other = load_other(args.parent_lib)
        for kind, n in (("snake", 1 << 20), ("crypto", 262144)):
            out["eager_ab"][f"{kind}_{n}"] = r = ab_eager(torch, pkg, dev, kind, n, other, args.blocks, args.window)
            print("A/B", kind, n, {k: (v["us_per_step"] if isinstance(v, dict) else v) for k, v in r.items()},
                  flush=True)
    out["gpu_after"] = gpu_info()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(out, f, indent=1)
    print(json.dumps({k: out[k] for k in ("gpu", "device_name")}))


if __name__ == "__main__":
    main()
