#!/usr/bin/env python
"""Eager in-place snake step time along the trajectory from reset (1,048,576 envs, G = 20, SAME_STEP, bench.py's
device-generated action tape), for this tree's libbeng and other builds of the same C ABI.

Every build gets its own env, reset with this tree's library and then stepped only through its own build's
beng_snake_step_inplace, so all envs walk the same trajectory when the builds compute the same results (checked at the
end: `obs_equal`).  Windows of --window-steps eager steps are timed between two CUDA events, the builds alternating
window by window, so the time per step can be read from the first steps after reset (length-1 snakes only) to the
steady state.  Records the GPU name, power limit and SM clocks beside the numbers.

    python profiles/snake_traj_probe.py [--lib NAME=PATH ...] [--windows W] [--window-steps S] [--out FILE]
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "profiles"))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--lib", action="append", default=[], metavar="NAME=PATH",
                    help="another build of libbeng.so to time on its own env (repeatable)")
    ap.add_argument("--windows", type=int, default=24)
    ap.add_argument("--window-steps", type=int, default=25)
    ap.add_argument("--out", default=None, help="also write the JSON result to this file")
    args = ap.parse_args()

    import torch

    import custom_gymnasium_environments_b200 as pkg
    from snake_l2_probe import gpu_info

    if not torch.cuda.is_available():
        raise SystemExit("snake_traj_probe.py needs a CUDA device")
    dev = torch.device("cuda", 0)
    L = pkg._lib
    libs = {"this_tree": L.load()}
    for spec in args.lib:
        name, path = spec.split("=", 1)
        lib = C.CDLL(os.path.abspath(path))
        lib.beng_snake_step_inplace.restype, lib.beng_snake_step_inplace.argtypes = \
            L.SIGNATURES["beng_snake_step_inplace"]
        libs[name] = lib
    n, W, pool = 1 << 20, args.window_steps, 256
    stream = torch.cuda.current_stream(dev)
    tapes = torch.empty((pool, n), dtype=torch.int64, device=dev)
    for t in range(pool):  # bench.py's tape: seed 0, env ids from 0
        L.check(libs["this_tree"].beng_fill_random_actions(tapes[t].data_ptr(), n, 1, 4, t, 0, 0, stream.cuda_stream),
                "beng_fill_random_actions")
    envs = {}
    for name in libs:
        envs[name] = pkg.BatchedSnakeEnv(n, 20, device=dev, seed=0)
        envs[name].reset()
    torch.cuda.synchronize(dev)
    out = {"gpu": gpu_info(), "n_envs": n, "window_steps": W,
           "libs": {"this_tree": "this tree's library", **dict(s.split("=", 1) for s in args.lib)},
           "us_per_step": {name: [] for name in libs}}
    names = list(libs)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    for w in range(args.windows):
        for name in (names if w % 2 == 0 else names[::-1]):
            env, lib = envs[name], libs[name]
            p, st, io = C.byref(env.params), C.byref(env._state), C.byref(env._ios[0])
            torch.cuda.synchronize(dev)
            e0.record(stream)
            for t in range(w * W, (w + 1) * W):
                L.check(lib.beng_snake_step_inplace(p, st, tapes[t % pool].data_ptr(), io, n, stream.cuda_stream),
                        "beng_snake_step_inplace")
            e1.record(stream)
            e1.synchronize()
            out["us_per_step"][name].append(round(e0.elapsed_time(e1) * 1e3 / W, 2))
    out["obs_equal"] = {name: bool(torch.equal(envs[name].obs, envs["this_tree"].obs)) for name in libs}
    out["gpu_after"] = gpu_info()
    for name in names:
        print(name, out["us_per_step"][name], flush=True)
    print(json.dumps(out))
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as f:
            f.write(json.dumps(out, indent=1) + "\n")


if __name__ == "__main__":
    main()
