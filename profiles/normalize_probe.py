#!/usr/bin/env python
"""Cost of VecNormalize per step on one GPU, next to the env step and a plain torch composition of the same semantics.

For each (env, num_envs) it times, eager and replayed from one CUDA graph of K steps, with device-resident actions:
  env      env.step alone
  train    VecNormalize(env).step in training mode (moments pass + apply pass)
  frozen   the same with training = False (apply pass only)
  torch    env.step followed by a torch composition of the same semantics (var_mean, Chan's update, clamp, ...)
Every figure is the median of --blocks windows of `reps` K-step calls, variants alternating window by window, timed with
CUDA events after a warm-up.  L2 is NOT flushed between steps (the env's step itself writes the observations the
normalization reads).  It also checks, from one shared state, that the torch composition and the CUDA path agree.

The byte model of one training step per env is 12 * dim + 26 B (observations read twice and written once, reward,
flags, returns and output reward), 8 * dim + 8 B frozen; `model_fraction` is that many bytes at 7.7 TB/s over the
measured added time.  Records the GPU name and power limit beside the numbers and writes one JSON file (--out).

    python profiles/normalize_probe.py [--blocks B] [--out FILE]
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
K = 10  # steps per captured loop
HBM_BYTES_PER_S = 7.7e12
CONFIGS = [("crypto", 262144), ("traffic", 65536), ("traffic", 1048576), ("climate", 1048576), ("builder", 1048576)]


def gpu_info():
    q = "name,power.limit,clocks.sm,clocks.max.sm"
    try:
        out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"],
                             capture_output=True, text=True, timeout=30).stdout.strip()
        return dict(zip(q.split(","), (v.strip() for v in out.split(","))))
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        return {"error": repr(e)}


def make_env(pkg, kind, n):
    if kind == "crypto":
        return pkg.BatchedCryptoTradingEnv(n, None, "discrete", seed=1)
    if kind == "traffic":
        return pkg.BatchedTrafficManagementEnv(n, seed=1)
    if kind == "climate":
        return pkg.BatchedSmartClimateEnv(n, seed=1)
    return pkg.BatchedWorldBuilderEnv(n, flatten_obs=True, seed=1)


def make_actions(torch, kind, env):
    n, g = env.num_envs, torch.Generator(device="cuda").manual_seed(0)
    if kind == "crypto" or kind == "builder":
        return torch.randint(0, 5, (n,), device="cuda", generator=g)
    if kind == "traffic":
        return torch.randint(0, 3, (n, env.num_intersections), device="cuda", generator=g)
    return {"ac_temp": torch.rand(n, device="cuda", generator=g) * 16 + 16,
            "lights": torch.randint(0, 2, (n, 4), device="cuda", generator=g).to(torch.int8)}


class TorchNormalize:
    """The VecNormalize semantics as plain torch ops on persistent device tensors (capturable)."""

    def __init__(self, torch, n, dim, clip=10.0, gamma=0.99, eps=1e-8):
        self.t, self.clip, self.gamma, self.eps = torch, clip, gamma, eps
        f64 = dict(dtype=torch.float64, device="cuda")
        self.mean, self.var, self.count = torch.zeros(dim, **f64), torch.ones(dim, **f64), torch.full((), 1e-4, **f64)
        self.rmean, self.rvar, self.rcount = torch.zeros((), **f64), torch.ones((), **f64), torch.full((), 1e-4, **f64)
        self.returns = torch.zeros(n, **f64)
        self.obs = torch.zeros(n, dim, dtype=torch.float32, device="cuda")
        self.rew = torch.zeros(n, dtype=torch.float32, device="cuda")

    def load(self, w):
        d = w.dim
        self.mean.copy_(w.obs_rms.data[:d]), self.var.copy_(w.obs_rms.data[d:2 * d]), self.count.copy_(w.obs_rms.data[-1])
        self.rmean.copy_(w.ret_rms.data[0]), self.rvar.copy_(w.ret_rms.data[1]), self.rcount.copy_(w.ret_rms.data[2])
        self.returns.copy_(w.returns)

    @staticmethod
    def _merge(torch, mean, var, count, x):
        b_var, b_mean = torch.var_mean(x, 0, correction=0)
        n = x.shape[0]
        delta = b_mean - mean
        tot = count + n
        m2 = var * count + b_var * n + delta * delta * count * n / tot
        mean.add_(delta * n / tot)
        var.copy_(m2 / tot)
        count.add_(n)

    def step(self, obs, reward, terminated, truncated, training=True):
        torch = self.t
        x = obs.double()
        if training:
            self._merge(torch, self.mean, self.var, self.count, x)
        self.obs.copy_(((x - self.mean) / torch.sqrt(self.var + self.eps)).clamp_(-self.clip, self.clip))
        if training:
            self.returns.mul_(self.gamma).add_(reward.double())
            self._merge(torch, self.rmean, self.rvar, self.rcount, self.returns)
        self.rew.copy_((reward.double() / torch.sqrt(self.rvar + self.eps)).clamp_(-self.clip, self.clip))
        self.returns.masked_fill_(terminated | truncated, 0.0)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--blocks", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "normalize_probe_b200.json"))
    args = ap.parse_args()
    import torch

    import custom_gymnasium_environments_b200 as pkg

    assert torch.cuda.is_available(), "the probe measures on a GPU"
    result = {"gpu": gpu_info(), "torch": torch.__version__, "steps_per_graph": K, "l2_flushed": False, "configs": []}
    for kind, n in CONFIGS:
        env = make_env(pkg, kind, n)
        w = pkg.VecNormalize(env)
        w.reset()
        act = make_actions(torch, kind, env)
        tn = TorchNormalize(torch, n, w.dim)

        # agreement from one shared state: the wrapper's statistics before a step feed the torch composition
        for _ in range(3):
            w.step(act)
        tn.load(w)
        w.step(act)
        tn.step(raw := (env.flat_obs if kind == "builder" else env.obs), env.reward, env.terminated, env.truncated)
        d = w.dim
        rel = lambda a, b: float(((a - b).abs() / b.abs().clamp_min(1e-300)).max())  # noqa: E731
        check = {"obs_max_abs_diff": float((w.obs - tn.obs).abs().max()),
                 "reward_max_abs_diff": float((w.reward - tn.rew).abs().max()),
                 "mean_max_rel_diff": rel(w.obs_rms.data[:d], tn.mean),
                 "var_max_rel_diff": rel(w.obs_rms.data[d:2 * d], tn.var),
                 "ret_var_rel_diff": rel(w.ret_rms.data[1:2], tn.rvar.reshape(1)),
                 "returns_equal": bool(torch.equal(w.returns, tn.returns))}
        del raw

        def run_env():
            env.step(act)

        def run_train():
            w.training = True
            w.step(act)

        def run_frozen():
            w.training = False
            w.step(act)

        def run_torch():
            o, r, te, tr, _ = env.step(act)
            tn.step(env.flat_obs if kind == "builder" else o, r, te, tr)

        eager = {"env": run_env, "train": run_train, "frozen": run_frozen, "torch": run_torch}
        graphs = {}
        for name, fn in eager.items():
            for _ in range(3):
                fn()
            torch.cuda.synchronize()
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g):
                for _ in range(K):
                    fn()
            graphs[name] = g
        w.training = True
        # reps per window: about 0.2 s of steps (one timed eager window sizes it)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(K):
            run_torch()
        e1.record()
        e1.synchronize()
        reps = max(2, int(0.2 / max(e0.elapsed_time(e1) * 1e-3, 1e-6)))
        samples = {f"{m}_{v}": [] for m in ("eager", "graph") for v in eager}
        for _ in range(args.blocks):
            for v, fn in eager.items():
                for _ in range(K):  # warm-up of this variant's state
                    fn()
                e0.record()
                for _ in range(reps):
                    for _ in range(K):
                        fn()
                e1.record()
                e1.synchronize()
                samples[f"eager_{v}"].append(e0.elapsed_time(e1) * 1e3 / (reps * K))
                graphs[v].replay()
                e0.record()
                for _ in range(reps):
                    graphs[v].replay()
                e1.record()
                e1.synchronize()
                samples[f"graph_{v}"].append(e0.elapsed_time(e1) * 1e3 / (reps * K))
        us = {k: statistics.median(s) for k, s in samples.items()}
        train_bytes, frozen_bytes = n * (12 * d + 26), n * (8 * d + 8)
        row = {"env": kind, "num_envs": n, "dim": d, "us_per_step": us, "spread_us": {k: [min(s), max(s)] for k, s in samples.items()},
               "check": check, "train_bytes": train_bytes, "frozen_bytes": frozen_bytes}
        for m in ("eager", "graph"):
            for v, b in (("train", train_bytes), ("frozen", frozen_bytes), ("torch", train_bytes)):
                added = us[f"{m}_{v}"] - us[f"{m}_env"]
                row[f"{m}_{v}_added_us"] = added
                if v != "torch":
                    row[f"{m}_{v}_model_fraction"] = (b / HBM_BYTES_PER_S * 1e6) / added if added > 0 else None
        result["configs"].append(row)
        print(json.dumps({k: row[k] for k in ("env", "num_envs", "dim")}), json.dumps(us), json.dumps(check), flush=True)
        del env, w, tn, graphs
        torch.cuda.empty_cache()
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
