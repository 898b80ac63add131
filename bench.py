#!/usr/bin/env python
"""Benchmark of the batched env-step hot path (BASELINE.json: env-steps/sec; headline = batched SnakeEnv, 1M envs/GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--env snake|crypto|traffic|climate|builder]   # this repo's CUDA engine
    python bench.py --impl reference [--gpus N] --steps K --warmup W [--env …]  # CPU arm: the reference's step loop
    python bench.py … --dump-outputs DIR   # also write the last timed step's outputs as DIR/*.npy (dump_step_outputs)

A "step" is ONE launch of the fused step kernel over the whole batch, inputs resident in HBM; `value` =
envs x steps x ranks / max-over-ranks device time (CUDA events).  `e2e` is the same metric through the
host-buffer C-ABI call (`beng_<env>_step_host`: pinned host actions in, numpy obs/reward/terminated out, copies
inside the timed region).  `roofline` uses SURVEY.md 8(d)'s algorithmic bytes per env-step against the measured HBM
copy bandwidth in MEASURED_PEAKS.json.  `cpu_baseline` times the UNMODIFIED reference class in its own per-env Python
step loop (oracle/ref_loader.py: /root/reference here, the byte-for-byte copies staged under oracle/_ref by
`python -m oracle.make_ref` on the GPU box; `kind: "reference"`, the oracle port only if neither exists) on the host
cores, rank 0 at N=1 only.  The default `--env snake` run appends device-timed crypto and traffic blocks (BASELINE
configs[2], [3]) as `secondary`.

Prints exactly one JSON line on stdout (rank 0).
"""
from __future__ import annotations

import argparse
import json
import multiprocessing as mp
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "env_steps_per_sec"
UNIT = "env-steps/s"
FALLBACK_HBM_GBS = 6650.0  # /opt/skills/guides/B200_PROFILING.md fallback when MEASURED_PEAKS.json is absent


class Workload:
    """Per-env benchmark description (BASELINE.json configs[1..3])."""

    def __init__(self, name, envs_per_gpu, bytes_per_env_step, n_choices, n_cols, dtype, label, obs_bytes,
                 result_bytes, cpu_single_steps):
        self.name, self.envs_per_gpu, self.bytes = name, envs_per_gpu, bytes_per_env_step
        self.n_choices, self.n_cols, self.dtype, self.label = n_choices, n_cols, dtype, label
        self.obs_bytes, self.result_bytes, self.cpu_single_steps = obs_bytes, result_bytes, cpu_single_steps


WORKLOADS = {
    # SURVEY.md 8(d): obs 400 W + action 8 R + reward 4 W + flags 2 W + state 16 R/W + ring 2 R/W
    "snake": Workload("snake", 1 << 20, 450, 4, 1, "u8",
                      "batched SnakeEnvClassic, G=20, random actions, SAME_STEP auto-reset (BASELINE.json configs[1])",
                      400, 4 + 1 + 1 + 4 + 4, 20000),
    # SURVEY.md 8(d): window read 1000 + candle 20 + obs 1044 W + action 8 + reward/flags 6 + scalars 112.
    # (The "+408 if closes are kept in float64" is NOT added although they are: the lower figure is the
    # conservative denominator.)
    "crypto": Workload("crypto", 1 << 18, 2190, 5, 1, "f64",
                       "batched CryptoTradingEnv, discrete actions, default TradingConfig, fp64 dynamics / fp32 obs, "
                       "SAME_STEP auto-reset (BASELINE.json configs[2])", 1044, 4 + 1 + 1, 300),
    # SURVEY.md 8(d): obs 520 W + actions 72 R + reward/flags 6 + lights 36 + vehicle pool 400 + counters 144 + scalars 32
    "traffic": Workload("traffic", 1 << 16, 1210, 3, 9, "i32",
                        "batched TrafficManagementEnv, default config (9 intersections, 50 vehicles, spawn 0.3), "
                        "SAME_STEP auto-reset (BASELINE.json configs[3])", 520, 4 + 1 + 1, 600),
    # SURVEY.md 8(f) rank 3 (no BASELINE config): state 5 x f64 + 4 x i32 read and written (112 + 112... = 80 + 32 each
    # way), obs 36 W, action 8 R, reward 4 W, flags 2 W
    "climate": Workload("climate", 1 << 20, 162, 2, 5, "f64",
                        "batched SmartClimateEnv (SURVEY.md 8f rank 3), default config, random Dict actions, "
                        "SAME_STEP auto-reset", 36, 4 + 1 + 1, 3000),
    # SURVEY.md 8(f) rank 3 (no BASELINE config): grid 100 R + 100 W (state = observation, rewritten in place),
    # scalar state 40 R + 40 W, resources/capacity/win_steps 24 W, action 8 R, reward 4 W, flags 2 W
    "builder": Workload("builder", 1 << 20, 318, 5, 1, "i32",
                        "batched WorldBuilderEnv (SURVEY.md 8f rank 3), 10x10 grid, Dict observation, random actions, "
                        "SAME_STEP auto-reset", 100 + 16 + 4 + 4, 4 + 1, 6000),
}


# ------------------------------------------------------------------------------------------------
# CPU arm: the reference's own per-env Python step loop, one env per process
# ------------------------------------------------------------------------------------------------
def reference_kind() -> str:
    """"reference" when the unmodified reference classes can be imported (/root/reference in the build container,
    oracle/_ref on the GPU box -- staged by `python -m oracle.make_ref`), else "port" (oracle/*_port.py)."""
    from oracle import ref_loader

    return "reference" if ref_loader.reference_available() else "port"


def _make_cpu_env(env_name, worker, kind):
    """-> (env, sample_action).  kind "reference": the UNMODIFIED reference class behind the stub gymnasium/pygame
    (oracle/ref_loader.py), seeded through the module-level RNGs it really uses; kind "port": oracle/*_port.py."""
    import random

    import numpy as np

    rng = random.Random(1234 + worker)
    randrange, uniform = rng.randrange, rng.uniform
    samplers = {
        "snake": lambda: randrange(4),
        "crypto": lambda: randrange(5),
        "builder": lambda: randrange(5),
        # MultiDiscrete([3]*9) sample, like env.action_space.sample() in traffic_management_env/test_env.py:266-278
        "traffic": lambda: np.array([randrange(3) for _ in range(9)]),
        # Dict action sample: ac_temp Box(16, 32, (1,)), lights MultiBinary(4)
        "climate": lambda: {"ac_temp": np.array([uniform(16.0, 32.0)], dtype=np.float32),
                            "lights": np.array([randrange(2) for _ in range(4)], dtype=np.int8)},
    }
    if kind == "reference":
        import logging

        from oracle import ref_loader

        random.seed(4321 + worker)      # snake / crypto / traffic draw from the process-global `random` ...
        np.random.seed(4321 + worker)   # ... crypto and world_builder also from `np.random`
        if env_name == "snake":
            env = ref_loader.load_snake().SnakeEnvClassic()
        elif env_name == "crypto":
            env = ref_loader.load_crypto().CryptoTradingEnv(action_type="discrete")
        elif env_name == "traffic":
            env = ref_loader.load_traffic()[0].TrafficManagementEnv()
        elif env_name == "climate":
            env = ref_loader.load_climate().SmartClimateEnv(log_level=logging.ERROR)
        else:
            env = ref_loader.load_builder()[0].WorldBuilderEnv()
    else:
        if env_name == "snake":
            from oracle.snake_port import SnakePort

            env = SnakePort(20, rng=rng)
        elif env_name == "crypto":
            from oracle.crypto_port import CryptoPort

            np.random.seed(1234 + worker)
            env = CryptoPort(action_type="discrete")
        elif env_name == "builder":
            from oracle.builder_port import BuilderPort

            np.random.seed(1234 + worker)
            env = BuilderPort()
        elif env_name == "climate":
            from oracle.climate_port import ClimatePort

            env = ClimatePort(seed=1234 + worker)
        else:
            from oracle.traffic_port import TrafficPort

            env = TrafficPort(rng=rng)
    return env, samplers[env_name]


def _cpu_worker_loop(args):
    """Step one env with random actions and reset-on-done for `n_steps` steps -- the loop shape of the reference's own
    harness, crypto_trading_env/test_crypto_trading.py:410-416.  Returns (steps, seconds)."""
    env_name, worker, n_steps, kind = args
    env, sample = _make_cpu_env(env_name, worker, kind)
    env.reset()
    step, reset = env.step, env.reset
    t0 = time.perf_counter()
    for _ in range(n_steps):
        _, _, term, trunc, _ = step(sample())
        if term or trunc:
            reset()
    return n_steps, time.perf_counter() - t0


def cpu_rate_single(env_name: str, seconds: float, kind: str) -> float:
    probe = WORKLOADS[env_name].cpu_single_steps
    n, dt = _cpu_worker_loop((env_name, 0, probe, kind))
    rate = n / dt
    n, dt = _cpu_worker_loop((env_name, 0, max(probe, int(rate * seconds)), kind))
    return n / dt


def cpu_rate_parallel(pool, env_name: str, procs: int, steps_per_proc: int, kind: str):
    t0 = time.perf_counter()
    res = pool.map(_cpu_worker_loop, [(env_name, w, steps_per_proc, kind) for w in range(procs)])
    wall = time.perf_counter() - t0
    return sum(r[0] for r in res) / wall, wall


def c_oracle_rate(env_name: str, seconds: float = 1.5) -> float:
    """Throughput of the plain-C oracle (1 thread), for context next to the Python port."""
    import numpy as np

    from oracle import c_oracle

    rng = np.random.default_rng(0)
    if env_name == "snake":
        n = 1 << 15
        orc = c_oracle.SnakeOracle(n, seed=0)
        acts = rng.integers(0, 4, (16, n))
    elif env_name == "crypto":
        n = 1 << 11
        orc = c_oracle.CryptoOracle(n, seed=0)
        acts = rng.integers(0, 5, (16, n))
    elif env_name == "builder":
        n = 1 << 14
        orc = c_oracle.BuilderOracle(n, seed=0)
        acts = rng.integers(0, 5, (16, n))
    elif env_name == "climate":
        n = 1 << 14
        orc = c_oracle.ClimateOracle(n, seed=0)
        ac = (rng.random((16, n)) * 16 + 16).astype(np.float32)
        li = rng.integers(0, 2, (16, n, 4)).astype(np.int8)
        orc.reset()
        t0 = time.perf_counter()
        k = 0
        while time.perf_counter() - t0 < seconds:
            orc.step(ac[k % 16], li[k % 16])
            k += 1
        return n * k / (time.perf_counter() - t0)
    else:
        n = 1 << 10
        orc = c_oracle.TrafficOracle(n, seed=0)
        acts = rng.integers(0, 3, (16, n, 9))
    orc.reset()
    orc.step(acts[0])
    t0 = time.perf_counter()
    k = 0
    while time.perf_counter() - t0 < seconds:
        orc.step(acts[k % 16])
        k += 1
    return n * k / (time.perf_counter() - t0)


def cpu_arm_description(env_name, kind, cores, per_proc):
    ref = {"snake": "snake_env_classic/snake_env.py SnakeEnvClassic, G=20",
           "crypto": "crypto_trading_env/crypto_trading_env.py CryptoTradingEnv, discrete actions",
           "traffic": "traffic_management_env/environment.py TrafficManagementEnv, default config",
           "climate": "smartclimate/env.py SmartClimateEnv, default config",
           "builder": "world_builder_env WorldBuilderEnv, 10x10 grid"}[env_name]
    what = (f"the UNMODIFIED reference class ({ref}) behind stub gymnasium/pygame" if kind == "reference"
            else f"pure-Python port (oracle/{env_name}_port.py) of {ref}")
    return (f"{what}: 1 env per process x {cores} processes x {per_proc} random-action steps with reset-on-done "
            f"(os.cpu_count() = {os.cpu_count()})")


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", 0))
    if rank != 0:
        return  # rank 0 alone runs the CPU arm
    w = WORKLOADS[args.env]
    cores = os.cpu_count() or 1
    kind = reference_kind()
    single = cpu_rate_single(args.env, 1.0, kind)
    budget_s = 60.0
    per_step = int(min(50000, max(20, single * budget_s / max(1, args.steps + args.warmup))))
    ctx = mp.get_context("fork")
    with ctx.Pool(cores) as pool:
        for _ in range(args.warmup):
            cpu_rate_parallel(pool, args.env, cores, per_step, kind)
        t0 = time.perf_counter()
        total = 0
        for _ in range(args.steps):
            res = pool.map(_cpu_worker_loop, [(args.env, k, per_step, kind) for k in range(cores)])
            total += sum(r[0] for r in res)
        wall = time.perf_counter() - t0
    value = total / wall
    baseline = {"value": value, "unit": UNIT, "cores": cores, "kind": kind,
                "sample": cpu_arm_description(args.env, kind, cores, per_step) + " per bench step",
                "single_core_value": single}
    if kind == "reference":  # the port's rate beside it, for continuity with round 1
        baseline["port_single_core_value"] = cpu_rate_single(args.env, 1.0, "port")
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * wall / max(1, args.steps),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": w.dtype, "data": "synthetic",
        "config": workload_config(args, per_gpu=args.envs_per_gpu),
        "cpu_baseline": baseline,
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
# clocks
# ------------------------------------------------------------------------------------------------
class ClockSampler:
    """Samples SM clock / throttle reasons through NVML while the timed region runs."""

    BAD = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20}
    NOTED = {"sw_power_cap": 0x4, "hw_power_brake": 0x80, "sync_boost": 0x10}

    def __init__(self, index: int, period_s: float = 0.02):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thread = None
        self.period = period_s
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = int(pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM))
        except Exception as e:  # pragma: no cover
            self.nv, self.err = None, repr(e)

    def _once(self):
        nv = self.nv
        self.samples.append(int(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM)))
        try:
            bits = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
        except Exception:
            bits = int(nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h))
        for name, bit in {**self.BAD, **self.NOTED}.items():
            if bits & bit:
                self.reasons.add(name)

    def _run(self):
        while not self._stop.is_set():
            try:
                self._once()
            except Exception:
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv:
            self._thread = threading.Thread(target=self._run, daemon=True)
            self._thread.start()

    def stop(self):
        if self._thread:
            self._stop.set()
            self._thread.join()

    def summary(self):
        if not self.nv:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml_unavailable"]}
        med = statistics.median(self.samples) if self.samples else None
        return {"sm_mhz": med, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(self.samples)}


# ------------------------------------------------------------------------------------------------
def workload_config(args, per_gpu, env_name=None):
    w = WORKLOADS[env_name or args.env]
    mb = per_gpu * w.bytes / 1e6
    if per_gpu * w.bytes < 2 * 126e6 and not getattr(args, "no_l2_flush", False):
        l2 = (f"L2 flushed between timed steps: one step moves only {mb:.0f} MB (< 126 MB L2), so every step is timed "
              "on its own CUDA events with an untimed 256 MB fill before it")
    else:
        l2 = (f"inputs larger than L2: each step streams {mb:.0f} MB through a 126 MB L2; the action tape cycles "
              "over >= 64 distinct tensors")
    return {"workload": w.label, "env": w.name,
            "envs_per_gpu": per_gpu, "global_envs": per_gpu * args.gpus, "max_steps": 1000,
            "actions": ("i.i.d. Dict actions (ac_temp ~ U(16, 32) float32, lights ~ Bernoulli(0.5) int8 x4), torch-generated "
                        "tape resident in HBM") if w.name == "climate" else
                       (f"i.i.d. uniform{{0..{w.n_choices - 1}}} int64, device-generated tape (Philox stream 1), "
                        "resident in HBM"),
            "l2_policy": l2,
            "parallelism": f"env-sharded x{args.gpus}, no data-path collective"}


def load_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    try:
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    except Exception:
        return FALLBACK_HBM_GBS, "fallback (B200_PROFILING.md 6.65 TB/s)"


def load_traffic(env_name, n_envs):
    """Per-launch DRAM bytes of the step kernel from the COMMITTED ncu capture (profiles/<env>_step_traffic.json,
    builder-run), scaled to this batch.  Not measured in this run: -> (bytes or None, where it comes from)."""
    path = os.path.join("profiles", f"{env_name}_step_traffic.json")
    try:
        with open(os.path.join(ROOT, path)) as f:
            d = json.load(f)
        return d["dram_bytes_per_env_step"] * n_envs, f"{path} (ncu --set full capture, builder-run; not measured in this run)"
    except Exception:
        return None, None


def make_env(pkg, env_name, n, dev, seed, base):
    if env_name == "snake":
        return pkg.BatchedSnakeEnv(n, 20, device=dev, seed=seed, env_id_base=base)
    if env_name == "crypto":
        return pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=dev, seed=seed, env_id_base=base)
    if env_name == "climate":
        return pkg.BatchedSmartClimateEnv(n, device=dev, seed=seed, env_id_base=base)
    if env_name == "builder":
        return pkg.BatchedWorldBuilderEnv(n, device=dev, seed=seed, env_id_base=base)
    return pkg.BatchedTrafficManagementEnv(n, device=dev, seed=seed, env_id_base=base)


def kernel_description(lib, env_name, n):
    import ctypes as C

    if env_name == "snake":
        t_, s_, c_ = C.c_int32(), C.c_int32(), C.c_int32()
        lib.beng_snake_launch_config(20, n, C.byref(t_), C.byref(s_), C.byref(c_))
        return (f"beng::snake_kernel<T={t_.value},STAGES={s_.value},IS_RESET=false,OWNROW=true>, "
                f"{c_.value} persistent CTAs/SM")
    if env_name == "crypto":
        return ("beng::crypto5_kernel: warp-specialised, 768 threads, 1 persistent CTA/SM: 8 dynamics warps (float64 "
                "state chain, 112 regs) run up to 16 units ahead of 16 observation warps (64 regs) that compose the 261-float "
                "rows from a 2-stage TMA tensor-load ring and drain 32-env tiles with bulk stores")
    if env_name == "climate":
        return ("beng::climate_step_persistent_kernel<T=128>: one thread per env, 5 persistent CTAs per SM walking 128-env "
                "tiles, the next tile's state and action words requested before the current tile is computed")
    if env_name == "builder":
        return ("beng::builder_kernel<T=64,IS_RESET=false,CELLS=100>: one thread per env, 64-env grid tile per CTA, "
                "occupancy bitmap per row")
    return ("beng::traffic_step_kernel<NI=9,IPW=3,72 regs,IS_RESET=false>: 128-thread CTA per 32 envs, three intersection "
            "warps (3 intersections each) + one env warp, 7 CTAs/SM")


API_NAMES = {"snake": "BatchedSnakeEnv.step_host -> beng_snake_step_host",
             "crypto": "BatchedCryptoTradingEnv.step_host -> beng_crypto_step_host",
             "climate": "BatchedSmartClimateEnv.step_host -> beng_climate_step_host",
             "builder": "BatchedWorldBuilderEnv.step_host -> beng_builder_step_host",
             "traffic": "BatchedTrafficManagementEnv.step_host -> beng_traffic_step_host"}


def pin_to_gpu_numa_node(local_rank):
    """Bind this process to the CPUs NVML names as local to its GPU, so that the pinned host buffers it allocates next
    (first touch) and the copy-issuing thread sit on the GPU's NUMA node.  -> (bound?, previous affinity)."""
    prev = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    try:
        import pynvml

        pynvml.nvmlInit()
        pynvml.nvmlDeviceSetCpuAffinity(pynvml.nvmlDeviceGetHandleByIndex(local_rank))
        return True, prev
    except Exception:
        return False, prev


def pcie_ceiling(torch, dev, nbytes):
    """Measured pinned-memory D2H and H2D `cudaMemcpyAsync` bandwidth (GB/s) for one buffer of `nbytes`."""
    nbytes = int(max(1 << 20, min(nbytes, 1 << 30)))
    d = torch.empty(nbytes, dtype=torch.uint8, device=dev)
    h = torch.empty(nbytes, dtype=torch.uint8, pin_memory=True)
    out = {}
    for name, (dst, src) in {"d2h": (h, d), "h2d": (d, h)}.items():
        dst.copy_(src, non_blocking=True)
        torch.cuda.synchronize(dev)
        best = 0.0
        for _ in range(3):
            t0 = time.perf_counter()
            dst.copy_(src, non_blocking=True)
            torch.cuda.synchronize(dev)
            best = max(best, nbytes / (time.perf_counter() - t0) / 1e9)
        out[name] = best
    return out


DUMP_MAX_BYTES = 64_000_000


def _flatten(name, value, out):
    if isinstance(value, dict):  # a Dict observation or the infos (nested "episode" dict, lazily computed entries)
        for k in value.keys():
            _flatten(f"{name}.{k}", value[k], out)
    else:
        out[name] = value


def dump_step_outputs(directory, step_out, n):
    """Write what one step() returned -- (obs, reward, terminated, truncated, infos) -- as <directory>/<name>.npy, dict
    entries under dotted names (obs.grid, info.episode.r, ...).  Values float32 holds exactly (float32 and narrower
    floats, bool, 8- and 16-bit integers) are written as float32, the rest as float64.  float64 holds integers exactly
    only up to 2**53 in magnitude, so a wider integer value (a 64-bit counter or hash) is refused rather than written
    rounded.  Arrays with one row per env keep
    the rows of a fixed sample of envs when all of them would pass DUMP_MAX_BYTES: the sample is drawn from a fixed seed
    and sorted, the same for every array, and written as env_index.npy, so that two runs with the same arguments write
    the same files and two builds can be compared array by array."""
    import numpy as np
    import torch

    narrow = (torch.float32, torch.float16, torch.bfloat16, torch.bool, torch.int8, torch.uint8, torch.int16)
    arrays = {}
    for name, value in zip(("obs", "reward", "terminated", "truncated", "info"), step_out):
        _flatten(name, value, arrays)
    arrays = {k: torch.as_tensor(v) for k, v in arrays.items()}
    for k, v in arrays.items():
        wide = v.to(torch.int64) if not v.dtype.is_floating_point and v.dtype != torch.bool and v.numel() else None
        if wide is not None and (int(wide.max()) > 2 ** 53 or int(wide.min()) < -2 ** 53):
            raise ValueError(f"--dump-outputs: {k} holds integers beyond 2**53, which float64 cannot store exactly")
    out_dtype = {k: torch.float32 if v.dtype in narrow else torch.float64 for k, v in arrays.items()}
    per_env = [k for k, v in arrays.items() if v.dim() >= 1 and v.shape[0] == n]
    row_bytes = 8 + sum(arrays[k][0].numel() * out_dtype[k].itemsize for k in per_env)  # 8: the env_index entry
    other_bytes = sum(v.numel() * out_dtype[k].itemsize for k, v in arrays.items() if k not in per_env)
    keep = min(n, (DUMP_MAX_BYTES - other_bytes - 128 * (len(arrays) + 1)) // row_bytes)  # 128: one .npy header
    index = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).choice(n, size=keep, replace=False))
    os.makedirs(directory, exist_ok=True)
    np.save(os.path.join(directory, "env_index.npy"), index.astype(np.float64))
    for k, v in arrays.items():
        if k in per_env and keep < n:
            v = v.index_select(0, torch.as_tensor(index, device=v.device))
        np.save(os.path.join(directory, f"{k}.npy"), v.to(out_dtype[k]).cpu().numpy())
    print(f"bench: wrote {len(arrays) + 1} arrays of the last timed step ({keep} of {n} envs) to {directory}",
          file=sys.stderr)


def bench_env(ctx, env_name, n, steps, warmup, e2e_steps):
    """Time one env's step kernel (device-resident) and its host-buffer C-ABI call (end to end) on every rank.
    Returns the measurement block on rank 0 (None elsewhere).  All ranks must call this in the same order."""
    torch, dist, pkg, lib, args = ctx["torch"], ctx["dist"], ctx["pkg"], ctx["lib"], ctx["args"]
    rank, local_rank, world, dev = ctx["rank"], ctx["local_rank"], ctx["world"], ctx["dev"]
    from custom_gymnasium_environments_b200.dist import all_reduce_episode_stats, summarize

    w = WORKLOADS[env_name]
    seed = 0
    base = rank * n  # contiguous global env-id slice per rank (weak scaling)
    env = make_env(pkg, env_name, n, dev, seed, base)
    env.reset()
    stream = torch.cuda.current_stream(dev)

    # action tapes, resident in HBM before the timed region (pool of distinct steps, cycled)
    pool = max(64, min(steps + warmup, args.action_pool))
    if env_name == "climate":  # Dict action: ac_temp float32 (n,), lights int8 (n, 4), torch-generated tapes
        gen = torch.Generator(device=dev).manual_seed(1234 + rank)
        ac_t = torch.rand((pool, n), device=dev, generator=gen) * 16.0 + 16.0
        li_t = torch.randint(0, 2, (pool, n, 4), device=dev, generator=gen).to(torch.int8)
        tapes = [{"ac_temp": ac_t[t], "lights": li_t[t]} for t in range(pool)]
        to_host = lambda a: {k: v.cpu().pin_memory() for k, v in a.items()}  # noqa: E731
    else:
        tape_shape = (pool, n) if w.n_cols == 1 else (pool, n, w.n_cols)
        tapes = torch.empty(tape_shape, dtype=torch.int64, device=dev)
        for t in range(pool):
            pkg._lib.check(lib.beng_fill_random_actions(tapes[t].data_ptr(), n, w.n_cols, w.n_choices, t, base, seed,
                                                        stream.cuda_stream), "beng_fill_random_actions")
        to_host = lambda a: a.cpu().pin_memory()  # noqa: E731
    torch.cuda.synchronize(dev)

    def barrier():
        if world > 1:
            dist.barrier()

    # ---- device-resident timing -----------------------------------------------------------------
    # Timing rule: inputs larger than L2, or L2 flushed between timed iterations.  Snake (472 MB/step) and crypto
    # (574 MB/step) stream far more than the 126 MB L2 every step.  Traffic at its BASELINE size moves ~79 MB per
    # step, which would stay L2-resident: there every step is timed on its own events with a 256 MB fill in between
    # (the warm, back-to-back figure is reported separately as `value_l2_warm`).
    flush = n * w.bytes < 2 * 126e6 and not args.no_l2_flush
    for t in range(warmup):
        env.step(tapes[t % pool])
    torch.cuda.synchronize(dev)
    barrier()
    sampler = ClockSampler(local_rank)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = lib.beng_launch_count()
    torch.cuda.synchronize(dev)
    sampler.start()
    ev0.record(stream)
    for t in range(steps):
        last = env.step(tapes[(warmup + t) % pool])
    ev1.record(stream)
    torch.cuda.synchronize(dev)
    launches = lib.beng_launch_count() - launches0
    ms_warm = ev0.elapsed_time(ev1)
    ms = ms_warm
    if flush:
        scratch = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
        pairs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        launches0 = lib.beng_launch_count()
        for t in range(steps):
            scratch.fill_(t & 0xFF)  # evicts the previous step's lines from L2 (not timed)
            pairs[t][0].record(stream)
            last = env.step(tapes[(warmup + t) % pool])
            pairs[t][1].record(stream)
        torch.cuda.synchronize(dev)
        launches = lib.beng_launch_count() - launches0
        ms = sum(a.elapsed_time(b) for a, b in pairs)
        del scratch
    sampler.stop()
    if args.dump_outputs and env_name == args.env and rank == 0:
        # here, not later: step() returns the env's own buffers, which the steps below overwrite
        dump_step_outputs(args.dump_outputs, last, n)
    barrier()
    ms_t = torch.tensor([ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(ms_t, op=dist.ReduceOp.MAX)
    ms_max = float(ms_t.item())
    value = n * world * steps / (ms_max * 1e-3)
    value_warm = n * world * steps / (ms_warm * 1e-3)

    # ---- launch-bound size (traffic at 65,536 envs: ~12 us of L2-warm kernel per ~13 us of Python enqueue): the same
    # back-to-back loop replayed from ONE CUDA graph, per GPU, this rank's own figure (no collective: a rank whose capture
    # failed reports None).  step() is a pure stream operation (tests/test_single_launch_gpu.py), so the capture is
    # just the loop.
    graph_warm = None
    if env_name == "traffic" and flush:
        try:
            k_graph = min(32, pool)
            graph = torch.cuda.CUDAGraph()
            torch.cuda.synchronize(dev)
            with torch.cuda.graph(graph):
                for t in range(k_graph):
                    env.step(tapes[t])
            reps = max(2, steps // k_graph)
            graph.replay()
            torch.cuda.synchronize(dev)
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record(stream)
            for _ in range(reps):
                graph.replay()
            g1.record(stream)
            torch.cuda.synchronize(dev)
            us = g0.elapsed_time(g1) * 1e3 / (reps * k_graph)
            graph_warm = {"env_steps_per_sec_per_gpu": n / (us * 1e-6), "us_per_step": us, "steps_per_graph": k_graph,
                          "note": "L2-warm back-to-back steps replayed from one CUDA graph (rank 0's GPU)"}
        except Exception as ex:  # noqa: BLE001 -- a diagnostic extra, never the headline
            graph_warm = {"error": str(ex)[:200]}

    # ---- end-to-end through the host-buffer C-ABI call -------------------------------------------
    e2e_steps = max(1, min(steps, e2e_steps))
    host_tapes = [to_host(tapes[t % pool]) for t in range(min(e2e_steps + 2, 8))]
    h2d = n * 8 if env_name == "climate" else n * 8 * w.n_cols
    d2h_full = n * (w.obs_bytes + w.result_bytes)
    d2h_lite = n * w.result_bytes

    def time_e2e(copy_obs):
        for t in range(2):
            env.step_host(host_tapes[t % len(host_tapes)], copy_obs=copy_obs)
        torch.cuda.synchronize(dev)
        barrier()
        t0 = time.perf_counter()
        for t in range(e2e_steps):
            # synchronous, as a caller of the reference's numpy API would see it: results are on the host on return
            env.step_host(host_tapes[t % len(host_tapes)], copy_obs=copy_obs)
        torch.cuda.synchronize(dev)
        dt = time.perf_counter() - t0
        dt_t = torch.tensor([dt], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(dt_t, op=dist.ReduceOp.MAX)
        return n * world * e2e_steps / float(dt_t.item()), float(dt_t.item()) / e2e_steps

    e2e_full, e2e_s_per_step = time_e2e(True)
    e2e_lite, _ = time_e2e(False)
    # the link ceiling for THIS rank's big D2H copy, measured with plain pinned cudaMemcpyAsync right after (all ranks
    # at once at N > 1, like the e2e loop itself), so that e2e can be read as a fraction of what the platform gives
    barrier()
    link = pcie_ceiling(torch, dev, n * w.obs_bytes)
    link_t = torch.tensor([link["d2h"], link["h2d"]], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(link_t, op=dist.ReduceOp.MIN)
    link_d2h, link_h2d = (float(v) for v in link_t.tolist())

    # ---- episode statistics: the only collective, outside the step loop ---------------------------
    if env_name == "snake":
        summary = summarize(all_reduce_episode_stats(env.stats))
    else:
        st = env.stats.clone()
        if world > 1:
            dist.all_reduce(st, op=dist.ReduceOp.SUM)
        v = st.tolist()
        summary = {"episodes": int(v[0]), "episode_return_mean": v[1] / max(v[0], 1),
                   "episode_len_mean": v[2] / max(v[0], 1)}
        if env_name == "builder":
            summary["wins"] = v[3]
        if env_name == "crypto":
            summary["final_value_mean"] = v[3] / max(v[0], 1)
    del env, tapes
    torch.cuda.empty_cache()
    if rank != 0:
        return None

    peak, peak_src = load_peak()
    per_launch_ms = ms / max(1, steps)  # rank-0 kernel time; the timed region is back-to-back step launches
    achieved = n * w.bytes / (per_launch_ms * 1e-3) / 1e9
    traffic, traffic_src = load_traffic(env_name, n)
    e2e_gbs = (h2d + d2h_full) / e2e_s_per_step / 1e9  # per rank: every rank moves its own buffers
    return {
        "value": value, "ms_per_step": ms_max / max(1, steps), "steps": steps, "warmup": warmup,
        "config": workload_config(args, per_gpu=n, env_name=env_name),
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_source": traffic_src, "peak_source": peak_src,
                     "algorithmic_bytes_per_env_step": w.bytes,
                     # north_star's literal definition: ncu-measured DRAM bytes against "about 8 TB/s"
                     "frac_ncu_dram_of_nominal_8tbs": (traffic / (per_launch_ms * 1e-3) / 8e12) if traffic else None,
                     "kernel": kernel_description(lib, env_name, n), "kernel_ms": per_launch_ms},
        "e2e": {"value": e2e_full, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h_full,
                "steps": e2e_steps, "api": API_NAMES[env_name] + " (pinned host buffers, synchronous per step, full "
                                                                  "observation copied back)",
                "pcie_gbs": e2e_gbs, "pcie_ceiling_gbs": {"d2h": link_d2h, "h2d": link_h2d},
                "pcie_frac": e2e_gbs / link_d2h if link_d2h else None,
                "pcie_note": "per-rank host<->device bytes per second inside the e2e loop (kernel time included) against "
                             "a plain pinned cudaMemcpyAsync D2H of the observation buffer measured in this run"
                             + (" with all ranks copying at once (min over ranks)" if world > 1 else ""),
                "numa_bound": ctx["numa_bound"]},
        "e2e_obs_on_device": {"value": e2e_lite, "unit": UNIT, "h2d_bytes_per_step": h2d,
                              "d2h_bytes_per_step": d2h_lite,
                              "note": "same call with obs_host=NULL: reward/terminated/info to host, observation "
                                      "stays in HBM for an on-device policy"},
        "gpu_launches": int(launches),
        "l2_flushed_between_steps": bool(flush),
        "value_l2_warm": value_warm if flush else None,
        "l2_warm_cuda_graph": graph_warm,
        "clocks": sampler.summary(),
        "episodes": summary,
    }


def run_b200_arm(args):
    import torch
    import torch.distributed as dist

    nccl_logs = None
    if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", "INFO") and not os.environ.get("NCCL_DEBUG_FILE"):
        # NCCL's banner and communicator lines would precede the JSON line on stdout.  Each rank logs to its own file
        # (eight ranks writing to one stderr pipe garble each other's lines); rank 0 replays the version and
        # "comm ... rank R nranks N" lines to stderr at the end, where whoever asked for them sees them whole.  stdout
        # carries the JSON line only.  The files go to one temporary directory per user that every rank of the host
        # can name before NCCL starts, never into the source tree.
        import tempfile

        nccl_logs = os.path.join(tempfile.gettempdir(), f"bench_nccl_logs_{os.getuid()}")
        os.makedirs(nccl_logs, exist_ok=True)
        os.environ["NCCL_DEBUG_FILE"] = os.path.join(nccl_logs, "nccl.%h.%p.log")
    t_start = time.time()

    import custom_gymnasium_environments_b200 as pkg
    from custom_gymnasium_environments_b200.dist import init_process_group

    rank, local_rank, world = init_process_group()
    if world != args.gpus:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun --nproc-per-node {args.gpus}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the engine has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    numa_bound, prev_affinity = pin_to_gpu_numa_node(local_rank)
    ctx = {"torch": torch, "dist": dist, "pkg": pkg, "lib": pkg._lib.load(), "args": args, "rank": rank,
           "local_rank": local_rank, "world": world, "dev": dev, "numa_bound": numa_bound}
    if world > 1:  # one tiny all-reduce up front: creates the NCCL communicator (and its log lines) before any timing
        dist.all_reduce(torch.zeros(1, device=dev))

    w = WORKLOADS[args.env]
    head = bench_env(ctx, args.env, args.envs_per_gpu, args.steps, args.warmup, args.e2e_steps)
    secondary = {}
    if args.env == "snake" and not args.no_secondary:
        # BASELINE.json configs[2] and configs[3] in the same driver-run record: shorter device-timed runs of the crypto
        # and traffic step kernels at their own BASELINE sizes (same timing rules; no CPU leg).
        # Their own fixed step counts, whatever --steps/--warmup say: the crypto step gets ~20 % dearer once episodes start
        # to end on the portfolio bounds (from step ~120 of the synchronised batch on; sparse in-kernel resets), so a short
        # run right after reset() would flatter it -- 150 warm-up steps, then steps 150..450 are timed.
        for name, sec_steps, sec_warmup in (("crypto", 300, 150), ("traffic", 300, 50)):
            blk = bench_env(ctx, name, WORKLOADS[name].envs_per_gpu, sec_steps, sec_warmup, min(args.e2e_steps, 10))
            if blk is not None:
                blk.update(metric=METRIC, unit=UNIT, dtype=WORKLOADS[name].dtype, n_gpus=world)
                secondary[name] = blk

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    line = {"metric": METRIC, "value": head.pop("value"), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": head.pop("ms_per_step"), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": w.dtype, "data": "synthetic"}
    head.pop("steps"), head.pop("warmup")
    line.update(head)
    if secondary:
        line["secondary"] = secondary
    if world == 1 and not args.no_cpu_baseline:
        if prev_affinity is not None:
            os.sched_setaffinity(0, prev_affinity)  # the CPU arm uses every host core again
        cores = os.cpu_count() or 1
        kind = reference_kind()
        single = cpu_rate_single(args.env, 2.0, kind)
        mctx = mp.get_context("fork")
        with mctx.Pool(cores) as pool_:
            per_proc = max(20, int(single * 10.0))
            par, wall = cpu_rate_parallel(pool_, args.env, cores, per_proc, kind)
        line["cpu_baseline"] = {
            "value": par, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": cpu_arm_description(args.env, kind, cores, per_proc) + f" ({wall:.1f} s wall)",
            "single_core_value": single, "c_oracle_single_thread_value": c_oracle_rate(args.env)}
        if kind == "reference":
            line["cpu_baseline"]["port_single_core_value"] = cpu_rate_single(args.env, 1.0, "port")
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    if nccl_logs:
        import glob

        for path in sorted(glob.glob(os.path.join(nccl_logs, "nccl.*.log"))):
            if os.path.getmtime(path) < t_start - 1:
                continue
            with open(path, errors="replace") as f:
                for ln in f:
                    if "nranks" in ln or "NCCL version" in ln:
                        sys.stderr.write(ln)
        sys.stderr.flush()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2000)
    ap.add_argument("--warmup", type=int, default=200)
    ap.add_argument("--impl", choices=["b200", "reference"], default="b200")
    ap.add_argument("--env", choices=sorted(WORKLOADS), default="snake",
                    help="snake = the BASELINE.json headline (configs[1]); crypto = configs[2]; traffic = configs[3]; "
                         "climate, builder = SURVEY.md 8(f) rank 3 (no BASELINE config)")
    ap.add_argument("--envs-per-gpu", type=int, default=None)
    ap.add_argument("--action-pool", type=int, default=256, help="distinct pre-generated action steps kept in HBM")
    ap.add_argument("--e2e-steps", type=int, default=20)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true",
                    help="snake only: skip the crypto and traffic blocks that the default run appends as `secondary`")
    ap.add_argument("--no-l2-flush", action="store_true", help="traffic only: time back-to-back steps (L2-warm)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="b200 arm only: after the timed steps, write what the last one returned (--env's step(), rank 0) as "
                         "DIR/<name>.npy, float32/float64, at most 64 MB in all (a fixed sample of envs when larger)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this repo's CUDA engine computed; the reference arm has nothing to dump")
    sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)
    args.warmup = max(args.warmup, 3)
    if args.envs_per_gpu is None:
        args.envs_per_gpu = WORKLOADS[args.env].envs_per_gpu
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_b200_arm(args)


if __name__ == "__main__":
    main()
