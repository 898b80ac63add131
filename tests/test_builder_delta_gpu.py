"""BatchedWorldBuilderEnv.step_host(delta_obs=True) on the GPU: the host grid mirror patched from per-env change records
must equal, byte for byte, what the full-copy path returns, and equal env.grid on the device, after every step."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import c_oracle
from test_builder_delta import tape
from test_snake_delta_gpu import CountingLib

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    p._lib.load()
    return p


def pair(pkg, n, G, mode, flatten=False, seed=5, debug=False):
    envs = [pkg.BatchedWorldBuilderEnv(n, G, flatten_obs=flatten, device=DEV, seed=seed, autoreset_mode=mode,
                                       debug_checks=debug) for _ in range(2)]
    for e in envs:
        e.reset()
    return envs


def same_bytes(x, y):
    return x.dtype == y.dtype and x.shape == y.shape and x.tobytes() == y.tobytes()


def step_both(full, delta, act):
    out_f = full.step_host(act)
    out_d = delta.step_host(act, delta_obs=True)
    assert len(out_f) == len(out_d) == 5
    assert not out_d[0]["grid"].flags.writeable
    assert list(out_f[0]) == list(out_d[0])
    for k in out_f[0]:
        assert same_bytes(out_f[0][k], out_d[0][k]), k
    for x, y in zip(out_f[1:4], out_d[1:4]):
        assert same_bytes(x, y)
    assert out_f[4] == out_d[4] == {}
    assert np.array_equal(out_d[0]["grid"], delta.grid.cpu().numpy())  # the mirror equals the device grid
    if full.flatten_obs:
        assert torch.equal(full.flat_obs, delta.flat_obs)
    return out_f


@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("G,n", [(10, 10007), (15, 130), (7, 31), (4, 333), (2, 1)])
def test_delta_matches_full_copy(pkg, G, n, mode):
    full, delta = pair(pkg, n, G, mode)
    delta.lib = counting = CountingLib(delta.lib)
    steps = 300
    for t in range(steps):
        step_both(full, delta, tape("random" if t % 3 else "build", G * 7 + n, n, t))
    # the first call seeds the mirror with a full copy, every later one moves records only
    assert counting.calls["beng_builder_step_host"] == 1
    assert counting.calls["beng_builder_step_host_delta"] == steps - 1
    assert counting.calls["beng_builder_apply_obs_delta"] == steps - 1
    assert full.episode_stats() == delta.episode_stats()
    assert torch.equal(full.invalid_count, delta.invalid_count)


def test_delta_with_flatten_obs(pkg):
    """step_host returns the Dict form either way; the device's flattened observation must match too."""
    n, G = 4099, 10
    full, delta = pair(pkg, n, G, "next_step", flatten=True)
    for t in range(100):
        step_both(full, delta, tape("random", 17, n, t))


def test_invalidating_calls_fall_back_to_one_full_copy(pkg):
    n, G = 4099, 10
    full, delta = pair(pkg, n, G, "next_step")
    counting = delta.lib = CountingLib(delta.lib)
    g = torch.Generator(device=DEV).manual_seed(1)
    t = 0

    def delta_steps(k=3):
        nonlocal t
        counting.calls.clear()
        for _ in range(k):
            step_both(full, delta, tape("random", 9, n, t))
            t += 1
        assert counting.calls["beng_builder_step_host"] == 1, counting.calls
        assert counting.calls["beng_builder_step_host_delta"] == k - 1, counting.calls

    def both(fn):
        for e in (full, delta):
            fn(e)
        delta_steps()

    delta_steps()
    sd = full.state_dict()
    mask = torch.rand(n, device=DEV, generator=g) < 0.3
    act = torch.randint(0, 5, (n,), device=DEV, generator=g)
    both(lambda e: e.reset())
    both(lambda e: e.reset(seed=123))
    both(lambda e: e.reset(options={"reset_mask": mask}))
    both(lambda e: e.step(act))
    both(lambda e: e.step_host(act.cpu().numpy(), copy_obs=False))
    both(lambda e: e.load_state_dict(sd))
    both(lambda e: (e.step(act), e.step(act)))


def test_full_batch(pkg):
    n = 1 << 20
    full, delta = pair(pkg, n, 10, "same_step")
    for t in range(30):
        step_both(full, delta, c_oracle.action_tape(3, 0, n, t, 5))


# Runs in a process of its own (see the test below) and prints one JSON line.
PROFILED_STEPS = r"""
import json, sys
sys.path.insert(0, sys.argv[1])
import torch
import custom_gymnasium_environments_b200 as pkg
from oracle import c_oracle

n = 8192
env = pkg.BatchedWorldBuilderEnv(n, device="cuda:0")
env.reset()
lib = pkg._lib.load()
act = [c_oracle.action_tape(4, 0, n, t, 5) for t in range(8)]
for a in act[:3]:  # the first call seeds the mirror with a full copy
    env.step_host(a, delta_obs=True)
torch.cuda.synchronize()
with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
    before = lib.beng_launch_count()
    for a in act[3:]:
        env.step_host(a, delta_obs=True)
    torch.cuda.synchronize()
launches = lib.beng_launch_count() - before
kernels = [e.name for e in prof.events()
           if e.device_type == torch.autograd.DeviceType.CUDA and not e.name.startswith("Memcpy")]
prof.export_chrome_trace(sys.argv[2])
copies = [e for e in json.load(open(sys.argv[2]))["traceEvents"] if e.get("cat") == "gpu_memcpy"]
print(json.dumps({"n": n, "launches": launches, "kernels": kernels,
                  "d2h": sum(e["args"]["bytes"] for e in copies if "DtoH" in e["name"]),
                  "h2d": sum(e["args"]["bytes"] for e in copies if "HtoD" in e["name"])}))
"""


def test_delta_step_is_one_kernel_and_moves_33_bytes_per_env(pkg, tmp_path):
    """Five profiled delta steps: five launches of one builder kernel, 33 B per env D2H and 8 B per env H2D.

    The profiler runs in a child process because its CUDA activity tracing is process-wide state.  With this session
    in the suite's process, the first session of test_single_launch_gpu.py, which runs later in the same process,
    recorded one of its five kernels."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    flags = ["-B"] + (["-s"] if sys.flags.no_user_site else [])
    run = subprocess.run([sys.executable, *flags, "-c", PROFILED_STEPS, root, str(tmp_path / "trace.json")],
                         cwd=str(tmp_path), capture_output=True, text=True, timeout=600)
    assert run.returncode == 0, run.stderr[-4000:]
    r = json.loads(run.stdout.strip().splitlines()[-1])
    n, kernels = r["n"], r["kernels"]
    assert r["launches"] == 5
    assert len(kernels) == 5 and len(set(kernels)) == 1 and "builder_kernel" in kernels[0], kernels
    assert r["d2h"] == 5 * 33 * n and r["h2d"] == 5 * 8 * n, r


def test_delta_obs_argument_errors(pkg):
    env = pkg.BatchedWorldBuilderEnv(16, device=DEV)
    env.reset()
    a = np.ones(16, np.int64)
    with pytest.raises(ValueError):
        env.step_host(a, delta_obs=True, sync=False)
    with pytest.raises(ValueError):
        env.step_host(a, delta_obs=True, copy_obs=False)
    for _ in range(2):
        obs = env.step_host(a, delta_obs=True)[0]
        assert not obs["grid"].flags.writeable
        with pytest.raises(ValueError):
            obs["grid"][0, 0, 0] = 1
    assert env.step_host(a)[0]["grid"].flags.writeable  # the full-copy path is unchanged


def test_debug_checks_on_invalid_actions_as_on_the_full_path(pkg):
    """step_host does not check on either path; the invalid action is counted, and the next step() raises."""
    n = 64
    full, delta = pair(pkg, n, 10, "same_step", debug=True)
    a = np.ones(n, np.int64)
    step_both(full, delta, a)
    bad = a.copy()
    bad[5] = 7
    step_both(full, delta, bad)
    assert full.invalid_count.item() == delta.invalid_count.item() == 1
    for e in (full, delta):
        with pytest.raises(ValueError, match="Invalid action"):
            e.step(torch.as_tensor(a, device=DEV))
