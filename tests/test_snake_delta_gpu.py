"""BatchedSnakeEnv.step_host(delta_obs=True) on the GPU: the host observation mirror patched from per-env change records
must equal, byte for byte, what the full-copy path returns, and equal env.obs on the device, after every step."""
import collections
import json

import numpy as np
import pytest
import torch

from oracle import c_oracle
from test_snake_delta import greedy_actions

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    assert torch.cuda.is_available(), "gpu tests need a CUDA device"
    p._lib.load()
    return p


class CountingLib:
    """Stands in for env.lib and counts the entry points called through it."""

    def __init__(self, lib):
        self._lib, self.calls = lib, collections.Counter()

    def __getattr__(self, name):
        self.calls[name] += 1
        return getattr(self._lib, name)


def pair(pkg, n, G, mode, max_steps=1000, tl=False, seed=5):
    envs = [pkg.BatchedSnakeEnv(n, G, device=DEV, seed=seed, autoreset_mode=mode, max_steps=max_steps,
                                time_limit_truncation=tl) for _ in range(2)]
    for e in envs:
        e.reset()
    return envs


def random_tape(seed, n, t):
    """Uniform actions with ~3 % out-of-space values (-1, 4): such an env is left untouched."""
    a = c_oracle.action_tape(seed, 0, n, t, 4)
    bad = c_oracle.action_tape(seed + 1, 0, n, t, 32) == 0
    return np.where(bad, np.where(a & 1, 4, -1), a)


def step_both(full, delta, act):
    out_f = full.step_host(act)
    out_d = delta.step_host(act, delta_obs=True)
    assert not out_d[0].flags.writeable
    for x, y in zip(out_f[:4], out_d[:4]):
        assert np.array_equal(x, y)
    for k in out_f[4]:
        assert np.array_equal(out_f[4][k], out_d[4][k]), k
    assert np.array_equal(out_d[0], delta.obs.cpu().numpy())  # the mirror equals the device observations
    return out_f


@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("G,n,max_steps,tl", [(20, 10007, 1000, False), (15, 333, 40, True), (8, 1, 25, False),
                                              (33, 10007, 60, True), (64, 333, 1000, False)])
def test_delta_matches_full_copy(pkg, G, n, max_steps, tl, mode):
    full, delta = pair(pkg, n, G, mode, max_steps, tl)
    delta.lib = counting = CountingLib(delta.lib)
    steps = 300
    for t in range(steps):
        step_both(full, delta, random_tape(G * 7 + n, n, t))
    # the first call seeds the mirror with a full copy, every later one moves records only
    assert counting.calls["beng_snake_step_host"] == 1
    assert counting.calls["beng_snake_step_host_delta"] == steps - 1
    assert counting.calls["beng_snake_apply_obs_delta"] == steps - 1
    assert full.episode_stats() == delta.episode_stats()


@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("G,n,steps", [(5, 64, 1500), (8, 64, 2500)])
def test_delta_greedy_long_snakes(pkg, G, n, steps, mode):
    """Greedy tapes on small boards: long snakes, ring wrap-around, and full boards without food."""
    full, delta = pair(pkg, n, G, mode, seed=11)
    max_len, no_food = 0, False
    obs = full.obs.cpu().numpy()
    for t in range(steps):
        st = {k: v.cpu().numpy() for k, v in full.export_state().items()}
        max_len = max(max_len, int(st["length"].max()))
        no_food |= bool((st["food_r"] < 0).any())
        obs = step_both(full, delta, greedy_actions(obs, st, G))[0]
    assert max_len >= G * G // 3
    if G == 5 and mode != "disabled":
        assert no_food


def test_invalidating_calls_fall_back_to_a_full_copy(pkg):
    n, G = 4099, 20
    full, delta = pair(pkg, n, G, "next_step", max_steps=30)
    g = torch.Generator(device=DEV).manual_seed(1)
    t = 0

    def delta_steps(k=3):
        nonlocal t
        for _ in range(k):
            step_both(full, delta, random_tape(9, n, t))
            t += 1

    def both(fn):
        for e in (full, delta):
            fn(e)
        delta_steps()

    delta_steps()
    sd = full.state_dict()
    mask = torch.rand(n, device=DEV, generator=g) < 0.3
    act = torch.randint(0, 4, (n,), device=DEV, generator=g)
    buf = torch.zeros((n, G, G), dtype=torch.int8, device=DEV)
    both(lambda e: e.reset())
    both(lambda e: e.reset(seed=123))
    both(lambda e: e.reset(options={"reset_mask": mask}))
    both(lambda e: e.step(act))
    both(lambda e: e.step(act, out_obs=buf))
    both(lambda e: e.step_host(act.cpu().numpy(), copy_obs=False))
    both(lambda e: e.load_state_dict(sd))
    both(lambda e: (e.step(act), e.step(act)))


def test_full_batch(pkg):
    n = 1 << 20
    full, delta = pair(pkg, n, 20, "same_step")
    for t in range(50):
        step_both(full, delta, c_oracle.action_tape(3, 0, n, t, 4))


def test_delta_step_is_one_kernel_and_moves_18_bytes_per_env(pkg, tmp_path):
    n = 8192
    env = pkg.BatchedSnakeEnv(n, device=DEV)
    env.reset()
    lib = pkg._lib.load()
    act = [c_oracle.action_tape(4, 0, n, t, 4) for t in range(8)]
    for a in act[:2]:
        env.step_host(a, delta_obs=True)
    trace = tmp_path / "trace.json"
    seen = {}

    def ready(p):
        seen["kernels"] = [e.name for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA
                           and not e.name.startswith("Memcpy")]
        p.export_chrome_trace(str(trace))

    # one untraced warm-up step inside the profiler, then five traced delta steps
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA],
                                schedule=torch.profiler.schedule(wait=0, warmup=1, active=5, repeat=1),
                                on_trace_ready=ready) as prof:
        for i, a in enumerate(act[2:]):
            if i == 1:
                before = lib.beng_launch_count()
            env.step_host(a, delta_obs=True)
            prof.step()
    assert lib.beng_launch_count() - before == 5
    kernels = seen["kernels"]
    assert len(kernels) == 5 and len(set(kernels)) == 1 and "snake_kernel" in kernels[0], kernels
    copies = [e for e in json.loads(trace.read_text())["traceEvents"] if e.get("cat") == "gpu_memcpy"]
    d2h = sum(e["args"]["bytes"] for e in copies if "DtoH" in e["name"])
    h2d = sum(e["args"]["bytes"] for e in copies if "HtoD" in e["name"])
    assert d2h == 5 * 18 * n and h2d == 5 * 8 * n, (d2h, h2d)


def test_delta_obs_argument_errors(pkg):
    env = pkg.BatchedSnakeEnv(16, device=DEV)
    env.reset()
    a = np.zeros(16, np.int64)
    with pytest.raises(ValueError):
        env.step_host(a, delta_obs=True, sync=False)
    with pytest.raises(ValueError):
        env.step_host(a, delta_obs=True, copy_obs=False)
    for _ in range(2):
        obs = env.step_host(a, delta_obs=True)[0]
        assert not obs.flags.writeable
        with pytest.raises(ValueError):
            obs[0, 0, 0] = 1
    assert env.step_host(a)[0].flags.writeable  # the full-copy path is unchanged
