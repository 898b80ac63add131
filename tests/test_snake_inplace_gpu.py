"""BatchedSnakeEnv.step() patches env.obs in place (beng_snake_step_inplace) while it holds the previous observation.
Every step must return, byte for byte, what the composing kernel (beng_snake_step, reached through out_obs=) returns
for a twin env with the same seed: observation, reward, flags, state, finished-env list and statistics."""
import collections
import ctypes as C

import numpy as np
import pytest
import torch

from test_snake_delta import greedy_actions

DEV = "cuda:0"
MODES = ("same_step", "next_step", "disabled")


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    p._lib.load()
    return p


class CountingLib:
    """Stands in for env.lib and counts the entry points called through it."""

    def __init__(self, lib):
        self._lib, self.calls = lib, collections.Counter()

    def __getattr__(self, name):
        self.calls[name] += 1
        return getattr(self._lib, name)


def make(pkg, n, G, mode, max_steps=1000, tl=False, seed=11):
    env = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=seed, autoreset_mode=mode, max_steps=max_steps,
                              time_limit_truncation=tl)
    env.lib = CountingLib(env.lib)
    return env


class Twin:
    """The env under test and a twin with the same seed that always composes full rows into a scratch buffer."""

    def __init__(self, pkg, n, G, mode, **kw):
        self.env, self.ref = make(pkg, n, G, mode, **kw), make(pkg, n, G, mode, **kw)
        self.scratch = torch.empty_like(self.ref.obs)
        self.G = G

    def reset(self, **kw):
        a, b = self.env.reset(**kw)[0], self.ref.reset(**kw)[0]
        assert torch.equal(a, b)
        self.scratch.copy_(b)

    def step(self, act, **kw):
        """env.step(act, **kw) against the twin's composing step; -> the env's step() result."""
        out = self.env.step(act, **kw)
        ref = self.ref.step(act, out_obs=self.scratch)
        check_equal(self.env, self.ref, out, ref)
        return out

    def check_state(self):
        assert torch.equal(self.env._core, self.ref._core)
        assert torch.equal(self.env._ring, self.ref._ring)
        assert torch.equal(self.env.stats, self.ref.stats)


def check_equal(env, ref, out, ref_out):
    for x, y in zip(out[:4], ref_out[:4]):
        assert torch.equal(x, y)
    fin = torch.sort(env.finished_envs()).values.long()  # (the list's order is unspecified)
    assert torch.equal(fin, torch.sort(ref.finished_envs()).values.long())
    for k in ("ep_return", "ep_length", "ep_score"):
        assert torch.equal(getattr(env, k)[fin], getattr(ref, k)[fin])
    assert torch.equal(env.stats, ref.stats)
    assert torch.equal(env.invalid_count, ref.invalid_count)


def device_tape(n, t, seed):
    """Uniform actions on the device with ~3 % out-of-space values (-1, 4): such an env is left untouched."""
    g = torch.Generator(device=DEV).manual_seed(seed * 100003 + t)
    a = torch.randint(0, 4, (n,), device=DEV, generator=g)
    bad = torch.randint(0, 32, (n,), device=DEV, generator=g) == 0
    return torch.where(bad, torch.where((a & 1) == 1, 4, -1), a)


def host_greedy(env):
    st = {k: v.cpu().numpy() for k, v in env.export_state().items()}
    return torch.as_tensor(greedy_actions(env.obs.cpu().numpy(), st, env.grid_size), device=DEV)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", MODES)
def test_full_batch_random(pkg, mode):
    n = 1 << 20
    tw = Twin(pkg, n, 20, mode, max_steps=40, tl=True)
    tw.reset()
    for t in range(64):
        tw.step(device_tape(n, t, 1))
        if t % 16 == 15:
            tw.check_state()
    tw.check_state()
    assert tw.env.lib.calls["beng_snake_step_inplace"] == 64 and tw.env.lib.calls["beng_snake_step"] == 0
    assert int(tw.env.stats[0]) > 0 or mode == "disabled"


@pytest.mark.gpu
@pytest.mark.parametrize("policy", ("random", "greedy"))
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("G,n", [(2, 37), (3, 1), (5, 4099), (8, 1031), (15, 300), (20, 4099), (33, 257), (64, 97)])
def test_ragged_counts_and_grids(pkg, G, n, mode, policy):
    """Random tapes die often and hit every reset path; greedy tapes grow long snakes, which exercises eating, the
    food rejection loop, a near-full G = 5 board, a full G = 2 board (no food) and the time limit."""
    tw = Twin(pkg, n, G, mode, max_steps=150, tl=G % 2 == 0)
    tw.reset()
    for t in range(200):
        act = host_greedy(tw.env) if policy == "greedy" else device_tape(n, t, G)
        tw.step(act)
    tw.check_state()
    assert tw.env.lib.calls["beng_snake_step_inplace"] == 200


@pytest.mark.gpu
def test_path_switching(pkg):
    """Every way of leaving env.obs stale or current, against a twin that always composes."""
    n, G = 3001, 20
    tw = Twin(pkg, n, G, "same_step", max_steps=60)
    env, calls = tw.env, tw.env.lib.calls
    tw.reset()
    t = iter(range(10_000))

    def step(expect, **kw):
        before = calls[expect]
        out = tw.step(device_tape(n, next(t), 3), **kw)
        assert calls[expect] == before + 1, (expect, dict(calls))
        return out

    for _ in range(5):
        step("beng_snake_step_inplace")
    other = torch.empty_like(env.obs)
    assert step("beng_snake_step", out_obs=other)[0].data_ptr() == other.data_ptr()
    step("beng_snake_step")  # env.obs missed a step: composed in full once, then patched again
    step("beng_snake_step_inplace")
    step("beng_snake_step", out_obs=env.obs)  # composes into env.obs itself, which stays current
    step("beng_snake_step_inplace")

    act = device_tape(n, next(t), 3).cpu().numpy()
    out, ref = env.step_host(act), tw.ref.step_host(act)
    for x, y in zip(out[:4], ref[:4]):
        assert np.array_equal(x, y)
    tw.scratch.copy_(tw.ref.obs)
    step("beng_snake_step_inplace")

    env.load_state_dict(tw.ref.state_dict())
    step("beng_snake_step")
    step("beng_snake_step_inplace")

    mask = (torch.arange(n, device=DEV) % 7 == 0)
    tw.reset(options={"reset_mask": mask})
    step("beng_snake_step_inplace")
    step("beng_snake_step_inplace")
    tw.check_state()


@pytest.mark.gpu
def test_invalid_actions_leave_the_row(pkg):
    n, G = 1000, 12
    tw = Twin(pkg, n, G, "same_step")
    tw.reset()
    for t in range(30):
        tw.step(device_tape(n, t, 4))
    before = tw.env.obs.clone()
    core = tw.env._core.clone()
    bad = torch.where(torch.arange(n, device=DEV) % 2 == 0, -1, 4)
    obs = tw.step(bad)[0]
    assert torch.equal(obs, before)
    assert torch.equal(tw.env._core, core)
    assert int(tw.env.invalid_count) == int(tw.ref.invalid_count) > 0


@pytest.mark.gpu
def test_cuda_graph_replay(pkg):
    """K in-place steps captured in one CUDA graph walk the trajectory of eager in-place steps."""
    n, G, K = 65536, 20, 8
    eager, graphed = make(pkg, n, G, "same_step", max_steps=25), make(pkg, n, G, "same_step", max_steps=25)
    eager.reset(), graphed.reset()
    tapes = [device_tape(n, t, 6) for t in range(K)]
    graphed.step(tapes[0])  # leaves env.obs current, so that the captured steps are in-place ones
    eager.step(tapes[0])
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    stream = torch.cuda.Stream()
    with torch.cuda.stream(stream):
        with torch.cuda.graph(graph, stream=stream):
            for t in range(K):
                graphed.step(tapes[t])
    assert graphed.lib.calls["beng_snake_step_inplace"] == K + 1
    for _ in range(3):
        graph.replay()
        for t in range(K):
            eager.step(tapes[t])
        torch.cuda.synchronize()
        assert torch.equal(graphed.obs, eager.obs)
        assert torch.equal(graphed._core, eager._core) and torch.equal(graphed._ring, eager._ring)
        assert torch.equal(graphed.reward, eager.reward) and torch.equal(graphed.stats, eager.stats)


def test_inplace_argument_errors(pkg):
    """Checked before anything touches the device: no GPU needed."""
    lib = pkg._lib.load()
    fn = lib.beng_snake_step_inplace
    p = pkg._lib.SnakeParams(20, 1000, 2, 0, 0, 0)
    st, io = pkg._lib.SnakeState(64, 64), pkg._lib.SnakeIO()
    io.obs, io.reward, io.terminated = 64, 64, 64
    ok = (C.byref(p), C.byref(st), 64, C.byref(io))
    before = lib.beng_launch_count()
    assert fn(*ok, 0, None) == 0  # n == 0: nothing to do, nothing launched
    assert fn(*ok, -1, None) == -1
    assert fn(None, C.byref(st), 64, C.byref(io), 16, None) == -1
    assert fn(C.byref(p), None, 64, C.byref(io), 16, None) == -1
    assert fn(C.byref(p), C.byref(st), None, C.byref(io), 16, None) == -1
    assert fn(C.byref(p), C.byref(st), 64, None, 16, None) == -1
    assert fn(C.byref(p), C.byref(st), 68, C.byref(io), 16, None) == -1  # actions not 8-byte aligned
    io.obs = 72
    assert fn(*ok, 16, None) == -1  # obs not 16-byte aligned
    io.obs, io.reward = 64, None
    assert fn(*ok, 16, None) == -1
    io.reward, st.core = 64, 72
    assert fn(*ok, 16, None) == -1  # state record not 16-byte aligned
    st.core, p.grid_size = 64, 65
    assert fn(*ok, 16, None) == -2
    assert lib.beng_launch_count() == before
