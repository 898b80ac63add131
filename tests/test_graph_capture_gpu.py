"""BatchedSnakeEnv.step() and BatchedCryptoTradingEnv.step() captured in a CUDA graph walk the trajectory of eager steps:
the per-step state they advance (snake's done-counter parity, crypto's window head) lives on the device and is advanced
by the launch itself, so a captured launch is the right program on every replay.  Every check runs against an eager
twin with the same seed and env_id_base."""
import ctypes as C

import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N = 2053  # not a multiple of 32
G = 20
INFO = ("reward64", "portfolio_value", "current_price", "trade_kind", "ep_return", "ep_length")


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import custom_gymnasium_environments_b200 as p
    return p


class Case:
    """One env kind: how to build it, the action tape, one step, and the comparison with the twin."""

    def __init__(self, pkg, kind, mode, steps=200):
        self.pkg, self.kind, self.mode = pkg, kind, mode
        gen = torch.Generator(device=DEV).manual_seed(17)
        if kind.startswith("snake"):
            self.tape = [torch.randint(0, 4, (N,), device=DEV, generator=gen) for _ in range(steps)]
        elif kind == "crypto_discrete":
            self.tape = [torch.randint(0, 5, (N,), device=DEV, generator=gen) for _ in range(steps)]
        else:
            self.tape = [torch.rand((N, 2), device=DEV, generator=gen) * 2 - 1 for _ in range(steps)]

    def make(self):
        if self.kind.startswith("snake"):
            env = self.pkg.BatchedSnakeEnv(N, G, device=DEV, seed=7, env_id_base=3, autoreset_mode=self.mode,
                                           max_steps=6)
            env.rollout = torch.zeros((len(self.tape), N, G, G), dtype=torch.int8, device=DEV)
        else:
            action_type = "discrete" if self.kind == "crypto_discrete" else "continuous"
            env = self.pkg.BatchedCryptoTradingEnv(N, None, action_type, device=DEV, seed=7, env_id_base=3,
                                                   autoreset_mode=self.mode, max_steps=5)
        env.reset()
        env.clock = 0
        return env

    def step(self, env, t):
        """Step t of the tape (the same call eagerly and under capture)."""
        if self.kind == "snake_out_obs":
            return env.step(self.tape[t], out_obs=env.rollout[t])
        return env.step(self.tape[t])

    def eager(self, env, t0, k):
        for t in range(t0, t0 + k):
            self.step(env, t)

    def check(self, a, b, what):
        sa, sb = a.state_dict(), b.state_dict()
        assert sa.keys() == sb.keys()
        for k in sa:
            if k == "stats" and self.kind.startswith("crypto"):  # float64 atomics: order of the sums may differ
                torch.testing.assert_close(sa[k], sb[k], rtol=1e-12, atol=0, msg=f"{what}: {k}")
            elif isinstance(sa[k], torch.Tensor):
                assert torch.equal(sa[k], sb[k]), (what, k)
            else:
                assert sa[k] == sb[k], (what, k)
        obs_a = a.rollout if self.kind == "snake_out_obs" else a.obs
        obs_b = b.rollout if self.kind == "snake_out_obs" else b.obs
        assert torch.equal(obs_a, obs_b), what
        for k in ("reward", "terminated", "truncated"):
            assert torch.equal(getattr(a, k), getattr(b, k)), (what, k)
        if self.kind.startswith("snake"):
            fa, fb = a.finished_envs(), b.finished_envs()
            assert torch.equal(torch.sort(fa).values, torch.sort(fb).values), what
            assert torch.equal(a.stats, b.stats), what
        else:
            for k in INFO:
                assert torch.equal(getattr(a, k), getattr(b, k)), (what, k)
            assert torch.equal(a.price_history(), b.price_history()), what


KINDS = ["snake_inplace", "snake_out_obs", "crypto_discrete", "crypto_continuous"]


def capture(case, env, t0, k):
    """A graph of steps t0 .. t0+k-1 of `env`, captured after the lazy set-up of the first eager step."""
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        case.eager(env, t0, k)
    return graph


@pytest.mark.parametrize("mode", ["same_step", "next_step"])
@pytest.mark.parametrize("k", [1, 3, 7])
@pytest.mark.parametrize("kind", KINDS)
def test_replay_equals_eager(pkg, kind, k, mode):
    case = Case(pkg, kind, mode)
    g_env, e_env = case.make(), case.make()
    case.step(g_env, 0), case.step(e_env, 0)
    graph = capture(case, g_env, 1, k)
    for r in range(3):
        graph.replay()
        case.eager(e_env, 1, k)
        torch.cuda.synchronize()
        case.check(g_env, e_env, f"replay {r}")
    if k >= 3:  # 10 steps or more against max_steps 5 / 6: auto-resets happened inside the graph
        assert e_env.episode_stats()["n_episodes"] > 0


@pytest.mark.parametrize("kind", KINDS)
def test_capture_alone_changes_nothing(pkg, kind):
    case = Case(pkg, kind, "same_step")
    g_env, e_env = case.make(), case.make()
    case.step(g_env, 0), case.step(e_env, 0)
    capture(case, g_env, 1, 3)  # never replayed
    for t in range(1, 8):
        case.step(g_env, t), case.step(e_env, t)
        torch.cuda.synchronize()
        case.check(g_env, e_env, f"eager step {t}")


@pytest.mark.parametrize("kind", KINDS)
def test_replays_and_eager_steps_interleave(pkg, kind):
    k = 3
    case = Case(pkg, kind, "same_step")
    g_env, e_env = case.make(), case.make()
    case.step(g_env, 0), case.step(e_env, 0)
    graph = capture(case, g_env, 1, k)
    graph.replay()
    case.step(g_env, 4)
    graph.replay()
    case.eager(e_env, 1, k), case.step(e_env, 4), case.eager(e_env, 1, k)
    torch.cuda.synchronize()
    case.check(g_env, e_env, "replay, eager step, replay")


@pytest.mark.parametrize("kind", KINDS)
def test_load_state_dict_then_replay(pkg, kind):
    k = 3
    case = Case(pkg, kind, "same_step")
    g_env, e_env, src = case.make(), case.make(), case.make()
    case.step(g_env, 0), case.step(e_env, 0)
    graph = capture(case, g_env, 1, k)
    graph.replay()
    case.eager(e_env, 1, k)
    case.eager(src, 10, 17)  # another point of the trajectory, another window head
    sd = src.state_dict()
    g_env.load_state_dict(sd), e_env.load_state_dict(sd)
    if kind == "snake_inplace":  # env.obs is stale after a load: one eager step composes it before the next replay
        case.step(g_env, 30), case.step(e_env, 30)
    graph.replay()
    case.eager(e_env, 1, k)
    torch.cuda.synchronize()
    case.check(g_env, e_env, "replay after load_state_dict")


def test_crypto_legacy_host_head_walks_the_same_trajectory(pkg):
    """beng_crypto_step with window_head_dev = NULL and the host advancing params.window_head."""
    case = Case(pkg, "crypto_discrete", "same_step")
    managed, legacy = case.make(), case.make()
    L, lib = pkg._lib, pkg._lib.load()
    io = L.CryptoIO.from_buffer_copy(legacy._io)
    io.window_head_dev = None
    p = L.CryptoParams.from_buffer_copy(legacy.params)
    p.window_head = 0
    stream = torch.cuda.current_stream().cuda_stream
    for t in range(12):
        managed.step(case.tape[t])
        L.check(lib.beng_crypto_step(C.byref(p), C.byref(legacy._state), case.tape[t].data_ptr(), C.byref(io), N,
                                     stream), "beng_crypto_step")
        p.window_head = (p.window_head + 1) % 50
        torch.cuda.synchronize()
        sm = managed.state_dict()
        assert sm["window_head"] == p.window_head
        for k in ("scal", "meta", "ep_return", "close", "ohlv"):
            assert torch.equal(sm[k], getattr(legacy, "_" + k)), (t, k)
        for k in ("obs", "reward", "terminated") + INFO:
            assert torch.equal(getattr(managed, k), getattr(legacy, k)), (t, k)
    assert int(legacy._head[0]) == 0  # the device head of the legacy env was never touched


def test_snake_legacy_ping_pong_counters_walk_the_same_trajectory(pkg):
    """beng_snake_step with two distinct counters and the host alternating them."""
    case = Case(pkg, "snake_inplace", "same_step")
    managed, legacy = case.make(), case.make()
    L, lib = pkg._lib, pkg._lib.load()
    counts = torch.zeros(2, dtype=torch.int32, device=DEV)
    ios = []
    for parity in (0, 1):
        io = legacy._make_io(legacy.obs)
        io.done_count, io.done_count_next = counts.data_ptr() + 4 * parity, counts.data_ptr() + 4 * (1 - parity)
        ios.append(io)
    stream = torch.cuda.current_stream().cuda_stream
    for t in range(40):
        managed.step(case.tape[t])
        L.check(lib.beng_snake_step(C.byref(legacy.params), C.byref(legacy._state), case.tape[t].data_ptr(),
                                    C.byref(ios[t % 2]), N, stream), "beng_snake_step")
        torch.cuda.synchronize()
        assert torch.equal(managed.obs, legacy.obs) and torch.equal(managed._core, legacy._core), t
        assert torch.equal(managed._ring, legacy._ring) and torch.equal(managed.stats, legacy.stats), t
        assert torch.equal(managed.reward, legacy.reward) and torch.equal(managed.terminated, legacy.terminated), t
        listed = legacy.done_env[:int(counts[t % 2])]
        assert torch.equal(torch.sort(managed.finished_envs()).values, torch.sort(listed).values), t
    assert managed.episode_stats()["n_episodes"] > 0
