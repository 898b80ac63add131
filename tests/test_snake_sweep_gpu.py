"""The in-place snake step visits its CTAs in ascending order on one launch and in descending order on the next (the
parity of the self-managed done-counter block picks the order), and writes the rows of non-eating length-2 snakes as
whole 32-byte sectors.  Neither may change a result: after every step the in-place env must equal, byte for byte, a
twin with the same seed whose steps compose every row (beng_snake_step) -- observations, state records, rings,
rewards, flags, episode outputs, statistics and the (sorted) finished-env list."""
import ctypes as C

import numpy as np
import pytest
import torch

DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    p._lib.load()
    return p


def random_tape(n, t, seed):
    g = torch.Generator(device=DEV).manual_seed(seed * 7919 + t)
    return torch.randint(0, 4, (n,), device=DEV, generator=g)


def assert_same(env, ref, obs, ref_obs):
    assert torch.equal(obs, ref_obs)
    for name in ("_core", "_ring", "reward", "terminated", "truncated", "ep_return", "ep_length", "ep_score", "stats"):
        assert torch.equal(getattr(env, name), getattr(ref, name)), name
    fin = torch.sort(env.finished_envs()).values  # (the list's order is unspecified)
    assert torch.equal(fin, torch.sort(ref.finished_envs()).values)


class EnvTwin:
    """`env` steps in place through BatchedSnakeEnv.step() (the device-managed counter contract); `ref`, same seed,
    composes full rows into its own obs with step(out_obs=...)."""

    def __init__(self, pkg, n, G=20, **kw):
        self.env = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=11, **kw)
        self.ref = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=11, **kw)
        self.env.reset(), self.ref.reset()
        self.ref_obs = self.ref.obs.clone()

    def step(self, a):
        self.env.step(a)
        self.ref_step(a)

    def ref_step(self, a):
        self.ref.step(a, out_obs=self.ref_obs)

    def check(self):
        assert_same(self.env, self.ref, self.env.obs, self.ref_obs)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("same_step", "next_step"))
@pytest.mark.parametrize("n", (1, 255, 257, 256 * 41 + 37))
def test_every_step_matches_composing_twin(pkg, n, mode):
    """Odd and even steps alike (the sweep direction flips every launch), the ragged last CTA included."""
    tw = EnvTwin(pkg, n, max_steps=30, autoreset_mode=mode)
    for t in range(75):
        tw.step(random_tape(n, t, n))
        tw.check()
    assert int(tw.env.stats[0]) > 0


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("same_step", "next_step"))
def test_full_batch_every_step(pkg, mode):
    n = 1 << 20
    tw = EnvTwin(pkg, n, max_steps=20, autoreset_mode=mode)
    for t in range(25):
        tw.step(random_tape(n, t, 3))
        tw.check()


@pytest.mark.gpu
def test_graph_replays_of_odd_length_between_eager_steps(pkg):
    """A graph of 3 steps flips the sweep direction an odd number of times, so each replay starts on the other
    direction than the one before; eager steps between replays shift it again."""
    n, k = 256 * 9 + 37, 3
    tw = EnvTwin(pkg, n, max_steps=25, autoreset_mode="same_step")
    tapes = [random_tape(n, t, 5) for t in range(k + 40)]
    tw.step(tapes[-1])  # env.obs is current: every step from here on is the in-place one
    tw.check()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        for a in tapes[:k]:
            tw.env.step(a)
    for r in range(12):
        graph.replay()
        for a in tapes[:k]:
            tw.ref_step(a)
        tw.check()
        for e in range(r % 3):  # 0, 1 or 2 eager steps
            tw.step(tapes[k + r * 2 + e])
            tw.check()
    assert int(tw.env.stats[0]) > 0


def obs_buffer(n, G, mis):
    """A zeroed (n, G, G) int8 view whose data pointer is `mis` bytes past a 32-byte boundary."""
    raw = torch.zeros(n * G * G + 64, dtype=torch.int8, device=DEV)
    off = (mis - raw.data_ptr()) % 32
    view = raw[off:off + n * G * G].view(n, G, G)
    assert view.data_ptr() % 32 == mis
    return view


def length2_states(n, G, seed):
    """Length-2 snakes everywhere on the board, the edge cells included: head, a tail next to it, food on a free cell
    (next to the head in the direction of the action for a quarter of the envs, i.e. a meal), a random direction (so
    that some actions turn the head into the tail) and a random action.  Returns (core, ring, obs, action) as numpy."""
    rng = np.random.default_rng(seed)
    cells = G * G
    moves = np.array([(-1, 0), (0, 1), (1, 0), (0, -1)])  # 0 up, 1 right, 2 down, 3 left
    core = np.zeros((n, 4), dtype=np.uint32)
    ring = np.zeros((n, cells), dtype=np.int16)
    obs = np.zeros((n, cells), dtype=np.int8)
    act = rng.integers(0, 4, n)
    for e in range(n):
        while True:
            hr, hc = rng.integers(0, G, 2)
            tr, tc = np.array([hr, hc]) + moves[rng.integers(0, 4)]
            if 0 <= tr < G and 0 <= tc < G:
                break
        head, tail = hr * G + hc, tr * G + tc
        fr, fc = np.array([hr, hc]) + moves[act[e]]
        food = fr * G + fc
        if e % 4 != 0 or not (0 <= fr < G and 0 <= fc < G) or food == tail:
            while True:
                food = int(rng.integers(0, cells))
                if food not in (head, tail):
                    break
        rh = int(rng.integers(0, cells))
        ring[e, rh], ring[e, (rh - 1) % cells] = head, tail
        obs[e, head] = obs[e, tail] = 1
        obs[e, food] = 2
        d = int(rng.integers(0, 4))
        core[e] = (hr | (hc << 8) | ((food // G) << 16) | ((food % G) << 24), d | (2 << 16), rh << 16,
                   int(rng.integers(0, 1 << 20)))
    return core.view(np.int32), ring, obs, act


@pytest.mark.gpu
@pytest.mark.parametrize("mis", (0, 16))
@pytest.mark.parametrize("G,n", [(2, 257), (3, 1031), (20, 20000), (64, 600)])
def test_constructed_length2_moves(pkg, G, n, mis):
    """Constructed length-2 snakes on buffers that start on a 32-byte boundary or 16 bytes past one, stepped through
    the C ABI: moves whose new head or cleared tail lies in a sector shared with the neighbouring row, moves into the
    snake's own tail, meals and wall deaths, then onwards with random actions."""
    env = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=7, max_steps=500, autoreset_mode="same_step")
    ref = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=7, max_steps=500, autoreset_mode="same_step")
    env.reset(), ref.reset()
    core, ring, obs, act = length2_states(n, G, seed=G * 2 + mis)
    for e in (env, ref):
        e._core.copy_(torch.from_numpy(core))
        e._ring.copy_(torch.from_numpy(ring))
    buf = obs_buffer(n, G, mis)
    buf.copy_(torch.from_numpy(obs).view(n, G, G))
    scratch = torch.empty_like(ref.obs)
    lib = pkg._lib
    io = env._make_io(buf)

    def step(a):
        lib.check(env.lib.beng_snake_step_inplace(C.byref(env.params), C.byref(env._state), a.data_ptr(), C.byref(io),
                                                  n, torch.cuda.current_stream().cuda_stream), "step_inplace")
        ref.step(a, out_obs=scratch)
        assert_same(env, ref, buf, scratch)

    a0 = torch.from_numpy(act).to(DEV)
    step(a0)
    length = env.export_state()["length"]
    assert int((length == 3).sum()) > 0  # meals
    assert int((env.reward == -10).sum()) > 0  # deaths: into the tail, into a wall
    # At G = 20 every other 400-byte row starts 16 bytes past a sector boundary whatever the buffer's alignment, so some
    # new heads lie in a 32-byte sector that reaches into the neighbouring row.  (At G = 64 a row is 128 sectors: on a
    # 32-byte aligned buffer no sector straddles two rows.)
    if G == 20:
        st = env.export_state()
        row = buf.data_ptr() + torch.arange(n, device=DEV, dtype=torch.int64) * G * G
        sec = (row + st["head_r"] * G + st["head_c"]) // 32 * 32
        assert int(((sec < row) | (sec + 32 > row + G * G)).sum()) > 0
    for t in range(40):
        step(random_tape(n, t, G))
