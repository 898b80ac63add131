"""beng_snake_step_inplace writes the rows of length-1 snakes as whole 32-byte sectors, except sectors that reach into a
neighbouring env's row.  Called here through the C ABI on observation buffers that start on a 32-byte boundary or 16
bytes past one (the ABI only asks for 16), every step must leave the buffer, the results and the state byte for byte
as the composing kernel (beng_snake_step) leaves them for a twin env with the same seed."""
import ctypes as C

import pytest
import torch

DEV = "cuda:0"


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    p._lib.load()
    return p


def obs_buffer(n, G, mis):
    """A zeroed (n, G, G) int8 view whose data pointer is `mis` bytes past a 32-byte boundary."""
    raw = torch.zeros(n * G * G + 64, dtype=torch.int8, device=DEV)
    off = (mis - raw.data_ptr()) % 32
    view = raw[off:off + n * G * G].view(n, G, G)
    assert view.data_ptr() % 32 == mis
    return view


class Twin:
    """`env` steps through beng_snake_step_inplace on `buf`; `ref` (same seed) composes full rows with beng_snake_step."""

    def __init__(self, pkg, n, G, mis, **kw):
        self.pkg, self.n, self.G = pkg, n, G
        self.env = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=5, **kw)
        self.ref = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=5, **kw)
        self.buf = obs_buffer(n, G, mis)
        self.scratch = torch.empty_like(self.ref.obs)
        self.env.reset(), self.ref.reset()
        self.buf.copy_(self.env.obs)

    def set_state(self, core, obs):
        """The same state record (and empty ring) in both envs, and the observation that goes with it."""
        for e in (self.env, self.ref):
            e._core.copy_(core)
            e._ring.zero_()
        self.buf.copy_(obs)

    def step(self, act):
        env = self.env
        env._parity ^= 1
        io = env._make_io(self.buf, env._parity)
        lib = self.pkg._lib
        lib.check(env.lib.beng_snake_step_inplace(C.byref(env.params), C.byref(env._state), act.data_ptr(),
                                                  C.byref(io), self.n, torch.cuda.current_stream().cuda_stream),
                  "beng_snake_step_inplace")
        ref_out = self.ref.step(act, out_obs=self.scratch)
        assert torch.equal(self.buf, self.scratch)
        for x, y in zip((env.reward, env.terminated, env.truncated), ref_out[1:4]):
            assert torch.equal(x, y)
        fin = torch.sort(env.finished_envs()).values  # (the list's order is unspecified)
        assert torch.equal(fin, torch.sort(self.ref.finished_envs()).values)
        assert torch.equal(env._core, self.ref._core)
        assert torch.equal(env.stats, self.ref.stats)

    def check_state(self):
        assert torch.equal(self.env._ring, self.ref._ring)


def random_tape(n, t, seed):
    g = torch.Generator(device=DEV).manual_seed(seed * 7919 + t)
    return torch.randint(0, 4, (n,), device=DEV, generator=g)


@pytest.mark.gpu
@pytest.mark.parametrize("mis", (0, 16))
@pytest.mark.parametrize("G,n", [(2, 37), (5, 4099), (8, 1031), (15, 300), (20, 4099), (33, 257), (64, 97)])
def test_aligned_and_misaligned_buffers(pkg, G, n, mis):
    tw = Twin(pkg, n, G, mis, max_steps=120, autoreset_mode="same_step")
    for t in range(160):
        tw.step(random_tape(n, t, G))
    tw.check_state()


def edge_tape(n, t, top):
    """Envs with index parity `top` climb to grid row 0 and zig-zag leftwards over rows 0 and 1; the others descend to
    row 19 and zig-zag rightwards over rows 19 and 18, until they hit the wall.  Actions 0 up, 1 right, 2 down, 3 left."""
    up = (torch.arange(n, device=DEV) % 2) == top
    a_up = 0 if t < 10 else (3, 2, 3, 0)[(t - 10) % 4]
    a_down = 2 if t < 9 else (1, 0, 1, 2)[(t - 9) % 4]
    return torch.where(up, a_up, a_down)


@pytest.mark.gpu
@pytest.mark.parametrize("mis", (0, 16))
@pytest.mark.parametrize("top", (0, 1))
def test_cells_at_row_edges(pkg, mis, top):
    """At G = 20 with a 32-byte aligned buffer, cells 0..15 of odd rows and 384..399 of even rows lie in sectors shared
    with the neighbouring row, and neighbours move inside such a sector in the same step; 16 bytes past a boundary it is
    the other way round.  Each choice of `top` sends the envs to the straddling edge cells for one alignment and to
    the whole sectors at the row edges for the other."""
    n, G = 4096, 20
    tw = Twin(pkg, n, G, mis, max_steps=1000, autoreset_mode="same_step")
    at_edge = 0
    for t in range(40):
        tw.step(edge_tape(n, t, top))
        st = tw.env.export_state()
        cell = st["head_r"] * G + st["head_c"]
        at_edge += int(((cell < 16) | (cell >= 384)).sum())
    tw.check_state()
    assert at_edge > 4 * n  # most envs spent several steps in the edge cells


def pack_core(head_r, head_c, food_r, food_c, direction, ctr):
    x = head_r | (head_c << 8) | (food_r << 16) | (food_c << 24)
    y = direction | (1 << 16)  # length 1, no flags
    return torch.stack([x, y, torch.zeros_like(x), ctr], 1).to(torch.int32)


@pytest.mark.gpu
@pytest.mark.parametrize("mis", (0, 16))
def test_length1_meals(pkg, mis):
    """Length-1 snakes set one step away from their food, every one of them eating: the new food is placed from the
    two body cells and lands in all kinds of sectors, among them the head's own."""
    n, G = 65536, 20
    tw = Twin(pkg, n, G, mis, max_steps=1000, autoreset_mode="same_step")
    g = torch.Generator(device=DEV).manual_seed(17)
    hr, hc = (torch.randint(1, G - 1, (n,), device=DEV, generator=g) for _ in range(2))
    act = torch.randint(0, 4, (n,), device=DEV, generator=g)
    fr = hr + (act == 2).long() - (act == 0).long()
    fc = hc + (act == 1).long() - (act == 3).long()
    ctr = torch.randint(0, 1 << 20, (n,), device=DEV, generator=g)
    core = pack_core(hr, hc, fr, fc, act, ctr)  # direction == action: never a reversal
    obs = torch.zeros(n, G * G, dtype=torch.int8, device=DEV)
    obs.scatter_(1, (hr * G + hc)[:, None], 1)
    obs.scatter_(1, (fr * G + fc)[:, None], 2)
    tw.set_state(core, obs.view(n, G, G))
    tw.step(act)
    tw.check_state()
    st = tw.env.export_state()
    assert bool((st["length"] == 2).all())
    base = tw.buf.data_ptr() + torch.arange(n, device=DEV) * G * G
    head_sec = (base + st["head_r"] * G + st["head_c"]) // 32
    food_sec = (base + st["food_r"] * G + st["food_c"]) // 32
    assert int((head_sec == food_sec).sum()) > 100
    for t in range(30):  # and on from there
        tw.step(random_tape(n, t, 99))
    tw.check_state()


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ("same_step", "next_step"))
def test_full_batch_misaligned(pkg, mode):
    n = 1 << 20
    tw = Twin(pkg, n, 20, 16, max_steps=40, autoreset_mode=mode, time_limit_truncation=True)
    for t in range(64):
        tw.step(random_tape(n, t, 1))
    tw.check_state()
    assert int(tw.env.stats[0]) > 0
