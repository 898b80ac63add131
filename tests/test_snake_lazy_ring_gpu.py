"""Length-2 snakes off the ring.  The state record caches the direction of the last move that moved the head and a
tail-known bit; a length-2 body is then the head and the cell one step against that move, and the ring is written from
length 3 on.  Both step kernels must keep the same rules: every step here is compared with the C oracle (observation,
reward, flags, exported state and bodies) and, byte for byte, with a composing twin (state records and rings too)."""
import numpy as np
import pytest
import torch

from oracle.c_oracle import SnakeOracle

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MOVES = ((-1, 0), (0, 1), (1, 0), (0, -1))  # 0 up, 1 right, 2 down, 3 left
BITS = 0x1C  # last_move (bits 2-3) and tail_known (bit 4) of the direction byte


@pytest.fixture(scope="module")
def pkg():
    import custom_gymnasium_environments_b200 as p

    p._lib.load()
    return p


def np_(t):
    return t.cpu().numpy()


def greedy_actions(obs, st, G):
    """Food-seeking policy that avoids walls and the body when it can (the rule of oracle/gen_golden.greedy_action)."""
    n = obs.shape[0]
    hr, hc, fr, fc, d = (st[k].astype(np.int64) for k in ("head_r", "head_c", "food_r", "food_c", "direction"))
    best, best_key = d.copy(), np.full(n, np.iinfo(np.int64).max)
    for a, (dr, dc) in enumerate(MOVES):
        nr, nc = hr + dr, hc + dc
        wall = (nr < 0) | (nr >= G) | (nc < 0) | (nc >= G)
        body = np.zeros(n, bool)
        ok = ~wall
        body[ok] = obs[np.nonzero(ok)[0], nr[ok], nc[ok]] == 1
        key = (wall | body) * 1_000_000 + (np.abs(nr - fr) + np.abs(nc - fc)) * 10 + a
        key = np.where(np.abs(a - d) == 2, np.iinfo(np.int64).max, key)
        upd = key < best_key
        best, best_key = np.where(upd, a, best), np.where(upd, key, best_key)
    return best


class Trio:
    """`env` steps in place (BatchedSnakeEnv.step), `ref` composes every row into its own buffer, `orc` is the C
    oracle; all three start from the same seed."""

    def __init__(self, pkg, n, G, mode, max_steps=1000, seed=13):
        self.n, self.G = n, G
        self.env = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=seed, autoreset_mode=mode, max_steps=max_steps)
        self.ref = pkg.BatchedSnakeEnv(n, G, device=DEV, seed=seed, autoreset_mode=mode, max_steps=max_steps)
        self.orc = SnakeOracle(n, G, max_steps=max_steps, seed=seed, autoreset=mode)
        self.env.reset(), self.ref.reset()
        assert np.array_equal(np_(self.env.obs), self.orc.reset())
        self.ref_obs = self.ref.obs.clone()

    def step(self, a):
        at = torch.from_numpy(np.ascontiguousarray(a, np.int64)).to(DEV)
        self.env.step(at)
        self.ref.step(at, out_obs=self.ref_obs)
        self.orc.step(a)

    def check(self, t, bodies=True):
        env, ref, orc = self.env, self.ref, self.orc
        assert torch.equal(env.obs, self.ref_obs), t
        for name in ("_core", "_ring", "reward", "terminated", "truncated", "ep_return", "ep_length", "ep_score",
                     "stats"):
            assert torch.equal(getattr(env, name), getattr(ref, name)), (name, t)
        assert np.array_equal(np_(env.obs), orc.obs), t
        assert np.array_equal(np_(env.reward), orc.reward), t
        assert np.array_equal(np_(env.terminated).astype(np.uint8), orc.terminated), t
        st, ost = env.export_state(with_body=bodies), orc.state()
        for k in ost:
            assert np.array_equal(np_(st[k]).astype(np.int64), ost[k].astype(np.int64)), (k, t)
        if bodies:
            check_bodies(np_(st["body"]), orc, range(self.n))
        return st


def check_bodies(body, orc, envs):
    for e in envs:
        want = orc.body(e)
        assert np.array_equal(body[e, :len(want)], want) and (body[e, len(want):] == -1).all(), e


def length2_tails(obs, st, G):
    """For every env: the tail cell of a length-2 snake (the body cell of the row that is not the head), else -1."""
    n = obs.shape[0]
    flat = (obs.reshape(n, -1) == 1).copy()
    head = st["head_r"].astype(np.int64) * G + st["head_c"]
    flat[np.arange(n), head] = False
    tail = np.argmax(flat, axis=1)
    return np.where((st["length"] == 2) & flat.any(axis=1), tail, -1)


def test_disabled_mode_length2_deaths_and_turns(pkg):
    """Auto-reset DISABLED: a length-2 snake that dies stays where it is (its direction may have turned) and keeps
    stepping, so its tail must still be the cell against its last move and not against its direction -- including a
    turn back into the tail right after a death that changed the direction."""
    n, G, T = 2048, 6, 260
    tr = Trio(pkg, n, G, "disabled")
    rng = np.random.default_rng(1)
    prev_died = np.zeros(n, bool)
    into_tail_after_death = length2_deaths = 0
    for t in range(T):
        ost = tr.orc.state()
        greedy = greedy_actions(tr.orc.obs, ost, G)
        a = np.where(rng.random(n) < 0.5, greedy, rng.integers(0, 4, n))
        # where a length-2 snake has just died, often turn toward its tail
        tails = length2_tails(tr.orc.obs, ost, G)
        hr, hc, d = ost["head_r"].astype(np.int64), ost["head_c"].astype(np.int64), ost["direction"].astype(np.int64)
        to_tail = np.full(n, -1)
        for k, (dr, dc) in enumerate(MOVES):
            to_tail = np.where((tails >= 0) & ((hr + dr) * G + hc + dc == tails) & (hr + dr >= 0) & (hr + dr < G)
                               & (hc + dc >= 0) & (hc + dc < G), k, to_tail)
        steer = prev_died & (to_tail >= 0) & (rng.random(n) < 0.5)
        a = np.where(steer, to_tail, a)
        # a turn into the tail that the reversal guard lets through only because the death turned the direction
        into_tail = prev_died & (to_tail >= 0) & (a == to_tail) & (np.abs(a - d) != 2)
        tr.step(a)
        st = tr.check(t, bodies=(t % 4 == 0))
        died = tr.orc.reward < 0
        assert (died[into_tail]).all(), t  # moving into the tail is a self-hit
        into_tail_after_death += int(into_tail.sum())
        length2_deaths += int((died & (ost["length"] == 2)).sum())
        prev_died = died
    assert int(np_(st["length"]).max()) >= 3
    assert length2_deaths > 100 and into_tail_after_death > 20, (length2_deaths, into_tail_after_death)


@pytest.mark.parametrize("mode", ["same_step", "next_step"])
@pytest.mark.parametrize("G,n,T", [(4, 512, 300), (7, 512, 400)])
def test_growth_and_ring_wrap(pkg, mode, G, n, T):
    """A greedy tape grows snakes 1 -> 2 -> 3 and on (the meal that makes length 3 writes the ring's first three
    entries); on small boards the ring wraps around many times.  Bodies, observations and rewards every step."""
    tr = Trio(pkg, n, G, mode, max_steps=250)
    rng = np.random.default_rng(G)
    wraps = meals_to_3 = 0
    for t in range(T):
        a = greedy_actions(tr.orc.obs, tr.orc.state(), G)
        noise = rng.random(n) < 0.05
        a = np.where(noise, rng.integers(0, 4, n), a)
        before = tr.env._core.clone()
        len_before = np_((before[:, 1] >> 16) & 0xFFFF)
        tr.step(a)
        tr.check(t)
        core = tr.env._core
        length = np_((core[:, 1] >> 16) & 0xFFFF)
        ring_head, ring_head_before = np_((core[:, 2] >> 16) & 0xFFFF), np_((before[:, 2] >> 16) & 0xFFFF)
        wraps += int(((len_before >= 3) & (length >= 3) & (ring_head < ring_head_before)).sum())
        meals_to_3 += int(((len_before == 2) & (length == 3)).sum())
    assert meals_to_3 > 50 and wraps > 20, (meals_to_3, wraps)
    assert int(tr.orc.length.max()) >= min(10, G * G - 2)
    if mode == "same_step":
        assert tr.env.episode_stats() == tr.orc.stats()


def old_format(env):
    """The state of `env` as the ring-for-length-2 layout stored it: the last-move and tail-known bits cleared, and
    every length-2 snake's tail and head written to the ring at tail_index and ring_head.  Returns (core, ring)."""
    st = env.export_state(with_body=True)
    core, ring = env._core.clone(), env._ring.clone()
    cells = env.grid_size ** 2
    core[:, 1] &= ~BITS
    two = torch.nonzero(st["length"] == 2).flatten()
    rh = ((core[two, 2] >> 16) & 0xFFFF).long()
    ring[two, rh] = st["body"][two, 0].to(torch.int16)
    ring[two, (rh - 1) % cells] = st["body"][two, 1].to(torch.int16)
    return core, ring


@pytest.mark.parametrize("in_place", [True, False])
@pytest.mark.parametrize("mode", ["same_step", "next_step"])
def test_old_format_states_continue_like_twin(pkg, mode, in_place):
    """A state record without the new bits (a checkpoint of the earlier layout, length-2 tails in the ring) steps
    exactly like its twin that has them: observations, rewards, flags, episode outputs, statistics, exported state
    and bodies; the first move of each length-2 snake sets the bits, after which the two keep matching."""
    n, G, T = 4096, 8, 60
    kw = dict(device=DEV, seed=21, autoreset_mode=mode, max_steps=120)
    twin, old = pkg.BatchedSnakeEnv(n, G, **kw), pkg.BatchedSnakeEnv(n, G, **kw)
    twin.reset(), old.reset()
    rng = np.random.default_rng(3)

    def tape():
        greedy = greedy_actions(np_(twin.obs), {k: np_(v) for k, v in twin.export_state().items()}, G)
        return torch.from_numpy(np.where(rng.random(n) < 0.3, rng.integers(0, 4, n), greedy)).to(DEV)

    for _ in range(40):  # grow a population of length-2 and longer snakes
        a = tape()
        twin.step(a), old.step(a)
    n2 = int((twin.export_state()["length"] == 2).sum())
    assert n2 > 300, n2
    assert int((twin._core[:, 1] & BITS != 0).sum()) > 0
    core, ring = old_format(twin)
    old._core.copy_(core), old._ring.copy_(ring)
    assert torch.equal(old.export_state(with_body=True)["body"], twin.export_state(with_body=True)["body"])
    outs = (torch.empty_like(twin.obs), torch.empty_like(old.obs))
    for t in range(T):
        a = tape()
        if in_place:
            twin.step(a), old.step(a)
            o_twin, o_old = twin.obs, old.obs
        else:
            twin.step(a, out_obs=outs[0]), old.step(a, out_obs=outs[1])
            o_twin, o_old = outs
        assert torch.equal(o_twin, o_old), t
        for name in ("reward", "terminated", "truncated", "ep_return", "ep_length", "ep_score", "stats"):
            assert torch.equal(getattr(twin, name), getattr(old, name)), (name, t)
        assert torch.equal(torch.sort(twin.finished_envs()).values, torch.sort(old.finished_envs()).values), t
        s_twin, s_old = twin.export_state(with_body=True), old.export_state(with_body=True)
        for k in s_twin:
            assert torch.equal(s_twin[k], s_old[k]), (k, t)
        if not in_place:
            twin.obs.copy_(outs[0])  # (keeps the greedy tape reading the current observation)


@pytest.mark.parametrize("mode", ["same_step", "next_step"])
def test_state_dict_round_trip(pkg, mode):
    """A checkpoint taken mid-rollout (length-2 snakes with the new bits among them) loads into a fresh env that then
    steps exactly like the original: its first step composes, the later ones patch in place."""
    n, G = 3000, 6
    kw = dict(device=DEV, seed=5, autoreset_mode=mode, max_steps=90)
    src, dst = pkg.BatchedSnakeEnv(n, G, **kw), pkg.BatchedSnakeEnv(n, G, seed=99, device=DEV, autoreset_mode=mode,
                                                                     max_steps=90)
    src.reset(), dst.reset()
    rng = np.random.default_rng(8)

    def tape():
        greedy = greedy_actions(np_(src.obs), {k: np_(v) for k, v in src.export_state().items()}, G)
        return torch.from_numpy(np.where(rng.random(n) < 0.2, rng.integers(0, 4, n), greedy)).to(DEV)

    for _ in range(30):
        src.step(tape())
    assert int((src.export_state()["length"] == 2).sum()) > 100
    dst.load_state_dict(src.state_dict())
    assert torch.equal(dst.export_state(with_body=True)["body"], src.export_state(with_body=True)["body"])
    for t in range(50):
        a = tape()
        src.step(a), dst.step(a)
        assert torch.equal(src.obs, dst.obs), t
        for name in ("_core", "_ring", "reward", "terminated", "stats"):
            assert torch.equal(getattr(src, name), getattr(dst, name)), (name, t)
        done = src.terminated  # (the episode outputs are written for finished envs only, and are not state)
        for name in ("ep_return", "ep_length", "ep_score"):
            assert torch.equal(getattr(src, name)[done], getattr(dst, name)[done]), (name, t)
