"""The host side of the delta-encoded snake observation path, without a GPU: beng_snake_apply_obs_delta replays change
records (include/beng.h, BENG_OBS_DELTA_*) onto a host copy of the observations.  The records here come from a numpy
reference encoder run on consecutive observations of the C oracle, so every kind of step (move, eat, death, invalid
action, auto-reset in all three modes, time limit, full board) passes through the applier."""
import ctypes as C

import numpy as np
import pytest

from oracle import c_oracle

CLEAR = 0x80000000
UNUSED = 3 << 12
NONE = UNUSED | (UNUSED << 14)
BAD_ARG, UNSUPPORTED = -1, -2


@pytest.fixture(scope="module")
def lib():
    from custom_gymnasium_environments_b200 import _lib

    return _lib.load()


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def encode(prev, cur):
    """Reference encoder: one record per env turning row `prev` into row `cur`.  Up to two changed cells are listed as
    pairs; otherwise the row is cleared and its nonzero cells are listed (a fresh snake: head and food)."""
    n = prev.shape[0]
    prev, cur = prev.reshape(n, -1), cur.reshape(n, -1)
    changed = prev != cur
    clear = changed.sum(1) > 2
    listed = np.where(clear[:, None], cur != 0, changed)
    assert (listed.sum(1) <= 2).all(), "a cleared row holds at most two nonzero cells"
    first_two = np.argsort(~listed, axis=1, kind="stable")[:, :2]  # listed cells first, in cell order
    value = np.take_along_axis(cur, first_two, 1).astype(np.uint32)
    used = np.take_along_axis(listed, first_two, 1)
    pairs = np.where(used, first_two.astype(np.uint32) | (value << 12), UNUSED).astype(np.uint32)
    return (np.where(clear, CLEAR, 0) | pairs[:, 0] | (pairs[:, 1] << 14)).astype(np.uint32)


def greedy_actions(obs, st, G):
    """Food-seeking policy of oracle/gen_golden.greedy_action, vectorised over envs: among the moves that are not a
    reversal, prefer one that does not die, then the one closest to the food, then the lowest action."""
    n = obs.shape[0]
    hr, hc, fr, fc, d = (st[k].astype(np.int64) for k in ("head_r", "head_c", "food_r", "food_c", "direction"))
    best = d.copy()
    best_key = np.full(n, np.iinfo(np.int64).max)
    for a, (dr, dc) in enumerate(((-1, 0), (0, 1), (1, 0), (0, -1))):
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


def tape(policy, seed, n, t, obs, st, G):
    """Actions of step t.  The random tape carries ~3 % out-of-space actions (the env is left untouched)."""
    if policy == "greedy":
        return greedy_actions(obs, st, G)
    a = c_oracle.action_tape(seed, 0, n, t, 4)
    bad = c_oracle.action_tape(seed + 1, 0, n, t, 32) == 0
    return np.where(bad, np.where(a & 1, 4, -1), a)


@pytest.mark.parametrize("policy,max_steps", [("random", 37), ("greedy", 1000), ("greedy", 60)])
@pytest.mark.parametrize("n", [1, 31, 333])
@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("G", [20, 15, 8, 5, 64])
def test_apply_replays_oracle_observations(lib, G, mode, n, policy, max_steps):
    seed = 1000 * G + n
    orc = c_oracle.SnakeOracle(n, G, max_steps=max_steps, seed=seed, autoreset=mode)
    orc.reset()
    mirrors = {nt: orc.obs.copy() for nt in (1, 3, 64)}
    steps = 200 if (policy == "greedy" and G <= 8) else 60
    kinds = set()
    for t in range(steps):
        prev = orc.obs.copy()
        orc.step(tape(policy, seed, n, t, orc.obs, orc.state(), G))
        rec = encode(prev, orc.obs)
        kinds.update({"clear" if r & CLEAR else "none" if r == NONE else "pairs" for r in rec.tolist()})
        for nt, m in mirrors.items():
            assert lib.beng_snake_apply_obs_delta(ptr(rec), ptr(m), n, G, nt) == 0
            assert np.array_equal(m, orc.obs), (nt, t)
    assert "pairs" in kinds
    if mode != "disabled" and policy == "random" and n > 1:
        assert "clear" in kinds  # auto-resets happened


def test_record_layout(lib):
    """Pair A before pair B, the clear before both; value 3 leaves a cell alone; NONE changes nothing."""
    G = 4
    obs = np.arange(3 * G * G, dtype=np.int8).reshape(3, G, G) % 3
    want = obs.copy()
    rec = np.array([(5 | 1 << 12) | ((5 | 2 << 12) << 14),      # A then B on one cell: B wins
                    CLEAR | (7 | 1 << 12) | (UNUSED << 14),      # cleared row, one cell set
                    NONE], np.uint32)
    want[0].flat[5] = 2
    want[1] = 0
    want[1].flat[7] = 1
    assert lib.beng_snake_apply_obs_delta(ptr(rec), ptr(obs), 3, G, 2) == 0
    assert np.array_equal(obs, want)


def test_argument_errors(lib):
    G, n = 8, 10
    obs = np.zeros((n, G, G), np.int8)
    rec = np.full(n, NONE, np.uint32)
    assert lib.beng_snake_apply_obs_delta(None, ptr(obs), n, G, 1) == BAD_ARG
    assert lib.beng_snake_apply_obs_delta(ptr(rec), None, n, G, 1) == BAD_ARG
    assert lib.beng_snake_apply_obs_delta(ptr(rec), ptr(obs), -1, G, 1) == BAD_ARG
    assert lib.beng_snake_apply_obs_delta(ptr(rec), ptr(obs), n, 1, 1) == UNSUPPORTED
    assert lib.beng_snake_apply_obs_delta(ptr(rec), ptr(obs), n, 65, 1) == UNSUPPORTED
    assert lib.beng_snake_apply_obs_delta(None, None, 0, G, 1) == 0
    for nt in (0, -3, 1000):  # <= 0 means one thread; more threads than envs is fine
        assert lib.beng_snake_apply_obs_delta(ptr(rec), ptr(obs), n, G, nt) == 0
    assert not obs.any()
    for bad in (NONE | (1 << 28), (G * G) | (1 << 12) | (UNUSED << 14), UNUSED | ((G * G + 3) << 14)):
        r = rec.copy()
        r[7] = bad
        assert lib.beng_snake_apply_obs_delta(ptr(r), ptr(obs), n, G, 3) == BAD_ARG, hex(bad)
    assert not obs.any()

    # the device entry point refuses missing or misaligned record buffers before touching the GPU
    from custom_gymnasium_environments_b200 import _lib

    p = _lib.SnakeParams(G, 1000, 2, 0, 0, 0)
    st = _lib.SnakeState(16, 16)
    io = _lib.SnakeIO(obs=16, reward=16, terminated=16)
    args = (C.byref(p), C.byref(st), 16, C.byref(io), n, 16)
    host = np.zeros(n + 1, np.uint32)
    assert lib.beng_snake_step_host_delta(*args, None, ptr(host), None, None, None, None, None, None) == BAD_ARG
    assert lib.beng_snake_step_host_delta(*args, 16, None, None, None, None, None, None, None) == BAD_ARG
    assert lib.beng_snake_step_host_delta(*args, 18, ptr(host), None, None, None, None, None, None) == BAD_ARG
    assert lib.beng_snake_step_host_delta(*args, 16, host.ctypes.data + 2, None, None, None, None, None, None) == BAD_ARG
