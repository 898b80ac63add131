"""The host side of the delta-encoded world-builder grid path, without a GPU: beng_builder_apply_obs_delta replays change
records (include/beng.h, BENG_BUILDER_DELTA_*) onto a host copy of the grids.  The records here come from a numpy
reference encoder run on consecutive grids of the C oracle, so every kind of step (build, failed build, full board,
pass, invalid action, auto-reset in all three modes) passes through the applier."""
import ctypes as C

import numpy as np
import pytest

from oracle import c_oracle

NONE, CLEAR = 0, 0x80000000
BAD_ARG, UNSUPPORTED = -1, -2


@pytest.fixture(scope="module")
def lib():
    from custom_gymnasium_environments_b200 import _lib

    return _lib.load()


def ptr(a):
    return a.ctypes.data_as(C.c_void_p)


def encode(prev, cur):
    """Reference encoder: one record per env turning row `prev` into row `cur`.  No change gives NONE, one cell going
    from empty to a building gives cell | value << 8, anything else must be a reset: CLEAR."""
    n = prev.shape[0]
    prev, cur = prev.reshape(n, -1), cur.reshape(n, -1)
    changed = prev != cur
    n_changed = changed.sum(1)
    cell = changed.argmax(1)
    old, new = prev[np.arange(n), cell], cur[np.arange(n), cell]
    build = (n_changed == 1) & (old == 0) & (new > 0)
    clear = (n_changed > 0) & ~build
    assert not cur[clear].any(), "a row that changed in any other way must have been reset to empty"
    rec = np.where(build, cell.astype(np.uint32) | (new.astype(np.uint32) << 8), NONE)
    return np.where(clear, CLEAR, rec).astype(np.uint32)


def tape(policy, seed, n, t):
    """Actions of step t.  "random": uniform over Discrete(5) with ~3 % out-of-space actions (-1, 5), which leave the
    env untouched; "build": buildings only, which fills small boards."""
    if policy == "build":
        return c_oracle.action_tape(seed, 0, n, t, 4) + 1
    a = c_oracle.action_tape(seed, 0, n, t, 5)
    bad = c_oracle.action_tape(seed + 1, 0, n, t, 32) == 0
    return np.where(bad, np.where(a & 1, 5, -1), a)


@pytest.mark.parametrize("policy", ["random", "build"])
@pytest.mark.parametrize("n", [1, 31, 333])
@pytest.mark.parametrize("mode", ["same_step", "next_step", "disabled"])
@pytest.mark.parametrize("G", [10, 15, 7, 4, 2])
def test_apply_replays_oracle_grids(lib, G, mode, n, policy):
    seed = 1000 * G + n
    orc = c_oracle.BuilderOracle(n, G, seed=seed, autoreset=mode)
    orc.reset()
    mirrors = {nt: orc.grid.copy() for nt in (1, 3, 64)}
    kinds, full_board = set(), False
    for t in range(80):
        prev = orc.grid.copy()
        orc.step(tape(policy, seed, n, t))
        rec = encode(prev, orc.grid)
        kinds.update({"clear" if r & CLEAR else "none" if r == NONE else "build" for r in rec.tolist()})
        full_board |= bool((orc.grid.reshape(n, -1) != 0).all(1).any())
        for nt, m in mirrors.items():
            assert lib.beng_builder_apply_obs_delta(ptr(rec), ptr(m), n, G, nt) == 0
            assert np.array_equal(m, orc.grid), (nt, t)
    assert "build" in kinds
    if mode != "disabled":
        assert "clear" in kinds  # auto-resets happened
    if policy == "build" and G <= 4 and n > 1:
        assert full_board


def test_record_layout(lib):
    """The clear before the cell write; value 0 with cell 0 leaves the cell alone; NONE changes nothing."""
    G = 4
    grid = (np.arange(4 * G * G, dtype=np.int8).reshape(4, G, G) % 5)
    want = grid.copy()
    rec = np.array([7 | 3 << 8,              # write 3 to cell 7
                    CLEAR | 15 | 4 << 8,     # cleared row, then cell 15 (the last) = 4
                    CLEAR,                   # cleared row only
                    NONE], np.uint32)
    want[0].flat[7] = 3
    want[1] = 0
    want[1].flat[15] = 4
    want[2] = 0
    assert lib.beng_builder_apply_obs_delta(ptr(rec), ptr(grid), 4, G, 2) == 0
    assert np.array_equal(grid, want)


def test_argument_errors(lib):
    G, n = 7, 10
    grid = np.zeros((n, G, G), np.int8)
    rec = np.full(n, NONE, np.uint32)
    assert lib.beng_builder_apply_obs_delta(None, ptr(grid), n, G, 1) == BAD_ARG
    assert lib.beng_builder_apply_obs_delta(ptr(rec), None, n, G, 1) == BAD_ARG
    assert lib.beng_builder_apply_obs_delta(ptr(rec), ptr(grid), -1, G, 1) == BAD_ARG
    assert lib.beng_builder_apply_obs_delta(ptr(rec), ptr(grid), n, 1, 1) == UNSUPPORTED
    assert lib.beng_builder_apply_obs_delta(ptr(rec), ptr(grid), n, 16, 1) == UNSUPPORTED
    assert lib.beng_builder_apply_obs_delta(None, None, 0, G, 1) == 0
    for nt in (0, -3, 1000):  # <= 0 means one thread; more threads than envs is fine
        assert lib.beng_builder_apply_obs_delta(ptr(rec), ptr(grid), n, G, nt) == 0
    assert not grid.any()
    malformed = [1 << 11, 1 << 30, CLEAR | (1 << 20),    # bits 11-30
                 5 << 8, 7 << 8 | 3,                     # value > 4
                 (G * G) | 1 << 8, 255 | 4 << 8,         # cell >= G*G with a value
                 3, CLEAR | 1]                           # cell != 0 without a value
    for bad in malformed:
        r = rec.copy()
        r[7] = bad
        r[8] = 1 | 1 << 8  # a valid record after the malformed one in the same chunk
        assert lib.beng_builder_apply_obs_delta(ptr(r), ptr(grid), n, G, 3) == BAD_ARG, hex(bad)
        assert not grid[7].any()  # a malformed record is not applied
    assert lib.beng_builder_apply_obs_delta(ptr(np.array([(G * G - 1) | 2 << 8], np.uint32)), ptr(grid), 1, G, 1) == 0
    assert grid[0].flat[G * G - 1] == 2

    # the device entry point refuses missing or misaligned record buffers before touching the GPU
    from custom_gymnasium_environments_b200 import _lib

    p = _lib.BuilderParams(G, 2, 0, 0)
    st = _lib.BuilderState(16)
    io = _lib.BuilderIO(grid=16, reward=16, terminated=16)
    args = (C.byref(p), C.byref(st), 16, C.byref(io), n, 16)
    host = np.zeros(n + 1, np.uint32)
    rest = (None,) * 6
    assert lib.beng_builder_step_host_delta(*args, None, ptr(host), *rest) == BAD_ARG
    assert lib.beng_builder_step_host_delta(*args, 16, None, *rest) == BAD_ARG
    assert lib.beng_builder_step_host_delta(*args, 18, ptr(host), *rest) == BAD_ARG
    assert lib.beng_builder_step_host_delta(*args, 16, host.ctypes.data + 2, *rest) == BAD_ARG
