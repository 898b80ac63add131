"""The C oracle of TrafficManagementEnv against golden vectors produced by the reference itself
(tests/golden/traffic_golden.npz) and, in the build container, the live reference.  Everything is integer
dynamics + float64 expressions of integers in the reference's order: the comparison is EXACT."""
import zlib

import numpy as np
import pytest

from oracle import golden_files, philox, ref_loader, replay
from oracle.c_oracle import TrafficOracle

CASES = ["random_default", "random_hi_ids", "all_zero", "all_ns", "all_ew", "alternate", "custom_grid"]


@pytest.fixture(scope="module")
def tgold():
    return golden_files.load("traffic")


def meta(g, name):
    n_envs, n_steps, seed, base, snap, rows, cols, ni, maxv = (int(x) for x in g[f"{name}/meta"])
    return dict(n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, snap=snap, grid=(rows, cols), ni=ni,
                max_vehicles=maxv, spawn_rate=float(g[f"{name}/spawn_rate"]))


def make_oracle(m, autoreset="same_step"):
    return TrafficOracle(m["n_envs"], m["grid"], m["ni"], m["max_vehicles"], m["spawn_rate"], seed=m["seed"],
                         env_id_base=m["base"], autoreset=autoreset)


def crc_rows(obs):
    return np.array([zlib.crc32(o.tobytes()) for o in obs], dtype=np.uint32)


@pytest.mark.parametrize("name", CASES)
def test_c_oracle_matches_golden_exactly(tgold, name):
    g, m = tgold, meta(tgold, name)
    orc = make_oracle(m)
    assert np.array_equal(orc.reset(), g[f"{name}/reset_obs"])
    for t in range(m["n_steps"]):
        obs, rew, term, trunc = orc.step(g[f"{name}/action"][:, t].astype(np.int64))
        assert np.array_equal(orc.reward64, g[f"{name}/reward"][:, t]), t
        assert np.array_equal(term, g[f"{name}/terminated"][:, t]) and not trunc.any()
        assert np.array_equal(crc_rows(obs), g[f"{name}/obs_crc"][:, t]), t
        st = orc.state()
        for k in ("num_vehicles", "timestep", "rng_counter", "phase", "qlen", "passed"):
            assert np.array_equal(st[k].astype(np.int64), g[f"{name}/{k}"][:, t].astype(np.int64)), (k, t)
        if t % m["snap"] == 0:
            assert np.array_equal(obs, g[f"{name}/snap_obs"][:, t // m["snap"]])
    assert orc.stats()["n_episodes"] == int(g[f"{name}/terminated"].sum())


def test_reference_facts(tgold):
    """SURVEY.md section 8(c) anchors as pinned by the reference's own outputs."""
    g = tgold
    ph = g["all_zero/phase"]
    assert (ph[:, 0] == 1).all()           # first update(): NS_GREEN with timer 0 advances to NS_YELLOW at once
    assert (ph[:, 1] == 1).all() and (ph[:, 2] == 1).all() and (ph[:, 3] == 2).all()   # yellow lasts 3, green at step 4
    assert (g["all_zero/rng_counter"][:, 2] <= 3 * 6).all()
    assert g["random_default/num_vehicles"].max() == 50          # the pool saturates at max_vehicles
    term = g["random_default/terminated"]
    assert term.sum() == 6 and (g["random_default/timestep"][term == 1] == 0).all()   # time limit -> terminated -> reset
    assert g["random_default/reset_obs"].shape[1] == 130


def test_modes_and_masked_reset(tgold):
    m = meta(tgold, "random_default")
    act = tgold["random_default/action"].astype(np.int64)
    dis, nxt, same = (make_oracle(m, k) for k in ("disabled", "next_step", "same_step"))
    for o in (dis, nxt, same):
        o.reset()
    for t in range(1003):
        for o in (dis, nxt, same):
            o.step(act[:, t])
        if t < 999:
            assert np.array_equal(dis.obs, same.obs) and np.array_equal(nxt.obs, same.obs)
    assert (dis.state()["timestep"] == 1003).all() and dis.terminated.all()
    assert (nxt.state()["timestep"] == 2).all() and (same.state()["timestep"] == 3).all()
    mask = np.array([1, 0, 1], np.uint8)
    same.reset(mask)
    assert same.state()["timestep"].tolist() == [0, 3, 0]


@pytest.mark.skipif(not ref_loader.reference_available(),
                    reason="needs the original project's sources (BENG_REFERENCE_ROOT=<its checkout>)")
def test_c_oracle_matches_live_reference():
    env_mod, utils_mod = ref_loader.load_traffic()
    n, T, seed = 3, 1100, 31
    tape = philox.action_tape(seed, np.arange(n, dtype=np.uint64), 0, T, 3, 9)
    orc = TrafficOracle(n, seed=seed)
    orc.reset()
    envs = []
    for e in range(n):
        rr = replay.ReplayRandom(seed, e)
        env_mod.random = utils_mod.random = rr
        env = env_mod.TrafficManagementEnv()
        obs, _ = env.reset()
        assert np.array_equal(obs, orc.obs[e])
        envs.append((env, rr))
    for t in range(T):
        orc.step(tape[:, t])
        st = orc.state()
        for e, (env, rr) in enumerate(envs):
            env_mod.random = utils_mod.random = rr
            obs, r, term, trunc, info = env.step(tape[e, t])
            if term:
                obs, _ = env.reset()
            assert r == orc.reward64[e] and term == bool(orc.terminated[e]) and np.array_equal(obs, orc.obs[e])
            assert rr.counter == st["rng_counter"][e]


def test_kernel_arithmetic_shortcuts_are_exact():
    """The step kernel replaces three IEEE divisions by cheaper sequences (csrc/traffic.cu: div_const, the reciprocal
    table of the mean waiting time, the multiply-shift for start // cols).  Each is restated here in exact rational
    arithmetic / NumPy and compared with the division it stands for."""
    from fractions import Fraction as F

    rng = np.random.default_rng(7)
    # (a) div_const<B> (csrc/beng_common.cuh): q = RN(x*y), r = fma(-B, q, x), result = fma(r, y, q), y = RN(1/B)  ==  x / B
    def div_const(x, b):
        y = 1.0 / b
        q = x * y
        r = float(F(x) - b * F(q))            # an FMA rounds the exact expression once
        return float(F(q) + F(r) * F(y))

    def div9(x):
        return div_const(x, 9)

    # smartclimate's time of day, (step % 1440) / 60 (csrc/climate.cu), uses the same sequence with B = 60
    assert all(div_const(float(m), 60) == m / 60.0 for m in range(1440))

    xs = [float(s) for s in range(0, 9181)]    # every possible sum of nine queue totals (9 * 4 * 255)
    for _ in range(20000):                     # sums of squared deviations as _calculate_reward forms them
        q = rng.integers(0, 60, size=9).astype(np.float64)
        xs.append(float(np.sum((q - np.sum(q) / 9.0) ** 2)))
    xs += list(rng.random(5000) * 2.0 ** rng.integers(-40, 40, size=5000))
    assert all(div9(x) == x / 9.0 for x in xs)

    # (b) float32(qw / cnt) == float32(float64(qw) * RN(1/cnt)) below the 100.0 clamp (and both sides clamp above it)
    cnt = np.arange(1, 256, dtype=np.int64)
    rcp = 1.0 / cnt.astype(np.float64)
    for qw in [np.arange(0, 4096, dtype=np.int64), rng.integers(0, 1 << 24, size=8192), rng.integers(0, 1 << 31, size=8192)]:
        a = qw[:, None].astype(np.float64)
        ref = np.minimum((a / cnt[None, :]).astype(np.float32), np.float32(100.0))
        got = np.minimum((a * rcp[None, :]).astype(np.float32), np.float32(100.0))
        assert np.array_equal(ref, got)

    # (c) start // cols for start < 25 as (start * ceil(2^16 / cols)) >> 16
    for cols in list(range(1, 4000)) + [65535, 65536, 65537, (1 << 31) - 1]:
        inv = (65536 + cols - 1) // cols
        assert all((s * inv) >> 16 == s // cols for s in range(25))
