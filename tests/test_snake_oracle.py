"""The CPU oracle restatements of SnakeEnvClassic against the golden vectors produced by the
reference itself (tests/golden/snake_golden.npz, oracle/gen_golden.py), and -- in the build
container, where /root/reference exists -- against the live reference."""
import zlib

import numpy as np
import pytest

from conftest import case_meta
from oracle import philox, ref_loader, replay
from oracle.c_oracle import SnakeOracle
from oracle.snake_port import SnakePort

CASES = ["random_g20", "random_g20_hi", "greedy_g20", "greedy_g8", "greedy_g5", "random_g15", "circle_g20",
         "reverse_g20"]


def crc_rows(obs):
    return np.array([zlib.crc32(o.tobytes()) for o in obs], dtype=np.uint32)


@pytest.mark.parametrize("name", CASES)
def test_c_oracle_matches_golden_same_step(golden, name):
    m = case_meta(golden, name)
    g = {k: golden[f"{name}/{k}"] for k in ("action", "reward", "terminated", "score", "length", "head_r", "head_c",
                                             "food_r", "food_c", "direction", "steps", "rng_counter", "obs_crc",
                                             "snap_obs", "reset_obs", "final_score", "final_steps")}
    orc = SnakeOracle(m["n_envs"], m["G"], seed=m["seed"], env_id_base=m["base"], autoreset="same_step")
    assert np.array_equal(orc.reset(), g["reset_obs"])
    n_ep = 0
    for t in range(m["n_steps"]):
        obs, rew, term, trunc = orc.step(g["action"][:, t].astype(np.int64))
        assert np.array_equal(rew, g["reward"][:, t]), t
        assert np.array_equal(term, g["terminated"][:, t]), t
        assert not trunc.any()
        assert np.array_equal(orc.score, g["score"][:, t]) and np.array_equal(orc.length, g["length"][:, t])
        assert np.array_equal(crc_rows(obs), g["obs_crc"][:, t]), t
        st = orc.state()
        for k in ("head_r", "head_c", "food_r", "food_c", "direction", "steps", "rng_counter"):
            assert np.array_equal(st[k].astype(np.int64), g[k][:, t].astype(np.int64)), (k, t)
        if t % m["snap_every"] == 0:
            assert np.array_equal(obs, g["snap_obs"][:, t // m["snap_every"]])
        done = term.astype(bool)
        if done.any():
            assert np.array_equal(orc.ep_score[done], g["final_score"][:, t][done])
            died = g["reward"][:, t][done] < 0
            assert np.array_equal(orc.ep_length[done], g["final_steps"][:, t][done] + died)
            assert np.array_equal(orc.ep_return[done], 10.0 * g["final_score"][:, t][done] - 10.0 * died)
            n_ep += int(done.sum())
    assert orc.stats()["n_episodes"] == n_ep == int(g["terminated"].sum())


@pytest.mark.parametrize("name", ["random_g20", "greedy_g8", "circle_g20"])
def test_python_port_matches_golden(golden, name):
    m = case_meta(golden, name)
    act, rew, term = (golden[f"{name}/{k}"] for k in ("action", "reward", "terminated"))
    crc, step_crc = golden[f"{name}/obs_crc"], golden[f"{name}/step_obs_crc"]
    for e in range(min(m["n_envs"], 4)):
        env = SnakePort(m["G"], rng=replay.ReplayRandom(m["seed"], m["base"] + e))
        obs, info = env.reset()
        assert np.array_equal(obs, golden[f"{name}/reset_obs"][e]) and info == {"score": 0, "snake_length": 1}
        for t in range(m["n_steps"]):
            obs, r, te, tr, info = env.step(int(act[e, t]))
            assert (r, te, tr) == (rew[e, t], bool(term[e, t]), False)
            assert zlib.crc32(obs.tobytes()) == step_crc[e, t]
            if te:
                obs, _ = env.reset()
            assert zlib.crc32(obs.tobytes()) == crc[e, t]


def test_disabled_mode_is_the_bare_reference_class(golden):
    """SURVEY.md 8(c) anchor: nine step(1) from reset, then a wall death that freezes everything but the
    direction; turning away afterwards moves on (the reference has no 'dead' flag)."""
    rows = golden["frozen/rows"]
    orc = SnakeOracle(1, 20, seed=0, env_id_base=0, autoreset="disabled")
    orc.reset()
    for t, (r, term, steps, hr, hc, d, score, length, crc) in enumerate(rows):
        obs, rew, te, _ = orc.step(np.array([1 if t < 12 else 0]))
        st = orc.state()
        assert (rew[0], te[0], st["steps"][0], st["head_r"][0], st["head_c"][0], st["direction"][0]) == \
               (r, term, steps, hr, hc, d), t
        assert orc.score[0] == score and zlib.crc32(obs[0].tobytes()) == int(crc)
    assert rows[9][0] == -10.0 and rows[9][1] == 1 and rows[9][2] == 9  # the 10th step(1) is the wall death
    assert rows[12][0] == 0.0 and rows[12][2] == 10                      # turning up afterwards moves on


def test_next_step_mode_is_same_step_delayed():
    n, T = 64, 400
    tape = philox.action_tape(11, np.arange(n, dtype=np.uint64), 0, T, 4)
    same = SnakeOracle(n, seed=11, autoreset="same_step")
    nxt = SnakeOracle(n, seed=11, autoreset="next_step")
    same.reset(), nxt.reset()
    # drive next_step with a per-env tape pointer that stalls for one step after each termination
    ptr = np.zeros(n, dtype=np.int64)
    pending = np.zeros(n, dtype=bool)
    for t in range(T // 2):
        a = tape[np.arange(n), ptr]
        nxt.step(a)
        was_pending = pending.copy()
        pending = nxt.terminated.astype(bool)
        assert not (was_pending & pending).any() and (nxt.reward[was_pending] == 0).all()
        ptr += ~was_pending
    # replay the consumed prefix through same_step and compare final states env by env
    for e in range(n):
        one = SnakeOracle(1, seed=11, env_id_base=e, autoreset="same_step")
        one.reset()
        for t in range(ptr[e]):
            one.step(tape[e, t:t + 1])
        s1, s2 = one.state(), nxt.state()
        if not pending[e]:
            for k in s1:
                assert s1[k][0] == s2[k][e], (k, e)


def test_invalid_action_is_counted_and_ignored():
    orc = SnakeOracle(3, seed=0)
    orc.reset()
    before = orc.state()
    orc.step(np.array([7, -1, 1]))
    after = orc.state()
    assert orc.invalid == 2
    assert after["steps"].tolist() == [0, 0, 1] and before["head_c"][0] == after["head_c"][0]


def test_full_board_leaves_no_food():
    """Engine/oracle convention where the reference would spin forever (documented divergence)."""
    G = 2
    orc = SnakeOracle(256, G, seed=5, autoreset="disabled")
    orc.reset()
    rng = np.random.default_rng(0)
    seen_full = False
    for t in range(200):
        obs, *_ = orc.step(rng.integers(0, 4, 256))
        full = orc.length == G * G
        if full.any():
            seen_full = True
            assert (obs[full] == 1).all()
            assert (orc.state()["food_r"][full] == -1).all()
    assert seen_full


@pytest.mark.skipif(not ref_loader.reference_available(),
                    reason="needs the original project's sources (BENG_REFERENCE_ROOT=<its checkout>)")
@pytest.mark.parametrize("G,seed,policy", [(20, 21, "random"), (8, 22, "greedy"), (6, 23, "greedy")])
def test_c_oracle_matches_live_reference(G, seed, policy):
    from oracle.gen_golden import greedy_action

    mod = ref_loader.load_snake()
    n, T = 12, 1500
    orc = SnakeOracle(n, G, seed=seed, autoreset="same_step")
    orc.reset()
    envs = []
    for e in range(n):
        rr = replay.ReplayRandom(seed, e)
        mod.random = rr
        env = mod.SnakeEnvClassic(grid_size=G)
        obs, _ = env.reset()
        assert np.array_equal(obs, orc.obs[e])
        envs.append((env, rr))
    tape = philox.action_tape(seed, np.arange(n, dtype=np.uint64), 0, T, 4)
    for t in range(T):
        acts = np.array([greedy_action(env, G) if policy == "greedy" else tape[e, t]
                         for e, (env, _) in enumerate(envs)], dtype=np.int64)
        orc.step(acts)
        for e, (env, rr) in enumerate(envs):
            mod.random = rr
            obs, r, term, trunc, info = env.step(int(acts[e]))
            if term:
                obs, _ = env.reset()
            assert np.array_equal(obs, orc.obs[e]) and r == orc.reward[e] and term == orc.terminated[e]
            assert rr.counter == orc.state()["rng_counter"][e]
