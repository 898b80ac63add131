"""CPU-side checks of the running observation / reward normalization: the float64 oracle against hand-computed cases,
the C ABI's argument checks (all before anything launches) and the ctypes binding against include/beng.h."""
import ctypes as C
import os
import re

import numpy as np
import pytest

from oracle.vecnormalize import RunningMeanStd, VecNormalizeOracle

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BAD_ARG = -1
ADDR = 1 << 20  # a 16-byte aligned stand-in device address: the checks below never dereference it


# ---------------------------------------------------------------------------------------------- oracle
def test_running_mean_std_first_update_by_hand():
    rms = RunningMeanStd((1,))
    rms.update(np.array([[1.0], [3.0]]))
    # batch mean 2, batch var 1, n 2 merged into (mean 0, var 1, count 1e-4)
    tot = 1e-4 + 2
    assert rms.count == tot
    assert rms.mean[0] == 2.0 * 2 / tot
    assert rms.var[0] == (1.0 * 1e-4 + 1.0 * 2 + 4.0 * 1e-4 * 2 / tot) / tot


def test_chan_combine_of_two_batches_equals_the_variance_of_their_concatenation():
    rng = np.random.default_rng(0)
    a = rng.normal(3.0, 2.0, (517, 4))
    b = rng.normal(-1.0, 0.5, (211, 4)) + np.array([0.0, 1e6, -5.0, 1e-3])
    rms = RunningMeanStd((4,))
    rms.mean, rms.var, rms.count = a.mean(0), a.var(0), float(len(a))  # the moments of batch a
    rms.update(b)
    both = np.concatenate([a, b])
    assert rms.count == len(both)
    np.testing.assert_allclose(rms.mean, both.mean(0), rtol=1e-13)
    np.testing.assert_allclose(rms.var, both.var(0), rtol=1e-9)


def test_oracle_step_reset_and_clip_by_hand():
    o = VecNormalizeOracle(2, 1, clip_obs=1.5, clip_reward=0.5, gamma=0.5, epsilon=0.0)
    obs = np.array([[0.0], [4.0]], np.float32)
    n0 = o.reset(obs)
    tot = 1e-4 + 2
    mean, var = 2.0 * 2 / tot, (1e-4 + 4.0 * 2 + 4.0 * 1e-4 * 2 / tot) / tot
    np.testing.assert_array_equal(n0[:, 0], np.clip((np.array([0.0, 4.0]) - mean) / np.sqrt(var), -1.5, 1.5)
                                  .astype(np.float32))
    assert np.all(np.abs(n0) <= 1.5)
    o.returns[:] = [2.0, 4.0]
    _, r = o.step(obs, np.array([1.0, -1.0], np.float32), np.array([True, False]), np.array([False, False]))
    assert o.ret_rms.count == 1e-4 + 2
    np.testing.assert_array_equal(o.returns, [0.0, 1.0])  # 2 * 0.5 + 1 -> zeroed (terminated); 4 * 0.5 - 1
    # returns before the reset were (2, 1): batch mean 1.5, var 0.25
    assert np.all(np.abs(r) <= 0.5) and r[0] == 0.5 and r[1] == -0.5
    o.training = False
    o.returns[:] = [3.0, 3.0]
    o.step(obs, np.zeros(2, np.float32), np.array([False, False]), np.array([False, True]))
    np.testing.assert_array_equal(o.returns, [3.0, 0.0])  # frozen: no update, finished envs still zeroed
    o.reset(obs, mask=np.array([True, False]))
    np.testing.assert_array_equal(o.returns, [0.0, 0.0])


# ---------------------------------------------------------------------------------------------- C ABI
def header_fields(struct):
    text = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "beng.h")).read(), flags=re.S)
    body = re.search(r"typedef struct %s \{(.*?)\} %s;" % (struct, struct), text, flags=re.S).group(1)
    return re.findall(r"(\w+);", body)


def test_normalize_bindings_match_header():
    from custom_gymnasium_environments_b200 import _lib

    assert [f[0] for f in _lib.NormalizeParams._fields_] == header_fields("beng_normalize_params")
    assert [f[0] for f in _lib.NormalizeIO._fields_] == header_fields("beng_normalize_io")
    assert C.sizeof(_lib.NormalizeParams) == 40 and C.sizeof(_lib.NormalizeIO) == 10 * 8
    text = open(os.path.join(ROOT, "include", "beng.h")).read()
    for name, value in (("BENG_NORM_OBS", _lib.NORM_OBS), ("BENG_NORM_REWARD", _lib.NORM_REWARD),
                        ("BENG_NORM_UPDATE", _lib.NORM_UPDATE)):
        assert re.search(r"#define %s %du" % (name, value), text), name
    assert {"beng_normalize", "beng_normalize_workspace_bytes"} <= set(_lib.SIGNATURES)


def test_workspace_bytes():
    from custom_gymnasium_environments_b200 import _lib

    lib = _lib.load()
    assert lib.beng_normalize_workspace_bytes(-1, 4) == 0 and lib.beng_normalize_workspace_bytes(4, 0) == 0
    # 16-byte header + one (sum, sum of squares) float64 pair per CTA and column (dim features + the returns)
    for n, dim in ((1, 1), (2053, 261), (262144, 261), (1 << 20, 9), (65536, 130)):
        ws = lib.beng_normalize_workspace_bytes(n, dim)
        assert (ws - 16) % ((dim + 1) * 16) == 0 and 1 <= (ws - 16) // ((dim + 1) * 16) <= min(n, 296)


def call_args(L, flags, **io_fields):
    p = L.NormalizeParams(10.0, 10.0, 1e-8, 0.99, flags, 0)
    io = L.NormalizeIO(*([ADDR] * 10))
    for k, v in io_fields.items():
        setattr(io, k, v)
    return p, io


ALL = 7


@pytest.mark.parametrize("case", [
    dict(n=64, dim=0), dict(n=-1, dim=4), dict(n=64, dim=4, flags=8),
    dict(n=64, dim=4, obs=None), dict(n=64, dim=4, obs=ADDR + 2), dict(n=64, dim=4, obs_rms=None),
    dict(n=64, dim=4, obs_rms=ADDR + 4), dict(n=64, dim=4, obs_out=ADDR + 1),
    dict(n=64, dim=4, reward=None), dict(n=64, dim=4, reward=ADDR + 2), dict(n=64, dim=4, returns=None),
    dict(n=64, dim=4, returns=ADDR + 4), dict(n=64, dim=4, ret_rms=None), dict(n=64, dim=4, reward_out=ADDR + 2),
    dict(n=64, dim=4, workspace=None), dict(n=64, dim=4, workspace=ADDR + 8),
    dict(n=64, dim=4, clip_obs=-1.0), dict(n=64, dim=4, epsilon=float("nan")), dict(n=64, dim=4, gamma=-0.5),
])
def test_bad_arguments_are_rejected_before_launch(case):
    from custom_gymnasium_environments_b200 import _lib as L

    lib = L.load()
    case = dict(case)
    n, dim, flags = case.pop("n"), case.pop("dim"), case.pop("flags", ALL)
    scalars = {k: case.pop(k) for k in ("clip_obs", "epsilon", "gamma") if k in case}
    p, io = call_args(L, flags, **case)
    for k, v in scalars.items():
        setattr(p, k, v)
    before = lib.beng_launch_count()
    assert lib.beng_normalize(C.byref(p), C.byref(io), n, dim, None) == BAD_ARG
    assert lib.beng_normalize(None, C.byref(io), 64, 4, None) == BAD_ARG
    assert lib.beng_normalize(C.byref(p), None, 64, 4, None) == BAD_ARG
    assert lib.beng_launch_count() == before


def test_pointers_a_call_does_not_need_are_not_checked():
    from custom_gymnasium_environments_b200 import _lib as L

    lib = L.load()
    before = lib.beng_launch_count()
    # n = 0: every check runs, nothing launches
    p, io = call_args(L, ALL, terminated=None, truncated=None, obs_out=None, reward_out=None)
    assert lib.beng_normalize(C.byref(p), C.byref(io), 0, 261, None) == 0
    # reward only: the observation side may be NULL
    p, io = call_args(L, L.NORM_REWARD | L.NORM_UPDATE, obs=None, obs_rms=None, obs_out=None)
    assert lib.beng_normalize(C.byref(p), C.byref(io), 0, 1, None) == 0
    # observations only, frozen: no reward side, no workspace
    p, io = call_args(L, L.NORM_OBS, reward=None, returns=None, ret_rms=None, reward_out=None, workspace=None)
    assert lib.beng_normalize(C.byref(p), C.byref(io), 0, 9, None) == 0
    # frozen observations without an output: nothing to do, nothing launches even for n > 0
    p, io = call_args(L, L.NORM_OBS, obs_out=None, workspace=None)
    assert lib.beng_normalize(C.byref(p), C.byref(io), 64, 9, None) == 0
    assert lib.beng_launch_count() == before
