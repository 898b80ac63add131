"""The host-side protocol every Batched*Env shares: reset-before-step, the reset_mask rules, the checkpoint keys, the
exact-shape rule for array actions, and the Dict action forms climate accepts."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
N = 64  # != 9, so that a transposed traffic action array has another shape
NAMES = ["snake", "crypto", "traffic", "climate", "builder"]

STATE_KEYS = {
    "snake": {"core", "ring"},
    "builder": {"words", "grid"},
    "traffic": {"light", "passed", "waiting", "qmeta", "qwait", "misc", "total_reward"},
    "climate": {"f64", "i32"},
    "crypto": {"scal", "meta", "ep_return", "close", "ohlv", "window_head", "config"},
}


@pytest.fixture(scope="module")
def pkg():
    if not torch.cuda.is_available():
        pytest.skip("needs a GPU")
    import custom_gymnasium_environments_b200 as p
    return p


def make(pkg, name, n=N):
    """-> (env, numpy actions of the right shape, numpy actions of a wrong shape)."""
    rng = np.random.default_rng(5)
    if name == "snake":
        return pkg.BatchedSnakeEnv(n, device=DEV), rng.integers(0, 4, n), rng.integers(0, 4, (n, 1))
    if name == "crypto":
        return pkg.BatchedCryptoTradingEnv(n, None, "discrete", device=DEV), rng.integers(0, 5, n), rng.integers(0, 5, n + 1)
    if name == "traffic":
        act = rng.integers(0, 3, (n, 9))
        return pkg.BatchedTrafficManagementEnv(n, device=DEV), act, np.ascontiguousarray(act.T)
    if name == "builder":
        return pkg.BatchedWorldBuilderEnv(n, device=DEV), rng.integers(0, 5, n), rng.integers(0, 5, (n, 1))
    act = {"ac_temp": rng.uniform(16, 32, n).astype(np.float32), "lights": rng.integers(0, 2, (n, 4)).astype(np.int8)}
    return pkg.BatchedSmartClimateEnv(n, device=DEV), act, dict(act, lights=act["lights"][:, :3])


@pytest.mark.parametrize("name", NAMES)
def test_step_before_reset_raises(pkg, name):
    env, act, _ = make(pkg, name)
    with pytest.raises(RuntimeError, match="reset"):
        env.step(act)
    with pytest.raises(RuntimeError, match="reset"):
        env.step_host(act)


@pytest.mark.parametrize("name", NAMES)
def test_reset_mask_rules(pkg, name):
    env, _, _ = make(pkg, name)
    with pytest.raises(RuntimeError, match="first reset"):
        env.reset(options={"reset_mask": torch.ones(N, dtype=torch.bool, device=DEV)})
    env.reset()
    with pytest.raises(ValueError, match="reset_mask"):
        env.reset(options={"reset_mask": torch.ones(N + 1, dtype=torch.bool, device=DEV)})
    env.reset(options={"reset_mask": torch.ones(N, dtype=torch.bool, device=DEV)})


def test_masked_reset_resets_only_the_selected_envs(pkg):
    env, act, _ = make(pkg, "climate")
    env.reset()
    for _ in range(5):
        env.step(act)
    before = env.state_dict()
    mask = torch.arange(N, device=DEV) % 3 == 0
    env.reset(options={"reset_mask": mask})
    after = env.state_dict()
    keep = ~mask
    assert torch.equal(before["f64"][:, keep], after["f64"][:, keep])
    assert torch.equal(before["i32"][:, keep], after["i32"][:, keep])
    assert (before["i32"][1] == 5).all()
    assert (env.current_step[mask] == 0).all() and (env.current_step[keep] == 5).all()


@pytest.mark.parametrize("name", NAMES)
def test_state_dict_keys(pkg, name):
    env, _, _ = make(pkg, name)
    env.reset()
    assert set(env.state_dict()) == STATE_KEYS[name] | {"stats", "seed", "env_id_base"}


@pytest.mark.parametrize("name", NAMES)
def test_wrongly_shaped_numpy_actions_raise(pkg, name):
    env, act, bad = make(pkg, name)
    env.reset()
    with pytest.raises(ValueError):
        env.step(bad)
    env.step(act)


def test_climate_accepts_ac_temp_as_n_or_n_by_1(pkg):
    """ac_temp as (n,) or (n, 1), numpy or CUDA: the same trajectory."""
    _, act, _ = make(pkg, "climate")
    forms = {
        "numpy (n,)": lambda a: a,
        "numpy (n, 1)": lambda a: a.reshape(N, 1),
        "cuda (n,)": lambda a: torch.from_numpy(a).to(DEV),
        "cuda (n, 1)": lambda a: torch.from_numpy(a).to(DEV).reshape(N, 1),
    }
    results = {}
    for form, f in forms.items():
        env = pkg.BatchedSmartClimateEnv(N, device=DEV)
        env.reset()
        for t in range(4):
            obs, rew, term, trunc, _ = env.step({"ac_temp": f(act["ac_temp"] + t), "lights": act["lights"]})
        results[form] = (obs.cpu(), rew.cpu(), env.state_dict())
    ref_obs, ref_rew, ref_sd = results["numpy (n,)"]
    for form, (obs, rew, sd) in results.items():
        assert torch.equal(obs, ref_obs) and torch.equal(rew, ref_rew), form
        for k in ("f64", "i32"):
            assert torch.equal(sd[k], ref_sd[k]), (form, k)
