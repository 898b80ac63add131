"""CPU checks of the measurement harness and the registration shim: the reference arm of bench.py runs here (it is the
Python port of the reference loop on the host cores) and prints the JSON line the driver parses; the registration ids
are the reference's."""
import json
import os
import subprocess
import sys
import types

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_bench(*args):
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *args], capture_output=True, text=True,
                         timeout=600, cwd=ROOT)
    assert out.returncode == 0, out.stderr[-2000:]
    lines = [ln for ln in out.stdout.splitlines() if ln.strip()]
    assert len(lines) == 1, "exactly ONE JSON line on stdout"
    return json.loads(lines[0])


def test_reference_arm_prints_the_contract_line():
    d = run_bench("--impl", "reference", "--steps", "2", "--warmup", "1")
    assert d["impl"] == "reference" and d["metric"] == "env_steps_per_sec" and d["unit"] == "env-steps/s"
    assert d["n_gpus"] == 1 and d["steps"] == 2 and d["higher_is_better"] is True and d["scaling"] == "weak"
    assert d["vs_baseline"] is None and d["data"] == "synthetic" and "workload" in d["config"]
    assert d["value"] > 0 and d["ms_per_step"] > 0
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("port", "reference") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    e = d["e2e"]
    assert e["value"] == d["value"] and e["unit"] == d["unit"]
    assert e["h2d_bytes_per_step"] == 0 and e["d2h_bytes_per_step"] == 0


def test_b200_arm_refuses_to_run_without_a_gpu():
    """No CPU fallback: without CUDA the product arm must fail loudly, not print a number."""
    import torch

    if torch.cuda.is_available():
        return
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "1", "--warmup", "1"],
                         capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0
    assert not any(ln.strip().startswith("{") and '"value"' in ln for ln in out.stdout.splitlines())


def load_dump(directory):
    return {f[:-4]: np.load(os.path.join(directory, f)) for f in sorted(os.listdir(directory))}


def test_dump_keeps_a_fixed_sample_of_envs_within_64_mb(tmp_path):
    """bench.dump_step_outputs on a step result larger than 64 MB: float32/float64 files, nested infos flattened, the
    same sampled rows in every per-env array, and the same files from two calls."""
    import torch

    import bench
    from custom_gymnasium_environments_b200.vector import LazyInfos

    n = 1 << 17
    g = torch.Generator().manual_seed(0)
    obs = torch.rand((n, 130), generator=g)
    term = torch.rand(n, generator=g) < 0.1
    info = LazyInfos({"episode": {"r": torch.randn(n, dtype=torch.float64, generator=g)}, "_episode": term})
    info.lazy["score"] = lambda: torch.arange(n, dtype=torch.int32)
    step_out = (obs, torch.randn(n, generator=g), term, torch.zeros(n, dtype=torch.bool), info)
    for tag in ("a", "b"):
        bench.dump_step_outputs(str(tmp_path / tag), step_out, n)
    a, b = load_dump(tmp_path / "a"), load_dump(tmp_path / "b")
    assert set(a) == {"env_index", "obs", "reward", "terminated", "truncated", "info._episode", "info.episode.r",
                      "info.score"}
    assert all(np.array_equal(a[k], b[k]) and a[k].dtype == b[k].dtype for k in a)
    assert sum(os.path.getsize(tmp_path / "a" / f"{k}.npy") for k in a) <= 64e6
    idx = a["env_index"].astype(np.int64)
    assert 0 < len(idx) < n and np.all(np.diff(idx) > 0)
    assert a["obs"].dtype == np.float32 and np.array_equal(a["obs"], obs.numpy()[idx])
    assert a["terminated"].dtype == np.float32 and np.array_equal(a["terminated"], term.numpy()[idx])
    assert a["info.episode.r"].dtype == np.float64 and np.array_equal(a["info.episode.r"], info["episode"]["r"].numpy()[idx])
    assert a["info.score"].dtype == np.float64 and np.array_equal(a["info.score"], idx)


def test_dump_refuses_what_it_cannot_write_exactly(tmp_path):
    """An integer float64 would round (beyond 2**53) is refused, and so is --dump-outputs on the reference arm, which
    computes nothing on the CUDA engine."""
    import torch

    import bench

    n = 8
    wide = torch.full((n,), 2 ** 53 + 1, dtype=torch.int64)
    with pytest.raises(ValueError, match="2\\*\\*53"):
        bench.dump_step_outputs(str(tmp_path / "d"), (torch.zeros(n), torch.zeros(n), wide, wide, {}), n)
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--dump-outputs", str(tmp_path / "r")], capture_output=True, text=True, timeout=600, cwd=ROOT)
    assert out.returncode != 0 and "--dump-outputs" in out.stderr and not out.stdout.strip()
    assert not (tmp_path / "r").exists()


@pytest.mark.gpu
def test_dump_outputs_is_the_last_timed_step_and_repeats_run_to_run(tmp_path):
    """--dump-outputs DIR after W warm-up and K timed steps (one launch each): every array equals what step() returns
    when the same seeded env is driven through the same W + K steps of the benchmark's action tape; the same arguments
    write the same arrays, and one more timed step writes a different last step."""
    import torch

    import bench
    import custom_gymnasium_environments_b200 as pkg

    n, warmup = 4096, 3
    common = ["--env", "snake", "--envs-per-gpu", str(n), "--warmup", str(warmup), "--e2e-steps", "1", "--no-secondary",
              "--no-cpu-baseline", "--no-l2-flush"]
    dumps = {}
    for tag, steps in (("a", 40), ("b", 40), ("c", 41)):
        d = run_bench(*common, "--steps", str(steps), "--dump-outputs", str(tmp_path / tag))
        assert d["steps"] == steps and d["gpu_launches"] == steps
        dumps[tag] = load_dump(tmp_path / tag)
    a, b, c = dumps["a"], dumps["b"], dumps["c"]
    assert {"env_index", "obs", "reward", "terminated", "truncated", "info.score", "info.snake_length"} <= set(a)
    assert a["obs"].shape == (n, 20, 20) and np.array_equal(a["env_index"], np.arange(n))
    assert all(v.dtype in (np.float32, np.float64) for v in a.values())
    assert set(a) == set(b) and all(np.array_equal(a[k], b[k]) for k in a)
    assert not np.array_equal(a["obs"], c["obs"])

    # the benchmark's env (seed 0, env ids 0..n-1) and tape (step t takes beng_fill_random_actions counter t)
    lib = pkg._lib.load()
    env = pkg.BatchedSnakeEnv(n, 20, device="cuda:0", seed=0, env_id_base=0)
    env.reset()
    actions = torch.empty(n, dtype=torch.int64, device="cuda:0")
    for t in range(warmup + 40):
        pkg._lib.check(lib.beng_fill_random_actions(actions.data_ptr(), n, 1, 4, t, 0, 0,
                                                    torch.cuda.current_stream().cuda_stream), "beng_fill_random_actions")
        out = env.step(actions)
    want = {}
    for name, value in zip(("obs", "reward", "terminated", "truncated", "info"), out):
        bench._flatten(name, value, want)
    assert set(a) == set(want) | {"env_index"}
    for k, v in want.items():
        assert np.array_equal(a[k], v.cpu().numpy().astype(a[k].dtype)), k
    assert (a["reward"] != 0).any()  # the compared step is not a trivial one: some snakes eat or die in it


def test_registration_ids_match_the_reference(monkeypatch):
    registry, calls = {}, []

    def register(id, entry_point, max_episode_steps=None, **kw):  # noqa: A002 (gymnasium's own argument name)
        registry[id] = entry_point
        calls.append((id, entry_point, max_episode_steps))

    gym = types.ModuleType("gymnasium")
    envs = types.ModuleType("gymnasium.envs")
    reg = types.ModuleType("gymnasium.envs.registration")
    reg.register, reg.registry = register, registry
    gym.envs, envs.registration = envs, reg
    for name, mod in (("gymnasium", gym), ("gymnasium.envs", envs), ("gymnasium.envs.registration", reg)):
        monkeypatch.setitem(sys.modules, name, mod)
    from custom_gymnasium_environments_b200 import registration

    registration.register_all()  # (importing the package may already have done it: registration is idempotent)
    got = {i: (e, m) for i, e, m in calls}
    assert set(got) == set(registry) == {"snake_env_classic-v0", "CryptoTrading-v0", "TrafficManagement-v0",
                                         "SmartClimateEnv-v0"}
    assert got["snake_env_classic-v0"][1] == got["CryptoTrading-v0"][1] == got["TrafficManagement-v0"][1] == 1000
    for env_id, (entry, _) in got.items():  # every entry point resolves to a class of this package
        module, cls = entry.split(":")
        assert hasattr(__import__(module, fromlist=[cls]), cls), env_id
    registration.register_all()
    assert len(calls) == 4  # nothing is registered twice


def test_facades_are_gymnasium_envs_when_gymnasium_is_importable(tmp_path):
    """gym.make() refuses entry points that do not inherit gymnasium.Env: with a gymnasium on the path the single-instance
    facades must subclass its Env (and the batched classes its VectorEnv).  Checked in a subprocess with a stub package."""
    pkg = tmp_path / "gymnasium"
    (pkg / "vector").mkdir(parents=True)
    (pkg / "envs").mkdir()
    (pkg / "__init__.py").write_text("class Env:\n    metadata = {}\n    render_mode = None\n")
    (pkg / "vector" / "__init__.py").write_text("class VectorEnv:\n    metadata = {}\n    closed = False\n")
    (pkg / "envs" / "__init__.py").write_text("")
    (pkg / "envs" / "registration.py").write_text(
        "registry = {}\n"
        "def register(id, entry_point, max_episode_steps=None, **kw):\n"
        "    registry[id] = entry_point\n")
    code = ("import gymnasium, gymnasium.vector, custom_gymnasium_environments_b200 as p\n"
            "for c in (p.SnakeEnvClassic, p.CryptoTradingEnv, p.TrafficManagementEnv, p.SmartClimateEnv, p.WorldBuilderEnv):\n"
            "    assert issubclass(c, gymnasium.Env), c\n"
            "for c in (p.BatchedSnakeEnv, p.BatchedCryptoTradingEnv, p.BatchedTrafficManagementEnv):\n"
            "    assert issubclass(c, gymnasium.vector.VectorEnv), c\n"
            "from gymnasium.envs.registration import registry\n"
            "assert 'snake_env_classic-v0' in registry and 'CryptoTrading-v0' in registry, registry\n"
            "print('ok')\n")
    out = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=300, cwd=ROOT,
                         env=dict(os.environ, PYTHONPATH=f"{tmp_path}{os.pathsep}{ROOT}"))
    assert out.returncode == 0 and "ok" in out.stdout, out.stdout + out.stderr
