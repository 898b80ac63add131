"""CPU-side checks: the C-ABI library loads and exports every symbol include/beng.h declares, the
product refuses to run without CUDA (no CPU fallback), host-side helpers, and the world_size-2
sharding / statistics reduction over gloo."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "beng.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(beng_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_declared_symbol():
    import custom_gymnasium_environments_b200 as pkg

    lib = ctypes.CDLL(pkg._lib.library_path())
    syms = declared_symbols()
    assert "beng_snake_step" in syms and "beng_snake_reset" in syms and "beng_snake_step_host" in syms
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/beng.h but not exported"
    assert set(pkg._lib.SIGNATURES) == set(syms), "ctypes SIGNATURES out of sync with include/beng.h"
    assert lib.beng_version() == 100 and lib.beng_compiled_arch() == 100


def test_struct_layouts_match_header():
    import custom_gymnasium_environments_b200 as pkg

    assert ctypes.sizeof(pkg._lib.SnakeParams) == 32
    assert ctypes.sizeof(pkg._lib.SnakeState) == 16
    assert ctypes.sizeof(pkg._lib.SnakeIO) == 14 * 8
    lib = pkg._lib.load()
    assert lib.beng_snake_core_bytes(1000) == 16000
    assert lib.beng_snake_ring_bytes(1000, 20) == 1000 * 400 * 2


def test_argument_errors_do_not_need_a_gpu():
    import custom_gymnasium_environments_b200 as pkg

    lib = pkg._lib.load()
    p = pkg._lib.SnakeParams(20, 1000, 2, 0, 0, 0)
    assert ctypes.sizeof(pkg._lib.CryptoParams) == 96 and ctypes.sizeof(pkg._lib.TrafficParams) == 56
    assert ctypes.sizeof(pkg._lib.BuilderParams) == 24 and ctypes.sizeof(pkg._lib.BuilderIO) == 12 * 8
    assert ctypes.sizeof(pkg._lib.ClimateParams) == 32 and ctypes.sizeof(pkg._lib.CryptoState) == 40
    st = pkg._lib.SnakeState(None, None)
    io = pkg._lib.SnakeIO()
    assert lib.beng_snake_step(ctypes.byref(p), ctypes.byref(st), None, ctypes.byref(io), 16, None) == -1
    assert lib.beng_fill_random_actions(None, 16, 1, 4, 0, 0, 0, None) == -1
    p.grid_size = 100
    st = pkg._lib.SnakeState(16, 16)
    io.obs = 16
    assert lib.beng_snake_reset(ctypes.byref(p), ctypes.byref(st), ctypes.byref(io), None, 16, 1, None) == -2


@pytest.mark.skipif(torch.cuda.is_available(), reason="CPU-only check")
def test_product_fails_loudly_without_cuda():
    import custom_gymnasium_environments_b200 as pkg

    with pytest.raises(RuntimeError, match="no CPU fallback"):
        pkg.BatchedSnakeEnv(8)
    with pytest.raises(RuntimeError):
        pkg.SnakeEnvClassic()


def test_missing_library_is_an_error(tmp_path, monkeypatch):
    from custom_gymnasium_environments_b200 import _lib

    monkeypatch.setattr(_lib, "_lib", None)
    monkeypatch.setattr(_lib, "LIB_PATH", str(tmp_path / "nope.so"))
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.load()


def test_product_never_imports_the_oracle():
    pkg_dir = os.path.join(ROOT, "custom_gymnasium_environments_b200")
    for dirpath, _, files in os.walk(pkg_dir):
        for f in files:
            if f.endswith((".py", ".cu", ".cuh", ".h")):
                text = open(os.path.join(dirpath, f)).read()
                assert not re.search(r"^\s*(from|import)\s+oracle", text, flags=re.M), f
                assert "liboracle" not in text, f


def test_spaces_and_batching():
    from custom_gymnasium_environments_b200.spaces import Box, Discrete, MultiDiscrete, batch_space

    d = Discrete(4)
    assert d.contains(3) and not d.contains(4) and not d.contains(1.0) and d.contains(np.int64(0))
    b = Box(0, 2, (20, 20), np.int8)
    assert b.shape == (20, 20) and b.dtype == np.int8 and b.contains(np.zeros((20, 20), np.int8))
    bb = batch_space(b, 5)
    assert bb.shape == (5, 20, 20)
    bd = batch_space(d, 7)
    assert isinstance(bd, MultiDiscrete) and bd.nvec.tolist() == [4] * 7
    assert 0 <= d.sample() < 4


def test_action_upload_shape_and_dtype_rules():
    """vector.as_device_actions with CPU buffers: a tensor of the buffer's dtype and shape is used as it is, anything
    else lands in the buffer in the buffer's dtype; arrays must have exactly the buffer's shape."""
    from custom_gymnasium_environments_b200.vector import as_device_actions

    buf = torch.zeros(5, dtype=torch.int64)
    same = torch.arange(5)
    assert as_device_actions(same, buf) is same
    for src in (torch.arange(6)[1:], torch.arange(5, dtype=torch.int32), torch.arange(5).reshape(5, 1),
                [0, 1, 2, 3, 4], np.arange(5, dtype=np.int16)):  # misaligned view, other dtype, other shape, list, numpy
        buf.zero_()
        out = as_device_actions(src, buf)
        assert out is buf and out.dtype == torch.int64 and out.tolist() == list(torch.as_tensor(src).reshape(5).tolist())
    for bad in (np.zeros((5, 1), np.int64), np.zeros(6, np.int64), np.zeros((1, 5), np.int64)):
        with pytest.raises(ValueError, match="shape"):
            as_device_actions(bad, buf)

    for dtype, src in ((torch.float32, np.array([[1.0, 2.0], [3.0, 4.0]])), (torch.int8, np.array([[1, 0], [0, 1]]))):
        buf = torch.zeros((2, 2), dtype=dtype)
        out = as_device_actions(src, buf)
        assert out is buf and out.dtype == dtype and np.array_equal(out.numpy(), src)
        with pytest.raises(ValueError, match="shape"):
            as_device_actions(src.T.reshape(4), buf)
        t = torch.tensor(src, dtype=dtype)
        out = as_device_actions(t, buf)
        assert out.dtype == dtype and torch.equal(out, t)


def test_shard_range_partitions_exactly():
    from custom_gymnasium_environments_b200.dist import shard_range

    for total, world in [(1 << 20, 8), (10, 3), (7, 8), (0, 2)]:
        spans = [shard_range(total, r, world) for r in range(world)]
        assert spans[0][0] == 0 and sum(c for _, c in spans) == total
        for (s0, c0), (s1, _) in zip(spans, spans[1:]):
            assert s0 + c0 == s1
    with pytest.raises(ValueError):
        shard_range(10, 2, 2)


_GLOO_WORKER = r"""
import os, sys, torch, torch.distributed as dist
sys.path.insert(0, sys.argv[1])
from custom_gymnasium_environments_b200.dist import all_reduce_episode_stats, init_process_group, shard_range, summarize
rank, local_rank, world = init_process_group("gloo")
start, count = shard_range(1000, rank, world)
stats = torch.tensor([count, -10 * count, 50 * count, rank + 1, 3 + rank], dtype=torch.int64)
red = all_reduce_episode_stats(stats)
assert red.tolist() == [1000, -10000, 50000, 3, 4], red.tolist()
assert stats.tolist()[0] == count  # input untouched
s = summarize(red)
assert s["episode_return_mean"] == -10.0 and s["score_max"] == 4
dist.barrier(); dist.destroy_process_group()
sys.stdout.write(f"rank {rank} ok {start} {count}\n"); sys.stdout.flush()
"""


def test_stats_all_reduce_gloo_world_size_2(tmp_path):
    script = tmp_path / "worker.py"
    script.write_text(_GLOO_WORKER)
    port = 29500 + (os.getpid() % 2000)
    cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node", "2", "--master-addr",
           "127.0.0.1", "--master-port", str(port), str(script), ROOT]
    env = dict(os.environ, CUDA_VISIBLE_DEVICES="", OMP_NUM_THREADS="1")
    res = subprocess.run(cmd, capture_output=True, text=True, timeout=240, env=env)
    assert res.returncode == 0, res.stdout + res.stderr
    assert "rank 0 ok 0 500" in res.stdout and "rank 1 ok 500 500" in res.stdout
