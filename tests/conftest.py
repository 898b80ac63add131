import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_sessionstart(session):
    """The in-tree libbeng.so normally travels with the repo snapshot.  If it is absent (a fresh checkout) compile it
    once -- the same nvcc command as __graft_entry__.build() -- and recompile it when a source changed since it was built
    (content hash, _build.is_stale), so that the tests exercise the CUDA library the tree describes instead of failing at
    import or silently testing an old binary; compiling is not a fallback, the product still refuses to run without the library."""
    from custom_gymnasium_environments_b200 import _build, _lib

    if "BENG_LIB_PATH" not in os.environ and _build.is_stale():  # missing, or built from other sources than the tree's
        _build.build_library(force=True)


@pytest.fixture(scope="session")
def golden():
    from oracle import golden_files

    return golden_files.load("snake")


@pytest.fixture(scope="session")
def golden_cases(golden):
    return [str(c) for c in golden["cases"]]


def case_meta(golden, name):
    G, n_envs, n_steps, seed, base, snap_every = (int(x) for x in golden[f"{name}/meta"])
    return dict(G=G, n_envs=n_envs, n_steps=n_steps, seed=seed, base=base, snap_every=snap_every)
