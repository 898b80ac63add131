"""The golden vectors under tests/golden/: what the reference returned for seeded action tapes, written by the
gen_golden*.py scripts and read by the parity tests.

One env's vectors may span several files, <env>_golden.npz, <env>_golden_1.npz, <env>_golden_2.npz, ..., so that no
file passes MAX_FILE_BYTES; `load` merges them back into one mapping of key -> array.
"""
from __future__ import annotations

import glob
import io
import os

import numpy as np

DIR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")
MAX_FILE_BYTES = 1_000_000


def paths(env: str) -> list:
    """-> the files of `env`'s vectors, the first one first."""
    rest = glob.glob(os.path.join(DIR, f"{env}_golden_[0-9]*.npz"))
    return [os.path.join(DIR, f"{env}_golden.npz")] + sorted(rest, key=lambda p: int(p[:-4].rsplit("_", 1)[1]))


def load(env: str) -> dict:
    """-> {key: array} over every file of `env`'s vectors."""
    out = {}
    for path in paths(env):
        with np.load(path) as f:
            out.update((k, f[k]) for k in f.files)
    return out


def _packed_bytes(arrays: dict) -> int:
    buf = io.BytesIO()
    np.savez_compressed(buf, **arrays)
    return buf.getbuffer().nbytes


def save(env: str, blob: dict) -> list:
    """Write `blob` (key -> array, kept in order) as `env`'s vectors, starting a new file whenever the current one would
    pass MAX_FILE_BYTES.  Zip members are compressed one by one, so a file's size is at most the sum of the sizes of its
    arrays saved alone.  -> the paths written."""
    parts, cur, cur_bytes = [], {}, 0
    for k, v in blob.items():
        nbytes = _packed_bytes({k: v})
        if cur and cur_bytes + nbytes > MAX_FILE_BYTES:
            parts.append(cur)
            cur, cur_bytes = {}, 0
        cur[k], cur_bytes = v, cur_bytes + nbytes
    parts.append(cur)
    for old in paths(env)[1:]:
        os.remove(old)
    out = [os.path.join(DIR, f"{env}_golden.npz" if i == 0 else f"{env}_golden_{i}.npz") for i in range(len(parts))]
    for path, arrays in zip(out, parts):
        np.savez_compressed(path, **arrays)
        if os.path.getsize(path) > MAX_FILE_BYTES:
            raise ValueError(f"{path}: one array alone passes {MAX_FILE_BYTES} bytes; store a smaller case")
    return out
