import os
import sys
import zlib

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
PART_BYTES = 900_000            # a golden record larger than this (compressed) is stored as <stem>.npz + <stem>.1.npz + ...


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class GoldenRecord(dict):
    """The arrays of one golden record; `files` lists their names, as on the `np.load` result."""

    @property
    def files(self):
        return list(self)


def _parts(stem):
    paths, k = [stem + ".npz"], 1
    while os.path.isfile(f"{stem}.{k}.npz"):
        paths.append(f"{stem}.{k}.npz")
        k += 1
    return paths


def load_golden(name, root=None):
    """Golden record `name` (e.g. "mmgcn_tiny.npz") of `root` (default tests/golden), joined from its part files."""
    rec = GoldenRecord()
    for path in _parts(os.path.join(root or GOLDEN, name[:-len(".npz")])):
        with np.load(path, allow_pickle=True) as z:
            rec.update((k, z[k]) for k in z.files)
    return rec


def save_golden(path, arrays):
    """Write `arrays` as the record `path` (a .npz path), in as many part files as keep each under PART_BYTES."""
    stem, parts, size = path[:-len(".npz")], [{}], 0
    for k, v in arrays.items():
        n = len(zlib.compress(np.asarray(v).tobytes()))
        if parts[-1] and size + n > PART_BYTES:
            parts.append({})
            size = 0
        parts[-1][k], size = v, size + n
    for old in _parts(stem)[len(parts):]:
        if os.path.isfile(old):
            os.remove(old)
    for i, part in enumerate(parts):
        np.savez_compressed(stem + (f".{i}" if i else "") + ".npz", **part)


@pytest.fixture(scope="session")
def golden():
    cache = {}

    def get(name):
        if name not in cache:
            cache[name] = load_golden(name)
        return cache[name]
    return get
