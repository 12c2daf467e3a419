import os
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")
# Intra-op threads of the process that wrote the golden vectors (oracle/gen_golden.py).  MKL splits a GEMM by thread
# count, so the CPU oracle reproduces the reference's outputs bit for bit only with the same count.
GOLDEN_INTRA_OP_THREADS = 8


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_sessionstart(session):
    """Keep libbmv.so in step with the sources (nvcc cross-compiles without a GPU); a stale or
    missing library must never be what the GPU tests exercise."""
    import shutil
    from boostmvsnerfs_b200 import build as _build
    if os.path.exists(_build.NVCC) or shutil.which("nvcc"):
        _build.build()


def pytest_collection_modifyitems(config, items):
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class Golden:
    """npz fixture written by oracle/gen_golden.py (reference inputs/outputs)."""

    def __init__(self, name):
        self._z = np.load(os.path.join(GOLDEN_DIR, name))

    def __contains__(self, key):
        return key in self._z.files

    def keys(self):
        return list(self._z.files)

    def np(self, key):
        return self._z[key]

    def t(self, key, device="cpu"):
        return torch.from_numpy(self._z[key]).to(device)


_cache = {}


def load_golden(name):
    if name not in _cache:
        _cache[name] = Golden(name)
    return _cache[name]


@pytest.fixture(scope="session")
def ops_golden():
    return load_golden("enerf_ops.npz")


@pytest.fixture
def golden_threads():
    """Runs a test with the intra-op thread count the golden vectors were written with."""
    old = torch.get_num_threads()
    torch.set_num_threads(GOLDEN_INTRA_OP_THREADS)
    yield
    torch.set_num_threads(old)
