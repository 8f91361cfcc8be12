import glob
import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(REPO, "ipdm-pytorch_b200")
GOLDEN = os.path.join(REPO, "tests", "golden")
for p in (REPO, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


def golden(name):
    """Arrays of tests/golden/<name>.npz merged with those of its parts <name>.1.npz, <name>.2.npz, ... (oracle/make_golden.py
    splits a case over several files to keep each file under 1 MB)."""
    paths = [os.path.join(GOLDEN, name + ".npz")] + sorted(glob.glob(os.path.join(GOLDEN, glob.escape(name) + ".[0-9]*.npz")))
    arrays = {}
    for path in paths:
        with np.load(path) as z:
            assert not set(z.files) & set(arrays), path
            arrays.update((k, z[k]) for k in z.files)
    return arrays


def rel_l2(a, b):
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.linalg.norm(a - b) / max(np.linalg.norm(b), 1e-30))


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda:0")
