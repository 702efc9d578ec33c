"""Shared fixtures.  `-m "not gpu"` runs here on CPU; `-m gpu` needs a B200 (driver runs it at round end)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


@pytest.fixture(scope="session")
def built():
    """Build everything once (oracle + CUDA library); cheap when already built."""
    import __graft_entry__ as g
    g.build()
    return True


@pytest.fixture(scope="session")
def oracle(built):
    from oracle.oracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def reference_vectors():
    """Outputs of the unmodified reference kernels on the seeded inputs of test_oracle_golden.py."""
    return dict(np.load(os.path.join(GOLDEN, "reference_vectors.npz")))


@pytest.fixture(scope="session")
def golden():
    return dict(np.load(os.path.join(GOLDEN, "golden.npz")))


@pytest.fixture(scope="session")
def digits():
    d = np.load(os.path.join(GOLDEN, "digits.npz"))
    return d["images"], d["labels"]


def model_names():
    return sorted(f[:-4] for f in os.listdir(os.path.join(GOLDEN, "models")) if f.endswith(".bnm"))


def load_model(name):
    from bitnetmcu_b200.model import Model
    return Model.load(os.path.join(GOLDEN, "models", name + ".bnm"))


def xorshift_images(n, img_bytes=256, seed=12345):
    """numpy restatement of the SURVEY.md 8c stream (low byte of xorshift32, one draw per pixel)."""
    out = np.empty(n * img_bytes, dtype=np.uint8)
    s = seed & 0xFFFFFFFF
    for i in range(out.size):
        s ^= (s << 13) & 0xFFFFFFFF
        s ^= s >> 17
        s ^= (s << 5) & 0xFFFFFFFF
        out[i] = s & 0xFF
    return out.view(np.int8).reshape(n, img_bytes)
