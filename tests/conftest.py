import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def golden():
    """golden(name) -> {array name: array} of tests/golden/<name>.npz, or of its parts <name>.0.npz,
    <name>.1.npz, ... merged in order (tests/golden/make_golden.py splits a fixture above 1 MB)."""
    def load(name):
        path = os.path.join(GOLDEN, name + ".npz")
        if os.path.exists(path):
            return dict(np.load(path))
        out, i = {}, 0
        while os.path.exists(os.path.join(GOLDEN, "%s.%d.npz" % (name, i))):
            out.update(np.load(os.path.join(GOLDEN, "%s.%d.npz" % (name, i))))
            i += 1
        if not out:
            raise FileNotFoundError("no golden fixture %s in %s" % (name, GOLDEN))
        return out
    return load
