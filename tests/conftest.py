import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        return np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False)
    return load


def pytest_sessionfinish(session, exitstatus):
    """Worst relative errors seen by the GPU parity tests (tests/parity.py) -> the JSON file A0_PARITY_RECORD names.
    Unset (the default), nothing is written: a test run leaves the tree as it found it."""
    path = os.environ.get("A0_PARITY_RECORD")
    if not path:
        return
    try:
        from tests import parity
        parity.dump(path)
    except Exception:
        pass
