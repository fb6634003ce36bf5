import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (select with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        return np.load(os.path.join(GOLDEN, name + ".npz"))
    return load
