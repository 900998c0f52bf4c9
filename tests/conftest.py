import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle"), os.path.join(ROOT, "tests"), os.path.join(ROOT, "tests", "emul")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    def load(name):
        return np.load(os.path.join(GOLDEN, name))
    return load
