import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: compares with the reference's own outputs (run live when its "
                                       "sources are available, else as stored under tests/golden)")


@pytest.fixture(scope="session")
def kat():
    with open(os.path.join(GOLDEN, "reference_kat.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def kat_arrays():
    return dict(np.load(os.path.join(GOLDEN, "reference_kat.npz")))


@pytest.fixture(scope="session")
def e2e_golden():
    with open(os.path.join(GOLDEN, "reference_e2e.json")) as f:
        doc = json.load(f)
    return doc, dict(np.load(os.path.join(GOLDEN, "reference_e2e.npz")))
