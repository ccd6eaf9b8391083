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


def load_golden(name):
    gv = dict(np.load(os.path.join(GOLDEN, name + ".npz")))
    if "inputs_sha256" in gv:
        from helpers import redraw_inputs
        gv.update(redraw_inputs(gv))
    return gv


@pytest.fixture(scope="session")
def golden():
    return load_golden
