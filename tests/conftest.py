import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture(scope="session")
def oracle():
    from oracle.pyoracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def emul():
    from tests.helpers import HostEmul
    return HostEmul()


def golden(name):
    return np.load(os.path.join(GOLDEN, name + ".npz"))


@pytest.fixture(scope="session")
def gpu_lib():
    """The CUDA library with a visible device; GPU tests fail loudly when either is missing."""
    import bvh_b200.api as api
    api.lib()
    assert api.device_count() > 0, "no CUDA device visible: GPU tests must run on the B200 box"
    return api
