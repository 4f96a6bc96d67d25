import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import ffi
    ffi.build()
    return ffi.Oracle()


@pytest.fixture(scope="session")
def model0():
    from percepnet_b200.weights import synth_model
    return synth_model(0)


@pytest.fixture(scope="session")
def model_hot():
    from percepnet_b200.weights import synth_model
    return synth_model(7, gain=3.0)
