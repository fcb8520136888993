import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box via gpurun)")
    config.addinivalue_line("markers", "reference: needs a checkout of the original NeuralOC project, named by NOC_REFERENCE")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
