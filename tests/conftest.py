import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "slow: takes more than a few seconds")


@pytest.fixture(scope="session")
def oracle():
    """The CPU oracle (C restatement of the reference path); test-side checker only."""
    import oracle_lib
    return oracle_lib.port()


@pytest.fixture(scope="session")
def gpu():
    """Bind the product library to cuda:0; fails (does not skip) when the CUDA path is unusable."""
    import clap_b200
    clap_b200.init(0)
    return clap_b200
