import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


@pytest.fixture(scope="session")
def orc():
    from oracle import orc as _orc
    _orc.build()
    return _orc


@pytest.fixture(scope="session")
def ctx():
    import powdr_b200
    c = powdr_b200.Context(0)
    c.set_fri_params(8, 4)          # small FRI parameters for the parity tests (oracle wrappers default to the same)
    yield c
    c.close()
