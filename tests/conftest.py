import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run with -m gpu on the B200 box)")


@pytest.fixture(scope="session")
def port():
    import oracle
    return oracle.Port()


@pytest.fixture(scope="session")
def ref():
    """The reference engine's recorded results on the case sets of tests/inputs.py."""
    from tests import inputs
    return inputs.RefResults()


@pytest.fixture(scope="session")
def native():
    from k4os.compression.lz4_b200 import build, _native
    build.build()
    return _native.lib()


def has_gpu() -> bool:
    try:
        from k4os.compression.lz4_b200 import _native
        return _native.lib().k4lz4_device_count() > 0
    except Exception:
        return False
