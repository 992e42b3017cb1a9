import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device")


@pytest.fixture(scope="session")
def oracle():
    from oracle import pyoracle
    return pyoracle.Oracle()


@pytest.fixture(scope="session")
def ref_cpu():
    from tests import refgolden
    return refgolden.Reference("cpu")


@pytest.fixture(scope="session")
def ref_avx2():
    from tests import refgolden
    return refgolden.Reference("avx2")
