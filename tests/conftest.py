import importlib
import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200); run with -m gpu")


@pytest.fixture(scope="session")
def pcpx():
    """The ctypes binding over libpcpx.so (the product's C ABI)."""
    return importlib.import_module("point-cloud-processing_b200")


@pytest.fixture(scope="session")
def oracle():
    from oracle_lib import Oracle

    return Oracle()


@pytest.fixture(scope="session")
def ref():
    """The reference's own headers behind a C bridge; None when oracle/_ref was not built
    (it can only be built with PCP_REFERENCE naming a checkout of the reference)."""
    from oracle_lib import RefBridge, build_oracle, have_ref

    build_oracle()
    return RefBridge() if have_ref() else None


@pytest.fixture(scope="session")
def emu():
    from emu_lib import Emu

    return Emu()
