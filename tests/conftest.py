import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle_py
    oracle_py.lib()
    return oracle_py


@pytest.fixture(scope="session")
def kflib():
    from roskfpos_b200 import lib
    lib.lib()
    return lib


def pytest_sessionfinish(session, exitstatus):
    """KFPOS_PARITY_REPORT=<file>: leave the observed parity numbers (stable fraction, tie count, worst error
    per test) there.  Unset, the suite writes nothing."""
    out = os.environ.get("KFPOS_PARITY_REPORT")
    if out:
        from tests import util
        util.write_parity_report(out)
