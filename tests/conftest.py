import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

GOLDEN = os.path.join(ROOT, "tests", "golden")
# data files of the upstream project (Vanlightly/vsr-tlaplus), stored unchanged: the shipped model configuration and the
# published 24-state counterexample
REF_CFG = os.path.join(GOLDEN, "VSR.cfg")
REF_TRACE = os.path.join(GOLDEN, "state_transfer_violation_trace.txt")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def pkg():
    """The product package; builds the native library if it is missing."""
    import _pkg
    so = os.path.join(ROOT, "vsr-tlaplus_b200", "libvsr_b200.so")
    if not os.path.exists(so) or not os.path.exists(os.path.join(ROOT, "oracle", "_build", "liboracle.so")):
        import __graft_entry__
        __graft_entry__.build()
    return _pkg.load()
