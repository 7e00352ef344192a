import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def orc():
    """The CPU oracle (plain-C restatement); built on demand with gcc."""
    from oracle import oracle as O
    return O.OracleLib()


@pytest.fixture(scope="session")
def ict():
    import invcompcamtrack_b200 as ict
    ict.lib()
    return ict
