import os
import shutil
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

from detectmateservice_b200.compat import ipc_tempdir  # noqa: E402

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture
def sock_dir():
    """Directory for the ipc:// sockets of one test (tmp_path can be too deep for an AF_UNIX address)."""
    d = ipc_tempdir()
    yield d
    shutil.rmtree(d, ignore_errors=True)
