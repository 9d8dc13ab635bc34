import os
import sys
import warnings

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
warnings.filterwarnings("ignore", category=DeprecationWarning)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    gdir = os.path.join(ROOT, "tests", "golden")
    if gdir not in sys.path:
        sys.path.insert(0, gdir)
    import make_golden
    return make_golden.load()
