import os
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests", "support")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def gold():
    from golden_file import GoldenFile
    return GoldenFile(os.path.join(ROOT, "tests", "golden", "reference_golden.npz"))


@pytest.fixture(scope="session")
def track():
    from oracle.track import TrackTable
    return TrackTable(0.4)
