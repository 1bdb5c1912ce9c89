import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "slow: long CPU test, excluded from the default CPU suite")


def pytest_collection_modifyitems(config, items):
    """`slow` tests run only with ZOPFLI_B200_SLOW=1 (they are reproductions of claims in DESIGN.md, not gates)"""
    if os.environ.get("ZOPFLI_B200_SLOW"):
        return
    skip = pytest.mark.skip(reason="slow: set ZOPFLI_B200_SLOW=1")
    for it in items:
        if "slow" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def ref():
    """the reference's answers (tests/golden/reference_answers.json; the live library while recording)"""
    import zref
    return zref.reference()


@pytest.fixture(scope="session")
def oracle():
    import zref
    return zref.Oracle()
