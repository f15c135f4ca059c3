import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

# The checkout of the reference msamtools v1.1.3 sources (not part of this repository), or None: the tests that run the
# reference's shell suites need it and skip without it.
from oracle import oracle as _orc  # noqa: E402

REFERENCE = _orc.reference_dir()
REF_TESTS = os.path.join(REFERENCE, "tests") if REFERENCE else ""
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200")


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as orc
    orc.build()
    orc.load()
    return orc


needs_reference = pytest.mark.skipif(not os.path.isdir(REF_TESTS), reason="the reference's sources are absent (MSAMTOOLS_REFERENCE, BASELINE.json reference_path)")
