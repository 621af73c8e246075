import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "omnirevolve-image-processor_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

# image_processor/ directory of a checkout of the original project; it is not part of this repository, so the tests that
# import it live are opt-in.  Everything else compares with outputs of it frozen under tests/golden/.
REFERENCE_DIR = os.environ.get("OMNI_REFERENCE_DIR", "")
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: imports the original project from OMNI_REFERENCE_DIR (skipped when it is unset)")


def pytest_collection_modifyitems(config, items):
    have_ref = bool(REFERENCE_DIR) and os.path.isdir(REFERENCE_DIR)
    for it in items:
        if "reference" in it.keywords and not have_ref:
            it.add_marker(pytest.mark.skip(reason="OMNI_REFERENCE_DIR does not name the original project's image_processor/"))


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN
