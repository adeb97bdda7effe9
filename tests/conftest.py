import os
import sys

import pytest

ROOT = os.path.abspath(os.path.join(os.path.dirname(__file__), ".."))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    """Committed fixtures converted from the reference's data artefacts
    (tests/golden/make_golden.py)."""
    import cases
    return cases.fixtures()


@pytest.fixture(scope="session")
def golden_meta():
    import json
    with open(os.path.join(ROOT, "tests", "golden", "fixtures.json")) as f:
        return json.load(f)
