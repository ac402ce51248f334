import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs a checkout of the original project at $SAA_REFERENCE_ROOT")


def pytest_collection_modifyitems(config, items):
    ref = os.environ.get("SAA_REFERENCE_ROOT", "")
    have_ref = bool(ref) and os.path.isfile(os.path.join(ref, "Tools", "Dynamic_solver.py"))
    skip_ref = pytest.mark.skip(reason="SAA_REFERENCE_ROOT does not name a checkout of the original project")
    for it in items:
        if "reference" in it.keywords and not have_ref:
            it.add_marker(skip_ref)
