import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: runs the reference package that build() stages under oracle/_ref")


def pytest_collection_modifyitems(config, items):
    from oracle import stage_reference
    have_ref = stage_reference.staged()
    skip_ref = pytest.mark.skip(reason="the reference package is not staged under oracle/_ref")
    for item in items:
        if "reference" in item.keywords and not have_ref:
            item.add_marker(skip_ref)
