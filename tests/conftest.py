import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "reference: needs the original Ofighters source tree (OFB_REFERENCE_ROOT)")


def pytest_collection_modifyitems(config, items):
    from oracle import ref_shim
    if not ref_shim.available():
        skip = pytest.mark.skip(reason="OFB_REFERENCE_ROOT does not name the original Ofighters source tree")
        for it in items:
            if "reference" in it.keywords:
                it.add_marker(skip)
