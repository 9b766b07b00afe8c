import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")
    config.addinivalue_line("markers", "needs_reference: needs a checkout of upstream SAMBLE named by SAMBLE_REFERENCE")


def pytest_collection_modifyitems(config, items):
    from tests.golden import ref_loader

    have_ref = ref_loader.available()
    skip_ref = pytest.mark.skip(reason="SAMBLE_REFERENCE does not name a checkout of upstream SAMBLE")
    for item in items:
        if "needs_reference" in item.keywords and not have_ref:
            item.add_marker(skip_ref)
