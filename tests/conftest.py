import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "ref: needs the reference binaries of oracle/_ref (built only from the reference sources)")


def pytest_collection_modifyitems(config, items):
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_sinkfeed"))
    for it in items:
        if "ref" in it.keywords and not have_ref:
            it.add_marker(pytest.mark.skip(reason="oracle/_ref/ref_sinkfeed not built (needs the reference sources)"))
