import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device")
    config.addinivalue_line(
        "markers", "needs_reference: imports the unmodified upstream environment from SY_REFERENCE_ROOT (oracle/ref_loader.py)"
    )


def pytest_collection_modifyitems(config, items):
    import ref_loader

    have_ref = ref_loader.reference_available()
    skip_ref = pytest.mark.skip(reason=f"unmodified upstream sources not found under {ref_loader.REFERENCE_ROOT} (SY_REFERENCE_ROOT)")
    for item in items:
        if "needs_reference" in item.keywords and not have_ref:
            item.add_marker(skip_ref)


@pytest.fixture(scope="session")
def golden_traces():
    import numpy as np

    return np.load(os.path.join(GOLDEN, "traces.npz"))
