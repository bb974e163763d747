import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def oracle():
    from oracle import cpu_oracle
    cpu_oracle.build()
    return cpu_oracle


@pytest.fixture(scope="session")
def reference(golden_dir):
    """The reference kernels' bit-exact outputs on the parity tests' inputs (tests/golden/reference_outputs.npz, see
    _util.ReferenceOutputs).  RI_RECORD_REFERENCE=<file.npz> records them from the reference backend (oracle/_ref)."""
    from _util import ReferenceOutputs
    rec = ReferenceOutputs(os.path.join(golden_dir, "reference_outputs.npz"), os.environ.get("RI_RECORD_REFERENCE"))
    yield rec
    rec.save()
