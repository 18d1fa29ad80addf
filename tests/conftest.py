import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (B200, sm_100a)")
    config.addinivalue_line("markers", "reference: needs a checkout of the reference (oracle/ref_import.py)")


def pytest_collection_modifyitems(config, items):
    import torch
    has_gpu = torch.cuda.is_available()
    from oracle import ref_import
    has_ref = ref_import.available()
    for item in items:
        if "gpu" in item.keywords and not has_gpu:
            item.add_marker(pytest.mark.skip(reason="no CUDA device"))
        if "reference" in item.keywords and not has_ref:
            item.add_marker(pytest.mark.skip(reason=f"no checkout of the reference at {ref_import.REFERENCE_ROOT}"))


@pytest.fixture(scope="session")
def golden():
    import torch

    def load(name):
        return torch.load(os.path.join(GOLDEN, name), map_location="cpu", weights_only=False)
    return load
