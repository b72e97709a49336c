import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: test needs a CUDA device (B200, sm_100a)")


def _has_gpu():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    path = os.path.join(ROOT, "tests", "golden", "golden.npz")
    return np.load(path)


@pytest.fixture(scope="session")
def ref_outputs():
    """What the unmodified reference CPU library answered for the inputs of the tests that compare with it
    (tests/golden/make_reference_outputs.py)."""
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_outputs.npz"))


@pytest.fixture(scope="session")
def ref_outputs_fullsize():
    """The same for the BASELINE-size configs of tests/test_fullsize_gpu.py (64 sampled queries each)."""
    return np.load(os.path.join(ROOT, "tests", "golden", "reference_outputs_fullsize.npz"))


@pytest.fixture(scope="session")
def res():
    import faiss_b200 as fb

    return fb.StandardGpuResources()
