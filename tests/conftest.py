import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden", "reference_vectors.npz")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA sm_100 device (run on the B200 box)")
    config.addinivalue_line("filterwarnings", "ignore::UserWarning")
    config.addinivalue_line("filterwarnings", "ignore::DeprecationWarning")


def pytest_collection_modifyitems(config, items):
    try:
        import torch
        has_gpu = torch.cuda.is_available()
    except Exception:
        has_gpu = False
    if has_gpu:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    return dict(np.load(GOLDEN))


@pytest.fixture(scope="session")
def golden_traj():
    return dict(np.load(os.path.join(os.path.dirname(GOLDEN), "trajectory_vectors.npz")))


@pytest.fixture(scope="session")
def lib_built():
    """Build (incrementally) and return the path of libcfm_b200.so."""
    from cfm_b200 import build
    return build.build()
