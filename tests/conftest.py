import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")

from oracle import golden  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_crops():
    return golden.load(os.path.join(GOLDEN, "crops.npz"))


@pytest.fixture(scope="session")
def golden_model():
    return golden.load(os.path.join(GOLDEN, "model.npz"))


@pytest.fixture(scope="session")
def golden_track():
    return golden.load(os.path.join(GOLDEN, "track.npz"))


def state_dict_from_npz(npz, prefix="w::"):
    import torch
    return {k[len(prefix):]: torch.from_numpy(np.array(npz[k])) for k in npz if k.startswith(prefix)}
