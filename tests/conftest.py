import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    import torch

    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    # the reference's 16 minibatch gradients are stored in a file of their own (each file stays under 1 MB)
    g = dict(np.load(os.path.join(ROOT, "tests", "golden", "ref_ppo_seed1.npz")))
    g.update(np.load(os.path.join(ROOT, "tests", "golden", "ref_ppo_seed1_grads.npz")))
    return g
