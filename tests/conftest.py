import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def pytest_collection_modifyitems(config, items):
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def golden_layers():
    """The layer cases of every layers_<kind>_<variant>.npz, as one mapping."""
    import glob
    import numpy as np
    parts = sorted(glob.glob(os.path.join(GOLDEN, "layers_*.npz")))
    assert parts, "tests/golden/layers_*.npz missing"
    out = {}
    for p in parts:
        with np.load(p) as z:
            out.update({k: z[k] for k in z.files})
    return out


@pytest.fixture(scope="session")
def golden_models():
    import numpy as np
    return np.load(os.path.join(GOLDEN, "models.npz"))
