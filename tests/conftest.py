import glob
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    # -m gpu tests must not silently pass on a box without a GPU
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


def golden_files(prefix):
    return sorted(glob.glob(os.path.join(GOLDEN, prefix + "*.npz")))


def load_npz(path):
    with np.load(path) as z:
        return {k: z[k] for k in z.files}


@pytest.fixture(scope="session")
def tcl():
    import tcl_b200
    tcl_b200._cabi.build()
    return tcl_b200


@pytest.fixture(scope="session")
def oracle_mod():
    import oracle
    oracle.build()
    return oracle
