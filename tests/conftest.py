import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "sub-cortical_segmentation_b200")
for p in (ROOT, PKG):
    if p not in sys.path:
        sys.path.insert(0, p)

GOLDEN = os.path.join(ROOT, "tests", "golden")
WEIGHTS = os.path.join(ROOT, "nets", "miccai2012_v1", "miccai2012_v1.pkl")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def gather_golden():
    """gather_golden.npz with the patch arrays of generate_training_set's output rebuilt: the unshuffled ones are the
    B_x_* patches, the shuffled ones those rows in the order T_shuf_perm (tests/golden/make_golden.py)"""
    G = dict(np.load(os.path.join(GOLDEN, "gather_golden.npz")))
    for k, mode in (("xa", "axial"), ("xc", "coronal"), ("xs", "saggital")):
        G["T_plain_" + k] = G["B_x_" + mode][:, None]
        G["T_shuf_" + k] = G["T_plain_" + k][G["T_shuf_perm"]]
    return G


@pytest.fixture(scope="session")
def weights_path():
    return WEIGHTS


@pytest.fixture(scope="session")
def oracle_params():
    from oracle import network
    return network.load_params(WEIGHTS)
