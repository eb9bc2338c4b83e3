import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
sys.path.insert(0, GOLDEN)
from golden_params import unpack_parameters  # noqa: E402


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def load_golden(name):
    g = dict(np.load(os.path.join(GOLDEN, name), allow_pickle=False))
    if "init_seed" in g:            # network parameters stored compactly (golden_params.py); restoring them needs torch
        unpack_parameters(g)
    return g


@pytest.fixture(scope="session")
def golden():
    return load_golden


def quad_state(g, tag):
    return {k: g[f"{k}_{tag}"] for k in ("x", "v", "R", "Om", "t", "t_last", "Rd_last", "obs", "step")}
