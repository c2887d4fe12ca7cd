import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def pytest_collection_modifyitems(config, items):
    """`gpu`-marked tests are skipped (not errored) on a machine without a CUDA device."""
    import torch
    if torch.cuda.is_available():
        return
    skip = pytest.mark.skip(reason="needs a CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


def rel_err(a, b):
    """max|a-b| relative to max(|b|, spread(b)) -- SURVEY.md section 8d parity definition."""
    import numpy as np
    a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
    denom = max(float(np.abs(b).max()), float(b.std()), 1e-30)
    return float(np.abs(a - b).max()) / denom
