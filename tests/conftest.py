import glob
import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if REPO not in sys.path:
    sys.path.insert(0, REPO)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _has_cuda():
    try:
        import torch

        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_cuda():
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


class Golden:
    """tests/golden/finc_golden_<part>.npz: outputs of the reference's own code
    (tests/golden/make_golden.py), whole cases split over files of under 1 MB."""

    def __init__(self):
        self.data, self.names = {}, []
        for path in sorted(glob.glob(os.path.join(REPO, "tests", "golden", "finc_golden_*.npz"))):
            with np.load(path) as part:
                self.names += [str(n) for n in part["__index__"]]
                self.data.update({k: part[k] for k in part.files if k != "__index__"})
        assert self.names, "tests/golden/finc_golden_*.npz missing"

    def case(self, name):
        pre = name + "/"
        return {k[len(pre):]: v for k, v in self.data.items() if k.startswith(pre)}


@pytest.fixture(scope="session")
def golden():
    return Golden()


def rel_err(a, b):
    """max-norm relative error: max|a-b| / max(max|b|, tiny)."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))


def elementwise_close(a, b, rtol=1e-5, floor=1e-1):
    """element-wise relative check with an absolute floor: |a - b| <= rtol * (|b| + floor * max|b|).
    Used NEXT to rel_err (max-norm): two fp32 evaluations in different orders differ by a few 1e-7 absolute
    on elements that cancel to ~0 whatever their size, hence the floor of rtol * floor * max|b| = 1e-6 max|b|."""
    a = np.asarray(a, dtype=np.float64)
    b = np.asarray(b, dtype=np.float64)
    return bool((np.abs(a - b) <= rtol * (np.abs(b) + floor * np.abs(b).max())).all())
