import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
# A checkout of the original yolo-from-scratch (train.py, eval.py, tests/), which is not part of this repository.
# Tests that need it skip without one; __graft_entry__.build() stages a copy into baseline/_ref when it finds one.
REFERENCE_DIR = os.environ.get("YOLO_FROM_SCRATCH_REFERENCE") or os.path.join(ROOT, "baseline", "_ref")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    from oracle.golden_store import expand

    def load(name):
        with np.load(os.path.join(GOLDEN, name + ".npz"), allow_pickle=False) as z:
            return expand(z)
    return load

