import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
for p in (ROOT, os.path.join(ROOT, "oracle")):
    if p not in sys.path:
        sys.path.insert(0, p)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden_dir():
    return os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="session")
def ref_ops():
    """The reference's own compiled ops (oracle/_ref), or None where they were not built: the tests then compare with
    the reference's outputs stored in tests/golden and with the C oracle, and say so in a warning."""
    import warnings

    import build_ref
    try:
        return build_ref.load("roiaware_pool3d_cuda"), build_ref.load("iou3d_nms_cuda")
    except ImportError as e:
        warnings.warn("%s: the op tests compare with the reference's stored outputs and the C oracle only" % e)
        return None

