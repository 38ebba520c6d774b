import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")
WEIGHTS = os.path.join(GOLDEN, "weights")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a B200 (run by the driver with -m gpu)")


@pytest.fixture(scope="session")
def built_lib():
    """Build (if stale) and return the path of librf_b200.so -- nvcc cross-compiles without a GPU."""
    from retinaface_b200.build import build_library
    return build_library()


@pytest.fixture(scope="session")
def golden_image():
    import cv2
    img = cv2.imread(os.path.join(GOLDEN, "data", "img.jpg"))
    assert img is not None and img.shape == (886, 1280, 3)
    return img


def caffemodel(name: str) -> str:
    return os.path.join(WEIGHTS, name + ".caffemodel")
