import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
MODEL_FILE = os.path.join(ROOT, "chunkflow_b200", "convnet", "unet3l.py")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")
    config.addinivalue_line("markers", "slow: minutes of CPU oracle time (still part of `-m gpu`)")


@pytest.fixture(scope="session")
def geometry():
    with open(os.path.join(GOLDEN, "geometry.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def golden():
    def load(name):
        with np.load(os.path.join(GOLDEN, name)) as z:
            return {k: z[k] for k in z.files}
    return load


@pytest.fixture(scope="session")
def pins():
    """What the original chunkflow computed on the pinning tests' inputs (tests/reference_pins.py)."""
    from reference_pins import Pins
    return Pins()


@pytest.fixture(scope="session")
def unet_model():
    from chunkflow_b200.lib import load_source
    return load_source(MODEL_FILE).load_model(None)


def has_gpu() -> bool:
    from chunkflow_b200 import _native
    try:
        return _native.load().cfb_device_count() > 0
    except Exception:
        return False
