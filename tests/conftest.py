import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


class SmallGolden:
    """tests/golden/small_cases.npz -- outputs of the unmodified reference function."""

    def __init__(self):
        self.z = np.load(os.path.join(GOLDEN_DIR, "small_cases.npz"))
        self.names = json.loads(str(self.z["__names__"]))
        self.versions = json.loads(str(self.z["__versions__"]))

    def case(self, name):
        kw = json.loads(str(self.z[f"{name}/kwargs"]))
        return (self.z[f"{name}/image"], self.z[f"{name}/depth"], kw,
                self.z[f"{name}/points"], self.z[f"{name}/colors"])


@pytest.fixture(scope="session")
def small_golden():
    return SmallGolden()


@pytest.fixture(scope="session")
def large_golden():
    with open(os.path.join(GOLDEN_DIR, "large_cases.json")) as f:
        return json.load(f)


def canon(a):
    """Bit pattern with the sign of zero and the NaN payload canonicalised.

    NumPy's selection leaves the order of -0.0/+0.0 ties unspecified, so the sign of a zero
    percentile (and of z == 0 outputs derived from it) is not pinned by the reference."""
    a = np.ascontiguousarray(a, dtype=np.float32) + np.float32(0.0)
    a = np.where(np.isnan(a), np.float32(np.nan), a)
    return np.ascontiguousarray(a).view(np.uint32)


def assert_bits_equal(got, want, what=""):
    assert got.shape == want.shape, f"{what}: shape {got.shape} != {want.shape}"
    g, w = canon(got), canon(want)
    bad = int((g != w).sum())
    assert bad == 0, f"{what}: {bad} of {g.size} float32 words differ"
