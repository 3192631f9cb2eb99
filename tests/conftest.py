import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _npz_groups(path):
    z = np.load(path)
    groups = {}
    for key in z.files:
        if "/" in key:
            g, f = key.split("/", 1)
            groups.setdefault(g, {})[f] = z[key]
        else:
            groups[key] = z[key]
    return groups


@pytest.fixture(scope="session")
def knn_golden():
    return _npz_groups(os.path.join(GOLDEN, "knn_cases.npz"))


@pytest.fixture(scope="session")
def gather_golden():
    return _npz_groups(os.path.join(GOLDEN, "gather_cases.npz"))


@pytest.fixture(scope="session")
def grid_golden():
    return _npz_groups(os.path.join(GOLDEN, "grid_cases.npz"))


@pytest.fixture(scope="session")
def oracle_ref_golden():
    return _npz_groups(os.path.join(GOLDEN, "oracle_ref_cases.npz"))


def sha256_of(a):
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def reference_knn(golden, name, oracle_idx):
    """The reference's KNN result ``name`` of oracle_ref_cases.npz, rebuilt from the oracle's result on the same
    inputs (the stored rows replaced) and checked against the sha256 of the reference's whole array."""
    case = golden[name]
    want = np.array(oracle_idx, dtype=np.int64)
    rows = case["rows"]
    want[rows[:, 0], rows[:, 1]] = case["vals"]
    assert sha256_of(want) == str(case["sha256"]), \
        "%s: the oracle's result differs from the reference's outside the stored rows" % name
    return want


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("gpu-marked test ran without a CUDA device")
    return torch.device("cuda:0")


def frame_point_sets(frame, n_points):
    from ffb6d_b200.synthetic import image_pyramid_np
    sets = {("cld", i): frame["cld"][: n_points // 4 ** i] for i in range(5)}
    for sr, p in image_pyramid_np(frame["dpt_xyz"]).items():
        sets[("img", sr)] = p
    return sets
