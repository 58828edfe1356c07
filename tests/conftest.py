import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
GOLDEN = os.path.join(ROOT, "tests", "golden")
DEFAULT_CONSTRUCT = "P2P-MS2v5-LacZ-PP7v4"


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def load_golden(stem):
    """tests/golden/<stem>.npz merged with its parts <stem>.1.npz, <stem>.2.npz, ... (a fixture is split to keep every
    file under 1 MB, tests/golden/make_golden.py); an array present in several parts is concatenated along its first
    axis, in part order."""
    out, path, k = {}, os.path.join(GOLDEN, stem + ".npz"), 1
    while True:
        with np.load(path) as z:
            for key in z.files:
                out[key] = np.concatenate([out[key], z[key]]) if key in out else z[key]
        path = os.path.join(GOLDEN, "%s.%d.npz" % (stem, k))
        if not os.path.exists(path):
            return out
        k += 1


@pytest.fixture(scope="session")
def cells_npz():
    return load_golden("cells")


@pytest.fixture(scope="session")
def results_npz():
    return load_golden("results")


@pytest.fixture(scope="session")
def chains_npz():
    return load_golden("chains")


@pytest.fixture(scope="session")
def orc():
    """The C oracle (test infrastructure)."""
    from oracle import c_oracle, forward_literal
    c_oracle.lib()
    return c_oracle, c_oracle.Construct.from_dict(forward_literal.CONSTRUCTS[DEFAULT_CONSTRUCT])


@pytest.fixture(scope="session")
def gpu_cells(cells_npz):
    """All 299 TestData cells resident on cuda:0 through the C ABI."""
    from transcriptioncycleinference_b200 import _lib
    from transcriptioncycleinference_b200.engine import Cells
    if _lib.device_count() < 1:
        pytest.skip("no CUDA device")
    c = Cells.from_packed(cells_npz["N"], cells_npz["off"], cells_npz["t"], cells_npz["ms2"], cells_npz["pp7"])
    yield c
    c.close()


def golden_theta(results, c):
    off = results["off"]
    s = slice(int(off[c]), int(off[c + 1]))
    return np.concatenate([[results["mean_v"][c], results["mean_tau"][c], results["mean_ton"][c],
                            results["mean_MS2_basal"][c], results["mean_PP7_basal"][c], results["mean_A"][c],
                            results["mean_R"][c]], results["mean_dR"][s]])


def random_theta(rng, N, wide=True):
    """theta drawn uniformly inside the bounds of TranscriptionCycleMCMC.m:242-254."""
    lo = np.concatenate([[0, 0, 0, 0, 0, 0, 0], -30 * np.ones(N)])
    hi = np.concatenate([[10, 20, 10, 50, 50, 1, 40], 30 * np.ones(N)])
    if not wide:   # the region chains actually visit
        lo[:7] = [0.5, 0, 0, 0, 0, 0, 5]; hi[:7] = [4, 6, 6, 3, 3, 1, 25]
        lo[7:] = -8; hi[7:] = 8
    return lo + (hi - lo) * rng.random(7 + N)
