import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `-m gpu`)")


def pytest_collection_modifyitems(config, items):
    """`gpu`-marked tests are skipped (not failed) on a box without CUDA."""
    try:
        import torch
        has_cuda = torch.cuda.is_available()
    except Exception:
        has_cuda = False
    if has_cuda:
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for item in items:
        if "gpu" in item.keywords:
            item.add_marker(skip)


GOLDEN_MAX_FILE_BYTES = 1_000_000
GOLDEN_LN_RHO_SAMPLE = 512


def load_golden(name):
    import numpy as np
    return np.load(os.path.join(GOLDEN_DIR, name + ".npz"), allow_pickle=False)


def save_golden(name, payload):
    """Writes tests/golden/<name>.npz.  A fixture that would exceed GOLDEN_MAX_FILE_BYTES keeps final_ln_rho for a fixed,
    seeded sample of GOLDEN_LN_RHO_SAMPLE rows, their indices in final_ln_rho_rows; every other array is stored whole."""
    import numpy as np
    path = os.path.join(GOLDEN_DIR, name + ".npz")
    np.savez_compressed(path, **payload)
    if os.path.getsize(path) > GOLDEN_MAX_FILE_BYTES:
        n = payload["final_ln_rho"].shape[0]
        rows = np.sort(np.random.default_rng(0).choice(n, size=min(n, GOLDEN_LN_RHO_SAMPLE), replace=False))
        payload = dict(payload, final_ln_rho=payload["final_ln_rho"][rows], final_ln_rho_rows=rows)
        np.savez_compressed(path, **payload)
    return path


def ln_rho_rows(g):
    """The rows of the fit that a fixture's final_ln_rho holds: all of them, unless save_golden sampled them."""
    return g["final_ln_rho_rows"] if "final_ln_rho_rows" in g.files else slice(None)


@pytest.fixture(scope="session")
def lib_built():
    """Build libbgmm.so if needed (nvcc cross-compiles without a GPU)."""
    from bayesml_b200 import build
    return build.build()
