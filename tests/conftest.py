import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real sm_100 GPU (run on the B200 box with -m gpu)")
    config.addinivalue_line("markers", "needs_reference: needs the reference repository at $LBIC_REFERENCE_ROOT "
                                       "(skipped where it is not set)")


def golden_cases():
    return sorted(f[5:-4] for f in os.listdir(GOLDEN) if f.startswith("case_") and f.endswith(".npz"))


def load_case(name):
    d = np.load(os.path.join(GOLDEN, f"case_{name}.npz"))
    return {k: d[k] for k in d.files}


def load_tables():
    d = np.load(os.path.join(GOLDEN, "tables.npz"))
    return {k: d[k] for k in d.files}


@pytest.fixture(scope="session")
def golden_tables():
    return load_tables()
