import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    import numpy as np

    # the reference-run vectors, split over two files (tools/make_golden.py) so that neither exceeds 1 MB
    g = {}
    for name in ("reference_vectors.npz", "reference_vectors_2.npz"):
        g.update(np.load(os.path.join(ROOT, "tests", "golden", name)))
    return g


@pytest.fixture(scope="session")
def port():
    from oracle import loader

    loader.build()
    return loader.port()


@pytest.fixture(scope="session")
def qlib():
    """The product library, built on demand (CPU-only build check; compute needs a GPU)."""
    import __graft_entry__ as g
    from qdsp_b200 import lib

    if not os.path.exists(lib.LIB_PATH):
        g.build()
    return lib.load()
