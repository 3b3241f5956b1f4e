import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with `pytest -m gpu`)")


@pytest.fixture(scope="session")
def oracle():
    """CPU oracle bindings (test infrastructure); builds liboracle.so.  What the reference itself computes is recorded under
    tests/golden/."""
    from oracle import pyoracle
    pyoracle.build(ref=False)
    return pyoracle


@pytest.fixture(scope="session")
def ref():
    """outputs of the unmodified reference kernels on a B200, recorded by tests/golden/make_ref_outputs.py: ref(prefix) -> record"""
    import numpy as np
    from tests import util
    z = np.load(os.path.join(ROOT, "tests", "golden", "ref_outputs_gpu_v1.npz"))
    return lambda prefix: util.load_record(z, prefix)


@pytest.fixture(scope="session")
def gpu_ctx():
    from line3dpp_b200 import capi
    ctx = capi.Context(0)   # raises without a GPU: the product has no CPU fallback
    yield ctx
    ctx.close()
