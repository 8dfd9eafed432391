import json
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLD_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


def _have_gpu() -> bool:
    try:
        import ctypes
        cudart = ctypes.CDLL("libcudart.so.12")
        n = ctypes.c_int(0)
        return cudart.cudaGetDeviceCount(ctypes.byref(n)) == 0 and n.value > 0
    except OSError:
        try:
            import torch
            return torch.cuda.is_available()
        except Exception:
            return False


HAVE_GPU = _have_gpu()


def pytest_collection_modifyitems(config, items):
    if HAVE_GPU:
        return
    skip = pytest.mark.skip(reason="no CUDA device in this container (GPU tests run under gpurun)")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def goldens():
    with open(os.path.join(GOLD_DIR, "goldens.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def reference_outputs():
    """stored results of the reference's functions on the inputs of the tests that compare with them; their provenance is
    the file's "source" (tests/golden/make_reference_outputs.py)"""
    with open(os.path.join(GOLD_DIR, "reference_outputs.json")) as f:
        return json.load(f)


@pytest.fixture(scope="session")
def reflib_if_built():
    """the compiled reference when oracle/_ref is built (make -C oracle REF=<checkout>), else None: the tests that check
    reference_outputs compare with it directly as well"""
    from oracle.oracle import RefLib, have_ref
    return RefLib() if have_ref() else None


@pytest.fixture(scope="session")
def instances():
    z = np.load(os.path.join(GOLD_DIR, "instances.npz"))
    out = {}
    for k in z.files:
        nm, what = k.split("__")
        out.setdefault(nm, {})[what] = z[k]
    return {nm: (v["xy"], int(v["wt"])) for nm, v in out.items()}


@pytest.fixture(scope="session")
def oracle():
    from oracle.oracle import Oracle
    return Oracle()


@pytest.fixture(scope="session")
def reflib():
    from oracle.oracle import RefLib, have_ref
    if not have_ref():
        pytest.skip("oracle/_ref/libtspref.so not available")
    return RefLib()


@pytest.fixture(scope="session")
def engine():
    from tsp_optimization_b200 import Engine
    e = Engine(0)
    yield e
    e.close()
