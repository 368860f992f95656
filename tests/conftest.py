import importlib
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def tw():
    """The product binding (loads lib3dworld_b200.so; builds it first if nvcc is around and it is missing)."""
    lib = os.path.join(ROOT, "3dworld_b200", "lib3dworld_b200.so")
    if not os.path.exists(lib):
        spec = importlib.util.spec_from_file_location("tw_build", os.path.join(ROOT, "3dworld_b200", "build.py"))
        m = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(m)
        m.build()
    return importlib.import_module("3dworld_b200")


@pytest.fixture(scope="session")
def scene(tw):
    return importlib.import_module("3dworld_b200.scene")


@pytest.fixture(scope="session")
def oracle():
    import oracle as O
    O.lib()
    return O


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference objects (oracle/_ref); built by build() where the 3DWorld sources exist (REFERENCE_ROOT, else BASELINE.json's reference_path)."""
    import refapi as R
    if not R.available():
        pytest.skip("oracle/_ref/libref3dworld.so not built (build() builds it where the 3DWorld sources exist: REFERENCE_ROOT, else BASELINE.json's reference_path)")
    R.lib().ref_set_threads(max(1, min(16, os.cpu_count() or 1)))
    return R


@pytest.fixture(scope="session")
def ctx(tw):
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    c = tw.Context(0)
    yield c
    c.close()


def bits_differ(a, b):
    """Number of elements whose fp32 bit patterns differ (NaN == NaN)."""
    a = np.ascontiguousarray(a, np.float32).ravel()
    b = np.ascontiguousarray(b, np.float32).ravel()
    assert a.shape == b.shape
    return int(np.sum((a.view(np.uint32) != b.view(np.uint32)) & ~(np.isnan(a) & np.isnan(b))))


@pytest.fixture(scope="session")
def beq():
    return bits_differ
