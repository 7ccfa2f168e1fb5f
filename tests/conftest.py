import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session", autouse=True)
def _built():
    """Build product + checker libraries once (nvcc cross-compiles without a GPU)."""
    import __graft_entry__ as g
    g.build()


@pytest.fixture(scope="session")
def golden_dir():
    return GOLDEN


@pytest.fixture(scope="session")
def sort_model():
    return open(os.path.join(GOLDEN, "sort6_model.bin"), "rb").read()


_host_stub = None


def load_host_stub():
    """Compile tests/host_stub.c (allocation, sampler RNG, tokenizer: what a host program links beside the shim) in a
    temporary directory and load it with RTLD_GLOBAL, so that libnano_infer_b200.so can be loaded and called.  The
    directory is removed once the library is mapped."""
    global _host_stub
    if _host_stub is None:
        import ctypes as C
        import subprocess
        import tempfile
        with tempfile.TemporaryDirectory(prefix="nb200_host_stub_") as td:
            so = os.path.join(td, "libnano_host_stub.so")
            subprocess.run(["gcc", "-O2", "-Wall", "-fPIC", "-shared", "-I" + os.path.join(ROOT, "include"),
                            os.path.join(ROOT, "tests", "host_stub.c"), "-o", so], check=True)
            _host_stub = C.CDLL(so, mode=C.RTLD_GLOBAL)
    return _host_stub


def sha256(a) -> str:
    import hashlib
    return hashlib.sha256(np.ascontiguousarray(a).tobytes()).hexdigest()


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def assert_bits_equal(a, b, what=""):
    a = np.ascontiguousarray(a); b = np.ascontiguousarray(b)
    assert a.shape == b.shape, f"{what}: shape {a.shape} vs {b.shape}"
    ne = np.nonzero(a.view(np.uint8).reshape(-1) != b.view(np.uint8).reshape(-1))[0]
    assert ne.size == 0, f"{what}: {ne.size} differing bytes, first at byte {ne[:4]}"
