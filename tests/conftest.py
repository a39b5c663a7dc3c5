import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def _ensure_built():
    """A fresh checkout has no libowrx_b200.so / oracle .so (git-ignored) and an edited source leaves a stale one: (re)compile
    (nvcc cross-compiles without a GPU).  The build is incremental (mtime-based): an up-to-date tree compiles nothing."""
    import __graft_entry__
    __graft_entry__.build()


def pytest_configure(config):
    _ensure_built()
    config.addinivalue_line("markers", "gpu: needs a B200 (run with -m gpu on the GPU box)")


def _have_gpu():
    try:
        from openwebrx_b200 import _native as N
        import ctypes as C
        n = C.c_int()
        return N.lib.owrx_device_count(C.byref(n)) == 0 and n.value > 0
    except Exception:
        return False


@pytest.fixture(scope="session")
def gpu():
    if not _have_gpu():
        pytest.fail("GPU test selected but no CUDA device / libowrx_b200.so is usable (no CPU fallback exists)")
    return 0
