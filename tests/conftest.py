import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    from oracle import oracle as O

    O.build()
    return O


@pytest.fixture(scope="session")
def emu_lib():
    """The product sources compiled against tests/emu's serial CUDA stand-in (test infrastructure)."""
    import subprocess

    from stitching_b200 import _lib

    emu_dir = os.path.join(ROOT, "tests", "emu")
    subprocess.check_call(["make", "-C", emu_dir, "-s"])
    return _lib.bind(os.path.join(emu_dir, "libstitch_b200_emu.so"))


@pytest.fixture()
def use_emu(emu_lib, monkeypatch):
    """Route the Python drop-ins through the emulation library for this test only.

    Pooled page-locked buffers (host_pool) and device twins (device_array) are released through whichever library is bound
    at that moment, so the ones left over are released on each side of the switch, each by the library that made them:
    the emulation's cudaFree is free(), the real one's is not."""
    import gc

    from stitching_b200 import _lib, host_pool

    def release_leftovers():
        gc.collect()
        host_pool.trim()

    release_leftovers()
    monkeypatch.setattr(_lib, "_lib", emu_lib)
    yield emu_lib
    release_leftovers()


@pytest.fixture(scope="session")
def cuda_lib():
    """The real library on a real GPU; fails (does not skip) when it cannot run."""
    from stitching_b200 import _lib

    L = _lib.lib()
    _lib.check(L.sb_init(int(os.environ.get("LOCAL_RANK", "0"))), "sb_init")
    return L
