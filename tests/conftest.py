import os
import sys
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def gpu_lib():
    """the product library on a real GPU; fails loudly if it is missing"""
    from openjph_b200 import _lib
    L = _lib.lib()
    assert L.ojb_device_count() > 0, "no CUDA device visible"
    return L


@pytest.fixture(scope="session")
def emu_lib():
    """SIMT-emulator build of the same sources (CPU test tier only)"""
    import emu
    return emu.emu_lib()


@pytest.fixture
def ref(request):
    """the reference's answers: its build in oracle/_ref when present, else the stored ones (tests/refgolden.py),
    replayed through the library the test checks (the product library in the GPU tier, the emulator build otherwise)"""
    import refharness
    lib = None if "gpu_lib" in request.fixturenames else request.getfixturevalue("emu_lib")
    return refharness.active(lib)
