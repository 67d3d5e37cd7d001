import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


def _has_gpu():
    try:
        import torch
        return torch.cuda.is_available()
    except Exception:
        return False


def pytest_collection_modifyitems(config, items):
    if _has_gpu():
        return
    skip = pytest.mark.skip(reason="no CUDA device")
    for it in items:
        if "gpu" in it.keywords:
            it.add_marker(skip)


@pytest.fixture(scope="session")
def emu_lib():
    """TEST-ONLY single-thread emulation of the device code (g++ -DT4_EMU): lets the bit-exact logic of the
    engine be checked against the oracle without a GPU.  Exports t4emu_* symbols; never shipped."""
    import __graft_entry__
    from trust4_b200 import api
    lib = api.Lib(__graft_entry__.build_emu(), "t4emu_")
    lib.check(lib.init(0, 2 << 30))
    return lib


@pytest.fixture(scope="session")
def gpu_lib():
    from trust4_b200 import api
    lib = api.default_lib()
    lib.check(lib.init(0, 8 << 30))
    return lib


@pytest.fixture
def ref(request):
    """The reference's classes: live from oracle/_ref/libt4ref.so where it is built, else the results recorded from it
    under tests/golden/ref (tests/refharness.py)."""
    import refharness
    refharness.use_tape(request.node.nodeid)
    yield refharness
    refharness.end_tape()


@pytest.fixture
def ref_live():
    """The compiled reference itself, for tests of the oracle (they have nothing to check without it)."""
    import refharness
    if not refharness.available():
        pytest.skip("oracle/_ref/libt4ref.so not built: needs the reference sources (make -C oracle)")
    return refharness
