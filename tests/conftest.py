import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def pytest_addoption(parser):
    parser.addoption("--emulate", action="store_true", default=False,
                     help="TEST HARNESS: run the `-m gpu` tests against the kernels under the CPU SIMT emulator "
                          "(tests/emul/simt) instead of a GPU - slow; e.g. pytest tests -m gpu --emulate")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box)")


@pytest.fixture(scope="session")
def checkers():
    """Build oracle/liboracle.so (+ oracle/_ref when /root/reference exists)."""
    import _bind
    _bind.build_checkers()
    return _bind


@pytest.fixture(scope="session")
def oracle(checkers):
    return checkers.Oracle()


@pytest.fixture(scope="session")
def product(request):
    """The CUDA product library; built in-tree if missing.  Never falls back to a CPU path."""
    from youtokentome_b200 import _lib
    if request.config.getoption("--emulate"):  # never the default: the GPU tests are the parity tests proper
        from _emu import emu_lib
        os.environ.setdefault("YT_EMU_SMS", "8")
        _lib._lib = emu_lib()
        return _lib._lib
    if not os.path.exists(_lib.LIB_PATH):
        _lib.build()
    return _lib.lib()
