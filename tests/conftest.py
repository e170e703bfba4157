import os
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a real B200 (run with -m gpu on the GPU box)")


@pytest.fixture(scope="session")
def oracle():
    import zhelpers
    return zhelpers.Oracle()


@pytest.fixture(scope="session")
def ref():
    """The unmodified reference compiled into oracle/_ref (skips when that build is absent)."""
    import zhelpers
    if not os.path.exists(zhelpers.REF_PATH):
        pytest.skip("oracle/_ref/libzref.so not built (needs /root/reference)")
    return zhelpers.Ref()


@pytest.fixture(scope="session")
def reference_codec(oracle):
    """compress2 / uncompress / deflate with a strategy as the reference computes them: the unmodified reference build
    when oracle/_ref has it, else the oracle, whose compress2 and uncompress tests/test_oracle_pin.py holds byte for byte
    to outputs recorded from the reference (tests/golden).  The oracle has no strategies: those streams then come from
    the system zlib."""
    import zhelpers
    if os.path.exists(zhelpers.REF_PATH):
        return zhelpers.Ref()
    return zhelpers.OracleAsReference(oracle)


@pytest.fixture(scope="session")
def lib():
    from zlib_b200 import load
    return load()


@pytest.fixture(scope="session")
def gpu_lib(lib):
    """libzb200.so initialised on cuda:0; fails loudly (never skips) when used under -m gpu."""
    rc = lib.dll.zb200_init(-1)
    assert rc == 0, f"zb200_init failed: {lib.last_error()}"
    return lib
