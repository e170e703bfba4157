"""CPU: zb200_inflate_batch_size and its device form refuse bad arguments, and without a B200 refuse to work at all."""
import ctypes as C

import numpy as np
import pytest

from zlib_b200 import binding as zb


def _size(lib, off, wrap=zb.WRAP_ZLIB, n=None):
    off = np.asarray(off, dtype=np.uint64)
    n = len(off) - 1 if n is None else n
    src = np.zeros(int(off.max()) + 8 if len(off) else 8, dtype=np.uint8)
    ol = np.zeros(max(n, 1), dtype=np.uint64)
    st = np.zeros(max(n, 1), dtype=np.int32)
    return lib.dll.zb200_inflate_batch_size(src.ctypes.data, off.ctypes.data, n, ol.ctypes.data, None, st.ctypes.data,
                                            wrap, 0, None)


def test_bad_arguments_refused(lib):
    assert _size(lib, [0, 10, 4]) == zb.Z_STREAM_ERROR
    assert b"must not decrease" in lib.dll.zb200_last_error()
    for wrap in (-1, 4):
        assert _size(lib, [0, 4], wrap=wrap) == zb.Z_STREAM_ERROR
        assert b"wrap" in lib.dll.zb200_last_error()
        assert lib.dll.zb200_inflate_batch_size_dev(None, None, 0, None, None, None, None, wrap, 0, None) == zb.Z_STREAM_ERROR
    assert lib.dll.zb200_inflate_batch_size(None, None, 3, None, None, None, zb.WRAP_ZLIB, 0, None) == zb.Z_STREAM_ERROR
    assert lib.dll.zb200_inflate_batch_size_dev(None, None, 3, None, None, None, None, zb.WRAP_ZLIB, 0, None) == zb.Z_STREAM_ERROR


def test_no_cpu_path(lib):
    if lib.dll.zb200_device_count() > 0:
        pytest.skip("a GPU is present")
    assert _size(lib, [0, 4, 9]) == zb.Z_STREAM_ERROR
    assert b"no CPU path" in lib.dll.zb200_last_error()
    dummy = C.c_void_p(8)
    assert lib.dll.zb200_inflate_batch_size_dev(dummy, dummy, 2, dummy, None, dummy, None, zb.WRAP_ZLIB, 0, None) == zb.Z_STREAM_ERROR
    assert b"no CPU path" in lib.dll.zb200_last_error()
