"""CPU: zb200_zip_list parses central directories on the host, field by field as Python's zipfile reads them."""
import io
import struct
import zipfile

import pytest

from zlib_b200 import binding as zb


def _zip(members, compression=zipfile.ZIP_DEFLATED, level=None, comment=b""):
    b = io.BytesIO()
    with zipfile.ZipFile(b, "w", compression, compresslevel=level) as z:
        for name, data in members:
            z.writestr(name, data)
        z.comment = comment
    return b.getvalue()


class _NoSeek(io.RawIOBase):
    """A write-only stream without tell/seek: zipfile then writes data descriptors (flag bit 3)."""
    def __init__(self):
        self.buf = bytearray()

    def writable(self):
        return True

    def write(self, b):
        self.buf += b
        return len(b)


def _zip_descriptors(members):
    out = _NoSeek()
    with zipfile.ZipFile(out, "w", zipfile.ZIP_DEFLATED) as z:
        for name, data in members:
            with z.open(name, "w") as f:
                f.write(data)
    return bytes(out.buf)


MEMBERS = [("a.txt", b"hello, hello! " * 5000), ("empty", b""), ("dir/", b""), ("dür/ü.bin", bytes(range(256)) * 40),
           ("r.bin", b"\x00\x01" * 70000)]


def _agree(lib, arc):
    got = lib.zip_list(arc)
    want = zipfile.ZipFile(io.BytesIO(arc)).infolist()
    assert len(got) == len(want)
    for g, w in zip(got, want):
        assert g.name == w.filename
        assert (g.local_off, g.comp_len, g.raw_len, g.crc32, g.method, g.flags) == \
            (w.header_offset, w.compress_size, w.file_size, w.CRC, w.compress_type, w.flag_bits)
    return got


@pytest.mark.parametrize("compression,level", [(zipfile.ZIP_STORED, None), (zipfile.ZIP_DEFLATED, 1),
                                               (zipfile.ZIP_DEFLATED, 6), (zipfile.ZIP_DEFLATED, 9)])
def test_list_matches_zipfile(lib, compression, level):
    got = _agree(lib, _zip(MEMBERS, compression, level))
    assert [e.raw_len for e in got] == [len(d) for _, d in MEMBERS]
    assert got[3].flags & 0x800                           # the UTF-8 name


def test_list_comment_and_leading_bytes(lib):
    arc = _zip(MEMBERS, comment=b"an archive comment " * 100)
    _agree(lib, arc)
    got = _agree(lib, b"#!/bin/sh\nexit 0\n" * 30 + arc)
    assert got[0].local_off == len(b"#!/bin/sh\nexit 0\n") * 30


def test_list_data_descriptors(lib):
    arc = _zip_descriptors(MEMBERS[:2] + MEMBERS[3:])
    got = _agree(lib, arc)
    assert all(e.flags & 8 for e in got)


def test_list_empty_archive(lib):
    assert _agree(lib, _zip([])) == []


def test_list_capacity(lib):
    import ctypes as C
    import numpy as np
    arc = _zip(MEMBERS)
    recs = np.zeros(8, dtype=zb._zip_entry_dtype())
    n = C.c_size_t(2)
    assert lib.dll.zb200_zip_list(arc, len(arc), recs.ctypes.data, C.byref(n)) == zb.Z_BUF_ERROR
    assert n.value == len(MEMBERS)
    n = C.c_size_t(len(MEMBERS))
    assert lib.dll.zb200_zip_list(arc, len(arc), recs.ctypes.data, C.byref(n)) == zb.Z_OK
    assert n.value == len(MEMBERS)
    assert recs.dtype.itemsize == 48


def _rc(lib, arc):
    import ctypes as C
    import numpy as np
    recs = np.zeros(64, dtype=zb._zip_entry_dtype())
    n = C.c_size_t(64)
    return lib.dll.zb200_zip_list(arc, len(arc), recs.ctypes.data, C.byref(n))


def test_list_refuses_damaged_archives(lib):
    arc = _zip(MEMBERS)
    end = arc.rindex(b"PK\x05\x06")
    assert _rc(lib, arc) == zb.Z_OK
    assert _rc(lib, arc[:end + 10]) == zb.Z_STREAM_ERROR             # truncated inside the end record
    assert _rc(lib, arc[:end]) == zb.Z_STREAM_ERROR                  # no end record at all
    assert _rc(lib, arc[len(arc) // 2:]) == zb.Z_STREAM_ERROR        # the directory is not where the end record says
    multi = arc[:end + 4] + struct.pack("<H", 1) + arc[end + 6:]     # number of this disk = 1
    assert _rc(lib, multi) == zb.Z_STREAM_ERROR
    multi = arc[:end + 8] + struct.pack("<H", 1) + arc[end + 10:]    # entries on this disk != total entries
    assert _rc(lib, multi) == zb.Z_STREAM_ERROR
    # a ZIP64 end locator in front of the end record (as written for archives beyond ZIP32)
    loc = b"PK\x06\x07" + struct.pack("<IQI", 0, end, 1)
    assert _rc(lib, arc[:end] + loc + arc[end:]) == zb.Z_STREAM_ERROR
    big = arc[:end + 12] + struct.pack("<I", 0xFFFFFFFF) + arc[end + 16:]   # directory size 0xFFFFFFFF
    assert _rc(lib, big) == zb.Z_STREAM_ERROR
