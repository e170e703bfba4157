"""ctypes binding of libzb200.so: every symbol of include/zlib.h and include/zb200.h.

Mirrors the reference's C interface one to one (same names, argument order and
return codes as h/zlib.h in ChrisHird/ZLIB), so tests read like the reference's
example.c.  Loading is RTLD_LOCAL|RTLD_DEEPBIND: the library exports the same
names as the system libz that CPython itself links, and must never interpose.
"""
from __future__ import annotations

import ctypes as C
import os
from typing import Optional, Tuple, Union

LIB_PATH = os.path.join(os.path.dirname(os.path.abspath(__file__)), "libzb200.so")

Z_OK, Z_STREAM_END, Z_NEED_DICT = 0, 1, 2
Z_ERRNO, Z_STREAM_ERROR, Z_DATA_ERROR, Z_MEM_ERROR, Z_BUF_ERROR, Z_VERSION_ERROR = -1, -2, -3, -4, -5, -6
Z_NO_FLUSH, Z_PARTIAL_FLUSH, Z_SYNC_FLUSH, Z_FULL_FLUSH, Z_FINISH, Z_BLOCK = 0, 1, 2, 3, 4, 5
Z_DEFLATED = 8
WRAP_RAW, WRAP_ZLIB, WRAP_GZIP = 0, 1, 2
DOS_DATETIME = 46 << 25 | 10 << 21 | 18 << 16            # 2026-10-18 00:00:00 in zip.c's dosDate layout
ZB200_DEFLATE_NOT_LAST, ZB200_DEFLATE_NO_HEADER, ZB200_DEFLATE_NO_TRAILER = 1, 2, 4
ZLIB_VERSION = b"1.2.3"
ZB200_UNZ_BADZIPFILE, ZB200_UNZ_CRCERROR = -103, -105          # minizip's unzip.h values


class z_stream(C.Structure):
    """h/zlib.h:82-101 (112 bytes on LP64)."""
    _fields_ = [
        ("next_in", C.c_void_p), ("avail_in", C.c_uint), ("total_in", C.c_ulong),
        ("next_out", C.c_void_p), ("avail_out", C.c_uint), ("total_out", C.c_ulong),
        ("msg", C.c_char_p), ("state", C.c_void_p),
        ("zalloc", C.c_void_p), ("zfree", C.c_void_p), ("opaque", C.c_void_p),
        ("data_type", C.c_int), ("adler", C.c_ulong), ("reserved", C.c_ulong),
    ]


Buf = Union[bytes, bytearray, memoryview, int, "C.Array"]


def _ptr(buf) -> Tuple[C.c_void_p, Optional[object]]:
    """(pointer, keep-alive) for bytes-like objects, numpy arrays or raw addresses."""
    if buf is None:
        return C.c_void_p(0), None
    if isinstance(buf, int):
        return C.c_void_p(buf), None
    if isinstance(buf, bytes):
        return C.cast(C.c_char_p(buf), C.c_void_p), buf
    if hasattr(buf, "ctypes") and hasattr(buf, "nbytes"):        # numpy
        return C.c_void_p(buf.ctypes.data), buf
    if hasattr(buf, "data_ptr"):                                  # torch tensor
        return C.c_void_p(buf.data_ptr()), buf
    if isinstance(buf, C.Array):
        return C.cast(buf, C.c_void_p), buf
    mv = memoryview(buf)
    arr = (C.c_char * mv.nbytes).from_buffer(mv.obj if not mv.readonly else bytearray(mv))
    return C.cast(arr, C.c_void_p), arr


def _stream(stream) -> C.c_void_p:
    if stream is None:
        return C.c_void_p(0)
    if isinstance(stream, int):
        return C.c_void_p(stream)
    return C.c_void_p(stream.cuda_stream)                         # torch.cuda.Stream


class gz_header(C.Structure):
    """h/zlib.h:105-121."""
    _fields_ = [("text", C.c_int), ("time", C.c_ulong), ("xflags", C.c_int), ("os", C.c_int),
                ("extra", C.c_void_p), ("extra_len", C.c_uint), ("extra_max", C.c_uint),
                ("name", C.c_void_p), ("name_max", C.c_uint), ("comment", C.c_void_p), ("comm_max", C.c_uint),
                ("hcrc", C.c_int), ("done", C.c_int)]


class ZipEntry:
    """One member as zb200_zip_list reports it; `raw` is the 48-byte zb200_zip_entry record."""
    __slots__ = ("name", "local_off", "comp_len", "raw_len", "crc32", "method", "flags", "raw")

    def __init__(self, name, rec):
        self.name = name
        self.local_off, self.comp_len, self.raw_len = int(rec["local_off"]), int(rec["comp_len"]), int(rec["raw_len"])
        self.crc32, self.method, self.flags = int(rec["crc32"]), int(rec["method"]), int(rec["flags"])
        self.raw = rec.copy()

    def __repr__(self):
        return (f"ZipEntry({self.name!r}, local_off={self.local_off}, comp_len={self.comp_len}, raw_len={self.raw_len}, "
                f"crc32={self.crc32:#010x}, method={self.method}, flags={self.flags:#x})")


def _zip_entry_dtype():
    import numpy as np
    return np.dtype([("local_off", "<u8"), ("comp_len", "<u8"), ("raw_len", "<u8"), ("name_off", "<u8"), ("crc32", "<u4"),
                     ("method", "<u2"), ("flags", "<u2"), ("name_len", "<u2"), ("reserved16", "<u2"), ("reserved32", "<u4")])


def _nbytes(buf) -> int:
    if hasattr(buf, "data_ptr"):                                  # torch tensor
        return buf.numel() * buf.element_size()
    if hasattr(buf, "nbytes"):
        return int(buf.nbytes)
    return len(buf)


class Lib:
    """One loaded copy of libzb200.so."""

    def __init__(self, path: str = LIB_PATH):
        if not os.path.exists(path):
            raise ImportError(
                f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(zlib_b200 has no fallback implementation)")
        self.path = path
        self.dll = C.CDLL(path, mode=os.RTLD_LOCAL | os.RTLD_DEEPBIND)
        d = self.dll
        ul, ui, vp, sz = C.c_ulong, C.c_uint, C.c_void_p, C.c_size_t
        u32p, u64p, i32p = C.POINTER(C.c_uint32), C.POINTER(C.c_uint64), C.POINTER(C.c_int32)
        zsp = C.POINTER(z_stream)
        sig = {
            # zlib.h
            "zlibVersion": (C.c_char_p, []), "zlibCompileFlags": (ul, []), "zError": (C.c_char_p, [C.c_int]),
            "get_crc_table": (C.POINTER(ul), []), "inflateSyncPoint": (C.c_int, [zsp]),
            "deflate": (C.c_int, [zsp, C.c_int]), "deflateEnd": (C.c_int, [zsp]),
            "deflateSetDictionary": (C.c_int, [zsp, vp, ui]), "deflateCopy": (C.c_int, [zsp, zsp]),
            "deflateReset": (C.c_int, [zsp]), "deflateParams": (C.c_int, [zsp, C.c_int, C.c_int]),
            "deflateTune": (C.c_int, [zsp, C.c_int, C.c_int, C.c_int, C.c_int]),
            "deflateBound": (ul, [zsp, ul]), "deflatePrime": (C.c_int, [zsp, C.c_int, C.c_int]),
            "deflateSetHeader": (C.c_int, [zsp, vp]),
            "inflate": (C.c_int, [zsp, C.c_int]), "inflateEnd": (C.c_int, [zsp]),
            "inflateSetDictionary": (C.c_int, [zsp, vp, ui]), "inflateSync": (C.c_int, [zsp]),
            "inflateCopy": (C.c_int, [zsp, zsp]), "inflateReset": (C.c_int, [zsp]),
            "inflatePrime": (C.c_int, [zsp, C.c_int, C.c_int]), "inflateGetHeader": (C.c_int, [zsp, vp]),
            "compress": (C.c_int, [vp, C.POINTER(ul), vp, ul]),
            "compress2": (C.c_int, [vp, C.POINTER(ul), vp, ul, C.c_int]),
            "compressBound": (ul, [ul]), "uncompress": (C.c_int, [vp, C.POINTER(ul), vp, ul]),
            "adler32": (ul, [ul, vp, ui]), "adler32_combine": (ul, [ul, ul, C.c_long]),
            "crc32": (ul, [ul, vp, ui]), "crc32_combine": (ul, [ul, ul, C.c_long]),
            "deflateInit_": (C.c_int, [zsp, C.c_int, C.c_char_p, C.c_int]),
            "inflateInit_": (C.c_int, [zsp, C.c_char_p, C.c_int]),
            "deflateInit2_": (C.c_int, [zsp, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]),
            "inflateInit2_": (C.c_int, [zsp, C.c_int, C.c_char_p, C.c_int]),
            # zb200.h
            "zb200_init": (C.c_int, [C.c_int]), "zb200_device_count": (C.c_int, []),
            "zb200_last_error": (C.c_char_p, []), "zb200_build_info": (C.c_char_p, []),
            "zb200_alloc_pinned": (vp, [sz]), "zb200_free_pinned": (None, [vp]),
            "zb200_alloc_device": (vp, [sz]), "zb200_free_device": (None, [vp]),
            "zb200_copy": (C.c_int, [vp, vp, sz, vp]), "zb200_sync": (C.c_int, [vp]),
            "zb200_copy_async": (C.c_int, [vp, vp, sz, vp]),
            "zb200_host_register": (C.c_int, [vp, sz]), "zb200_host_unregister": (C.c_int, [vp]),
            "zb200_ipc_export": (C.c_int, [vp, vp]), "zb200_ipc_open": (C.c_int, [vp, C.POINTER(vp)]), "zb200_ipc_close": (C.c_int, [vp]),
            "zb200_checksum": (C.c_int, [vp, sz, u32p, u32p, vp]),
            "zb200_checksum_dev": (C.c_int, [vp, sz, vp, vp]),
            "zb200_checksum_batch": (C.c_int, [vp, vp, sz, vp, vp, vp]),
            "zb200_deflate": (C.c_int, [vp, sz, vp, C.POINTER(sz), C.c_int, C.c_int, vp]),
            "zb200_deflate_shard": (C.c_int, [vp, sz, vp, sz, vp, C.POINTER(sz), C.c_int, C.c_int, C.c_int, u32p, u32p, vp]),
            "zb200_deflate_shard_begin": (C.c_int, [C.POINTER(vp), vp, sz, vp, sz, vp, sz, C.c_int, C.c_int, C.c_int, vp]),
            "zb200_deflate_shard_end": (C.c_int, [vp, C.POINTER(sz), u32p, u32p]),
            "zb200_deflate_batch": (C.c_int, [vp, vp, sz, vp, vp, vp, vp, vp, vp, C.c_int, C.c_int, vp]),
            "zb200_zip_bound": (sz, [vp, vp, sz]),
            "zb200_zip_build": (C.c_int, [vp, vp, vp, sz, C.c_int, C.c_uint32, vp, C.POINTER(sz)]),
            "zb200_zip_segment": (C.c_int, [vp, vp, vp, sz, C.c_int, C.c_uint32, vp, C.POINTER(sz), vp]),
            "zb200_zip_directory": (C.c_int, [vp, vp, sz, C.c_uint32, C.c_uint64, vp, C.POINTER(sz)]),
            "zb200_zip_list": (C.c_int, [vp, sz, vp, C.POINTER(sz)]),
            "zb200_zip_extract": (C.c_int, [vp, sz, vp, sz, vp, vp, vp, vp, vp]),
            "zb200_gunzip": (C.c_int, [vp, sz, vp, C.POINTER(sz), C.POINTER(sz), vp]),
            "zb200_bgzf_bound": (sz, [sz]),
            "zb200_bgzf_compress": (C.c_int, [vp, sz, vp, C.POINTER(sz), C.c_int, vp]),
            "zb200_inflate_batch": (C.c_int, [vp, vp, sz, vp, vp, vp, vp, C.c_int, vp]),
            "zb200_inflate_batch_dev": (C.c_int, [vp, vp, sz, vp, vp, vp, vp, C.c_int, vp]),
            "zb200_inflate_batch_size": (C.c_int, [vp, vp, sz, vp, vp, vp, C.c_int, C.c_uint64, vp]),
            "zb200_inflate_batch_size_dev": (C.c_int, [vp, vp, sz, vp, vp, vp, vp, C.c_int, C.c_uint64, vp]),
            "zb200_multi_devices": (C.c_int, []),
            "zb200_multi_deflate": (C.c_int, [vp, sz, vp, C.POINTER(sz), C.c_int, C.c_int, C.c_int, u32p, u32p]),
            "zb200_multi_checksum": (C.c_int, [vp, sz, C.c_int, u32p, u32p]),
            "zb200_multi_inflate_batch": (C.c_int, [vp, vp, sz, vp, vp, vp, vp, C.c_int, C.c_int]),
            "zb200_kernel_launches": (C.c_uint64, []),
            "zb200_profile": (None, [C.c_int]), "zb200_profile_report": (C.c_int, [C.c_char_p, sz]),
        }
        self.missing = []
        for name, (res, args) in sig.items():
            try:
                f = getattr(d, name)
            except AttributeError:
                self.missing.append(name)
                continue
            f.restype, f.argtypes = res, args
        self.signatures = sig

    # ---- errors ---------------------------------------------------------
    def last_error(self) -> str:
        return (self.dll.zb200_last_error() or b"").decode()

    def _check(self, rc: int, what: str):
        if rc != Z_OK:
            raise RuntimeError(f"{what} -> {rc}: {self.last_error()}")

    # ---- checksums ------------------------------------------------------
    def crc32(self, data: Buf, value: int = 0, length: Optional[int] = None) -> int:
        p, keep = _ptr(data)
        n = len(data) if length is None else length
        return self.dll.crc32(value, p, n)

    def adler32(self, data: Buf, value: int = 1, length: Optional[int] = None) -> int:
        p, keep = _ptr(data)
        n = len(data) if length is None else length
        return self.dll.adler32(value, p, n)

    def crc32_combine(self, c1: int, c2: int, len2: int) -> int:
        return self.dll.crc32_combine(c1, c2, len2)

    def adler32_combine(self, a1: int, a2: int, len2: int) -> int:
        return self.dll.adler32_combine(a1, a2, len2)

    def checksum(self, data: Buf, length: Optional[int] = None, stream=None) -> Tuple[int, int]:
        """(crc32(0,data), adler32(1,data)) in one GPU pass; data may be a device pointer."""
        p, keep = _ptr(data)
        n = len(data) if length is None else length
        crc, adl = C.c_uint32(0), C.c_uint32(0)
        self._check(self.dll.zb200_checksum(p, n, C.byref(crc), C.byref(adl), _stream(stream)), "zb200_checksum")
        return crc.value, adl.value

    def checksum_dev(self, d_ptr: int, length: int, d_out2: int, stream=None) -> None:
        self._check(self.dll.zb200_checksum_dev(C.c_void_p(d_ptr), length, C.c_void_p(d_out2), _stream(stream)),
                    "zb200_checksum_dev")

    # ---- one-shot codec ---------------------------------------------------
    def compress_bound(self, n: int) -> int:
        return self.dll.compressBound(n)

    def compress2(self, data: Buf, level: int = -1, cap: Optional[int] = None) -> Tuple[int, bytes]:
        n = len(data)
        cap = self.compress_bound(n) if cap is None else cap
        out = C.create_string_buffer(max(cap, 1))
        ol = C.c_ulong(cap)
        p, keep = _ptr(data)
        rc = self.dll.compress2(out, C.byref(ol), p, n, level)
        return rc, (out.raw[:ol.value] if rc == Z_OK else b"")

    def uncompress(self, data: Buf, cap: int) -> Tuple[int, bytes]:
        out = C.create_string_buffer(max(cap, 1))
        ol = C.c_ulong(cap)
        p, keep = _ptr(data)
        rc = self.dll.uncompress(out, C.byref(ol), p, len(data))
        return rc, (out.raw[:ol.value] if rc == Z_OK else b"")

    def deflate(self, src: Buf, src_len: int, dst: Buf, dst_cap: int, level: int = 6, wrap: int = WRAP_ZLIB,
                stream=None) -> int:
        """zb200_deflate on host or device buffers; returns the compressed length."""
        ps, k1 = _ptr(src)
        pd, k2 = _ptr(dst)
        ol = C.c_size_t(dst_cap)
        self._check(self.dll.zb200_deflate(ps, src_len, pd, C.byref(ol), level, wrap, _stream(stream)), "zb200_deflate")
        return ol.value

    def deflate_shard(self, src: Buf, src_len: int, dict_: Buf, dict_len: int, dst: Buf, dst_cap: int, level: int,
                      wrap: int, flags: int, stream=None) -> Tuple[int, int, int]:
        ps, k1 = _ptr(src)
        pk, k3 = _ptr(dict_)
        pd, k2 = _ptr(dst)
        ol = C.c_size_t(dst_cap)
        crc, adl = C.c_uint32(0), C.c_uint32(0)
        self._check(self.dll.zb200_deflate_shard(ps, src_len, pk, dict_len, pd, C.byref(ol), level, wrap, flags,
                                                 C.byref(crc), C.byref(adl), _stream(stream)), "zb200_deflate_shard")
        return ol.value, crc.value, adl.value

    def deflate_shard_begin(self, src: Buf, src_len: int, dict_: Buf, dict_len: int, dst: Buf, dst_cap: int, level: int,
                            wrap: int, flags: int, stream=None):
        """First half of deflate_shard: everything enqueued; returns the job handle for deflate_shard_end."""
        ps, k1 = _ptr(src)
        pk, k3 = _ptr(dict_)
        pd, k2 = _ptr(dst)
        job = C.c_void_p(0)
        self._check(self.dll.zb200_deflate_shard_begin(C.byref(job), ps, src_len, pk, dict_len, pd, dst_cap, level, wrap, flags,
                                                       _stream(stream)), "zb200_deflate_shard_begin")
        return job

    def deflate_shard_end(self, job) -> Tuple[int, int, int]:
        ol = C.c_size_t(0)
        crc, adl = C.c_uint32(0), C.c_uint32(0)
        self._check(self.dll.zb200_deflate_shard_end(job, C.byref(ol), C.byref(crc), C.byref(adl)), "zb200_deflate_shard_end")
        return ol.value, crc.value, adl.value

    def checksum_batch(self, bufs, stream=None):
        """zb200_checksum_batch over a list of bytes objects -> ([crc32], [adler32])."""
        import numpy as np
        n = len(bufs)
        off = np.zeros(n + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(b) for b in bufs], dtype=np.uint64)
        base = np.frombuffer(b"".join(bufs) + b"\0" * 8, dtype=np.uint8)
        crc = np.zeros(max(n, 1), dtype=np.uint32)
        adl = np.zeros(max(n, 1), dtype=np.uint32)
        self._check(self.dll.zb200_checksum_batch(base.ctypes.data, off.ctypes.data, n, crc.ctypes.data, adl.ctypes.data,
                                                  _stream(stream)), "zb200_checksum_batch")
        return [int(x) for x in crc[:n]], [int(x) for x in adl[:n]]

    def deflate_batch(self, bufs, level: int = 6, wrap: int = WRAP_ZLIB, caps=None, stream=None):
        """zb200_deflate_batch over a list of bytes objects -> (streams, statuses, crcs, adlers)."""
        import numpy as np
        n = len(bufs)
        caps = [self.compress_bound(len(b)) + 16 for b in bufs] if caps is None else caps
        src_off = np.zeros(n + 1, dtype=np.uint64)
        dst_off = np.zeros(n + 1, dtype=np.uint64)
        src_off[1:] = np.cumsum([len(b) for b in bufs], dtype=np.uint64)
        dst_off[1:] = np.cumsum(caps, dtype=np.uint64)
        src = np.frombuffer(b"".join(bufs) + b"\0" * 8, dtype=np.uint8)
        dst = np.zeros(int(dst_off[-1]) + 8, dtype=np.uint8)
        dst_len = np.zeros(max(n, 1), dtype=np.uint64)
        crc = np.zeros(max(n, 1), dtype=np.uint32)
        adl = np.zeros(max(n, 1), dtype=np.uint32)
        status = np.full(max(n, 1), -99, dtype=np.int32)
        self._check(self.dll.zb200_deflate_batch(src.ctypes.data, src_off.ctypes.data, n, dst.ctypes.data, dst_off.ctypes.data,
                                                 dst_len.ctypes.data, crc.ctypes.data, adl.ctypes.data, status.ctypes.data,
                                                 level, wrap, _stream(stream)), "zb200_deflate_batch")
        outs = [bytes(dst[int(dst_off[i]):int(dst_off[i]) + int(dst_len[i])]) if status[i] == 0 else b"" for i in range(n)]
        return outs, [int(x) for x in status[:n]], [int(x) for x in crc[:n]], [int(x) for x in adl[:n]]

    def zip_build(self, files, level: int = 6, dos_datetime: int = DOS_DATETIME):
        """zb200_zip_build over {name: bytes} -> archive bytes."""
        import numpy as np
        names = list(files)
        n = len(names)
        arr = (C.c_char_p * max(n, 1))(*[nm.encode() for nm in names])
        off = np.zeros(n + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(files[nm]) for nm in names], dtype=np.uint64)
        src = np.frombuffer(b"".join(files[nm] for nm in names) + b"\0" * 8, dtype=np.uint8)
        cap = self.dll.zb200_zip_bound(arr, off.ctypes.data, n)
        out = C.create_string_buffer(max(cap, 1))
        ol = C.c_size_t(cap)
        self._check(self.dll.zb200_zip_build(arr, src.ctypes.data, off.ctypes.data, n, level, dos_datetime, out, C.byref(ol)),
                    "zb200_zip_build")
        return out.raw[:ol.value]

    def zip_segment(self, names, datas, level: int = 6, dos_datetime: int = DOS_DATETIME):
        """zb200_zip_segment over parallel lists of names and bytes -> (segment bytes, [(local_off, comp_len, raw_len, crc32)])."""
        import numpy as np
        n = len(names)
        arr = (C.c_char_p * max(n, 1))(*[nm.encode() for nm in names])
        off = np.zeros(n + 1, dtype=np.uint64)
        off[1:] = np.cumsum([len(d) for d in datas], dtype=np.uint64)
        src = np.frombuffer(b"".join(datas) + b"\0" * 8, dtype=np.uint8)
        cap = self.dll.zb200_zip_bound(arr, off.ctypes.data, n)
        out = np.empty(max(cap, 1), dtype=np.uint8)
        members = np.zeros((max(n, 1), 4), dtype=np.uint64)     # zb200_zip_member: 3 x u64, then {u32 crc32, u32 reserved}
        ol = C.c_size_t(cap)
        self._check(self.dll.zb200_zip_segment(arr, src.ctypes.data, off.ctypes.data, n, level, dos_datetime, out.ctypes.data,
                                               C.byref(ol), members.ctypes.data), "zb200_zip_segment")
        metas = [(int(m[0]), int(m[1]), int(m[2]), int(m[3]) & 0xFFFFFFFF) for m in members[:n]]
        return out[:ol.value].tobytes(), metas

    def zip_directory(self, names, metas, cd_offset: int, dos_datetime: int = DOS_DATETIME):
        """zb200_zip_directory: central directory + end record for members given as (local_off, comp_len, raw_len, crc32)."""
        import numpy as np
        n = len(names)
        arr = (C.c_char_p * max(n, 1))(*[nm.encode() for nm in names])
        members = np.zeros((max(n, 1), 4), dtype=np.uint64)
        for i, m in enumerate(metas):
            members[i] = (m[0], m[1], m[2], m[3])
        cap = 22 + sum(46 + len(nm.encode()) for nm in names)
        out = C.create_string_buffer(cap)
        ol = C.c_size_t(cap)
        self._check(self.dll.zb200_zip_directory(arr, members.ctypes.data, n, dos_datetime, cd_offset, out, C.byref(ol)),
                    "zb200_zip_directory")
        return out.raw[:ol.value]

    def zip_list(self, archive):
        """zb200_zip_list -> [ZipEntry]; names decoded as zipfile does (UTF-8 with flag bit 11, else cp437).
        `archive`: bytes, a numpy array or a CUDA torch tensor of uint8."""
        import numpy as np
        p, keep = _ptr(archive)
        size = _nbytes(archive)
        cnt = C.c_size_t(0)
        rc = self.dll.zb200_zip_list(p, size, None, C.byref(cnt))
        if rc not in (Z_OK, Z_BUF_ERROR):
            self._check(rc, "zb200_zip_list")
        recs = np.zeros(max(cnt.value, 1), dtype=_zip_entry_dtype())
        if cnt.value:
            self._check(self.dll.zb200_zip_list(p, size, recs.ctypes.data, C.byref(cnt)), "zb200_zip_list")
        recs = recs[:cnt.value]
        names = []
        if cnt.value:
            lo = int(recs["name_off"].min())
            hi = int((recs["name_off"] + recs["name_len"]).max())
            if hasattr(archive, "data_ptr"):
                blob = archive[lo:hi].cpu().numpy().tobytes()
            else:
                blob = bytes(memoryview(archive).cast("B")[lo:hi]) if not hasattr(archive, "ctypes") else archive[lo:hi].tobytes()
            for r in recs:
                raw = blob[int(r["name_off"]) - lo:int(r["name_off"]) - lo + int(r["name_len"])]
                names.append(raw.decode("utf-8") if int(r["flags"]) & 0x800 else raw.decode("cp437"))
        return [ZipEntry(nm, r) for nm, r in zip(names, recs)]

    def zip_extract(self, archive, entries=None, caps=None, stream=None):
        """zb200_zip_extract -> (outputs, statuses).  entries: ZipEntry list (default: every member, from zip_list); caps:
        slot sizes (default raw_len).  With the archive in a CUDA torch tensor the outputs are views of one CUDA tensor,
        otherwise bytes."""
        import numpy as np
        if entries is None:
            entries = self.zip_list(archive)
        n = len(entries)
        recs = np.zeros(max(n, 1), dtype=_zip_entry_dtype())
        for i, e in enumerate(entries):
            recs[i] = e.raw
        caps = [e.raw_len for e in entries] if caps is None else list(caps)
        dst_off = np.zeros(n + 1, dtype=np.uint64)
        dst_off[1:] = np.cumsum(caps, dtype=np.uint64)
        on_dev = hasattr(archive, "data_ptr") and getattr(archive, "is_cuda", False)
        if on_dev:
            import torch
            dst = torch.empty(int(dst_off[-1]) + 8, dtype=torch.uint8, device=archive.device)
        else:
            dst = np.zeros(int(dst_off[-1]) + 8, dtype=np.uint8)
        dst_len = np.zeros(max(n, 1), dtype=np.uint64)
        status = np.full(max(n, 1), -99, dtype=np.int32)
        pa, keep = _ptr(archive)
        pd, keep2 = _ptr(dst)
        self._check(self.dll.zb200_zip_extract(pa, _nbytes(archive), recs.ctypes.data, n, pd, dst_off.ctypes.data,
                                               dst_len.ctypes.data, status.ctypes.data, _stream(stream)), "zb200_zip_extract")
        if on_dev:
            outs = [dst[int(dst_off[i]):int(dst_off[i]) + int(dst_len[i])] for i in range(n)]
        else:
            outs = [dst[int(dst_off[i]):int(dst_off[i]) + int(dst_len[i])].tobytes() for i in range(n)]
        return outs, [int(x) for x in status[:n]]

    def _out_like(self, data, n):
        """An output buffer of n bytes: a CUDA tensor when `data` is one, else numpy."""
        import numpy as np
        if hasattr(data, "data_ptr") and getattr(data, "is_cuda", False):
            import torch
            return torch.empty(max(n, 1), dtype=torch.uint8, device=data.device)
        return np.empty(max(n, 1), dtype=np.uint8)

    def gunzip(self, data, stream=None):
        """zb200_gunzip: every member of a gzip file -> bytes, or a CUDA tensor when `data` is one.  Raises RuntimeError
        (the library's message names the member) on damaged data.  A first guess of 4x the input is retried once at the
        size the library reports."""
        p, keep = _ptr(data)
        n = _nbytes(data)
        cap = max(4 * n, 1 << 20)
        for _ in range(2):
            out = self._out_like(data, cap)
            po, keep2 = _ptr(out)
            ol, cnt = C.c_size_t(cap), C.c_size_t(0)
            rc = self.dll.zb200_gunzip(p, n, po, C.byref(ol), C.byref(cnt), _stream(stream))
            if rc != Z_BUF_ERROR:
                break
            cap = ol.value
        self._check(rc, "zb200_gunzip")
        self.last_members = cnt.value
        return out[:ol.value] if hasattr(out, "data_ptr") else out[:ol.value].tobytes()

    def bgzf_compress(self, data, level: int = 6, stream=None):
        """zb200_bgzf_compress -> BGZF bytes, or a CUDA tensor when `data` is one."""
        p, keep = _ptr(data)
        n = _nbytes(data)
        cap = self.dll.zb200_bgzf_bound(n)
        out = self._out_like(data, cap)
        po, keep2 = _ptr(out)
        ol = C.c_size_t(cap)
        self._check(self.dll.zb200_bgzf_compress(p, n, po, C.byref(ol), level, _stream(stream)), "zb200_bgzf_compress")
        return out[:ol.value] if hasattr(out, "data_ptr") else out[:ol.value].tobytes()

    def inflate_batch(self, streams, caps, wrap: int = WRAP_ZLIB, stream=None):
        """zb200_inflate_batch over a list of bytes objects; returns (outputs, statuses)."""
        import numpy as np
        n = len(streams)
        src_off = np.zeros(n + 1, dtype=np.uint64)
        dst_off = np.zeros(n + 1, dtype=np.uint64)
        src_off[1:] = np.cumsum([len(x) for x in streams], dtype=np.uint64)
        dst_off[1:] = np.cumsum(caps, dtype=np.uint64)
        src = np.frombuffer(b"".join(streams) + b"\0" * 8, dtype=np.uint8)
        dst = np.zeros(int(dst_off[-1]) + 8, dtype=np.uint8)
        dst_len = np.zeros(max(n, 1), dtype=np.uint64)
        status = np.full(max(n, 1), -99, dtype=np.int32)
        self._check(self.dll.zb200_inflate_batch(src.ctypes.data, src_off.ctypes.data, n, dst.ctypes.data,
                                                 dst_off.ctypes.data, dst_len.ctypes.data, status.ctypes.data,
                                                 wrap, _stream(stream)), "zb200_inflate_batch")
        outs = [bytes(dst[int(dst_off[i]):int(dst_off[i]) + int(dst_len[i])]) for i in range(n)]
        return outs, [int(x) for x in status[:n]]

    def inflate_batch_dev(self, d_src, d_src_off, n, d_dst, d_dst_off, d_dst_len, d_status, wrap=WRAP_ZLIB, stream=None):
        self._check(self.dll.zb200_inflate_batch_dev(C.c_void_p(d_src), C.c_void_p(d_src_off), n, C.c_void_p(d_dst),
                                                     C.c_void_p(d_dst_off), C.c_void_p(d_dst_len), C.c_void_p(d_status),
                                                     wrap, _stream(stream)), "zb200_inflate_batch_dev")

    def inflate_batch_size(self, streams, wrap: int = WRAP_ZLIB, limit: int = 0, stream=None):
        """zb200_inflate_batch_size over a list of bytes objects -> (out_len, src_used, status) lists: what inflate_batch
        would produce for each stream, found without producing it (zlib Adler-32 and gzip CRC-32 are not verified)."""
        import numpy as np
        n = len(streams)
        src_off = np.zeros(n + 1, dtype=np.uint64)
        src_off[1:] = np.cumsum([len(x) for x in streams], dtype=np.uint64)
        src = np.frombuffer(b"".join(streams) + b"\0" * 8, dtype=np.uint8)
        out_len = np.zeros(max(n, 1), dtype=np.uint64)
        src_used = np.zeros(max(n, 1), dtype=np.uint64)
        status = np.full(max(n, 1), -99, dtype=np.int32)
        self._check(self.dll.zb200_inflate_batch_size(src.ctypes.data, src_off.ctypes.data, n, out_len.ctypes.data,
                                                      src_used.ctypes.data, status.ctypes.data, wrap, limit,
                                                      _stream(stream)), "zb200_inflate_batch_size")
        return [int(x) for x in out_len[:n]], [int(x) for x in src_used[:n]], [int(x) for x in status[:n]]

    def decompress_batch(self, streams, wrap: int = WRAP_ZLIB, limit: int = 0, stream=None):
        """Sizes the batch with inflate_batch_size, then decodes it into slots of exactly those sizes -> (outputs,
        statuses).  `limit` bounds every slot (0 = none): a stream longer than that reports Z_BUF_ERROR."""
        out_len, _, _ = self.inflate_batch_size(streams, wrap=wrap, limit=limit, stream=stream)
        return self.inflate_batch(streams, out_len, wrap=wrap, stream=stream)

    # ---- streaming API driven the way example.c drives it ----------------
    def deflate_stream(self, data: bytes, level=6, wbits=15, in_chunk=1 << 16, out_chunk=1 << 16, flushes=None,
                       dictionary=None, strategy=0):
        """deflateInit2 + deflate(...) loop + deflateEnd; `flushes` maps input offsets to flush values."""
        strm = z_stream()
        rc = self.dll.deflateInit2_(C.byref(strm), level, Z_DEFLATED, wbits, 8, strategy, ZLIB_VERSION, C.sizeof(z_stream))
        if rc != Z_OK:
            return rc, b""
        if dictionary is not None:
            rc = self.dll.deflateSetDictionary(C.byref(strm), dictionary, len(dictionary))
            assert rc == Z_OK, rc
        src = C.create_string_buffer(bytes(data), len(data) + 1)
        outbuf = C.create_string_buffer(out_chunk)
        out = bytearray()
        pos = 0
        flushes = dict(flushes or {})
        base = C.addressof(src)
        while True:
            n = min(in_chunk, len(data) - pos)
            cut = min([o for o in flushes if pos < o <= pos + n], default=None)
            if cut is not None:
                n = cut - pos
            strm.next_in, strm.avail_in = base + pos, n
            pos += n
            flush = Z_FINISH if pos == len(data) else flushes.get(pos, Z_NO_FLUSH)
            while True:
                strm.next_out, strm.avail_out = C.addressof(outbuf), out_chunk
                rc = self.dll.deflate(C.byref(strm), flush)
                out += outbuf.raw[:out_chunk - strm.avail_out]
                if rc == Z_STREAM_END:
                    break
                if rc not in (Z_OK, Z_BUF_ERROR):
                    self.dll.deflateEnd(C.byref(strm))
                    return rc, bytes(out)
                if strm.avail_in == 0 and strm.avail_out != 0:
                    break
            if rc == Z_STREAM_END:
                break
        adler, tin, tout = strm.adler, strm.total_in, strm.total_out
        rc = self.dll.deflateEnd(C.byref(strm))
        assert tin == len(data) and tout == len(out), (tin, tout, len(out))
        self.last_adler = adler
        return rc, bytes(out)

    def inflate_stream(self, comp: bytes, wbits=15, in_chunk=1 << 16, out_chunk=1 << 16, flush=Z_NO_FLUSH,
                       dictionary=None):
        """inflateInit2 + inflate(...) loop + inflateEnd -> (last rc, output, msg, total_in)."""
        strm = z_stream()
        rc = self.dll.inflateInit2_(C.byref(strm), wbits, ZLIB_VERSION, C.sizeof(z_stream))
        if rc != Z_OK:
            return rc, b"", None, 0
        if dictionary is not None and wbits < 0:
            assert self.dll.inflateSetDictionary(C.byref(strm), dictionary, len(dictionary)) == Z_OK
        src = C.create_string_buffer(bytes(comp), len(comp) + 1)
        outbuf = C.create_string_buffer(out_chunk)
        out = bytearray()
        pos, base = 0, C.addressof(src)
        rc = Z_OK
        stall = 0
        while rc == Z_OK or rc == Z_BUF_ERROR:
            if strm.avail_in == 0 and pos < len(comp):
                n = min(in_chunk, len(comp) - pos)
                strm.next_in, strm.avail_in = base + pos, n
                pos += n
            strm.next_out, strm.avail_out = C.addressof(outbuf), out_chunk
            before = (strm.total_in, strm.total_out)
            rc = self.dll.inflate(C.byref(strm), flush)
            out += outbuf.raw[:out_chunk - strm.avail_out]
            if rc == Z_NEED_DICT and dictionary is not None:
                rc = self.dll.inflateSetDictionary(C.byref(strm), dictionary, len(dictionary))
                continue
            if (strm.total_in, strm.total_out) == before:
                stall += 1
                if stall > 2 or (pos >= len(comp) and strm.avail_in == 0):
                    break
            else:
                stall = 0
        msg, tin = strm.msg, strm.total_in
        self.last_adler = strm.adler
        self.dll.inflateEnd(C.byref(strm))
        return rc, bytes(out), (msg.decode() if msg else None), tin

    def synth(self, n: int, kind: int = 1, seed: int = 1, offset: int = 0):
        """numpy uint8 array of synthetic corpus bytes (SURVEY.md 8(d)); generated by libzbsynth.so, not by this library."""
        from . import synth as _synth
        return _synth.synth(n, kind, seed, offset)

    def profile(self, enable: bool) -> None:
        self.dll.zb200_profile(1 if enable else 0)

    def profile_report(self):
        """{kernel: (total_ms, launches)} since profile(True)."""
        buf = C.create_string_buffer(8192)
        self.dll.zb200_profile_report(buf, 8192)
        out = {}
        for item in buf.value.decode().split(";"):
            if "=" in item:
                k, v = item.split("=")
                ms, cnt = v.split(":")
                out[k] = (float(ms), int(cnt))
        return out

    def kernel_launches(self) -> int:
        return self.dll.zb200_kernel_launches()


_default: Optional[Lib] = None


def load(path: str = LIB_PATH) -> Lib:
    global _default
    if _default is None or _default.path != path:
        _default = Lib(path)
    return _default
