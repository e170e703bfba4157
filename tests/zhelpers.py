"""Test-side handles on the CPU oracle (oracle/libzoracle.so) and on the compiled
reference (oracle/_ref/libzref.so).  Test infrastructure only."""
import ctypes as C
import os
import random
import subprocess

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
ORACLE_PATH = os.path.join(ORACLE_DIR, "libzoracle.so")
REF_PATH = os.path.join(ORACLE_DIR, "_ref", "libzref.so")
GOLDEN = os.path.join(ROOT, "tests", "golden")


def build_oracle():
    src = os.path.join(ORACLE_DIR, "zoracle.c")
    if (not os.path.exists(ORACLE_PATH)) or os.path.getmtime(ORACLE_PATH) < os.path.getmtime(src):
        subprocess.check_call(["make", "-s", "-C", ORACLE_DIR, ORACLE_PATH])


class Oracle:
    def __init__(self):
        build_oracle()
        d = self.dll = C.CDLL(ORACLE_PATH, mode=os.RTLD_LOCAL)
        u32, sz, cp = C.c_uint32, C.c_size_t, C.c_char_p
        d.zo_crc32.restype, d.zo_crc32.argtypes = u32, [u32, C.c_void_p, sz]
        d.zo_adler32.restype, d.zo_adler32.argtypes = u32, [u32, C.c_void_p, sz]
        d.zo_crc32_combine.restype, d.zo_crc32_combine.argtypes = u32, [u32, u32, C.c_int64]
        d.zo_adler32_combine.restype, d.zo_adler32_combine.argtypes = u32, [u32, u32, C.c_int64]
        d.zo_compress_bound.restype, d.zo_compress_bound.argtypes = sz, [sz]
        d.zo_deflate.restype = C.c_int
        d.zo_deflate.argtypes = [C.c_void_p, sz, C.c_void_p, sz, C.POINTER(sz), C.c_int, C.c_int]
        d.zo_inflate.restype = C.c_int
        d.zo_inflate.argtypes = [C.c_void_p, sz, C.c_void_p, sz, C.POINTER(sz), C.POINTER(sz), C.c_int]
        d.zo_last_msg.restype = cp
        d.zo_last_max_dist.restype, d.zo_last_max_dist.argtypes = sz, []

    @staticmethod
    def _p(data):
        if data is None:
            return None
        if hasattr(data, "ctypes"):
            return C.c_void_p(data.ctypes.data)
        return C.cast(C.c_char_p(bytes(data)) if not isinstance(data, bytes) else C.c_char_p(data), C.c_void_p)

    def crc32(self, data, value=0):
        return self.dll.zo_crc32(value, self._p(data), len(data) if data is not None else 0)

    def adler32(self, data, value=1):
        return self.dll.zo_adler32(value, self._p(data), len(data) if data is not None else 0)

    def crc32_combine(self, a, b, n):
        return self.dll.zo_crc32_combine(a, b, n)

    def adler32_combine(self, a, b, n):
        return self.dll.zo_adler32_combine(a, b, n)

    def compress_bound(self, n):
        return self.dll.zo_compress_bound(n)

    def deflate(self, data, level=6, wrap=1):
        n = len(data)
        cap = self.compress_bound(n) + 64
        out = C.create_string_buffer(cap)
        ol = C.c_size_t(0)
        rc = self.dll.zo_deflate(self._p(data), n, out, cap, C.byref(ol), level, wrap)
        assert rc == 0, rc
        return out.raw[:ol.value]

    def inflate(self, comp, cap, wrap=1):
        """(rc, output bytes, consumed input bytes)"""
        out = C.create_string_buffer(max(cap, 1))
        ol, iu = C.c_size_t(0), C.c_size_t(0)
        rc = self.dll.zo_inflate(self._p(comp), len(comp), out, cap, C.byref(ol), C.byref(iu), wrap)
        return rc, out.raw[:ol.value], iu.value

    def last_msg(self):
        m = self.dll.zo_last_msg()
        return m.decode() if m else None

    def last_max_dist(self):
        """The largest distance the last inflate() decoded."""
        return self.dll.zo_last_max_dist()


class Ref:
    """ctypes view of the reference's own zlib.h ABI (oracle/_ref/libzref.so)."""

    def __init__(self):
        d = self.dll = C.CDLL(REF_PATH, mode=os.RTLD_LOCAL | os.RTLD_DEEPBIND)
        ul = C.c_ulong
        d.crc32.restype, d.crc32.argtypes = ul, [ul, C.c_void_p, C.c_uint]
        d.adler32.restype, d.adler32.argtypes = ul, [ul, C.c_void_p, C.c_uint]
        d.crc32_combine.restype, d.crc32_combine.argtypes = ul, [ul, ul, C.c_long]
        d.adler32_combine.restype, d.adler32_combine.argtypes = ul, [ul, ul, C.c_long]
        d.compress2.restype, d.compress2.argtypes = C.c_int, [C.c_void_p, C.POINTER(ul), C.c_void_p, ul, C.c_int]
        d.uncompress.restype, d.uncompress.argtypes = C.c_int, [C.c_void_p, C.POINTER(ul), C.c_void_p, ul]
        d.compressBound.restype, d.compressBound.argtypes = ul, [ul]
        d.zlibVersion.restype = C.c_char_p
        d.zlibCompileFlags.restype = ul
        d.get_crc_table.restype = C.POINTER(ul)

    _p = staticmethod(Oracle._p)

    def crc32(self, data, value=0):
        return self.dll.crc32(value, self._p(data), len(data) if data is not None else 0)

    def adler32(self, data, value=1):
        return self.dll.adler32(value, self._p(data), len(data) if data is not None else 0)

    def compress2(self, data, level=6):
        n = len(data)
        cap = self.dll.compressBound(n)
        out = C.create_string_buffer(cap)
        ol = C.c_ulong(cap)
        rc = self.dll.compress2(out, C.byref(ol), self._p(data), n, level)
        assert rc == 0, rc
        return out.raw[:ol.value]

    def uncompress(self, comp, cap):
        out = C.create_string_buffer(max(cap, 1))
        ol = C.c_ulong(cap)
        rc = self.dll.uncompress(out, C.byref(ol), self._p(comp), len(comp))
        return rc, (out.raw[:ol.value] if rc == 0 else b"")

    def deflate_stream(self, data, level=6, wbits=15, strategy=0):
        """deflateInit2 + deflate(Z_FINISH) + deflateEnd of the reference itself (for strategies and window sizes)."""
        from zlib_b200.binding import z_stream, ZLIB_VERSION
        d = self.dll
        d.deflateInit2_.restype = C.c_int
        d.deflateInit2_.argtypes = [C.POINTER(z_stream), C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_char_p, C.c_int]
        d.deflate.restype, d.deflate.argtypes = C.c_int, [C.POINTER(z_stream), C.c_int]
        d.deflateEnd.restype, d.deflateEnd.argtypes = C.c_int, [C.POINTER(z_stream)]
        strm = z_stream()
        assert d.deflateInit2_(C.byref(strm), level, 8, wbits, 8, strategy, ZLIB_VERSION, C.sizeof(z_stream)) == 0
        n = len(data)
        cap = n + (n >> 3) + 1024
        src = C.create_string_buffer(bytes(data), n + 1)
        out = C.create_string_buffer(cap)
        strm.next_in, strm.avail_in = C.addressof(src), n
        strm.next_out, strm.avail_out = C.addressof(out), cap
        assert d.deflate(C.byref(strm), 4) == 1
        z = out.raw[:strm.total_out]
        assert d.deflateEnd(C.byref(strm)) == 0
        return z


class OracleAsReference:
    """The calls of Ref that the GPU gates use, answered by the oracle (system zlib for deflate strategies)."""

    def __init__(self, oracle):
        self.oracle = oracle

    def compress2(self, data, level=6):
        return self.oracle.deflate(data, level)

    def uncompress(self, comp, cap):
        rc, out, _ = self.oracle.inflate(comp, cap)
        return rc, (out if rc == 0 else b"")

    def deflate_stream(self, data, level=6, wbits=15, strategy=0):
        import zlib
        co = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strategy)
        return co.compress(bytes(data)) + co.flush()


def unzip_with_oracle(path, oracle):
    """{name: bytes} of every member of the ZIP archive at `path`: the central directory as Python's zipfile reads it,
    each member's data found through its own local header and decoded by the oracle's raw inflate; the decoded length
    and CRC-32 must be the ones the directory records."""
    import struct
    import zipfile
    blob = open(path, "rb").read()
    out = {}
    for info in zipfile.ZipFile(path).infolist():
        sig = struct.unpack_from("<I", blob, info.header_offset)[0]
        name_len, extra_len = struct.unpack_from("<HH", blob, info.header_offset + 26)
        assert sig == 0x04034B50, (info.filename, hex(sig))
        start = info.header_offset + 30 + name_len + extra_len
        raw = blob[start:start + info.compress_size]
        if info.compress_type == zipfile.ZIP_DEFLATED:
            rc, data, used = oracle.inflate(raw, info.file_size, 0)
            assert rc == 0 and used == len(raw), (info.filename, rc, oracle.last_msg())
        else:
            assert info.compress_type == zipfile.ZIP_STORED, (info.filename, info.compress_type)
            data = raw
        assert len(data) == info.file_size and oracle.crc32(data) == info.CRC, info.filename
        out[info.filename] = data
    return out


def corpus(kind, n, seed=0):
    """Small deterministic test inputs (pure Python, independent of the product's generator)."""
    rng = random.Random(seed * 1000003 + kind * 7919 + n)
    if kind == 0:
        return rng.randbytes(n)
    if kind == 1:
        words = [bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz") for _ in range(rng.randint(2, 10))) for _ in range(300)]
        out = bytearray()
        while len(out) < n:
            out += rng.choice(words) + (b" " if rng.random() < 0.9 else b"\n")
        return bytes(out[:n])
    if kind == 2:
        return bytes(n)
    if kind == 3:
        out = bytearray()
        i = 0
        while len(out) < n:
            out += i.to_bytes(4, "little") + rng.randint(0, 255).to_bytes(4, "little") + bytes(4) + rng.getrandbits(32).to_bytes(4, "little")
            i += 1
        return bytes(out[:n])
    if kind == 4:
        return bytes(rng.choice(b"ab") for _ in range(n))
    raise ValueError(kind)


# ---- CRC-32 / Adler-32 algebra in plain Python: references for checksums of buffers too long to hold on the host ----
# Reflected CRC-32 polynomial arithmetic as RFC 1952 defines the CRC; independent of every library under test.
CRC_POLY = 0xEDB88320
ADLER_BASE = 65521


def _gf2_mul(a, b):
    """a * b mod P, both in the reflected representation (bit 31 = x^0)."""
    p = 0
    for i in range(31, -1, -1):
        if (a >> i) & 1:
            p ^= b
        b = (b >> 1) ^ CRC_POLY if b & 1 else b >> 1
    return p


def _x8n(n):
    """x^(8 n) mod P by square and multiply."""
    acc, sq = 1 << 31, 1 << 23                   # x^0, x^8
    while n:
        if n & 1:
            acc = _gf2_mul(acc, sq)
        sq = _gf2_mul(sq, sq)
        n >>= 1
    return acc


def crc32_cat(c1, c2, len2):
    """CRC-32 of A || B from crc(A), crc(B) and len(B)."""
    return _gf2_mul(c1, _x8n(len2)) ^ c2


def crc32_drop_prefix(c12, c1, len2):
    """CRC-32 of B from crc(A || B), crc(A) and len(B)."""
    return c12 ^ _gf2_mul(c1, _x8n(len2))


def adler32_cat(a1, a2, len2):
    s1 = ((a1 & 0xFFFF) + (a2 & 0xFFFF) - 1) % ADLER_BASE
    s2 = ((a1 >> 16) + (a2 >> 16) + len2 * ((a1 & 0xFFFF) - 1)) % ADLER_BASE
    return (s2 << 16) | s1


def adler32_drop_prefix(a12, a1, len2):
    s1 = ((a12 & 0xFFFF) - (a1 & 0xFFFF) + 1) % ADLER_BASE
    s2 = ((a12 >> 16) - (a1 >> 16) - len2 * ((a1 & 0xFFFF) - 1)) % ADLER_BASE
    return (s2 << 16) | s1
