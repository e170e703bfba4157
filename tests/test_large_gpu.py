"""GPU: the 64-bit entry points past 4 GiB, against references that do not use this library -- the system zlib (run
incrementally, or decoding in pieces), the known plaintext, Python's gzip, and the plain-Python CRC-32 / Adler-32
algebra of zhelpers (checked against zlib in test_large_cpu.py).

Lengths are chosen at the edges where 32-bit arithmetic or a launch shape changes: 2^32 - 1 .. 2^32 + 5 bytes, the
checksum kernel's rounds (R = SMs x 32 warps x 1024 iterations x 512 bytes; seven rounds of CTAs pass the 1024 + 1
records one fold thread each can take), a compressed stream past 2^34 bytes (2^32 words of the decoder's bit reader),
gzip members whose ISIZE wraps.  Large buffers are built on the device from a pool of tiles of an odd length, so that
tile edges never line up with a chunk or CTA edge, and each tile exists once on the host: the CPU references stream
over the tile sequence.  Device memory in use is printed at every case (run with -s to see it)."""
import concurrent.futures as cf
import ctypes as C
import gzip
import random
import zlib

import numpy as np
import pytest

import zhelpers

pytestmark = pytest.mark.gpu

GiB = 1 << 30
TILE = (4 << 20) + 17
Z_OK, Z_BUF_ERROR = 0, -5
RAW, ZLIB, GZIP = 0, 1, 2                                      # ZB200_WRAP_*
WBITS = {RAW: -15, ZLIB: 15, GZIP: 31}
NOT_LAST = 1                                                    # ZB200_DEFLATE_NOT_LAST
_peak = [0]


def _torch():
    import torch
    return torch


def _mem(tag):
    torch = _torch()
    free, total = torch.cuda.mem_get_info()
    _peak[0] = max(_peak[0], total - free)
    print(f"[{tag}] device memory in use {(total - free) / GiB:.1f} GiB (peak so far {_peak[0] / GiB:.1f} GiB)")


def _release():
    import gc
    gc.collect()
    _torch().cuda.empty_cache()


def _round_bytes():
    return _torch().cuda.get_device_properties(0).multi_processor_count * 32 * 1024 * 512


def _vp(t, off=0):
    return C.c_void_p(t.data_ptr() + off)


def _u64(xs):
    return np.array(xs, dtype=np.uint64)


class Tiled:
    """n bytes: tiles of TILE bytes from a pool of synth() outputs, in a seeded order."""

    def __init__(self, lib, n, seed, kinds=(0, 1, 2, 3)):
        self.host = [lib.synth(TILE, kind=k, seed=s) for k in kinds for s in (seed, seed + 1, seed + 2)]
        rng = random.Random(seed)
        self.order = [rng.randrange(len(self.host)) for _ in range(-(-n // TILE))]
        self.n = n

    def pieces(self, a, b):
        i = a // TILE
        while a < b:
            t0 = i * TILE
            hi = min(TILE, b - t0)
            yield memoryview(self.host[self.order[i]])[a - t0:hi]
            a, i = t0 + hi, i + 1

    def device(self):
        torch = _torch()
        dtiles = [torch.from_numpy(t).cuda() for t in self.host]
        buf = torch.empty(self.n, dtype=torch.uint8, device="cuda")
        for i, t in enumerate(self.order):
            a = i * TILE
            b = min(self.n, a + TILE)
            buf[a:b].copy_(dtiles[t][:b - a])
        return buf

    def sums(self, marks):
        """{m: (crc32, adler32) of bytes [0, m)} in one pass of the system zlib (CRC and Adler on two threads)."""
        marks = sorted(set(marks) | {0})

        def run(fn, v):
            out, pos = {}, 0
            for m in marks:
                for p in self.pieces(pos, m):
                    v = fn(p, v)
                out[m], pos = v, m
            return out

        with cf.ThreadPoolExecutor(2) as ex:
            fc, fa = ex.submit(run, zlib.crc32, 0), ex.submit(run, zlib.adler32, 1)
            c, a = fc.result(), fa.result()
        return {m: (c[m], a[m]) for m in marks}


def _range_sums(S, a, b):
    """(crc32, adler32) of bytes [a, b) from the prefix sums S."""
    return (zhelpers.crc32_drop_prefix(S[b][0], S[a][0], b - a), zhelpers.adler32_drop_prefix(S[b][1], S[a][1], b - a))


class Expect:
    """Compares output arriving in pieces with expected plaintext arriving in (other) pieces."""

    def __init__(self, pieces):
        self.it, self.cur, self.pos = iter(pieces), np.empty(0, np.uint8), 0

    def take(self, out):
        got = np.frombuffer(out, dtype=np.uint8)
        i = 0
        while i < len(got):
            if not len(self.cur):
                self.cur = np.frombuffer(next(self.it), dtype=np.uint8)
            k = min(len(self.cur), len(got) - i)
            assert np.array_equal(got[i:i + k], self.cur[:k]), f"plaintext differs in [{self.pos}, {self.pos + k})"
            self.cur, i, self.pos = self.cur[k:], i + k, self.pos + k


def cpu_inflate(stream, wbits, expect_pieces, n, zdict=None, whole=True):
    """Decode `stream` with the system zlib in pieces; the output must be exactly the n bytes of expect_pieces, and
    (whole=True) the stream must end there with nothing after it."""
    d = zlib.decompressobj(wbits, zdict=zdict) if zdict is not None else zlib.decompressobj(wbits)
    e = Expect(expect_pieces)
    mv, pos = memoryview(stream), 0
    while not d.eof:
        if d.unconsumed_tail:
            buf = d.unconsumed_tail
        elif pos < len(mv):
            buf, pos = mv[pos:pos + (8 << 20)], pos + (8 << 20)
        else:
            break
        e.take(d.decompress(buf, 64 << 20))
    e.take(d.flush())
    assert e.pos == n, (e.pos, n)
    if whole:
        assert d.eof and not d.unused_data and not d.unconsumed_tail and pos >= len(mv)
    return True


def zeros_pieces(n, tiles=()):
    """n bytes of zeros with (offset, array) pieces placed in them, in pieces."""
    z = bytes(64 << 20)
    pos = 0
    for off, arr in list(tiles) + [(n, None)]:
        while pos < off:
            k = min(len(z), off - pos)
            yield memoryview(z)[:k]
            pos += k
        if arr is not None:
            yield memoryview(arr)
            pos += len(arr)


def deflate_dev(lib, src, n, level, wrap, src_off=0):
    torch = _torch()
    cap = lib.compress_bound(n) + 64
    dst = torch.empty(cap, dtype=torch.uint8, device="cuda")
    ol = C.c_size_t(cap)
    rc = lib.dll.zb200_deflate(_vp(src, src_off), n, _vp(dst), C.byref(ol), level, wrap, None)
    assert rc == Z_OK, (rc, lib.last_error())
    return dst[:ol.value]


def uncompress_dev(lib, z, cap):
    torch = _torch()
    out = torch.empty(max(cap, 1), dtype=torch.uint8, device="cuda")
    ol = C.c_ulong(cap)
    rc = lib.dll.uncompress(_vp(out), C.byref(ol), _vp(z), z.numel())
    return rc, out[:ol.value]


def inflate_batch_dev_arrays(lib, src, src_off, dst, dst_off, wrap):
    n = len(src_off) - 1
    so, do = _u64(src_off), _u64(dst_off)
    dl = np.zeros(max(n, 1), np.uint64)
    st = np.full(max(n, 1), -99, np.int32)
    rc = lib.dll.zb200_inflate_batch(_vp(src), so.ctypes.data, n, _vp(dst), do.ctypes.data, dl.ctypes.data, st.ctypes.data,
                                     wrap, None)
    assert rc == Z_OK, (rc, lib.last_error())
    return [int(x) for x in dl[:n]], [int(x) for x in st[:n]]


def checksum_dev(lib, ptr, n):
    torch = _torch()
    out = torch.zeros(2, dtype=torch.int32, device="cuda")
    rc = lib.dll.zb200_checksum_dev(C.c_void_p(ptr), n, _vp(out), None)
    assert rc == Z_OK, (n, rc, lib.last_error())
    torch.cuda.synchronize()
    v = out.cpu().numpy().view(np.uint32)
    return int(v[0]), int(v[1])


def checksum_host(lib, ptr, n):
    crc, adl = C.c_uint32(0), C.c_uint32(0)
    rc = lib.dll.zb200_checksum(C.c_void_p(ptr), n, C.byref(crc), C.byref(adl), None)
    assert rc == Z_OK, (n, rc, lib.last_error())
    return crc.value, adl.value


def _gzip_trailer(z):
    t = z[-8:].cpu().numpy().tobytes()
    return int.from_bytes(t[:4], "little"), int.from_bytes(t[4:], "little")


# ---- a compressed stream past 2^34 bytes: the decoder's 32-bit word indices --------------------------------------------

def _skewed_tile(j, n=GiB):
    """1 GiB of bytes with the top bit set one time in four (about 7.8 bits of entropy: dynamic blocks that barely
    compress), from seed j on the device."""
    torch = _torch()
    g = torch.Generator(device="cuda")
    g.manual_seed(7000 + j)
    x = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=g)
    y = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=g)
    return x & (y | 0x7F)


def test_stream_past_2_34_compressed_bytes(gpu_lib):
    """17 GiB of near-incompressible data as one zlib stream of more than 2^34 bytes (1 GiB shards chained by their
    32 KiB dictionaries, as a multi-GPU writer does), decoded by uncompress() in parallel segments."""
    torch = _torch()
    lib = gpu_lib
    ntile = 17
    _mem("2^34: start")
    cap = ntile * (lib.compress_bound(GiB) + 64) + 16
    z = torch.empty(cap, dtype=torch.uint8, device="cuda")
    z[0], z[1] = 0x78, 0x01
    pos, adler, starts, tail = 2, 1, [], None
    for j in range(ntile):
        t = _skewed_tile(j)
        ol, crc, adl = C.c_size_t(cap - pos - 4), C.c_uint32(0), C.c_uint32(0)
        dict_p, dict_n = (_vp(tail), tail.numel()) if tail is not None else (None, 0)
        rc = lib.dll.zb200_deflate_shard(_vp(t), GiB, dict_p, dict_n, _vp(z, pos), C.byref(ol), 1, RAW,
                                         NOT_LAST if j + 1 < ntile else 0, C.byref(crc), C.byref(adl), None)
        assert rc == Z_OK, (j, rc, lib.last_error())
        starts.append(pos)
        pos += ol.value
        adler = zhelpers.adler32_cat(adler, adl.value, GiB)
        tail = t[-32768:].clone()
        del t
    z[pos:pos + 4] = torch.tensor(list(adler.to_bytes(4, "big")), dtype=torch.uint8, device="cuda")
    zlen = pos + 4
    z = z[:zlen]
    n = ntile * GiB
    print(f"2^34: {n} bytes -> {zlen} bytes compressed")
    assert zlen > (1 << 34) + (64 << 20), zlen                 # well past the wrap of a 32-bit word index
    assert zlen < 0.995 * n                                    # Huffman-coded blocks, not stored ones
    _mem("2^34: stream built")

    # the system zlib on the first shard, the last one and the one that holds compressed byte 2^34, each from its own
    # start (the previous shard ends on a sync marker) with the 32 KiB in front of it as the dictionary
    k = max(j for j in range(ntile) if starts[j] <= (1 << 34))
    ends = starts[1:] + [zlen - 4]

    def host_tile(j):
        return _skewed_tile(j).cpu().numpy()

    jobs = []
    with cf.ThreadPoolExecutor(3) as ex:
        for j in sorted({0, k, ntile - 1}):
            seg = z[0 if j == 0 else starts[j]:ends[j]].cpu().numpy()
            zd = None if j == 0 else host_tile(j - 1)[-32768:].tobytes()
            jobs.append(ex.submit(cpu_inflate, seg, 15 if j == 0 else -15, [host_tile(j)], GiB, zd, j == ntile - 1))
        for f in jobs:
            assert f.result()
    _release()

    lib.profile(True)
    rc, out = uncompress_dev(lib, z, n)
    prof = lib.profile_report()
    lib.profile(False)
    _mem("2^34: decoded")
    assert rc == Z_OK, (rc, lib.last_error())
    assert out.numel() == n
    assert any("k_inflate_segments" in name for name in prof), sorted(prof)
    assert not any("k_inflate_stream" in name for name in prof), sorted(prof)     # not the one-warp fallback
    del z
    _release()
    for j in range(ntile):
        assert torch.equal(out[j * GiB:(j + 1) * GiB], _skewed_tile(j)), j
    del out
    _release()


# ---- one tiled buffer of about 24 GiB for the checksum, deflate and inflate cases -------------------------------------

def _lengths():
    R = _round_bytes()
    ls = [(1 << 32) - 1, 1 << 32, (1 << 32) + 1]
    for k in range(1, 7):
        ls += [k * R + 511, k * R + 512]
    ls.append(24 * GiB + 1001)
    return ls


ODD = 7                                                         # a base 7 bytes past an allocation: a 9-byte head
BATCH_SMALL = [1000, 77777]                                     # zb200_checksum_batch: small buffers, then one past 4 GiB
BIG_JOB = (1 << 32) + 5
DEFLATE_SIZES = ((1 << 32) - 1, 1 << 32, (1 << 32) + 5)


@pytest.fixture(scope="module")
def big(gpu_lib):
    ls = _lengths()
    n = max(ls) + 4096
    t = Tiled(gpu_lib, n, seed=21)
    marks = {m for L in ls for m in (L, ODD, ODD + L)}
    marks |= set(DEFLATE_SIZES)
    b0 = sum(BATCH_SMALL)
    marks |= {BATCH_SMALL[0], b0, b0 + BIG_JOB, BIG_JOB, BIG_JOB + 100000, BIG_JOB + 100000 + 777}
    sums = t.sums(marks)
    dev = t.device()
    _mem("tiled buffer")
    yield t, dev, sums
    del dev
    _release()


def test_checksum_dev_lengths_and_offsets(gpu_lib, big):
    t, dev, S = big
    for L in _lengths():
        for off in (0, ODD):
            want = _range_sums(S, off, off + L)
            assert checksum_dev(gpu_lib, dev.data_ptr() + off, L) == want, (L, off)


def test_checksum_pinned_and_pageable(gpu_lib, big):
    torch = _torch()
    t, dev, S = big
    R = _round_bytes()
    for L in ((1 << 32) + 1, 6 * R + 512):
        n = ODD + L
        for pinned in (True, False):
            host = torch.empty(n, dtype=torch.uint8, pin_memory=pinned)
            host.copy_(dev[:n])
            for off in (0, ODD):
                assert checksum_host(gpu_lib, host.data_ptr() + off, L) == _range_sums(S, off, off + L), (L, off, pinned)
            del host
            _mem(f"checksum from host (pinned {pinned}), {L} bytes")


def test_checksum_batch_past_4g(gpu_lib, big):
    t, dev, S = big
    off = np.cumsum([0] + BATCH_SMALL + [BIG_JOB]).astype(np.uint64)
    n = len(off) - 1
    crc, adl = np.zeros(n, np.uint32), np.zeros(n, np.uint32)
    rc = gpu_lib.dll.zb200_checksum_batch(_vp(dev), off.ctypes.data, n, crc.ctypes.data, adl.ctypes.data, None)
    assert rc == Z_OK, gpu_lib.last_error()
    for i in range(n):
        assert (int(crc[i]), int(adl[i])) == _range_sums(S, int(off[i]), int(off[i + 1])), i


def test_deflate_and_inflate_past_4g(gpu_lib, big):
    """zb200_deflate of 2^32 - 1, 2^32, 2^32 + 5 bytes in raw, zlib and gzip: trailers against the CPU sums, one stream
    per wrap decoded whole by the system zlib, every stream decoded by zb200_inflate_batch and the zlib ones by
    uncompress(); compress2 from pinned host memory."""
    torch = _torch()
    lib = gpu_lib
    t, dev, S = big
    full = {ZLIB: (1 << 32) - 1, GZIP: 1 << 32, RAW: (1 << 32) + 5}
    host_streams = {}
    for wrap in (RAW, ZLIB, GZIP):
        for n in DEFLATE_SIZES:
            z = deflate_dev(lib, dev, n, 1, wrap)
            assert z.numel() <= lib.compress_bound(n)
            crc, adl = S[n]
            if wrap == GZIP:
                assert _gzip_trailer(z) == (crc, n & 0xFFFFFFFF), n          # exactly 2^32 gives ISIZE 0
            elif wrap == ZLIB:
                assert int.from_bytes(z[-4:].cpu().numpy().tobytes(), "big") == adl, n
            if full[wrap] == n:
                host_streams[wrap] = (z.cpu().numpy(), n)
            out = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
            dl, st = inflate_batch_dev_arrays(lib, z, [0, z.numel()], out, [0, n + 64], wrap)
            assert st == [Z_OK] and dl == [n], (wrap, n, st, dl)
            assert torch.equal(out[:n], dev[:n]), (wrap, n)
            del out
            if wrap == ZLIB:
                rc, out = uncompress_dev(lib, z, n)
                assert rc == Z_OK and out.numel() == n, (n, rc, lib.last_error())
                assert torch.equal(out, dev[:n]), n
                del out
            del z
            _release()
            _mem(f"deflate wrap {wrap}, {n} bytes")
    with cf.ThreadPoolExecutor(3) as ex:
        fs = [ex.submit(cpu_inflate, s, WBITS[w], t.pieces(0, n), n) for w, (s, n) in host_streams.items()]
        for f in fs:
            assert f.result()
    del host_streams
    # compress2 from pinned host memory, decoded on the device against the plaintext
    n = (1 << 32) + 5
    src = torch.empty(n, dtype=torch.uint8, pin_memory=True)
    src.copy_(dev[:n])
    cap = lib.compress_bound(n)
    dst = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
    ol = C.c_ulong(cap)
    assert lib.dll.compress2(_vp(dst), C.byref(ol), _vp(src), n, 1) == Z_OK, lib.last_error()
    del src
    assert int.from_bytes(dst[ol.value - 4:ol.value].numpy().tobytes(), "big") == S[n][1]
    z = dst[:ol.value].cuda()
    del dst
    rc, out = uncompress_dev(lib, z, n)
    assert rc == Z_OK and torch.equal(out, dev[:n])
    del out, z
    _release()


def test_deflate_noise_past_4g(gpu_lib):
    """Incompressible input just past 4 GiB: stored blocks whose stream itself passes 2^32 bytes."""
    torch = _torch()
    lib = gpu_lib
    n = (1 << 32) + 1001
    g = torch.Generator(device="cuda")
    g.manual_seed(77)
    noise = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda", generator=g)
    z = deflate_dev(lib, noise, n, 1, ZLIB)
    assert (1 << 32) < z.numel() <= lib.compress_bound(n), z.numel()
    assert cpu_inflate(z.cpu().numpy(), 15, [noise.cpu().numpy()], n)
    rc, out = uncompress_dev(lib, z, n)
    assert rc == Z_OK and torch.equal(out, noise), (rc, lib.last_error())
    _mem("noise")
    del out, z, noise
    _release()


def test_deflate_batch_past_4g(gpu_lib, big):
    """A job of 2^32 + 5 bytes, then small jobs whose source and destination offsets lie past 2^32."""
    torch = _torch()
    lib = gpu_lib
    t, dev, S = big
    src_off = _u64([0, BIG_JOB, BIG_JOB + 100000, BIG_JOB + 100000 + 777])
    n = len(src_off) - 1
    caps = [lib.compress_bound(int(src_off[i + 1] - src_off[i])) + 16 for i in range(n)]
    dst_off = np.cumsum([0] + caps).astype(np.uint64)
    dst = torch.empty(int(dst_off[-1]) + 8, dtype=torch.uint8, device="cuda")
    dl, crc, adl = np.zeros(n, np.uint64), np.zeros(n, np.uint32), np.zeros(n, np.uint32)
    st = np.full(n, -99, np.int32)
    rc = lib.dll.zb200_deflate_batch(_vp(dev), src_off.ctypes.data, n, _vp(dst), dst_off.ctypes.data, dl.ctypes.data,
                                     crc.ctypes.data, adl.ctypes.data, st.ctypes.data, 1, ZLIB, None)
    assert rc == Z_OK and list(st) == [0] * n, (rc, list(st), lib.last_error())
    assert int(dst_off[1]) > 1 << 32
    streams = []
    for i in range(n):
        a, b = int(src_off[i]), int(src_off[i + 1])
        assert (int(crc[i]), int(adl[i])) == _range_sums(S, a, b), i
        streams.append((dst[int(dst_off[i]):int(dst_off[i]) + int(dl[i])].cpu().numpy(), a, b))
    del dst
    _release()
    with cf.ThreadPoolExecutor(n) as ex:
        fs = [ex.submit(cpu_inflate, s, 15, t.pieces(a, b), b - a) for s, a, b in streams]
        for f in fs:
            assert f.result()


def test_inflate_batch_dev_offsets_past_4g(gpu_lib, big):
    """zb200_inflate_batch_dev with small streams whose source and destination offsets lie beyond 2^32."""
    torch = _torch()
    lib = gpu_lib
    t, dev, S = big
    plains = [b"".join(bytes(p) for p in t.pieces(a, a + m)) for a, m in ((3, 100000), (TILE - 5, 70001), (9, 1))]
    streams = [zlib.compress(p, 6) for p in plains]
    base = (1 << 32) - 40
    src_off = [base]
    for s in streams:
        src_off.append(src_off[-1] + len(s))
    src = torch.zeros(src_off[-1] + 64, dtype=torch.uint8, device="cuda")
    for s, o in zip(streams, src_off):
        src[o:o + len(s)] = torch.frombuffer(bytearray(s), dtype=torch.uint8).cuda()
    dst_off = [(1 << 32) + 11]
    for p in plains:
        dst_off.append(dst_off[-1] + len(p) + 5)
    dst = torch.zeros(dst_off[-1] + 64, dtype=torch.uint8, device="cuda")
    n = len(streams)
    d_src_off = torch.tensor(src_off, dtype=torch.int64, device="cuda")
    d_dst_off = torch.tensor(dst_off, dtype=torch.int64, device="cuda")
    d_len = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_st = torch.full((n,), -99, dtype=torch.int32, device="cuda")
    lib.inflate_batch_dev(src.data_ptr(), d_src_off.data_ptr(), n, dst.data_ptr(), d_dst_off.data_ptr(), d_len.data_ptr(),
                          d_st.data_ptr(), ZLIB)
    torch.cuda.synchronize()
    assert d_st.cpu().tolist() == [Z_OK] * n, lib.last_error()
    assert d_len.cpu().tolist() == [len(p) for p in plains]
    for p, o in zip(plains, dst_off):
        assert dst[o:o + len(p)].cpu().numpy().tobytes() == p
    del src, dst
    _release()


def test_block_finder_stream_past_4g(gpu_lib):
    """A system-zlib stream (no sync markers: the decoder finds block starts itself) of more than 4 GiB of output and
    more than 512 MiB of input, i.e. bit positions past 2^32: uncompress() and zb200_inflate_batch."""
    torch = _torch()
    lib = gpu_lib
    n = (1 << 32) + 12345
    t = Tiled(lib, n, seed=41, kinds=(0, 1, 3))
    c = zlib.compressobj(1)
    parts = [c.compress(p) for p in t.pieces(0, n)]
    parts.append(c.flush())
    zs = b"".join(parts)
    del parts
    assert len(zs) > (1 << 29), len(zs)
    dev = t.device()
    z = torch.frombuffer(bytearray(zs), dtype=torch.uint8).cuda()
    del zs
    _mem("block finder")
    rc, out = uncompress_dev(lib, z, n)
    assert rc == Z_OK and torch.equal(out, dev), (rc, lib.last_error())
    del out
    out = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    dl, st = inflate_batch_dev_arrays(lib, z, [0, z.numel()], out, [0, n + 64], ZLIB)
    assert st == [Z_OK] and dl == [n]
    assert torch.equal(out[:n], dev)
    del out, z, dev
    _release()


# ---- at and past six rounds of the checksum kernel: every call that checksums a whole buffer ---------------------------

def test_six_rounds_plus_one_unit(gpu_lib):
    """6R + 512 bytes and more (seven rounds of CTAs): checksum, deflate, uncompress() and a gzip member.  Mostly zeros,
    with a few tiles spread through, checked by the system zlib."""
    torch = _torch()
    lib = gpu_lib
    R = _round_bytes()
    n = 6 * R + 512 + 3
    tiles = [lib.synth(TILE, kind=k, seed=50 + k) for k in (0, 1, 2)]
    place = [(5, tiles[0]), (n // 3 + 1, tiles[1]), (n - TILE - 9, tiles[2])]
    plain = torch.zeros(n, dtype=torch.uint8, device="cuda")
    for o, a in place:
        plain[o:o + len(a)] = torch.from_numpy(a).cuda()
    crc = adl = None
    for p in zeros_pieces(n, place):
        crc = zlib.crc32(p, crc or 0)
        adl = zlib.adler32(p, 1 if adl is None else adl)
    assert checksum_dev(lib, plain.data_ptr(), n) == (crc, adl)
    _mem("six rounds: plaintext")

    z = deflate_dev(lib, plain, n, 1, ZLIB)
    zh = z.cpu().numpy()
    assert cpu_inflate(zh, 15, zeros_pieces(n, place), n)
    rc, out = uncompress_dev(lib, z, n)
    assert rc == Z_OK and out.numel() == n, (rc, lib.last_error())
    assert torch.equal(out, plain)
    del out, z
    _release()
    _mem("six rounds: uncompress")

    # one gzip member of zeros
    plain.zero_()
    zg = deflate_dev(lib, plain, n, 1, GZIP)
    assert _gzip_trailer(zg) == (_zeros_crc(n), n & 0xFFFFFFFF)
    out = torch.empty(n, dtype=torch.uint8, device="cuda")
    ol, members = C.c_size_t(n), C.c_size_t(0)
    rc = lib.dll.zb200_gunzip(_vp(zg), zg.numel(), _vp(out), C.byref(ol), C.byref(members), None)
    assert rc == Z_OK and ol.value == n and members.value == 1, (rc, lib.last_error())
    assert _all_zero(out)
    del out, zg, plain
    _release()


def _all_zero(t):
    """No nonzero byte in t, checked 1 GiB at a time (a reduction over the whole tensor would allocate a temporary of
    several times its size)."""
    return not any(bool(t[i:i + GiB].any()) for i in range(0, t.numel(), GiB))


def _zeros_crc(n):
    c, z = 0, bytes(64 << 20)
    while n:
        k = min(n, len(z))
        c = zlib.crc32(memoryview(z)[:k], c)
        n -= k
    return c


def test_gunzip_members_at_and_past_4g(gpu_lib, big):
    """[1 MiB member, member of exactly 2^32 bytes (ISIZE 0), member of 2^32 + 3 zeros, 1 MiB member] in one file."""
    torch = _torch()
    lib = gpu_lib
    t, dev, S = big
    m = 1 << 20
    zeros = torch.zeros((1 << 32) + 3, dtype=torch.uint8, device="cuda")
    parts = [(dev, 10, m), (dev, 0, 1 << 32), (zeros, 0, zeros.numel()), (dev, 5000, m + 1)]
    members = [deflate_dev(lib, src, ln, 1, GZIP, src_off=o) for src, o, ln in parts]
    assert _gzip_trailer(members[1]) == (S[1 << 32][0], 0)
    assert _gzip_trailer(members[2]) == (_zeros_crc(zeros.numel()), 3)
    gz = torch.cat(members)
    total = sum(ln for _, _, ln in parts)
    out = torch.empty(total, dtype=torch.uint8, device="cuda")
    ol, cnt = C.c_size_t(total), C.c_size_t(0)
    rc = lib.dll.zb200_gunzip(_vp(gz), gz.numel(), _vp(out), C.byref(ol), C.byref(cnt), None)
    assert rc == Z_OK and ol.value == total and cnt.value == 4, (rc, ol.value, cnt.value, lib.last_error())
    pos = 0
    for src, o, ln in parts:
        assert torch.equal(out[pos:pos + ln], src[o:o + ln]), pos
        pos += ln
    ol = C.c_size_t(total - 1)
    rc = lib.dll.zb200_gunzip(_vp(gz), gz.numel(), _vp(out), C.byref(ol), C.byref(cnt), None)
    assert rc == Z_BUF_ERROR, rc
    _mem("gunzip")
    # Python's gzip accepts the members it can afford to decode here (the 2^32-byte member is the stream that
    # test_deflate_and_inflate_past_4g decodes with the system zlib)
    for i in (0, 2, 3):
        src, o, ln = parts[i]
        got = gzip.decompress(members[i].cpu().numpy().tobytes())
        assert len(got) == ln
        if i == 2:
            assert got.count(0) == ln
        else:
            assert got == src[o:o + ln].cpu().numpy().tobytes()
    del out, gz, members, zeros
    _release()
    _mem("end of file")
