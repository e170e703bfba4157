"""GPU: regression cases for the round-1 review findings.

  * the lean decode loop must meet its input limit wherever its word index moves (one-bit length and distance codes at
    an odd bit phase never crossed a word at the top of the loop): long runs decoded through small feeds, and streams
    truncated inside a block through uncompress() / zb200_inflate_batch();
  * deflateInit2 / inflateInit2 with windowBits below 15: match distances stay inside the declared window
    (qcsrc/deflate.c:270-279, h/deflate.h:276) and a stream declaring a larger window than the caller opened is refused
    (qcsrc/inflate.c:622).
"""
import random
import zlib

import pytest

import zhelpers
from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu


def _runs(n, seed):
    """Byte runs of a few values: the reference's dynamic blocks for these use 1- and 2-bit codes."""
    rng = random.Random(seed)
    out = bytearray()
    while len(out) < n:
        out += bytes([rng.choice(b"\x00\x00\x00a")]) * rng.choice([1, 3, 258, 600, 5000, 70000])
    return bytes(out[:n])


def test_runs_through_small_feeds(gpu_lib, oracle, reference_codec):
    for seed, n in ((1, 1 << 20), (2, 3 << 20), (3, 300000)):
        data = _runs(n, seed) if seed != 2 else bytes(n)
        for z in (reference_codec.compress2(data, 9), oracle.deflate(data, 6), zlib.compress(data, 1)):
            for in_chunk in (64, 77, 100):
                rc, out, msg, tin = gpu_lib.inflate_stream(z, 15, in_chunk, 1 << 20)
                assert rc == zb.Z_STREAM_END and msg is None, (seed, in_chunk, rc, msg)
                assert tin == len(z) and out == data, (seed, in_chunk, tin, len(z))
            rc, out = gpu_lib.uncompress(z, len(data))
            assert rc == zb.Z_OK and out == data


def test_truncated_inside_a_block(gpu_lib, oracle):
    rng = random.Random(5)
    cases = []
    for seed in range(6):
        data = _runs(200000 + 1000 * seed, 10 + seed) if seed % 2 == 0 else zhelpers.corpus(1, 150000, seed)
        z = oracle.deflate(data, 6)
        for _ in range(12):
            cut = rng.randrange(3, len(z) - 1)
            cases.append((z[:cut], len(data)))
    outs, st = gpu_lib.inflate_batch([c for c, _ in cases], [n for _, n in cases])
    for (c, n), s in zip(cases, st):
        want, _, _ = oracle.inflate(c, n)
        assert s == want == zb.Z_DATA_ERROR, (len(c), s, want)     # uncompr.c:53-55: out of input is a data error
        rc, _ = gpu_lib.uncompress(c, n)
        assert rc == want


@pytest.mark.parametrize("wbits", [8, 9, 10, 12, 14])
def test_small_window_deflate(gpu_lib, oracle, wbits):
    data = zhelpers.corpus(1, 400000, wbits) + zhelpers.corpus(3, 100000, wbits)
    eff = max(wbits, 9)                                            # deflate.c:270
    for level in (1, 6):
        rc, z = gpu_lib.deflate_stream(data, level, wbits, 1 << 20, 1 << 20)
        assert rc == zb.Z_OK
        assert (z[0] >> 4) + 8 == eff                              # CINFO
        assert zlib.decompressobj(eff).decompress(z) == data       # system zlib sizes its window from the caller's wbits
        rc2, out, _ = oracle.inflate(z, len(data))
        assert rc2 == 0 and out == data
        rc, raw = gpu_lib.deflate_stream(data, level, -wbits, 1 << 20, 1 << 20)
        assert rc == zb.Z_OK and zlib.decompressobj(-eff).decompress(raw) == data
        rc, gz = gpu_lib.deflate_stream(data, level, 16 + wbits, 1 << 20, 1 << 20)
        assert rc == zb.Z_OK and zlib.decompressobj(16 + eff).decompress(gz) == data
    # a dictionary longer than the window: only what the window can reach may be used
    dictionary = zhelpers.corpus(1, 40000, 99)
    rc, z = gpu_lib.deflate_stream(dictionary[-3000:] + data[:50000], 6, wbits, 1 << 20, 1 << 20, dictionary=dictionary)
    assert rc == zb.Z_OK
    d = zlib.decompressobj(eff, zdict=dictionary)
    assert d.decompress(z) == dictionary[-3000:] + data[:50000]


def test_inflate_refuses_a_larger_window_than_opened(gpu_lib, oracle):
    data = zhelpers.corpus(1, 100000, 4)
    z15 = oracle.deflate(data, 6)                                  # CINFO 7
    rc, out, msg, _ = gpu_lib.inflate_stream(z15, 12, 4096, 4096)
    assert rc == zb.Z_DATA_ERROR and msg == "invalid window size"
    rc, out, msg, _ = gpu_lib.inflate_stream(z15, 15, 4096, 4096)
    assert rc == zb.Z_STREAM_END and out == data
    rc, z10 = gpu_lib.deflate_stream(data, 6, 10, 1 << 20, 1 << 20)
    assert rc == zb.Z_OK
    for w in (10, 12, 15):
        rc, out, msg, _ = gpu_lib.inflate_stream(z10, w, 4096, 4096)
        assert rc == zb.Z_STREAM_END and out == data, (w, rc, msg)
    rc, out, msg, _ = gpu_lib.inflate_stream(z10, 9, 4096, 4096)
    assert rc == zb.Z_DATA_ERROR and msg == "invalid window size"


def test_partial_flush_and_prime(gpu_lib, oracle):
    """Z_PARTIAL_FLUSH ends on the ten bits of an empty static block and leaves the stream unaligned (trees.c:892), it is
    not served as a sync flush any more; deflatePrime (deflate.c:404-414) puts bits in front of the first block."""
    import ctypes as C
    rng = random.Random(77)
    data = zhelpers.corpus(1, 300000, 12) + zhelpers.corpus(3, 50000, 13)
    marker = b"\x00\x00\xff\xff"
    for level in (1, 6, 0):
        cuts = sorted(rng.sample(range(1000, len(data) - 1000), 9))
        flushes = {c: zb.Z_PARTIAL_FLUSH for c in cuts}
        flushes[cuts[4]] = zb.Z_SYNC_FLUSH
        rc, z = gpu_lib.deflate_stream(data, level, -15, 1 << 20, 1 << 20, flushes)
        assert rc == zb.Z_OK
        assert zlib.decompress(z, -15) == data
        rc2, out, used = oracle.inflate(z, len(data), 0)
        assert rc2 == 0 and out == data and used == len(z)
        if level:
            assert z.count(marker) <= 2, z.count(marker)           # the sync flush (and chance), not one per partial flush
        rc, zs = gpu_lib.deflate_stream(data, level, 15, 1 << 20, 1 << 20, {c: zb.Z_SYNC_FLUSH for c in cuts})
        assert rc == zb.Z_OK and zs.count(marker) >= 9 and zlib.decompress(zs) == data
    # every alignment: partial flushes after inputs of 1..40 bytes leave 0..7 bits pending each time
    small = zhelpers.corpus(1, 4000, 14)
    flushes = {i * 97 + (i % 40) + 1: zb.Z_PARTIAL_FLUSH for i in range(1, 40)}
    rc, z = gpu_lib.deflate_stream(small, 6, 15, 1 << 20, 1 << 20, flushes)
    assert rc == zb.Z_OK and zlib.decompress(z) == small
    # deflatePrime: ten primed bits that happen to be an empty static block keep a raw stream decodable
    strm = zb.z_stream()
    assert gpu_lib.dll.deflateInit2_(C.byref(strm), 6, zb.Z_DEFLATED, -15, 8, 0, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
    assert gpu_lib.dll.deflatePrime(C.byref(strm), 17, 0) == zb.Z_STREAM_ERROR
    assert gpu_lib.dll.deflatePrime(C.byref(strm), 10, 2) == zb.Z_OK
    src = C.create_string_buffer(data, len(data))
    dst = C.create_string_buffer(len(data) + 1000)
    strm.next_in, strm.avail_in = C.addressof(src), len(data)
    strm.next_out, strm.avail_out = C.addressof(dst), len(data) + 1000
    assert gpu_lib.dll.deflate(C.byref(strm), zb.Z_FINISH) == zb.Z_STREAM_END
    raw = dst.raw[:strm.total_out]
    assert gpu_lib.dll.deflateEnd(C.byref(strm)) == zb.Z_OK
    assert raw[0] == 0x02 and zlib.decompress(raw, -15) == data     # 010 + seven zero bits come first
    # deflateParams mid-stream (deflate.c:416-451): what was gathered leaves under the old level with a partial flush
    strm = zb.z_stream()
    assert gpu_lib.dll.deflateInit_(C.byref(strm), 9, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
    half = len(data) // 2
    strm.next_in, strm.avail_in = C.addressof(src), half
    strm.next_out, strm.avail_out = C.addressof(dst), len(data) + 1000
    assert gpu_lib.dll.deflate(C.byref(strm), zb.Z_NO_FLUSH) == zb.Z_OK
    assert gpu_lib.dll.deflateParams(C.byref(strm), 0, 0) == zb.Z_OK
    strm.next_in, strm.avail_in = C.addressof(src) + half, 1000
    assert gpu_lib.dll.deflate(C.byref(strm), zb.Z_NO_FLUSH) == zb.Z_OK
    assert gpu_lib.dll.deflateParams(C.byref(strm), 1, 0) == zb.Z_OK
    strm.next_in, strm.avail_in = C.addressof(src) + half + 1000, len(data) - half - 1000
    assert gpu_lib.dll.deflate(C.byref(strm), zb.Z_FINISH) == zb.Z_STREAM_END
    z = dst.raw[:strm.total_out]
    gpu_lib.dll.deflateEnd(C.byref(strm))
    assert zlib.decompress(z) == data
    strm = zb.z_stream()
    assert gpu_lib.dll.deflateInit_(C.byref(strm), 6, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
    strm.next_in, strm.avail_in = C.addressof(src), 5000
    strm.next_out, strm.avail_out = C.addressof(dst), 100000
    assert gpu_lib.dll.deflate(C.byref(strm), zb.Z_NO_FLUSH) == zb.Z_OK
    strm.avail_out = 0
    assert gpu_lib.dll.deflateParams(C.byref(strm), 1, 0) == zb.Z_BUF_ERROR     # deflate.c:440 via deflate(): no room for the flush
    gpu_lib.dll.deflateEnd(C.byref(strm))
