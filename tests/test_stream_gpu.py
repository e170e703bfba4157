"""GPU: the streaming zlib.h ABI (deflate/inflate with arbitrary buffer sizes, flushes, dictionaries) and the
reference's own callers -- example.c, minizip, miniunz -- linked against libzb200.so."""
import os
import random
import subprocess
import zlib

import pytest

import zhelpers
from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu
REFDIR = os.path.join(zhelpers.ORACLE_DIR, "_ref")

EXAMPLE_LINES = [  # what the reference's own build prints (SURVEY.md section 4)
    "uncompress(): hello, hello!", "gzread(): hello, hello!", "gzgets() after gzseek:  hello!",
    "inflate(): hello, hello!", "large_inflate(): OK", "after inflateSync(): hello, hello!",
    "inflate with dictionary: hello, hello!"]


def test_streaming_deflate_buffer_sizes(gpu_lib, oracle):
    rng = random.Random(1)
    for t in range(12):
        data = zhelpers.corpus(rng.randrange(5), rng.choice([0, 1, 14, 5000, 70000, 300000]), t)
        for in_chunk, out_chunk in ((1, 1), (7, 13), (4096, 16384), (1 << 20, 1 << 20)):
            if len(data) > 6000 and in_chunk < 4096:
                continue
            for wbits in (15, -15, 31):
                rc, z = gpu_lib.deflate_stream(data, rng.choice([1, 6]), wbits, in_chunk, out_chunk)
                assert rc == zb.Z_OK, (t, in_chunk, wbits, rc)
                assert zlib.decompress(z, wbits) == data
                if wbits == 15:
                    assert gpu_lib.last_adler == oracle.adler32(data)
                    rc2, out, used = oracle.inflate(z, len(data))
                    assert rc2 == 0 and out == data and used == len(z)


def test_flush_points_and_full_flush(gpu_lib, oracle):
    data = zhelpers.corpus(1, 200000, 9)
    flushes = {3: zb.Z_FULL_FLUSH, 1000: zb.Z_SYNC_FLUSH, 70000: zb.Z_PARTIAL_FLUSH, 150000: zb.Z_FULL_FLUSH}
    rc, z = gpu_lib.deflate_stream(data, 6, 15, 1 << 20, 1 << 20, flushes)
    assert rc == zb.Z_OK
    assert z.count(b"\x00\x00\xff\xff") >= 3                  # SYNC and FULL flushes leave the empty stored block (PARTIAL an empty static one)
    rc2, out, _ = oracle.inflate(z, len(data))
    assert rc2 == 0 and out == data
    # after a full flush the tail is decodable on its own as raw deflate (history forgotten)
    d = zlib.decompressobj(-15)
    i = z.index(b"\x00\x00\xff\xff") + 4
    assert (d.decompress(z[i:-4]) + d.flush()) == data[3:]


def test_streaming_inflate_buffer_sizes(gpu_lib, oracle):
    rng = random.Random(2)
    for t in range(10):
        data = zhelpers.corpus(rng.randrange(5), rng.choice([0, 1, 14, 5000, 70000, 400000]), 40 + t)
        z = oracle.deflate(data, rng.choice([0, 1, 6, 9]))
        for in_chunk, out_chunk in ((1, 1), (5, 3), (16384, 8192), (1 << 20, 1 << 16), (100, 1 << 20)):
            if len(data) > 6000 and min(in_chunk, out_chunk) < 100:
                continue
            rc, out, msg, tin = gpu_lib.inflate_stream(z, 15, in_chunk, out_chunk)
            assert rc == zb.Z_STREAM_END and out == data and msg is None and tin == len(z), (t, in_chunk, out_chunk, rc, msg)
            assert gpu_lib.last_adler == oracle.adler32(data)
        raw = oracle.deflate(data, 6, 0)
        rc, out, msg, tin = gpu_lib.inflate_stream(raw, -15, 16384, 16384, zb.Z_SYNC_FLUSH)   # the way unzip.c calls it
        assert rc == zb.Z_STREAM_END and out == data and tin == len(raw)


def test_streaming_inflate_errors(gpu_lib, oracle):
    data = zhelpers.corpus(1, 50000, 3)
    z = bytearray(oracle.deflate(data, 6))
    z[len(z) // 2] ^= 0x10
    rc, out, msg, _ = gpu_lib.inflate_stream(bytes(z), 15, 4096, 4096)
    assert rc == zb.Z_DATA_ERROR and msg is not None
    assert msg == oracle.last_msg() or oracle.inflate(bytes(z), len(data))[0] == -3
    z = oracle.deflate(data, 6)
    rc, out, msg, _ = gpu_lib.inflate_stream(z[:-1] + bytes([z[-1] ^ 1]), 15, 4096, 4096)
    assert rc == zb.Z_DATA_ERROR and msg == "incorrect data check" and out == data
    rc, out, msg, _ = gpu_lib.inflate_stream(z[:len(z) // 2], 15, 4096, 4096, zb.Z_FINISH)
    assert rc == zb.Z_BUF_ERROR


def test_dictionary_round_trip(gpu_lib, oracle):
    dictionary = b"hello, " * 200
    data = b"hello, hello! " * 500
    rc, z = gpu_lib.deflate_stream(data, 9, 15, 1 << 20, 1 << 20, dictionary=dictionary)
    assert rc == zb.Z_OK and (z[1] & 0x20)
    d = zlib.decompressobj(zdict=dictionary)
    assert d.decompress(z) == data
    rc, out, msg, _ = gpu_lib.inflate_stream(z, 15, 1 << 20, 1 << 20, dictionary=dictionary)
    assert rc == zb.Z_STREAM_END and out == data
    rc, out, msg, _ = gpu_lib.inflate_stream(z, 15, 1 << 20, 1 << 20, dictionary=b"wrong dictionary")
    assert rc == zb.Z_DATA_ERROR


def _need(path):
    """The reference's own programs are built by oracle/Makefile only when it is given the reference sources (REF=<dir>);
    they are not part of this repository."""
    if not os.path.exists(path):
        pytest.skip(f"{path} not built: oracle/Makefile needs REF=<reference zlib sources>")
    return path


def _extract_and_compare(path, files, out, oracle, names=None):
    """Python's zipfile extracts the archive into `out`, the oracle decodes every member on its own; both must give
    back `files` bit-exact (every member, or the ones in `names` for the extracted copies)."""
    import zipfile
    zipfile.ZipFile(path).extractall(out)
    for name in (files if names is None else names):
        assert (out / name).read_bytes() == files[name], name
    decoded = zhelpers.unzip_with_oracle(path, oracle)
    assert sorted(decoded) == sorted(files)
    for name, data in files.items():
        assert decoded[name] == data, name


def test_reference_example_c_against_libzb200(gpu_lib):
    """The reference's acceptance program (qcsrc/example.c + its gzio.c) linked against our library."""
    exe = _need(os.path.join(REFDIR, "example_zb200"))
    r = subprocess.run([exe, "/tmp/zb200_example.gz"], capture_output=True, text=True, timeout=300, cwd="/tmp")
    assert r.returncode == 0, r.stdout + r.stderr
    lines = [l.strip() for l in r.stdout.splitlines()]
    assert lines[0].startswith("zlib version 1.2.3 = 0x1230, compile flags = 0xa9")
    assert lines[1:] == EXAMPLE_LINES


def test_minizip_miniunz_both_directions(gpu_lib, tmp_path):
    """ZIP written by minizip-on-libzb200 is extracted bit-exact by the reference miniunz, and vice versa."""
    files = {}
    for i, (kind, n) in enumerate([(1, 4096), (3, 70000), (0, 20000), (1, 1 << 20), (2, 300000), (1, 0)]):
        name = f"f{i:05d}.bin"
        files[name] = zhelpers.corpus(kind, n, 70 + i)
        (tmp_path / name).write_bytes(files[name])
    for writer, reader in (("minizip_zb200", "miniunz"), ("minizip", "miniunz_zb200"), ("minizip_zb200", "miniunz_zb200")):
        w, r = _need(os.path.join(REFDIR, writer)), _need(os.path.join(REFDIR, reader))
        arc = tmp_path / f"{writer}.zip"
        out = tmp_path / f"x_{writer}_{reader}"
        out.mkdir()
        p = subprocess.run([w, "-o", "-6", str(arc)] + sorted(files), cwd=tmp_path, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout + p.stderr
        p = subprocess.run([r, "-o", str(arc)], cwd=out, capture_output=True, text=True, timeout=600)
        assert p.returncode == 0, p.stdout + p.stderr
        for name, data in files.items():
            assert (out / name).read_bytes() == data, (writer, reader, name)   # miniunz's exit code is not trusted
        import zipfile
        assert zipfile.ZipFile(arc).testzip() is None


def test_gzip_stream_decoding(gpu_lib):
    """inflateInit2(windowBits + 16 / + 32) through the streaming ABI in small pieces; strm->adler carries the CRC-32;
    a damaged CRC is 'incorrect data check', a damaged ISIZE 'incorrect length check' (inflate.c:1099-1112)."""
    import zlib
    data = gpu_lib.synth(700000, kind=1, seed=9).tobytes()
    co = zlib.compressobj(6, zlib.DEFLATED, 31)
    z = co.compress(data) + co.flush()
    for wbits in (31, 47):
        rc, out, msg, tin = gpu_lib.inflate_stream(z, wbits=wbits, in_chunk=5000, out_chunk=30000)
        assert rc == zb.Z_STREAM_END and out == data and tin == len(z)
        assert gpu_lib.last_adler == zlib.crc32(data)
    rc, out, msg, tin = gpu_lib.inflate_stream(zlib.compress(data, 6), wbits=47, in_chunk=7000, out_chunk=50000)
    assert rc == zb.Z_STREAM_END and out == data                 # auto-detect also takes a zlib stream
    bad = bytearray(z); bad[-6] ^= 4
    rc, out, msg, tin = gpu_lib.inflate_stream(bytes(bad), wbits=31)
    assert rc == zb.Z_DATA_ERROR and msg == "incorrect data check"
    bad = bytearray(z); bad[-1] ^= 4
    rc, out, msg, tin = gpu_lib.inflate_stream(bytes(bad), wbits=31)
    assert rc == zb.Z_DATA_ERROR and msg == "incorrect length check"
    # our own gzip output read back by our own gzip decoder
    rc, zz = gpu_lib.deflate_stream(data, level=6, wbits=31)
    assert rc == zb.Z_OK
    rc, out, msg, tin = gpu_lib.inflate_stream(zz, wbits=31, in_chunk=1 << 20, out_chunk=1 << 20)
    assert rc == zb.Z_STREAM_END and out == data


def test_inflate_get_header(gpu_lib):
    """inflateGetHeader (inflate.c:1211-1227, header walk :634-759): the gzip header fields reach the caller's gz_header
    while the stream is fed three bytes at a time; buffers clip; a zlib stream under windowBits + 32 reports done = -1."""
    import ctypes as C
    import struct
    data = zhelpers.corpus(1, 50000, 77)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    body = co.compress(data) + co.flush()
    extra, name, comment = b"EX\x04\x00abcd", b"file name.txt", b"a comment that is longer than the buffer"
    hdr = bytes([31, 139, 8, 1 | 2 | 4 | 8 | 16]) + struct.pack("<IBB", 1234567890, 2, 3)
    hdr += struct.pack("<H", len(extra)) + extra + name + b"\0" + comment + b"\0"
    hdr += struct.pack("<H", zlib.crc32(hdr) & 0xffff)
    member = hdr + body + struct.pack("<II", zlib.crc32(data), len(data))
    assert zlib.decompress(member, 31) == data
    for wbits in (31, 47):
        strm = zb.z_stream()
        assert gpu_lib.dll.inflateInit2_(C.byref(strm), wbits, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
        ebuf, nbuf, cbuf = C.create_string_buffer(64), C.create_string_buffer(64), C.create_string_buffer(10)
        head = zb.gz_header()
        head.extra, head.extra_max = C.addressof(ebuf), 64
        head.name, head.name_max = C.addressof(nbuf), 64
        head.comment, head.comm_max = C.addressof(cbuf), 10
        assert gpu_lib.dll.inflateGetHeader(C.byref(strm), C.byref(head)) == zb.Z_OK and head.done == 0
        src = C.create_string_buffer(member, len(member))
        out = C.create_string_buffer(len(data) + 16)
        strm.next_out, strm.avail_out = C.addressof(out), len(data) + 16
        pos, rc, done_at = 0, zb.Z_OK, None
        while rc in (zb.Z_OK, zb.Z_BUF_ERROR) and pos < len(member):
            n = 3 if pos < len(hdr) + 6 else len(member) - pos
            strm.next_in, strm.avail_in = C.addressof(src) + pos, n
            rc = gpu_lib.dll.inflate(C.byref(strm), zb.Z_NO_FLUSH)
            pos += n - strm.avail_in
            if head.done == 1 and done_at is None:
                done_at = pos
        assert rc == zb.Z_STREAM_END and out.raw[:len(data)] == data
        assert done_at is not None and len(hdr) <= done_at <= len(hdr) + 3
        assert (head.text, head.time, head.xflags, head.os, head.hcrc, head.done) == (1, 1234567890, 2, 3, 1, 1)
        assert head.extra_len == len(extra) and ebuf.raw[:len(extra)] == extra
        assert nbuf.raw[:len(name) + 1] == name + b"\0"
        assert cbuf.raw == comment[:10]                           # clipped to comm_max, no terminator
        gpu_lib.dll.inflateEnd(C.byref(strm))
    # a zlib stream where gzip was allowed: done = -1; plain zlib decoding refuses the call
    strm = zb.z_stream()
    assert gpu_lib.dll.inflateInit2_(C.byref(strm), 47, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
    head = zb.gz_header()
    assert gpu_lib.dll.inflateGetHeader(C.byref(strm), C.byref(head)) == zb.Z_OK
    z = zlib.compress(data)
    src = C.create_string_buffer(z, len(z))
    out = C.create_string_buffer(len(data))
    strm.next_in, strm.avail_in, strm.next_out, strm.avail_out = C.addressof(src), len(z), C.addressof(out), len(data)
    assert gpu_lib.dll.inflate(C.byref(strm), zb.Z_FINISH) == zb.Z_STREAM_END and head.done == -1
    gpu_lib.dll.inflateEnd(C.byref(strm))
    strm = zb.z_stream()
    assert gpu_lib.dll.inflateInit2_(C.byref(strm), 15, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
    assert gpu_lib.dll.inflateGetHeader(C.byref(strm), C.byref(head)) == zb.Z_STREAM_ERROR
    gpu_lib.dll.inflateEnd(C.byref(strm))


def test_inflate_finish_whole_buffer_takes_parallel_decoder(gpu_lib):
    """inflateInit + inflate(Z_FINISH) with the whole stream and the whole buffer -- uncompress() spelled out
    (uncompr.c:26-61) -- decodes a chunked stream through the segment-parallel path: Z_STREAM_END, totals, adler and
    avail_in as the reference leaves them (bytes after the trailer stay with the caller)."""
    import ctypes as C
    n = (6 << 20) + 77
    data = gpu_lib.synth(n, kind=1, seed=31).tobytes()
    rc, z = gpu_lib.compress2(data, 1)
    assert rc == zb.Z_OK
    import struct
    gz = b"\x1f\x8b\x08\x00\x00\x00\x00\x00\x00\x03" + z[2:-4] + struct.pack("<II", zlib.crc32(data), n) + b"more"
    for wbits, stream in ((15, z + b"trailing"), (-15, z[2:-4] + b"xy"), (31, gz), (47, gz)):
        strm = zb.z_stream()
        assert gpu_lib.dll.inflateInit2_(C.byref(strm), wbits, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
        src = C.create_string_buffer(stream, len(stream))
        out = C.create_string_buffer(n + 100)
        strm.next_in, strm.avail_in, strm.next_out, strm.avail_out = C.addressof(src), len(stream), C.addressof(out), n + 100
        gpu_lib.profile(True)
        rc = gpu_lib.dll.inflate(C.byref(strm), zb.Z_FINISH)
        rep = gpu_lib.profile_report()
        gpu_lib.profile(False)
        assert rc == zb.Z_STREAM_END and any("k_inflate_segments" in k for k in rep)
        assert out.raw[:n] == data and strm.total_out == n and strm.avail_out == 100
        extra = 8 if wbits == 15 else 2 if wbits < 0 else 4
        assert strm.avail_in == extra and strm.total_in == len(stream) - extra
        if wbits == 15:
            assert strm.adler == zlib.adler32(data)
        elif wbits > 15:
            assert strm.adler == zlib.crc32(data)
        assert gpu_lib.dll.inflate(C.byref(strm), zb.Z_FINISH) == zb.Z_STREAM_END
        gpu_lib.dll.inflateEnd(C.byref(strm))


def test_inflate_prime(gpu_lib):
    """inflatePrime (inflate.c:128-142): the first bits of a raw deflate stream handed over as primed bits, the rest as
    bytes that start right after them, decode to the same output; priming is refused once input is pending."""
    import ctypes as C
    data = zhelpers.corpus(1, 30000, 78)
    co = zlib.compressobj(6, zlib.DEFLATED, -15)
    z = co.compress(data) + co.flush()
    val = int.from_bytes(z, "little")
    for bits in (0, 1, 3, 8, 11, 16):
        rest = (val >> bits).to_bytes(len(z), "little")
        strm = zb.z_stream()
        assert gpu_lib.dll.inflateInit2_(C.byref(strm), -15, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
        assert gpu_lib.dll.inflatePrime(C.byref(strm), bits, val & ((1 << bits) - 1)) == zb.Z_OK
        src = C.create_string_buffer(rest, len(rest))
        out = C.create_string_buffer(len(data) + 8)
        strm.next_in, strm.avail_in, strm.next_out, strm.avail_out = C.addressof(src), len(rest), C.addressof(out), len(data) + 8
        assert gpu_lib.dll.inflate(C.byref(strm), zb.Z_FINISH) == zb.Z_STREAM_END
        assert out.raw[:len(data)] == data and strm.total_out == len(data)
        gpu_lib.dll.inflateEnd(C.byref(strm))
    strm = zb.z_stream()
    assert gpu_lib.dll.inflateInit2_(C.byref(strm), -15, zb.ZLIB_VERSION, C.sizeof(zb.z_stream)) == zb.Z_OK
    assert gpu_lib.dll.inflatePrime(C.byref(strm), 17, 0) == zb.Z_STREAM_ERROR
    assert gpu_lib.dll.inflatePrime(C.byref(strm), 3, 5) == zb.Z_OK
    assert gpu_lib.dll.inflatePrime(C.byref(strm), 3, 5) == zb.Z_STREAM_ERROR      # primed bits are pending input
    gpu_lib.dll.inflateEnd(C.byref(strm))


def test_zip_archive_from_one_gpu_batch(gpu_lib, oracle, tmp_path):
    """BASELINE config 5 in small: many files compressed by ONE zb200_deflate_batch call and laid out as a ZIP32
    archive by zb200_zip_build; Python's zipfile extracts every member bit-exact, the oracle's inflate agrees."""
    import random
    import zipfile
    rng = random.Random(31)
    files = {}
    for i in range(120):
        n = int(4096 * (2 ** rng.uniform(0, 9)))                 # 4 KiB .. 2 MiB, log-uniform
        if i in (3, 4):
            n = i - 3                                            # an empty and a one-byte member
        files[f"f{i:05d}.bin"] = zhelpers.corpus(rng.choice([0, 1, 1, 3, 3, 4]), n, 900 + i)
    arc = gpu_lib.zip_build(files, level=6)
    path = tmp_path / "batch.zip"
    path.write_bytes(arc)
    zf = zipfile.ZipFile(path)
    assert zf.testzip() is None and len(zf.namelist()) == len(files)
    assert sum(i.compress_size for i in zf.infolist()) < 0.8 * sum(len(v) for v in files.values())
    _extract_and_compare(path, files, tmp_path / "x", oracle)


def test_zip_segments_concatenate(gpu_lib, oracle, tmp_path):
    """The multi-GPU form of config 5 on one GPU: two segments (zb200_zip_segment, laid out on the device) concatenated
    and closed by zb200_zip_directory are one archive that Python's zipfile and the oracle's inflate extract bit-exact;
    members of several MiB exercise the piecewise copy kernel at every relative misalignment."""
    import zipfile
    rng = random.Random(32)
    names = [f"s/{'x' * (i % 7)}f{i:04d}.dat" for i in range(60)]
    datas = [zhelpers.corpus(rng.choice([0, 1, 3, 4]), int(1000 * 2 ** rng.uniform(0, 11)) + i % 5, 700 + i) for i in range(60)]
    datas[7] = b""
    datas[8] = gpu_lib.synth((3 << 20) + 3, kind=1, seed=4).tobytes()
    datas[40] = gpu_lib.synth((2 << 20) + 1, kind=2, seed=5).tobytes()     # noise: stored blocks
    seg_a, meta_a = gpu_lib.zip_segment(names[:25], datas[:25], level=1)
    seg_b, meta_b = gpu_lib.zip_segment(names[25:], datas[25:], level=6)
    metas = meta_a + [(m[0] + len(seg_a), m[1], m[2], m[3]) for m in meta_b]
    assert [m[3] for m in metas] == [zlib.crc32(d) for d in datas]
    arc = seg_a + seg_b + gpu_lib.zip_directory(names, metas, len(seg_a) + len(seg_b))
    path = tmp_path / "two_segments.zip"
    path.write_bytes(arc)
    zf = zipfile.ZipFile(path)
    assert zf.testzip() is None and zf.namelist() == names
    _extract_and_compare(path, dict(zip(names, datas)), tmp_path / "x", oracle)


def test_strategies(gpu_lib, oracle, reference_codec):
    """deflateInit2 strategies (deflate.c:1485-1494, 1594-1612, trees.c:986): every one decodes; Z_RLE only emits
    distance-1 matches, Z_HUFFMAN_ONLY none, Z_FIXED only fixed blocks; sizes are gated against the REFERENCE build
    running the same strategy and level, and order like the reference's."""
    import zlib
    data = (zhelpers.corpus(1, 200000, 5) + bytes(50000) + zhelpers.corpus(3, 100000, 6) + b"ab" * 30000)
    sizes = {}
    for strategy in (0, 1, 2, 3, 4):
        for level in (1, 6):
            rc, z = gpu_lib.deflate_stream(data, level=level, wbits=15, strategy=strategy)
            assert rc == zb.Z_OK
            assert zlib.decompress(z) == data
            rc2, out, used = oracle.inflate(z, len(data))
            assert rc2 == 0 and out == data
            sizes[(strategy, level)] = len(z)
            want = len(reference_codec.deflate_stream(data, level, 15, strategy))
            assert len(z) <= (1.06 if strategy == 4 else 1.03) * want + 64, (strategy, level, len(z), want)   # fixed codes punish every extra token
            if strategy >= 2:
                assert (z[1] >> 6) == 0                               # FLEVEL = fastest (deflate.c:628)
    assert sizes[(2, 6)] > sizes[(3, 6)] > sizes[(0, 6)]              # Huffman only > RLE > default
    assert sizes[(1, 6)] >= sizes[(0, 6)]


def test_zip_ten_thousand_files(gpu_lib, oracle, tmp_path):
    """BASELINE config 5 at its file count: 10 000 members (4 KiB .. 256 KiB, log-uniform, ~0.4 GB) in ONE zb200_zip_build
    call; Python's zipfile checks every member's CRC and extracts all of them, the oracle's inflate decodes all of them
    bit-exact."""
    import zipfile
    rng = random.Random(55)
    sizes = [int(4096 * 2 ** rng.uniform(0, 6)) for _ in range(10000)]
    blob = gpu_lib.synth(sum(sizes), kind=1, seed=56).tobytes()
    files, pos = {}, 0
    for i, n in enumerate(sizes):
        files[f"f{i:05d}.bin"] = blob[pos:pos + n]
        pos += n
    arc = gpu_lib.zip_build(files, level=1)
    path = tmp_path / "ten_thousand.zip"
    path.write_bytes(arc)
    zf = zipfile.ZipFile(path)
    assert len(zf.namelist()) == 10000 and zf.testzip() is None
    out = tmp_path / "x"
    _extract_and_compare(path, files, out, oracle, rng.sample(sorted(files), 500) + ["f00000.bin", "f09999.bin"])
    assert len(os.listdir(out)) == 10000
