"""GPU: zb200_gunzip decodes every member of a gzip file as gzip.decompress does; zb200_bgzf_compress writes BGZF."""
import ctypes as C
import gzip
import struct
import zlib

import numpy as np
import pytest

from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

KIB, MIB = 1 << 10, 1 << 20
BGZF_HEADER = bytes.fromhex("1f8b08040000000000ff060042430200")
BGZF_EOF = bytes.fromhex("1f8b08040000000000ff0600424302001b0003000000000000000000")


def _synth(lib, n, kind, seed):
    return bytes(lib.synth(n, kind=kind, seed=seed))


def _gunzip(lib, data, cap=None):
    """zb200_gunzip on host bytes -> (rc, output, members, dst_len)."""
    cap = max(4 * len(data), 1 << 20) if cap is None else cap
    out = np.empty(max(cap, 1), dtype=np.uint8)
    src = np.frombuffer(data, dtype=np.uint8) if data else np.zeros(1, dtype=np.uint8)
    ol, cnt = C.c_size_t(cap), C.c_size_t(0)
    rc = lib.dll.zb200_gunzip(src.ctypes.data, len(data), out.ctypes.data, C.byref(ol), C.byref(cnt), None)
    return rc, out[:ol.value].tobytes() if rc == zb.Z_OK else b"", cnt.value, ol.value


def _members(blob):
    """Walks a BGZF file: [(header, member length, isize)]; asserts the framing of every member."""
    out, p = [], 0
    while p < len(blob):
        h = blob[p:p + 18]
        assert h[:16] == BGZF_HEADER, (p, h.hex())
        bsize = struct.unpack("<H", h[16:18])[0]
        n = bsize + 1
        assert n <= 65536 and p + n <= len(blob)
        isize = struct.unpack("<I", blob[p + n - 4:p + n])[0]
        out.append((h, n, isize))
        p += n
    return out


@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_bgzf_round_trip_and_structure(gpu_lib, level):
    import torch
    big = _synth(gpu_lib, 64 * MIB + 12345, 1, level + 1)
    for n in (0, 1, 65279, 65280, 65281, MIB + 7, 64 * MIB + 12345):
        data = big[:n]
        for kind in ("host", "pinned", "device"):
            if kind == "host":
                blob = gpu_lib.bgzf_compress(data, level)
            elif kind == "pinned":
                pin = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8)[:n].pin_memory()
                blob = gpu_lib.bgzf_compress(pin, level)
                blob = blob if isinstance(blob, bytes) else bytes(blob)
            else:
                d = torch.frombuffer(bytearray(data) or bytearray(1), dtype=torch.uint8)[:n].cuda()
                blob = gpu_lib.bgzf_compress(d, level).cpu().numpy().tobytes()
            assert blob.endswith(BGZF_EOF), (n, kind)
            if n == 0:
                assert blob == BGZF_EOF
            assert gzip.decompress(blob) == data, (n, kind)
            mem = _members(blob)
            blocks = (n + 65279) // 65280
            assert len(mem) == blocks + 1
            for k, (_, _, isize) in enumerate(mem[:-1]):
                assert isize == (65280 if k + 1 < blocks else n - 65280 * (blocks - 1)), (n, k)
            if kind == "host":
                rc, out, cnt, _ = _gunzip(gpu_lib, blob)
                assert rc == zb.Z_OK and out == data and cnt == blocks + 1, (n, rc, cnt, gpu_lib.last_error())


def _hand_member(data, name=None, comment=None, extra=None, hcrc=False, level=6):
    flg = (4 if extra is not None else 0) | (8 if name else 0) | (16 if comment else 0) | (2 if hcrc else 0)
    h = bytearray(b"\x1f\x8b\x08" + bytes([flg]) + b"\x00\x00\x00\x00\x00\x03")
    if extra is not None:
        h += struct.pack("<H", len(extra)) + extra
    if name:
        h += name + b"\0"
    if comment:
        h += comment + b"\0"
    if hcrc:
        h += struct.pack("<H", zlib.crc32(bytes(h)) & 0xFFFF)
    co = zlib.compressobj(level, zlib.DEFLATED, -15)
    return bytes(h) + co.compress(data) + co.flush() + struct.pack("<II", zlib.crc32(data), len(data) & 0xFFFFFFFF)


def _pieces(lib, count, seed):
    text = _synth(lib, 2 * MIB, 0, seed)
    rng = np.random.default_rng(seed)
    out = []
    for k in range(count):
        n = int(rng.integers(0, 200 * KIB)) if k % 7 else 0        # empty members too
        a = int(rng.integers(0, len(text) - n + 1))
        out.append(text[a:a + n])
    return out


def _gzip_members(lib, datas, style, k0=0):
    out = []
    for k, d in enumerate(datas):
        s = style if style != "mixed" else ("py", "hand", "batch")[(k + k0) % 3]
        if s == "py":
            out.append(gzip.compress(d, compresslevel=(0, 1, 6, 9)[(k + k0) % 4], mtime=0))
        elif s == "hand":
            out.append(_hand_member(d, name=b"f%d.txt" % k, comment=b"c" * (k % 5), extra=b"ab\x02\x00xy" if k % 2 else None,
                                    hcrc=k % 3 == 0))
        else:
            outs, st, _, _ = lib.deflate_batch([d], 6, zb.WRAP_GZIP)
            assert st == [0]
            out.append(outs[0])
    return out


@pytest.mark.parametrize("count", [1, 2, 50])
@pytest.mark.parametrize("style", ["py", "hand", "batch", "mixed"])
def test_generic_files_match_gzip_decompress(gpu_lib, count, style):
    datas = _pieces(gpu_lib, count, count * 10 + len(style))
    mem = _gzip_members(gpu_lib, datas, style)
    blob = b"".join(mem)
    want = gzip.decompress(blob)
    assert want == b"".join(datas)
    rc, out, cnt, _ = _gunzip(gpu_lib, blob)
    assert rc == zb.Z_OK and out == want and cnt == count, (rc, cnt, gpu_lib.last_error())
    # zero padding between and after members
    padded = b"".join(m + b"\0" * (k % 3) * 5 for k, m in enumerate(mem)) + b"\0" * 17
    assert gzip.decompress(padded) == want
    rc, out, cnt, _ = _gunzip(gpu_lib, padded)
    assert rc == zb.Z_OK and out == want and cnt == count, (rc, cnt, gpu_lib.last_error())


def test_long_member_between_small_ones(gpu_lib):
    big = _synth(gpu_lib, 64 * MIB + 999, 0, 77)
    small = _pieces(gpu_lib, 6, 78)
    co = zlib.compressobj(6, zlib.DEFLATED, 31)                  # system zlib: no sync markers, the block finder's work
    mem = _gzip_members(gpu_lib, small[:3], "mixed") + [co.compress(big) + co.flush()] + _gzip_members(gpu_lib, small[3:], "mixed")
    blob = b"".join(mem)
    want = b"".join(small[:3]) + big + b"".join(small[3:])
    gpu_lib.profile(True)
    rc, out, cnt, _ = _gunzip(gpu_lib, blob)
    report = gpu_lib.profile_report()
    gpu_lib.profile(False)
    assert rc == zb.Z_OK and out == want and cnt == 7, (rc, cnt, gpu_lib.last_error())
    assert any("k_inflate_segments" in k for k in report), report   # the long member in parallel, not on one warp


def _early_end(gzip_member, junk=b"\x01\x02\x03\x04\x05\x06\x07\x09" * 3):
    """The member with junk between its deflate data and its trailer: the span in front of the next member still ends in
    the right CRC-32 and ISIZE, but the deflate data end before it."""
    return gzip_member[:-8] + junk + gzip_member[-8:]


@pytest.mark.parametrize("n", [50 * KIB, MIB + 5])                 # one warp; planned segments (this library's markers)
def test_data_ending_before_the_trailer_is_refused(gpu_lib, n):
    data = _synth(gpu_lib, n, 0, 31)
    outs, st, _, _ = gpu_lib.deflate_batch([data], 6, zb.WRAP_GZIP)
    tail = gzip.compress(b"next member", mtime=0)
    blob = _early_end(outs[0]) + tail
    gpu_lib.profile(True)
    _refused(gpu_lib, blob, 0)
    report = gpu_lib.profile_report()
    gpu_lib.profile(False)
    if n > 128 * KIB:
        assert any("k_inflate_segments" in k for k in report), report
    rc, out, cnt, _ = _gunzip(gpu_lib, outs[0] + tail)
    assert rc == zb.Z_OK and out == data + b"next member" and cnt == 2


def test_header_scan_is_bounded(gpu_lib):
    """1f 8b 08 with FNAME and FHCRC set, and no NUL anywhere: every position is a header whose name never ends."""
    import time
    blob = b"\x1f\x8b\x08\x0a" * (4 * MIB)
    with pytest.raises(Exception):
        gzip.decompress(blob)
    gpu_lib.profile(True)
    t0 = time.perf_counter()
    rc, _, cnt, _ = _gunzip(gpu_lib, blob)
    wall = time.perf_counter() - t0
    report = gpu_lib.profile_report()
    gpu_lib.profile(False)
    assert rc == zb.Z_DATA_ERROR and cnt == 0, (rc, gpu_lib.last_error())
    assert report["k_gz_scan"][0] < 1000.0 and wall < 30.0, (report, wall)


def test_spurious_candidates(gpu_lib):
    inner = _gzip_members(gpu_lib, _pieces(gpu_lib, 6, 91), "mixed")
    payload = b"head" + b"".join(inner) + b"tail" + b"".join(inner[:2])
    outer = gzip.compress(payload, compresslevel=0, mtime=0)
    after = _gzip_members(gpu_lib, _pieces(gpu_lib, 3, 92), "py")
    blob = outer + b"".join(after)
    want = gzip.decompress(blob)
    rc, out, cnt, _ = _gunzip(gpu_lib, blob)
    assert rc == zb.Z_OK and out == want and cnt == 4, (rc, cnt, gpu_lib.last_error())
    # the same inner members inside a BGZF file written at level 0
    bg = gpu_lib.bgzf_compress(payload * 3, 0)
    rc, out, cnt, _ = _gunzip(gpu_lib, bg)
    assert rc == zb.Z_OK and out == payload * 3 and cnt == len(_members(bg)), (rc, cnt, gpu_lib.last_error())


def _ten(lib):
    datas = _pieces(lib, 10, 5)
    datas = [d or b"x" * 1000 for d in datas]
    return datas, [gzip.compress(d, compresslevel=6, mtime=0) for d in datas]


def _refused(lib, blob, index, python_too=True):
    if python_too:
        with pytest.raises(Exception):
            gzip.decompress(blob)
    rc, _, cnt, _ = _gunzip(lib, blob)
    assert rc == zb.Z_DATA_ERROR, (rc, lib.last_error())
    if index is not None:
        assert cnt == index, (cnt, index, lib.last_error())
    assert ("member %d" % cnt) in lib.last_error()


def test_refusals(gpu_lib):
    datas, mem = _ten(gpu_lib)
    m = [bytearray(x) for x in mem]
    m[5][len(m[5]) // 2] ^= 0x55                                  # damaged data of member 5
    _refused(gpu_lib, b"".join(map(bytes, m)), 5)
    m = [bytearray(x) for x in mem]
    m[3][-8] ^= 1                                                 # CRC-32
    _refused(gpu_lib, b"".join(map(bytes, m)), 3)
    m = [bytearray(x) for x in mem]
    m[7][-2] ^= 1                                                 # ISIZE
    _refused(gpu_lib, b"".join(map(bytes, m)), 7)
    _refused(gpu_lib, b"".join(mem)[:-5], 9)                      # truncated last member
    _refused(gpu_lib, b"".join(mem) + b"garbage", 10)             # trailing garbage
    _refused(gpu_lib, b"\0\0\0" + b"".join(mem), 0)               # leading zeros
    m = [bytearray(x) for x in mem]
    m[4][3] |= 0x20                                               # reserved FLG bit: zlib refuses, Python does not
    _refused(gpu_lib, b"".join(map(bytes, m)), 4, python_too=False)
    m = list(mem)
    m[2] = bytearray(_hand_member(datas[2], name=b"n", hcrc=True))
    m[2][12] ^= 0xFF                                              # wrong FHCRC: zlib refuses, Python does not
    blob = b"".join(map(bytes, m))
    assert gzip.decompress(blob) == b"".join(datas)
    _refused(gpu_lib, blob, 2, python_too=False)


def test_buffer_too_small(gpu_lib):
    _, mem = _ten(gpu_lib)
    blob = b"".join(mem)
    want = gzip.decompress(blob)
    rc, _, _, need = _gunzip(gpu_lib, blob, cap=len(want) - 1)
    assert rc == zb.Z_BUF_ERROR and need == len(want), (rc, need)
    rc, out, cnt, _ = _gunzip(gpu_lib, blob, cap=len(want))
    assert rc == zb.Z_OK and out == want and cnt == 10
    assert _gunzip(gpu_lib, b"")[:3] == (zb.Z_OK, b"", 0)


def test_route_does_not_grow_with_members(gpu_lib):
    data = _synth(gpu_lib, 2000 * 65280, 1, 3)
    used = []
    for blocks in (200, 2000):
        blob = gpu_lib.bgzf_compress(data[:blocks * 65280], 1)
        _gunzip(gpu_lib, blob)                                    # warm
        gpu_lib.profile(True)
        before = gpu_lib.kernel_launches()
        rc, out, cnt, _ = _gunzip(gpu_lib, blob)
        used.append(gpu_lib.kernel_launches() - before)
        report = gpu_lib.profile_report()
        gpu_lib.profile(False)
        assert rc == zb.Z_OK and out == data[:blocks * 65280] and cnt == blocks + 1
        assert report["k_gz_scan"][1] == 1, report
    assert used[0] == used[1], used


def test_buffers(gpu_lib):
    import torch
    datas = _pieces(gpu_lib, 40, 12)
    big = _synth(gpu_lib, 80 * MIB, 2, 13)                                  # noise: the file stays above 64 MiB
    blob = b"".join(_gzip_members(gpu_lib, datas, "mixed")) + gpu_lib.bgzf_compress(big, 1)
    want = b"".join(datas) + big
    assert len(blob) >= 64 * MIB
    assert gpu_lib.gunzip(blob) == want                                     # pageable, >= 64 MiB
    pin = torch.frombuffer(bytearray(blob), dtype=torch.uint8).pin_memory()
    assert gpu_lib.gunzip(pin) == want                                      # pinned
    d = torch.frombuffer(bytearray(blob), dtype=torch.uint8).cuda()
    out = gpu_lib.gunzip(d)                                                 # device in, device out
    assert out.is_cuda and out.cpu().numpy().tobytes() == want
