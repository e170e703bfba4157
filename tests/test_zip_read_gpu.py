"""GPU: zb200_zip_extract reads archives back -- every member bit-exact, every failure with its own status."""
import io
import os
import random
import struct
import zipfile
import zlib

import numpy as np
import pytest

import zhelpers
from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

KIB, MIB = 1 << 10, 1 << 20


def _synth(lib, n, kind, seed):
    return bytes(lib.synth(n, kind=kind, seed=seed))


def _members(lib):
    rng = random.Random(7)
    return {
        "zero": b"",
        "one": b"x",
        "four_k.txt": _synth(lib, 4 * KIB, 0, 1),
        "chunk.txt": _synth(lib, 128 * KIB, 0, 2),
        "chunk_plus_one.txt": _synth(lib, 128 * KIB + 1, 0, 3),
        "text.txt": _synth(lib, 5 * MIB + 12345, 0, 4),
        "records.bin": _synth(lib, 3 * MIB + 7, 1, 5),
        "noise.bin": _synth(lib, 1 * MIB + 3, 2, 6),           # stored chunks: no markers, the one-stream fallback
        "medium.txt": _synth(lib, rng.randrange(300 * KIB, 900 * KIB), 0, 7),
    }


def _check(lib, arc, files, entries=None, outs=None, st=None):
    entries = lib.zip_list(arc) if entries is None else entries
    if outs is None:
        outs, st = lib.zip_extract(arc, entries)
    for e, o, s in zip(entries, outs, st):
        data = files[e.name]
        assert s == zb.Z_OK, (e.name, s)
        assert bytes(o) == data, e.name
        assert e.crc32 == zlib.crc32(data), e.name
    return entries, outs, st


@pytest.mark.parametrize("level", [0, 1, 6, 9])
def test_own_archives(gpu_lib, level):
    files = _members(gpu_lib)
    arc = gpu_lib.zip_build(files, level=level)
    entries, _, _ = _check(gpu_lib, arc, files)
    assert [e.name for e in entries] == list(files)


def _pyzip(files, compression, level=None, lead=b""):
    b = io.BytesIO()
    with zipfile.ZipFile(b, "w", compression, compresslevel=level) as z:
        for name, data in files.items():
            z.writestr(name, data)
    return lead + b.getvalue()


class _NoSeek(io.RawIOBase):
    def __init__(self):
        self.buf = bytearray()

    def writable(self):
        return True

    def write(self, b):
        self.buf += b
        return len(b)


def test_python_zipfile_archives(gpu_lib):
    files = _members(gpu_lib)
    del files["text.txt"]                                      # the one-stream fallback takes each long member: keep it short
    for compression, level in ((zipfile.ZIP_STORED, None), (zipfile.ZIP_DEFLATED, 1), (zipfile.ZIP_DEFLATED, 6),
                               (zipfile.ZIP_DEFLATED, 9)):
        _check(gpu_lib, _pyzip(files, compression, level), files)
    _check(gpu_lib, _pyzip(files, zipfile.ZIP_DEFLATED, 6, lead=b"leading bytes " * 99), files)
    out = _NoSeek()
    with zipfile.ZipFile(out, "w", zipfile.ZIP_DEFLATED) as z:
        for name, data in files.items():
            with z.open(name, "w") as f:
                f.write(data)
    entries, _, _ = _check(gpu_lib, bytes(out.buf), files)
    assert all(e.flags & 8 for e in entries)


def test_minizip_archives(gpu_lib, tmp_path):
    ref = os.path.join(zhelpers.ROOT, "oracle", "_ref")
    tools = [os.path.join(ref, t) for t in ("minizip", "minizip_zb200")]
    tools = [t for t in tools if os.path.exists(t)]
    if not tools:
        pytest.skip("oracle/_ref/minizip not built (needs the reference)")
    import subprocess
    files = {"a.txt": _synth(gpu_lib, 700 * KIB, 0, 11), "b.bin": _synth(gpu_lib, 2 * MIB, 1, 12), "c": b"c" * 10}
    for name, data in files.items():
        (tmp_path / name).write_bytes(data)
    for k, tool in enumerate(tools):
        out = tmp_path / f"m{k}.zip"
        subprocess.check_call([tool, "-o", "-6", str(out)] + list(files), cwd=tmp_path, stdout=subprocess.DEVNULL)
        _check(gpu_lib, out.read_bytes(), files)


def test_subset_order_and_statuses(gpu_lib):
    files = _members(gpu_lib)
    arc = bytearray(gpu_lib.zip_build(files, level=6))
    full = gpu_lib.zip_list(bytes(arc))
    _, outs, _ = _check(gpu_lib, bytes(arc), files, full)
    sub = full[::-2]
    o2, s2 = gpu_lib.zip_extract(bytes(arc), sub)
    assert s2 == [0] * len(sub)
    by_name = {e.name: o for e, o in zip(full, outs)}
    assert [bytes(o) for o in o2] == [by_name[e.name] for e in sub]
    # a slot one byte short
    caps = [e.raw_len for e in full]
    big = [i for i, e in enumerate(full) if e.raw_len > 1 * MIB]
    for i in (2, big[0]):
        c2 = list(caps)
        c2[i] -= 1
        _, st = gpu_lib.zip_extract(bytes(arc), full, caps=c2)
        assert st[i] == zb.Z_BUF_ERROR and all(s == 0 for k, s in enumerate(st) if k != i), st
    # encrypted flag and method 12, written into both headers of one member each
    enc, m12 = full[3], full[5]
    a2 = bytearray(arc)
    cd = {e.name: e.raw["name_off"] - 46 for e in full}
    a2[cd[enc.name] + 8] |= 1
    a2[enc.local_off + 6] |= 1
    struct.pack_into("<H", a2, cd[m12.name] + 10, 12)
    struct.pack_into("<H", a2, m12.local_off + 8, 12)
    ents = gpu_lib.zip_list(bytes(a2))
    _, st = gpu_lib.zip_extract(bytes(a2), ents)
    want = [zb.Z_OK] * len(ents)
    want[3], want[5] = zb.Z_STREAM_ERROR, zb.ZB200_UNZ_BADZIPFILE
    assert st == want


def _damaged(lib, arc, files, edit, want, idx):
    a2 = bytearray(arc)
    edit(a2)
    ents = lib.zip_list(bytes(a2))
    outs, st = lib.zip_extract(bytes(a2), ents)
    assert st[idx] in want, (idx, st[idx], want)
    for k, (e, o, s) in enumerate(zip(ents, outs, st)):
        if k != idx:
            assert s == zb.Z_OK and bytes(o) == files[e.name], (k, e.name, s)


def test_damage_one_member_at_a_time(gpu_lib):
    files = _members(gpu_lib)
    arc = gpu_lib.zip_build(files, level=6)
    ents = gpu_lib.zip_list(arc)
    cd = [e.raw["name_off"] - 46 for e in ents]
    data_at = [e.local_off + 30 + len(e.name.encode()) for e in ents]
    for i, e in enumerate(ents):
        if e.comp_len > 16:                                     # a flipped byte inside the deflate data
            p = data_at[i] + e.comp_len // 2

            def flip(a, p=p):
                a[p] ^= 0x5A
            _damaged(gpu_lib, arc, files, flip, (zb.Z_DATA_ERROR, zb.ZB200_UNZ_CRCERROR), i)

        def crc(a, i=i):                                        # CRC stated in both headers: coherent, but wrong
            for at in (cd[i] + 16, ents[i].local_off + 14):
                struct.pack_into("<I", a, at, ents[i].crc32 ^ 0x00010000)
        _damaged(gpu_lib, arc, files, crc, (zb.ZB200_UNZ_CRCERROR,), i)

        def method(a, i=i):                                     # local header disagrees with the directory
            struct.pack_into("<H", a, ents[i].local_off + 8, 0)
        _damaged(gpu_lib, arc, files, method, (zb.ZB200_UNZ_BADZIPFILE,), i)

        def namelen(a, i=i):
            struct.pack_into("<H", a, ents[i].local_off + 26, len(ents[i].name) + 1)
        _damaged(gpu_lib, arc, files, namelen, (zb.ZB200_UNZ_BADZIPFILE,), i)

        for d in (-1, 1):
            if e.raw_len + d < 0:
                continue

            def rawlen(a, i=i, d=d):                            # raw length stated in both headers
                for at in (cd[i] + 24, ents[i].local_off + 22):
                    struct.pack_into("<I", a, at, ents[i].raw_len + d)
            _damaged(gpu_lib, arc, files, rawlen, (zb.Z_DATA_ERROR,), i)


def test_crc_in_directory_with_data_descriptors(gpu_lib):
    files = {"a": _synth(gpu_lib, 400 * KIB, 0, 21), "b": _synth(gpu_lib, 3000, 1, 22)}
    out = _NoSeek()
    with zipfile.ZipFile(out, "w", zipfile.ZIP_DEFLATED) as z:
        for name, data in files.items():
            with z.open(name, "w") as f:
                f.write(data)
    arc = bytes(out.buf)
    ents = gpu_lib.zip_list(arc)
    for i in range(2):
        def crc(a, i=i):                                        # flag bit 3: the local header carries no CRC to compare
            struct.pack_into("<I", a, ents[i].raw["name_off"] - 46 + 16, ents[i].crc32 ^ 1)
        _damaged(gpu_lib, arc, files, crc, (zb.ZB200_UNZ_CRCERROR,), i)


def test_device_resident(gpu_lib):
    import torch
    files = _members(gpu_lib)
    arc = gpu_lib.zip_build(files, level=1)
    host_outs, host_st = gpu_lib.zip_extract(arc)
    d_arc = torch.frombuffer(bytearray(arc), dtype=torch.uint8).cuda()
    ents = gpu_lib.zip_list(d_arc)
    assert [(e.name, e.local_off, e.crc32) for e in ents] == [(e.name, e.local_off, e.crc32) for e in gpu_lib.zip_list(arc)]
    outs, st = gpu_lib.zip_extract(d_arc, ents)
    torch.cuda.synchronize()
    assert st == host_st == [0] * len(ents)
    assert all(o.is_cuda for o in outs)
    assert [o.cpu().numpy().tobytes() for o in outs] == host_outs
    # pinned host buffers give the same bytes
    import ctypes as C
    p = gpu_lib.dll.zb200_alloc_pinned(len(arc))
    try:
        C.memmove(p, arc, len(arc))
        pin = np.ctypeslib.as_array(C.cast(p, C.POINTER(C.c_uint8)), shape=(len(arc),))
        o3, s3 = gpu_lib.zip_extract(pin, ents)
        assert s3 == host_st and o3 == host_outs
    finally:
        gpu_lib.dll.zb200_free_pinned(C.c_void_p(p))


def _launches(lib, nsmall):
    rng = random.Random(nsmall)
    text = _synth(lib, 2 * 24 * MIB + 4 * MIB, 0, 31)
    files = {}
    for i in range(nsmall):
        o = 48 * MIB + rng.randrange(0, 2 * MIB)
        files[f"s{i:05d}"] = text[o:o + rng.randrange(1, 60000)]
    files["big0.txt"] = text[:24 * MIB]
    files["big1.txt"] = text[24 * MIB:48 * MIB]
    arc = lib.zip_build(files, level=6)
    ents = lib.zip_list(arc)
    lib.zip_extract(arc, ents)                                  # warm: buffers of the context grown
    lib.profile(True)
    before = lib.kernel_launches()
    outs, st = lib.zip_extract(arc, ents)
    used = lib.kernel_launches() - before
    report = lib.profile_report()
    lib.profile(False)
    assert st == [0] * len(ents)
    assert all(bytes(o) == files[e.name] for e, o in zip(ents, outs))
    return used, report


def test_large_members_take_the_segment_route(gpu_lib):
    used_many, report = _launches(gpu_lib, 2000)
    assert any("k_inflate_segments" in k for k in report), report
    assert not any("k_find_blocks_probe" in k for k in report), report
    # one marker search for the whole call: the one-stream fallback would search again for every member it takes
    assert report["k_find_markers"][1] == 1, report
    used_few, _ = _launches(gpu_lib, 200)
    assert used_many == used_few, (used_many, used_few)


def test_one_damaged_long_member_leaves_the_others_planned(gpu_lib):
    text = _synth(gpu_lib, 12 * MIB, 0, 41)
    files = {f"big{k}.txt": text[k * 3 * MIB:(k + 1) * 3 * MIB] for k in range(4)}
    files["small"] = text[:5000]
    arc = bytearray(gpu_lib.zip_build(files, level=6))
    ents = gpu_lib.zip_list(bytes(arc))
    e = ents[1]
    arc[e.local_off + 30 + len(e.name) + e.comp_len // 3] ^= 0x5A
    gpu_lib.profile(True)
    outs, st = gpu_lib.zip_extract(bytes(arc), ents)
    report = gpu_lib.profile_report()
    gpu_lib.profile(False)
    assert st[1] in (zb.Z_DATA_ERROR, zb.ZB200_UNZ_CRCERROR), st
    for k, (e, o, s) in enumerate(zip(ents, outs, st)):
        if k != 1:
            assert s == zb.Z_OK and bytes(o) == files[e.name], (k, s)
    assert report["k_find_markers"][1] <= 2, report            # the call's search, and at most one fallback: the damaged member


def _extract_at(lib, arc, ents, buf_ptr, base, caps):
    """zb200_zip_extract with the slots starting `base` bytes into the caller's buffer."""
    import ctypes as C
    n = len(ents)
    recs = np.zeros(n, dtype=zb._zip_entry_dtype())
    for i, e in enumerate(ents):
        recs[i] = e.raw
    dst_off = np.zeros(n + 1, dtype=np.uint64)
    dst_off[0] = base
    dst_off[1:] = base + np.cumsum(caps, dtype=np.uint64)
    dst_len = np.zeros(n, dtype=np.uint64)
    status = np.full(n, -99, dtype=np.int32)
    rc = lib.dll.zb200_zip_extract(arc, len(arc), recs.ctypes.data, n, C.c_void_p(buf_ptr), dst_off.ctypes.data,
                                   dst_len.ctypes.data, status.ctypes.data, None)
    assert rc == 0, lib.last_error()
    return dst_off, dst_len, status


@pytest.mark.parametrize("kind", ["pageable", "pinned", "pageable_64MiB"])
def test_slots_inside_a_larger_host_buffer(gpu_lib, kind):
    """Output lands in the slots only: bytes in front of dst_off[0] and behind dst_off[n] are the caller's."""
    import ctypes as C
    if kind == "pageable_64MiB":                                # staged through the library's host threads
        text = _synth(gpu_lib, 80 * MIB, 0, 51)
        files = {"a.txt": text[:40 * MIB], "b.txt": text[40 * MIB:], "c": b"c" * 999}
    else:
        files = _members(gpu_lib)
    arc = gpu_lib.zip_build(files, level=1)
    ents = gpu_lib.zip_list(arc)
    caps = [e.raw_len + 7 for e in ents]
    base, tail = 3 * MIB + 5, 1 * MIB
    size = base + sum(caps) + tail
    pin = None
    if kind == "pinned":
        pin = gpu_lib.dll.zb200_alloc_pinned(size)
        buf = np.ctypeslib.as_array(C.cast(pin, C.POINTER(C.c_uint8)), shape=(size,))
    else:
        buf = np.empty(size, dtype=np.uint8)
    try:
        buf[:] = 0xAB
        dst_off, dst_len, status = _extract_at(gpu_lib, arc, ents, buf.ctypes.data, base, caps)
        assert list(status) == [0] * len(ents)
        for i, e in enumerate(ents):
            a = int(dst_off[i])
            assert int(dst_len[i]) == e.raw_len and buf[a:a + e.raw_len].tobytes() == files[e.name], e.name
        assert (buf[:base] == 0xAB).all() and (buf[int(dst_off[-1]):] == 0xAB).all()
    finally:
        if pin:
            gpu_lib.dll.zb200_free_pinned(C.c_void_p(pin))


def test_member_of_three_gib(gpu_lib):
    """A ZIP32 member above 3 GiB: decoded by the segment route, its CRC-32 in a checksum window of its own."""
    import ctypes as C
    import torch
    n = (3 << 30) + 12345
    src = gpu_lib.synth(n, kind=0, seed=61)
    names = (C.c_char_p * 2)(b"huge.txt", b"small.txt")
    off = np.array([0, n, n + 1000], dtype=np.uint64)
    src2 = np.empty(n + 1000 + 8, dtype=np.uint8)
    src2[:n] = src
    src2[n:n + 1000] = src[:1000]
    cap = gpu_lib.dll.zb200_zip_bound(names, off.ctypes.data, 2)
    arc = np.empty(cap, dtype=np.uint8)
    ol = C.c_size_t(cap)
    assert gpu_lib.dll.zb200_zip_build(names, src2.ctypes.data, off.ctypes.data, 2, 1, zb.DOS_DATETIME, arc.ctypes.data,
                                       C.byref(ol)) == 0, gpu_lib.last_error()
    d_arc = torch.from_numpy(arc[:ol.value]).cuda()
    ents = gpu_lib.zip_list(d_arc)
    assert [e.raw_len for e in ents] == [n, 1000]
    gpu_lib.profile(True)
    outs, st = gpu_lib.zip_extract(d_arc, ents)
    report = gpu_lib.profile_report()
    gpu_lib.profile(False)
    assert st == [0, 0], (st, gpu_lib.last_error())
    d_src = torch.from_numpy(src2[:n + 1000]).cuda()
    assert torch.equal(outs[0], d_src[:n]) and torch.equal(outs[1], d_src[n:])
    assert report["k_find_markers"][1] == 1, report            # planned, not the one-stream fallback
