"""GPU: the streaming half of zlib.h call by call.  inflate() is held to the system zlib call for call (tests/zcalls.py
drives both libraries through the same script); deflate(), whose compressed bytes legitimately differ, is held to
zlib.h's rules for return codes and totals, and its output to what zlib decodes from it after every flush.

  A  every prefix of a stream, in one call and continued in a second
  B  random input pieces and output room over long window-chain streams
  C  receivers of flushed streams, with the sync markers stripped and put back as permessage-deflate does
  D  a reader of concatenated members (inflate, inflateReset, continue from next_in)
  E  inflateCopy at every call boundary, inflateReset against a fresh stream
  F  inflateSync after damage, with the marker split between calls
  G  the deflate() contract over levels, strategies, wraps, windows and flush scripts
  H  the declared window: no distance past the reference's MAX_DIST
  I  the 32 MiB gather boundary of deflate()
  J  deflateCopy and deflateReset
  K  deflateBound and deflateSetHeader"""
import ctypes as C
import gzip
import random
import struct
import zlib

import pytest

import deflate_cases as dc
import deflate_writer as dw
import zcalls
from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

Z_OK, Z_STREAM_END, Z_NEED_DICT, Z_DATA_ERROR, Z_BUF_ERROR = zb.Z_OK, zb.Z_STREAM_END, zb.Z_NEED_DICT, zb.Z_DATA_ERROR, zb.Z_BUF_ERROR
NO, PARTIAL, SYNC, FULL, FINISH = zb.Z_NO_FLUSH, zb.Z_PARTIAL_FLUSH, zb.Z_SYNC_FLUSH, zb.Z_FULL_FLUSH, zb.Z_FINISH
Z_FIXED = 4
JUNK = b"\x07junk after the stream"
MARKER = dc.MARKER
MIB = 1 << 20


@pytest.fixture(scope="module")
def zbz(gpu_lib):
    return zcalls.Api(gpu_lib.dll, "zb200")


@pytest.fixture(scope="module")
def sysz():
    api = zcalls.system_zlib()
    if api is None:
        pytest.fail("no system zlib (libz.so.1) to hold inflate() to")
    return api


def profiled(lib, fn):
    """fn() with per-kernel timing on -> (result, {kernel name: launches})."""
    lib.profile(True)
    try:
        r = fn()
        rep = lib.profile_report()
    finally:
        lib.profile(False)
    return r, {k: v[1] for k, v in rep.items()}


def ran(rep, name):
    return any(name in k for k in rep)


def text(n, seed=0):
    rng = random.Random(seed)
    words = [bytes(rng.choice(b"abcdefghijklmnopqrstuvwxyz") for _ in range(rng.randint(2, 9))) for _ in range(400)]
    out = bytearray()
    while len(out) < n:
        out += rng.choice(words) + (b" " if rng.random() < 0.9 else b".\n")
    return bytes(out[:n])


def noise(n, seed=0):
    return random.Random(seed + 99).randbytes(n)


def alternating(n, seed=0):
    """32 KiB of text, 32 KiB of random bytes, and so on."""
    out = bytearray()
    k = 0
    while len(out) < n:
        out += (text if k % 2 == 0 else noise)(32768, seed + k)
        k += 1
    return bytes(out[:n])


INPUTS = {"text": text, "random": noise, "zeros": lambda n, seed=0: bytes(n), "alternating": alternating}


def sys_deflate(data, level=6, wbits=15, strategy=0, mem_level=8, flushes=(), zdict=None):
    """System zlib; `flushes` is a list of (input offset, flush) -> (stream, [stream length at each flush])."""
    co = zlib.compressobj(level, zlib.DEFLATED, wbits, mem_level, strategy, **({"zdict": zdict} if zdict else {}))
    out, at, pos = bytearray(), [], 0
    for off, fl in flushes:
        out += co.compress(data[pos:off]) + co.flush(fl)
        at.append(len(out))
        pos = off
    out += co.compress(data[pos:]) + co.flush()
    return bytes(out), at


class Pair:
    """An inflate stream in this library and one in zlib, for the same windowBits; every script starts from inflateReset."""

    def __init__(self, zbz, sysz, wbits):
        self.ours, self.ref = zcalls.Stream(zbz, "inflate", wbits), zcalls.Stream(sysz, "inflate", wbits)
        self.raw = wbits < 0

    def run(self, script):
        """-> (our records, zlib's records, first difference or None)."""
        got, want = [], []
        for st, recs in ((self.ours, got), (self.ref, want)):
            st.pending = b""
            assert st.call("reset").rc == Z_OK
            recs += [st.call(*step) for step in script]
        return got, want, zcalls.inflate_diff(got, want, self.raw)

    def close(self):
        self.ours.close()
        self.ref.close()


def block_stops(sysz, z, wbits):
    """Byte offsets where zlib's inflate(Z_BLOCK) stops in z: the header end and every block boundary."""
    st = zcalls.Stream(sysz, "inflate", wbits)
    stops, left = [], z
    for _ in range(100000):
        r = st.call("inflate", left, 1 << 22, zb.Z_BLOCK)
        left = b""
        stops.append(r.total_in)
        if r.rc != Z_OK or (r.used == 0 and not r.out):
            break
    st.close()
    return stops


def cut_points(sysz, z, wbits, rng, every=2048):
    """Every offset of a stream up to `every` bytes; else +-16 bytes around every block start, sync marker, header end
    and trailer start, and 200 random offsets."""
    if len(z) <= every:
        return list(range(len(z) + 1))
    marks = block_stops(sysz, z, wbits) + [len(z) - 8, len(z) - 4]
    i = z.find(MARKER)
    while i >= 0:
        marks.append(i)
        i = z.find(MARKER, i + 1)
    pts = {p + d for p in marks for d in range(-16, 17)} | {rng.randrange(len(z) + 1) for _ in range(200)}
    return sorted(p for p in pts if 0 <= p <= len(z))


# ---- A. every prefix -------------------------------------------------------------------------------------------------
def prefix_streams(kind):
    """(name, stream, windowBits, dictionary) of the group."""
    if kind == "catalogue":
        out = []
        for c in dc.catalogue():
            cutc = c.kind == "cut"
            out.append((c.name + "/raw", c.raw, -15, None))
            out.append((c.name + "/zlib", dw.zlib_wrap(c.raw, c.plain, trailer=not cutc), 15, None))
            out.append((c.name + "/gzip", dw.gzip_wrap(c.raw, c.plain, trailer=not cutc), 31, None))
        return out
    data = text(60000, 5) + noise(3000, 5) + text(20000, 6)
    out = [("sys_level%d" % lv, sys_deflate(data, lv)[0], 15, None) for lv in (0, 1, 6, 9)]
    out += [("sys_fixed", sys_deflate(data, 6, strategy=zlib.Z_FIXED)[0], 15, None),
            ("sys_huffman", sys_deflate(data, 6, strategy=zlib.Z_HUFFMAN_ONLY)[0], 15, None),
            ("sys_raw9", sys_deflate(data[:30000], 9, -15)[0], -15, None),
            ("sys_gzip1", sys_deflate(data[:30000], 1, 31)[0], 31, None)]
    raw = sys_deflate(data[:9000], 6, -15)[0]
    head = b"\x1f\x8b\x08" + bytes([2 | 4 | 8 | 16]) + struct.pack("<I", 1234567) + b"\x00\x03"
    head += struct.pack("<H", 21) + b"XY\x11\x00" + bytes(range(17)) + b"file name.txt\x00" + b"a comment\x00"
    head += struct.pack("<H", zlib.crc32(head) & 0xFFFF)
    out.append(("gzip_all_header_fields", head + raw + struct.pack("<II", zlib.crc32(data[:9000]), 9000), 31, None))
    zd = text(5000, 9)
    out.append(("zlib_fdict", sys_deflate(data[:20000], 6, zdict=zd)[0], 15, zd))
    for w in range(9, 16):
        out.append(("zlib_wbits%d" % w, sys_deflate(data[:40000], 6, w)[0], w, None))
        out.append(("zlib_wbits%d_read15" % w, sys_deflate(data[:6000], 9, w)[0], 15, None))
    return out


@pytest.mark.parametrize("kind", ["catalogue", "zlib_made"])
def test_a_every_prefix(zbz, sysz, kind):
    """Each cut c of a stream: inflate(stream[:c]) with ample room must give what zlib gives for that prefix, call for
    call; the rest of the stream, with junk behind it, in a second call must end it with the junk left in avail_in."""
    rng = random.Random(1951)
    pairs, bad, n = {}, [], 0
    for name, z, wbits, zd in prefix_streams(kind):
        pair = pairs.get(wbits) or pairs.setdefault(wbits, Pair(zbz, sysz, wbits))
        for c in cut_points(sysz, z, wbits, rng):
            script = [("inflate", z[:c], 1 << 17, NO)]
            if zd is not None:
                script.append(("dict", b"", 0, zd))
            script.append(("inflate", z[c:] + JUNK, 1 << 17, NO))
            got, want, diff = pair.run(script)
            n += 1
            if diff:
                bad.append((name, c, len(z), diff))
            elif c == len(z) and want[-1].rc == Z_STREAM_END:
                assert got[-1].avail_in == len(JUNK), (name, got[-1])
    for p in pairs.values():
        p.close()
    assert n > 1000
    assert not bad, (len(bad), bad[:8])


# ---- B. random piece scripts over window-chain streams ---------------------------------------------------------------
PIECES = [0, 1, 7, 4096, None]                                  # None: all that is left
ROOMS = [0, 1, 257, 258, 32767, 32768, 32769, MIB - 1, MIB, MIB + 1, 3 * MIB]


def chain_stream():
    raw, plain = dc.long_stream(77, [32768 + 200000, 700000, 1500000, 40000], lead="chain")
    return raw, plain


def random_script(rng, z, steps):
    """`steps` calls of random input piece and room, then calls of all the rest and 3 MiB of room."""
    script, pos = [], 0
    for _ in range(steps):
        k = rng.choice(PIECES)
        k = len(z) - pos if k is None else min(k, len(z) - pos)
        script.append(("inflate", z[pos:pos + k], rng.choice(ROOMS), NO))
        pos += k
    script.append(("inflate", z[pos:], 3 * MIB, NO))
    script += [("inflate", b"", 3 * MIB, NO)] * 3
    return script


def test_b_random_pieces(gpu_lib, zbz, sysz):
    raw, plain = chain_stream()
    rng = random.Random(4)
    streams = [(raw, -15), (dw.zlib_wrap(raw, plain), 15)]
    bad = []

    def go():
        for z, wbits in streams:
            pair = Pair(zbz, sysz, wbits)
            for k in range(12):
                got, want, diff = pair.run(random_script(rng, z, rng.choice([5, 20, 60])))
                if diff:
                    bad.append((wbits, k, diff))
                elif zcalls.joined(got) != plain:
                    bad.append((wbits, k, "output is not the plaintext"))
            pair.close()
    _, rep = profiled(gpu_lib, go)
    assert not bad, bad[:6]
    assert ran(rep, "k_inflate_stream") and ran(rep, "k_slide_history"), rep


def test_b_finish_first_without_room(gpu_lib, zbz, sysz):
    """A first call with Z_FINISH, the whole stream and too little room: the one-stream decoder is tried (its marker
    search runs) and declines, the call decodes what fits, and later calls finish the stream."""
    raw, plain = chain_stream()
    z = dw.zlib_wrap(raw, plain)
    assert len(z) >= 65536
    bad = []
    for room in (len(plain) // 2, MIB - 1, 1):
        script = [("inflate", z, room, FINISH), ("inflate", b"", MIB, NO), ("inflate", b"", 3 * MIB, FINISH),
                  ("inflate", b"", 3 * MIB, NO)]
        got, rep = profiled(gpu_lib, lambda: zcalls.run(zbz, "inflate", script, wbits=15))
        want = zcalls.run(sysz, "inflate", script, wbits=15)
        diff = zcalls.inflate_diff(got, want)
        if diff:
            bad.append((room, diff))
        assert zcalls.joined(want) == plain and want[-2].rc == Z_STREAM_END
        assert ran(rep, "k_find_markers") or ran(rep, "k_find_blocks"), rep
        assert ran(rep, "k_inflate_stream"), rep
    assert not bad, bad


# ---- C. flush receivers ----------------------------------------------------------------------------------------------
def our_deflate(zbz, data, level, wbits, flushes, strategy=0):
    """This library's deflate(): input up to each flush point, then that flush; -> (stream, [length at each flush])."""
    st = zcalls.Stream(zbz, "deflate", wbits, level, 8, strategy)
    out, at, pos = bytearray(), [], 0
    for off, fl in list(flushes) + [(len(data), FINISH)]:
        r = st.call("deflate", data[pos:off], 2 * (off - pos) + 70000, fl)
        assert r.rc in (Z_OK, Z_STREAM_END) and r.avail_in == 0, r
        out += r.out
        at.append(len(out))
        pos = off
    assert r.rc == Z_STREAM_END
    st.close()
    return bytes(out), at[:-1]


@pytest.mark.parametrize("writer", ["zlib", "zb200"])
@pytest.mark.parametrize("flush", [SYNC, FULL, PARTIAL])
def test_c_flush_receivers(zbz, sysz, writer, flush):
    rng = random.Random(flush * 7 + (writer == "zlib"))
    data = alternating(300000, 3)
    offs = sorted(rng.sample(range(1, len(data)), 14) + [70000, 70001, 70003])
    fl = [(o, flush) for o in offs]
    bad = []
    for wbits in (-15, 15, 31):
        z, at = sys_deflate(data, 6, wbits, flushes=fl) if writer == "zlib" else our_deflate(zbz, data, 6, wbits, fl)
        bounds = [0] + at
        script = [("inflate", z[a:b], MIB, NO) for a, b in zip(bounds, bounds[1:])] + [("inflate", z[bounds[-1]:], MIB, NO)]
        variants = [script]
        if flush != PARTIAL:
            # permessage-deflate: each message without its 00 00 FF FF, the receiver appends it
            assert all(z[b - 4:b] == MARKER for b in at)
            msgs = [z[a:b - 4] for a, b in zip(bounds, bounds[1:])]
            variants.append([("inflate", m + MARKER, MIB, NO) for m in msgs] + script[-1:])
            variants.append([s for m in msgs for s in (("inflate", m, MIB, NO), ("inflate", MARKER, MIB, NO))] + script[-1:])
        for v, sc in enumerate(variants):
            pair = Pair(zbz, sysz, wbits)
            got, want, diff = pair.run(sc)
            pair.close()
            if diff:
                bad.append((wbits, v, diff))
                continue
            # up to each flush point, all input so far has come out and no input is left
            step = 2 if v == 2 else 1
            for i, off in enumerate(offs):
                r = got[(i + 1) * step - 1]
                if zcalls.joined(got[:(i + 1) * step]) != data[:off] or r.avail_in != 0:
                    bad.append((wbits, v, "flush %d at %d: %d bytes out, %d left" % (i, off, r.total_out, r.avail_in)))
                    break
            if zcalls.joined(got) != data:
                bad.append((wbits, v, "whole output differs"))
    assert not bad, bad[:6]


# ---- D. multi-member reader ------------------------------------------------------------------------------------------
def member_reader(api, z, wbits, piece):
    """inflate until Z_STREAM_END, inflateReset, continue from next_in -- in pieces of `piece` bytes -> records."""
    st = zcalls.Stream(api, "inflate", wbits)
    recs, pos, ended = [], 0, False
    for _ in range(200000):
        if ended:
            recs.append(st.call("reset"))
            ended = False
            if not st.pending and pos >= len(z):
                break
        k = min(piece, len(z) - pos)
        r = st.call("inflate", z[pos:pos + k], 4096, NO)
        pos += k
        recs.append(r)
        if r.rc == Z_STREAM_END:
            ended = True
        elif r.rc not in (Z_OK, Z_BUF_ERROR) or (pos >= len(z) and not r.out and not r.used):
            break
    st.close()
    return recs


def test_d_member_reader(zbz, sysz):
    rng = random.Random(12)
    parts = [text(rng.randint(0, 9000), k) if k % 3 else noise(rng.randint(0, 3000), k) for k in range(7)] + [b""]
    gz = b"".join(gzip.compress(p, compresslevel=rng.choice([1, 6, 9]), mtime=0) for p in parts)
    zl = b"".join(zlib.compress(p, rng.choice([0, 1, 6, 9])) for p in parts)
    bad = []
    for name, z, wbits in (("gzip", gz, 31), ("gzip_auto", gz, 47), ("zlib", zl, 15), ("gzip_junk", gz + JUNK, 31),
                           ("zlib_junk", zl + b"\x00" * 3, 15), ("gzip_trailing_zeros", gz + bytes(40), 31)):
        for piece in (1, 7, 4096):
            got = member_reader(zbz, z, wbits, piece)
            want = member_reader(sysz, z, wbits, piece)
            diff = zcalls.inflate_diff(got, want)
            if diff:
                bad.append((name, piece, diff))
            assert sum(r.rc == Z_STREAM_END for r in want) == len(parts), name
            assert zcalls.joined(want) == b"".join(parts)
    assert not bad, bad[:6]


# ---- E. inflateCopy and inflateReset ---------------------------------------------------------------------------------
def copy_stream():
    """A gzip member whose 7-byte pieces and 5-byte rooms stop calls inside the header, inside a dynamic block header
    (held as pending input), inside a stored block, with a match copy pending, and inside the trailer -> (stream,
    plaintext, {region: (first byte, end byte) in the stream}, the writer's matches as (position, length, distance))."""
    rng = random.Random(5)
    d = dw.Deflate()
    d.fixed(list(b"hello, hello, hello") + [(258, 7), (40, 3)])
    dyn = d.bitpos
    d.dynamic(list(rng.randbytes(40)) + [(258, 33), (100, 1)], dc.FLAT_LIT, dc.FLAT_DIST)
    empty = dw.Deflate()
    empty.dynamic([], dc.FLAT_LIT, dc.FLAT_DIST)                # the same header and an end-of-block code of 8 or 9 bits
    stored = d.bitpos
    d.stored(rng.randbytes(150))
    stored_end = d.bitpos
    d.fixed([(258, 1), (258, 100), 65, (30, 2)], final=True)
    raw, plain = d.result()
    head = b"\x1f\x8b\x08" + bytes([4 | 8]) + bytes(4) + b"\x00\x03" + struct.pack("<H", 9) + b"extra-fld" + b"a name\x00"
    z = head + raw + struct.pack("<II", zlib.crc32(plain), len(plain))
    h = len(head)
    regions = {"header": (0, h), "dynamic header": (h + dyn // 8, h + (dyn + empty.bitpos - 9) // 8),
               "stored block": (h + (stored + 3 + 7) // 8 + 4, h + stored_end // 8), "trailer": (len(z) - 8, len(z))}
    return z, plain, regions, list(d.copies)


def copy_run(api, z, at, piece=7, room=5):
    """Piecewise decode; inflateCopy before call `at`; both streams go on with the same calls (the copy finishes with one
    call of the rest) -> (original's records, copy's records)."""
    st = zcalls.Stream(api, "inflate", 31)
    orig, cp, other, pos, k = [], [], None, 0, 0
    while k < 4000 and not (orig and orig[-1].rc == Z_STREAM_END):
        if k == at:
            rc, other = st.copy()
            assert rc == Z_OK
        step = ("inflate", z[pos:pos + piece], room, NO)
        orig.append(st.call(*step))
        if other is not None and len(cp) < 4:
            cp.append(other.call(*step))
        pos += piece
        k += 1
        if orig[-1].rc not in (Z_OK, Z_BUF_ERROR):
            break
    if other is not None:
        cp.append(other.call("inflate", z[len(cp) * piece + at * piece:], 1 << 16, NO))
        other.close()
    st.close()
    return orig, cp


def test_e_inflate_copy_every_boundary(gpu_lib, zbz, sysz):
    z, plain, regions, copies = copy_stream()
    ref = copy_run(sysz, z, -1)[0]
    calls = len(ref)
    # the states the copies are taken in: a call boundary (7 bytes fed per call) strictly inside each region, and a call
    # that filled its room in the middle of a match
    for name, (lo, hi) in regions.items():
        assert any(lo < 7 * k < hi for k in range(1, calls)), (name, lo, hi)
    assert any(r.avail_out == 0 and any(p < r.total_out < p + n for p, n, _ in copies) for r in ref)
    bad = []

    def go():
        for at in range(calls):
            go, gc = copy_run(zbz, z, at)
            wo, wc = copy_run(sysz, z, at)
            for what, g, w in (("original", go, wo), ("copy", gc, wc)):
                diff = zcalls.inflate_diff(g, w)
                if diff:
                    bad.append((at, what, diff))
            assert zcalls.joined(wo) == plain
            assert zcalls.joined(wo[:at]) + zcalls.joined(wc) == plain
    _, rep = profiled(gpu_lib, go)
    assert not bad, bad[:6]
    assert ran(rep, "k_inflate_stream") and ran(rep, "k_slide_history"), rep


def test_e_inflate_reset_is_fresh(gpu_lib, zbz, sysz):
    """A stream reused after inflateReset -- left at the end, in an error, mid-stream, and waiting for a dictionary --
    decodes as a fresh one does."""
    _, rep = profiled(gpu_lib, lambda: reset_checks(zbz, sysz))
    assert ran(rep, "k_inflate_stream") and ran(rep, "k_slide_history"), rep


def reset_checks(zbz, sysz):
    z, plain = copy_stream()[:2]
    zd = text(3000, 2)
    zdict = sys_deflate(text(5000, 3), 6, zdict=zd)[0]
    before = {"end": [("inflate", z, MIB, NO)], "error": [("inflate", z[:40] + b"\xff" * 30, MIB, NO)],
              "middle": [("inflate", z[:100], 3, NO)]}
    script = [("inflate", z[:13], 5, NO), ("inflate", z[13:200], 100, NO), ("inflate", z[200:], MIB, NO),
              ("inflate", JUNK, 10, NO)]
    for api in (zbz, sysz):
        fresh = zcalls.run(api, "inflate", script, wbits=31)
        for name, pre in before.items():
            st = zcalls.Stream(api, "inflate", 31)
            for step in pre:
                st.call(*step)
            st.pending = b""
            assert st.call("reset").rc == Z_OK
            after = [st.call(*step) for step in script]
            st.close()
            assert after == fresh, (api.name, name)
        assert zcalls.joined(fresh) == plain
    assert zcalls.inflate_diff(zcalls.run(zbz, "inflate", script, wbits=31), zcalls.run(sysz, "inflate", script, wbits=31)) is None
    st = zcalls.Stream(zbz, "inflate", 15)
    assert st.call("inflate", zdict[:20], MIB, NO).rc == Z_NEED_DICT
    st.pending = b""
    assert st.call("reset").rc == Z_OK
    zz = zlib.compress(plain)
    assert [st.call("inflate", zz, MIB, NO)][0][:4] == ("inflate", Z_STREAM_END, len(zz), plain)
    st.close()


# ---- F. inflateSync --------------------------------------------------------------------------------------------------
def damaged(seed, wbits=-15):
    """A stream with a full-flush point every 8 KiB of input, damaged in its second segment so that zlib stops with
    Z_DATA_ERROR there -> (stream, end of the first call's input, marker offset behind the damage)."""
    data = text(80000, seed)
    z, at = sys_deflate(data, 6, wbits, flushes=[(o, FULL) for o in range(8192, len(data), 8192)])
    rng = random.Random(seed)
    sysz = zcalls.system_zlib()
    for _ in range(200):
        p = rng.randrange(at[0] + 20, at[1] - 60)
        bad = z[:p] + bytes(rng.randrange(256) for _ in range(6)) + z[p + 6:]
        e = at[1] - 24                                          # the first call ends 20 bytes before the marker
        r = zcalls.run(sysz, "inflate", [("inflate", bad[:e], MIB, NO)], wbits=wbits)[0]
        if r.rc == Z_DATA_ERROR and bad.find(MARKER, r.total_in) == at[1] - 4:
            return bad, e, at[1] - 4
    raise AssertionError("no damage found that zlib refuses")


@pytest.mark.parametrize("split", [None, 1, 2, 3])
def test_f_inflate_sync(zbz, sysz, split):
    bad = []
    for seed in range(6):
        z, e, m = damaged(seed)
        assert m > e
        if split is None:
            sync = [("sync", z[e:], 0, 0)]
        else:
            sync = [("sync", z[e:m + split], 0, 0), ("sync", z[m + split:], 0, 0)]
        script = [("inflate", z[:e], MIB, NO)] + sync + [("inflate", b"", MIB, NO), ("inflate", b"", MIB, NO)]
        got = zcalls.run(zbz, "inflate", script, wbits=-15)
        want = zcalls.run(sysz, "inflate", script, wbits=-15)
        assert want[0].rc == Z_DATA_ERROR and want[len(sync)].rc == Z_OK and want[-2].rc == Z_STREAM_END, want
        assert want[len(sync)].total_in == m + 4                # zlib resumes right behind the marker that was split
        diff = zcalls.inflate_diff(got, want, raw=True)
        if diff:
            bad.append((seed, diff))
    assert not bad, bad


# ---- G. deflate() contract, H. declared window -----------------------------------------------------------------------
def flush_script(rng, n, kind, wrap):
    """Steps of one deflate run: ("data", length, flush), ("params", level, strategy), ("prime", bits, value)."""
    steps, pos = [], 0
    if kind == "prime":
        bits = rng.randint(1, 16)
        steps.append(("prime", bits, rng.getrandbits(bits)))
    while pos < n:
        k = min(n - pos, rng.choice([1, 3, 7, rng.randint(1, 3000), rng.randint(1, 40000)]))
        pos += k
        if kind == "params" and rng.random() < 0.3:
            steps.append(("data", k, NO))
            lv, sg = rng.choice([(0, 0), (rng.randint(1, 9), Z_FIXED),
                                 (rng.randint(1, 9), 0), (rng.randint(0, 9), rng.randint(0, 4))])
            steps.append(("params", lv, sg))
        else:
            fl = rng.choice([NO, NO, SYNC, FULL, PARTIAL]) if kind in ("flushes", "prime") else NO
            steps.append(("data", k, fl))
            if fl != NO and rng.random() < 0.3:                 # flushes 1 to 7 bytes apart
                k2 = min(n - pos, rng.randint(1, 7))
                pos += k2
                steps.append(("data", k2, rng.choice([SYNC, FULL, PARTIAL])))
    return steps


def decode_so_far(out, wrap, wbits, prime, room=4 * MIB):
    """What zlib's streaming decoder yields from the output so far.  A raw stream behind `prime` = (bits, value) of
    deflatePrime is read from the byte that holds its first bit, the rest of that byte given to inflatePrime, so that
    stored blocks keep their alignment."""
    w = {0: -wbits, 1: wbits, 2: 16 + wbits}[wrap]
    if not prime:
        return zlib.decompressobj(w).decompress(out)
    k, r = divmod(prime[0], 8)
    assert int.from_bytes(out[:k + 1], "little") & ((1 << prime[0]) - 1) == prime[1]
    st = zcalls.Stream(zcalls.system_zlib(), "inflate", -15)
    if r:
        assert st.call("prime", b"", 0, (8 - r, out[k] >> r)).rc == Z_OK
    got = st.call("inflate", out[k + (1 if r else 0):], room, NO)
    st.close()
    assert got.rc in (Z_OK, Z_STREAM_END, Z_BUF_ERROR), got
    return got.out


def run_deflate_contract(zbz, data, level, strategy, wrap, wbits, steps, room_rng):
    """Runs the steps on this library; asserts zlib.h's rules after every call -> (stream, [problems])."""
    w = {0: -wbits, 1: wbits, 2: 16 + wbits}[wrap]
    st = zcalls.Stream(zbz, "deflate", w, level, 8, strategy)
    out, pos, probs, prime, last_flush = bytearray(), 0, [], None, NO
    full_at = None

    def check(tag, r, launched):
        if launched:
            if r.total_in != pos or r.total_out != len(out):
                probs.append((tag, "totals", r.total_in, pos, r.total_out, len(out)))
            want_adler = zlib.adler32(data[:pos]) if wrap == 1 else zlib.crc32(data[:pos]) if wrap == 2 else None
            if want_adler is not None and r.adler != want_adler:
                probs.append((tag, "adler", hex(r.adler), hex(want_adler)))

    for step in steps + [("data", 0, FINISH)]:
        if step[0] == "prime":
            r = st.call("prime", b"", 0, (step[1], step[2]))
            assert r.rc == Z_OK
            prime = (step[1], step[2])
            continue
        if step[0] == "params":
            r = st.call("params", b"", len(data) + 4096, (step[1], step[2]))
            out += r.out
            if r.rc != Z_OK and not (r.rc == Z_BUF_ERROR and last_flush == PARTIAL and r.total_in == pos):
                probs.append(("params", step[1:], r.rc))
            last_flush = PARTIAL
            continue
        _, k, fl = step
        piece = data[pos:pos + k]
        pos += k
        room = room_rng.choice([len(piece) + 1000, 3 * len(piece) + 70000, 1 << 22]) if fl != NO else 1 << 22
        r = st.call("deflate", piece, room, fl)
        out += r.out
        while r.rc == Z_OK and len(r.out) == room and fl != NO:
            r = st.call("deflate", b"", room, fl)                # zlib.h: call again while avail_out comes back 0
            out += r.out
        want_rc = Z_STREAM_END if fl == FINISH else Z_OK
        if fl == NO and not piece:
            want_rc = Z_BUF_ERROR
        if fl not in (NO, FINISH) and not piece and fl <= last_flush and r.avail_in == 0 and not r.out:
            want_rc = Z_BUF_ERROR                               # no new input and no stronger flush
        if r.rc != want_rc or r.avail_in:
            probs.append((step, "rc", r.rc, want_rc, r.avail_in))
            break
        last_flush = fl
        if fl != NO:
            check(step, r, True)
            if fl != FINISH:
                got = decode_so_far(bytes(out), wrap, wbits, prime)
                if got != data[:pos]:
                    probs.append((step, "decodes to %d of %d bytes" % (len(got), pos)))
                    break
            if fl == FULL:
                full_at = (len(out), pos)
    st.close()
    z = bytes(out)
    if not probs:
        if decode_so_far(z, wrap, wbits, prime) != data:
            probs.append("whole stream")
        if full_at and not prime:
            tail = zlib.decompressobj(-15).decompress(z[full_at[0]:])
            if tail != data[full_at[1]:]:
                probs.append(("after the last Z_FULL_FLUSH", len(tail), len(data) - full_at[1]))
    return z, prime, probs


def window_problems(oracle, z, wrap, wbits, n):
    """Decodes with the oracle; the largest distance must be inside MAX_DIST of the declared window."""
    rc, o, _ = oracle.inflate(z, n + 16, wrap)
    limit = 32768 if wbits == 15 else (1 << wbits) - 262
    if rc != 0:
        return ("oracle rc", rc)
    if oracle.last_max_dist() > limit:
        return ("distance", oracle.last_max_dist(), "window", wbits, "limit", limit)
    return None


def g_cases():
    rng = random.Random(2026)
    cases = []
    for strategy in range(5):
        for wrap in (0, 1, 2):
            for kind in INPUTS:
                script = rng.choice(["flushes", "flushes", "params"] + (["prime"] if wrap == 0 else []))
                cases.append((rng.randint(0, 9), strategy, wrap, 15 if script == "prime" else rng.choice([9, 12, 15]), kind, script))
    for level in (1, 6, 9):                                     # defect 1: Z_FIXED with partial flushes on random bytes
        for wbits in (9, 15):
            cases.append((level, Z_FIXED, rng.choice([0, 1, 2]), wbits, "random", "partial"))
        cases.append((level, 4, 1, 15, "random", "params_out_of_fixed"))
    for level in range(10):
        cases.append((level, rng.randint(0, 4), rng.randint(0, 2), rng.choice([9, 12, 15]), rng.choice(list(INPUTS)), "flushes"))
    return cases


@pytest.mark.parametrize("case", g_cases(), ids=lambda c: "L%d_s%d_w%d_b%d_%s_%s" % c)
def test_g_deflate_contract(zbz, oracle, case):
    level, strategy, wrap, wbits, kind, script = case
    rng = random.Random(repr(case))                              # the same script in every process
    n = 140000 if kind == "alternating" else 60000
    data = INPUTS[kind](n, 1)
    if script == "partial":
        steps, pos = [], 0
        while pos < n:
            k = min(n - pos, rng.choice([2000, 2100, 1, 5000]))
            pos += k
            steps.append(("data", k, PARTIAL))
    elif script == "params_out_of_fixed":
        steps = [("data", 2000, NO), ("params", 6, 0), ("data", 3000, NO), ("params", 6, 4), ("data", 2500, NO),
                 ("params", 0, 0), ("data", n - 7500, NO)]
    else:
        steps = flush_script(rng, n, script, wrap)
    z, prime, probs = run_deflate_contract(zbz, data, level, strategy, wrap, wbits, steps, rng)
    assert not probs, probs[:4]
    if wbits < 15 and not prime:
        assert window_problems(oracle, z, wrap, wbits, n) is None


@pytest.mark.parametrize("wbits", [9, 12, 15])
def test_h_dictionary_longer_than_window(zbz, oracle, wbits):
    """deflateSetDictionary with 40 000 bytes on a raw stream of a small window: the stream, behind stored blocks that
    carry the dictionary, decodes to dictionary + input, and reaches no further back than the window allows."""
    zd = text(40000, 8)
    data = zd[-3000:] + text(30000, 8)[:20000] + zd[5000:9000]
    for level in (1, 6, 9):
        st = zcalls.Stream(zbz, "deflate", -wbits, level)
        assert st.call("dict", b"", 0, zd).rc == Z_OK
        r = st.call("deflate", data, 1 << 20, FINISH)
        st.close()
        assert r.rc == Z_STREAM_END
        lead = b"".join(b"\x00" + struct.pack("<HH", len(b), len(b) ^ 0xFFFF) + b for b in (zd[:20000], zd[20000:]))
        rc, o, _ = oracle.inflate(lead + r.out, len(zd) + len(data) + 16, 0)
        assert rc == 0 and o == zd + data, (wbits, level, rc)
        limit = 32768 if wbits == 15 else (1 << wbits) - 262
        assert 0 < oracle.last_max_dist() <= limit, (wbits, level, oracle.last_max_dist())


# ---- I. the 32 MiB gather boundary -----------------------------------------------------------------------------------
@pytest.mark.parametrize("n,variant", [(32 * MIB - 1, ""), (32 * MIB, ""), (32 * MIB + 1, ""), (70 * MIB + 5, ""),
                                       (64 * MIB + 4000, "partial"), (32 * MIB + 5, "prime"),
                                       (32 * MIB, "finish_on_boundary")])
def test_i_gather_boundary(gpu_lib, zbz, n, variant):
    """Input in 1 MiB pieces with Z_NO_FLUSH, so that deflate() launches on its own every 32 MiB.  "partial": a
    Z_PARTIAL_FLUSH 3 bytes before 32 MiB, then 32 MiB more, so the bits it leaves pending enter an unforced batch.
    "prime": a raw stream behind 5 bits of deflatePrime, which the first unforced batch carries."""
    data = gpu_lib.synth(n, kind=1, seed=n & 0xFF).tobytes()
    wrap = 0 if variant == "prime" else 1
    st = zcalls.Stream(zbz, "deflate", -15 if wrap == 0 else 15, 1)
    prime = None
    if variant == "prime":
        prime = (5, 0x15)
        assert st.call("prime", b"", 0, prime).rc == Z_OK
    out, pos = bytearray(), 0
    while pos < n:
        k = min(MIB, n - pos)
        fl = NO
        if variant == "partial" and pos < 32 * MIB - 3 <= pos + k:
            k, fl = 32 * MIB - 3 - pos, PARTIAL
        if variant == "finish_on_boundary" and pos + k == n:
            fl = FINISH
        r = st.call("deflate", data[pos:pos + k], 64 * MIB, fl)
        pos += k
        out += r.out
        assert r.rc in ((Z_OK,) if fl != FINISH else (Z_STREAM_END,)) and r.avail_in == 0, (pos, r.rc)
        assert r.total_in == pos and r.total_out == len(out)
        if fl == PARTIAL:
            assert zlib.decompressobj().decompress(bytes(out)) == data[:pos]
    if variant != "finish_on_boundary":
        r = st.call("deflate", b"", 64 * MIB, FINISH)
        out += r.out
        assert r.rc == Z_STREAM_END
    assert r.total_out == len(out) and (wrap == 0 or r.adler == zlib.adler32(data))
    st.close()
    assert decode_so_far(bytes(out), wrap, 15, prime, room=n + MIB) == data


# ---- J. deflateCopy and deflateReset ---------------------------------------------------------------------------------
def test_j_deflate_copy_and_reset(zbz):
    rng = random.Random(31)
    data = alternating(200000, 4)
    for wrap, w in ((0, -15), (1, 12), (2, 31)):
        for trial in range(4):
            st = zcalls.Stream(zbz, "deflate", w, rng.choice([1, 6, 9]), 8, rng.choice([0, 1, 3]))
            cut = rng.randrange(1000, len(data) - 1000)
            pre = bytearray()
            # gather input; then, on odd trials, a flush whose output does not fit, so some of it is still held
            r = st.call("deflate", data[:cut], 1 << 22, NO)
            pre += r.out
            if trial % 2:
                r = st.call("deflate", b"", 100, SYNC)
                pre += r.out
                assert r.rc == Z_OK and len(r.out) == 100
            rc, cp = st.copy()
            assert rc == Z_OK
            tails = []
            for s in (st, cp):
                t = bytearray()
                for step in (("deflate", b"", 1 << 22, NO if not trial % 2 else SYNC), ("deflate", data[cut:cut + 500], 1 << 22, FULL),
                             ("deflate", data[cut + 500:], 1 << 22, FINISH)):
                    r = s.call(*step)
                    t += r.out
                assert r.rc == Z_STREAM_END, r
                tails.append(bytes(t))
                s.close()
            assert tails[0] == tails[1], (wrap, trial)
            z = bytes(pre) + tails[0]
            assert zlib.decompressobj(w).decompress(z) == data
        # deflateReset: the bytes of a fresh stream
        script = [("deflate", data[:70000], 1 << 22, NO), ("deflate", data[70000:90000], 1 << 22, PARTIAL),
                  ("deflate", data[90000:], 1 << 22, FINISH)]
        fresh = zcalls.run(zbz, "deflate", script, wbits=w, level=6)
        st = zcalls.Stream(zbz, "deflate", w, 6)
        st.call("deflate", data[:5000], 1 << 22, PARTIAL)
        st.call("deflate", data[5000:9000], 10, NO)
        st.pending = b""
        assert st.call("reset").rc == Z_OK
        again = [st.call(*s) for s in script]
        st.close()
        assert [(r.rc, r.out, r.total_in, r.total_out, r.adler) for r in again] == \
               [(r.rc, r.out, r.total_in, r.total_out, r.adler) for r in fresh], wrap


# ---- K. deflateBound and deflateSetHeader ----------------------------------------------------------------------------
BOUND_N = [0, 1, 2, 100, 65535, 65536, 131071, 131072, 131073, MIB + 7]


@pytest.mark.parametrize("wrap", [0, 1, 2])
def test_k_deflate_bound(zbz, wrap):
    """One deflate(Z_FINISH) into exactly deflateBound(strm, n) bytes ends the stream."""
    inputs = {kind: INPUTS[kind](MIB + 7, 6) for kind in ("random", "text")}
    bad = []
    for strategy in range(5):
        for level in (0, 1, 6, 9):
            for wbits in (9, 15):
                for mem in (1, 8, 9):
                    w = {0: -wbits, 1: wbits, 2: 16 + wbits}[wrap]
                    st = zcalls.Stream(zbz, "deflate", w, level, mem, strategy)
                    for kind, src in inputs.items():
                        for n in BOUND_N:
                            assert st.call("reset").rc == Z_OK
                            b = st.bound(n)
                            r = st.call("deflate", src[:n], b, FINISH)
                            if r.rc != Z_STREAM_END:
                                bad.append((strategy, level, wbits, mem, kind, n, b, r.rc))
                            elif n in (0, 100, MIB + 7) and zlib.decompressobj(w).decompress(r.out) != src[:n]:
                                bad.append((strategy, level, wbits, mem, kind, n, "does not decode"))
                    st.close()
    assert not bad, (len(bad), bad[:10])


def test_k_set_header(zbz, sysz):
    fields = [dict(), dict(name=b"x.txt"), dict(comment=b"about it", hcrc=1),
              dict(text=1, time=0x5F00AB12, os_=11, extra=b"AB\x04\x00wxyz", name=b"name", comment=b"c" * 300, hcrc=1),
              dict(extra=b"", hcrc=1)]
    data = text(50000, 3)
    for f in fields:
        for n in (0, 1000, 50000):
            st = zcalls.Stream(zbz, "deflate", 31, 6)
            assert st.set_header(**f) == Z_OK
            b = st.bound(n)
            r = st.call("deflate", data[:n], b, FINISH)
            st.close()
            assert r.rc == Z_STREAM_END, (f, n, b)
            z = r.out
            assert gzip.decompress(z) == data[:n]
            rd = zcalls.Stream(sysz, "inflate", 31)
            h = rd.get_header(room=512)
            ri = rd.call("inflate", z, n + 10, NO)
            rd.close()
            assert ri.rc == Z_STREAM_END and ri.out == data[:n], (f, ri.rc, ri.msg)
            assert h.done == 1 and h.hcrc == f.get("hcrc", 0) and h.text == f.get("text", 0)
            assert h.time == f.get("time", 0) and h.os == f.get("os_", 3)
            if "extra" in f:
                assert h.extra_len == len(f["extra"]) and C.string_at(h.extra, h.extra_len) == f["extra"]
            else:
                assert not h.extra
            for key, ptr in (("name", h.name), ("comment", h.comment)):
                if key in f:
                    assert C.string_at(ptr) == f[key]
                else:
                    assert not ptr
