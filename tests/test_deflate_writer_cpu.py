"""CPU: the hand-built DEFLATE catalogue (tests/deflate_cases.py) is what it claims to be, for both references: system
zlib and the oracle decode every valid case to the writer's plaintext and consume the whole stream; both refuse every
invalid case, the oracle with the expected message.  The GPU tests of the same catalogue trust it through this file."""
import time
import zlib

import numpy as np
import pytest

import deflate_cases as dc
import deflate_writer as dw

CATALOGUE = dc.catalogue()
BY_NAME = {c.name: c for c in CATALOGUE}


def test_catalogue_names_unique_and_short():
    assert len(BY_NAME) == len(CATALOGUE)
    assert all(len(c.raw) <= 65535 + 64 for c in CATALOGUE)     # short: one stored block of 65535 at most
    kinds = [c.kind for c in CATALOGUE]
    assert kinds.count("ok") >= 180 and kinds.count("bad") >= 25 and kinds.count("cut") == 3


@pytest.mark.parametrize("name", [c.name for c in CATALOGUE if c.kind == "ok"])
def test_valid_case(name, oracle):
    c = BY_NAME[name]
    d = zlib.decompressobj(-15)
    assert d.decompress(c.raw) == c.plain
    assert d.eof and d.unused_data == b""
    rc, out, used = oracle.inflate(c.raw, len(c.plain), 0)
    assert (rc, used) == (0, len(c.raw)) and out == c.plain
    for wrap, z in ((1, dw.zlib_wrap(c.raw, c.plain)), (2, dw.gzip_wrap(c.raw, c.plain))):
        assert zlib.decompress(z, {1: 15, 2: 31}[wrap]) == c.plain
        rc, out, used = oracle.inflate(z, len(c.plain), wrap)
        assert (rc, used) == (0, len(z)) and out == c.plain


def _oracle_shape(oracle, raw, n):
    """(rc, output length) of the oracle at capacities n (what it produces with room), n - 1, n + 17 and 0."""
    return [(r[0], len(r[1])) for r in (oracle.inflate(raw, cap, 0) for cap in (n, max(n - 1, 0), n + 17, 0))]


@pytest.mark.parametrize("name", [c.name for c in CATALOGUE if c.kind != "ok"])
def test_invalid_case(name, oracle):
    c = BY_NAME[name]
    d = zlib.decompressobj(-15)
    if c.kind == "bad":
        with pytest.raises(zlib.error) as e:
            d.decompress(c.raw)
        assert str(e.value).endswith(": " + c.msg), str(e.value)
    else:                                                       # cut: no error yet, but no end either
        d.decompress(c.raw)
        assert not d.eof
    rc, out, _ = oracle.inflate(c.raw, 1 << 20, 0)
    assert rc == -3 and oracle.last_msg() == c.msg
    n = len(out)
    if c.plain is not None:                                     # what the tokens meant up to the damage
        assert c.plain.startswith(out)
    shape = _oracle_shape(oracle, c.raw, n)
    # with room for everything in front of the damage the damage is reported; with less the output runs out first
    assert shape[0] == (-3, n) and shape[2] == (-3, n)
    assert shape[1][1] == max(n - 1, 0) and shape[3][1] == 0
    if n:   # out of room: a buffer error while input is left, else a data error (uncompr.c:53-55)
        assert shape[1][0] in (-5, -3) and shape[3][0] in (-5, -3)
    else:
        assert shape[1] == shape[3] == (-3, 0)


def test_case_contents():
    """Spot checks that the constructs the names promise are in the streams."""
    c = BY_NAME["hlit286_hdist30"]
    h = int.from_bytes(c.raw[5 + 32768:5 + 32768 + 3], "little")     # behind the stored block of noise
    assert (h & 7, (h >> 3) & 31, (h >> 8) & 31) == (0b101, 29, 29)  # final dynamic block, HLIT 286, HDIST 30
    for p in range(8):
        raw = BY_NAME["stored65535_phase%d" % p].raw
        assert raw[-65535 - 4:-65535] == b"\xff\xff\x00\x00"          # LEN / NLEN right in front of the data
    assert BY_NAME["dist32768_len3_258"].plain[32768:32771] == BY_NAME["dist32768_len3_258"].plain[:3]


def test_repeat16_first_is_otherwise_valid():
    """The case with a leading 16 is refused for that code alone: with three zeros in its place the same header is
    valid and decodes to the plaintext the wrappers' check values cover."""
    d = dw.Deflate()
    dc._repeat16_first(d, opening=[(0, 0)] * 3)
    raw, plain = d.result()
    assert zlib.decompress(raw, -15) == plain == BY_NAME["repeat16_first"].plain
    for p in (BY_NAME["repeat16_first"].raw, dc.long_stream(9, dc.chunked_sizes(4 * dc.CHUNK), bad_at=2,
                                                            bad_block=dc.long_invalid_blocks()["repeat16_first"])[0]):
        with pytest.raises(zlib.error, match="invalid bit length repeat"):
            zlib.decompress(p, -15)


def test_canonical_codes_rfc1951_example():
    """RFC 1951 3.2.2: lengths (3, 3, 3, 3, 3, 2, 4, 4) give codes 010 011 100 101 110 00 1110 1111."""
    codes = dw.canonical([3, 3, 3, 3, 3, 2, 4, 4])
    want = ["010", "011", "100", "101", "110", "00", "1110", "1111"]
    assert [int(w[::-1], 2) for w in want] == codes


def test_fixed_block_matches_zlib():
    """A fixed block of the writer decodes to the plaintext it computed."""
    data = b"abcabcabcabcabcabc" + bytes(range(256)) + b"x" * 300
    d = dw.Deflate()
    d.fixed(list(b"abc") + [(15, 3)] + list(range(256)) + [120, (258, 1), (41, 1)], final=True)
    raw, plain = d.result()
    assert plain == data and zlib.decompress(raw, -15) == data


def test_zip_writer_reads_back():
    import io
    import zipfile
    c1, c2 = BY_NAME["codes_15bit"], BY_NAME["repeat_codes_min_max"]
    arc, offs = dw.zip_archive([("a.bin", c1.raw, c1.plain), ("dir/b.bin", c2.raw, c2.plain)])
    z = zipfile.ZipFile(io.BytesIO(arc))
    assert z.read("a.bin") == c1.plain and z.read("dir/b.bin") == c2.plain
    assert arc[offs[0]:offs[0] + len(c1.raw)] == c1.raw


def test_long_streams_build_fast_and_decode():
    """The long streams of the GPU tests: layouts as intended (markers, sizes), bit-exact for system zlib, and built in
    seconds (a 16 MiB stream included)."""
    t0 = time.time()
    raw, plain = dc.long_stream(5, dc.chunked_sizes((16 << 20) + 12345), lead="period")
    assert time.time() - t0 < 20
    assert len(plain) == (16 << 20) + 12345 and zlib.decompress(raw, -15) == plain
    assert raw.count(b"\x00\x00\xff\xff") == len(dc.chunked_sizes(len(plain))) - 1
    for lead in ("far", "run", "none"):
        sizes = dc.chunked_sizes((1 << 20) + 77777)
        raw, plain = dc.long_stream(7, sizes, lead=lead)
        assert len(plain) == sum(sizes) and zlib.decompress(raw, -15) == plain
        # every marker ends a piece: the piece sizes are the output between markers
        d = zlib.decompressobj(-15)
        pos, outs = 0, []
        for k in range(len(sizes) - 1):
            m = raw.index(b"\x00\x00\xff\xff", pos) + 4
            outs.append(len(d.decompress(raw[pos:m])))
            pos = m
        assert outs == sizes[:-1]
    raw, plain = dc.long_stream(8, [40000, 70000, 50000, 90000], markers=False)
    assert b"\x00\x00\xff\xff" not in raw and zlib.decompress(raw, -15) == plain and len(plain) == 250000


@pytest.mark.parametrize("lead", ["chain", "period"])
def test_chain_streams_every_tail_depends_on_the_one_in_front(lead):
    """In the chain streams every tail of the 128 KiB layout holds bytes that come from the segment in front (the
    dependent tails form one chain through the stream, longer than any number of parallel rounds); the chain stream's
    output has no period of 32 KiB, so a byte read from a wrong ring slot is a wrong byte."""
    d = dc.long_writer(16, dc.chunked_sizes((2 << 20) + 1234), lead=lead)
    raw, plain = d.result()
    assert zlib.decompress(raw, -15) == plain
    starts = list(range(0, len(plain), dc.CHUNK))
    assert dc.tails_with_window_symbols(d.copies, starts, len(plain)) == list(range(1, len(starts)))
    a = np.frombuffer(plain, dtype=np.uint8)
    differ = int((a[32768:] != a[:-32768]).sum())
    if lead == "chain":
        assert differ > len(plain) // 2
    else:
        assert differ == 0
    # the other leads: every tail is noise of its own segment
    d = dc.long_writer(7, dc.chunked_sizes((1 << 20) + 77777), lead="far")
    assert dc.tails_with_window_symbols(d.copies, starts[:9], d.pos) == []


def test_far_in_first_segment(oracle):
    """A distance past the output in segment 0: refused by both references; the writer's plaintext (and so the check
    values) is what a decoder that read zeros in front of the output would produce."""
    d = dc.long_writer(22, dc.chunked_sizes(4 * dc.CHUNK + 20000), bad_at=0, bad_block=dc.far_in_first_segment)
    raw, plain = d.result()
    assert len(plain) == 4 * dc.CHUNK + 20000 and raw.count(dc.MARKER) == 4
    with pytest.raises(zlib.error, match="invalid distance too far back"):
        zlib.decompress(raw, -15)
    assert oracle.inflate(raw, len(plain), 0)[0] == -3 and oracle.last_msg() == "invalid distance too far back"
    assert plain[2 + 20480:2 + 20480 + 100] == bytes(100) and plain[2 + 20480 + 100:2 + 20480 + 258] == plain[:158]


@pytest.mark.parametrize("name", sorted(dc.long_invalid_blocks()))
def test_long_stream_with_invalid_block(name, oracle):
    raw, plain = dc.long_stream(9, dc.chunked_sizes(4 * dc.CHUNK), bad_at=2, bad_block=dc.long_invalid_blocks()[name])
    with pytest.raises(zlib.error):
        zlib.decompress(raw, -15)
    rc, out, _ = oracle.inflate(raw, 4 * dc.CHUNK, 0)
    assert rc == -3 and len(out) >= 2 * dc.CHUNK
