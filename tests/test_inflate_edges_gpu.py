"""GPU: the hand-built DEFLATE catalogue (tests/deflate_cases.py, checked against system zlib and the oracle by
tests/test_deflate_writer_cpu.py) through every inflate route -- the batch kernel, the streaming ABI, the one-stream
segment decoder of uncompress() with each way of finding segment starts, the planned segment decode of zb200_zip_extract,
zb200_gunzip, and a batch of a few long streams -- against the oracle: status, output, and where the API reports them
input used and message.  Every test also asserts which kernels ran, so a case meant for one decoder cannot pass on
another."""
import ctypes as C
import functools
import gzip
import random

import numpy as np
import pytest

import deflate_cases as dc
import deflate_writer as dw
from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

CATALOGUE = dc.catalogue()
WBITS = {zb.WRAP_RAW: -15, zb.WRAP_ZLIB: 15, zb.WRAP_GZIP: 31}


def wrapped(raw, plain, wrap, cut=False):
    if wrap == zb.WRAP_ZLIB:
        return dw.zlib_wrap(raw, plain, trailer=not cut)
    if wrap == zb.WRAP_GZIP:
        return dw.gzip_wrap(raw, plain, trailer=not cut)
    return raw


def profiled(lib, fn):
    """fn() with per-kernel timing on -> (result, {kernel: launches})."""
    lib.profile(True)
    try:
        r = fn()
        rep = lib.profile_report()
    finally:
        lib.profile(False)
    return r, {k: v[1] for k, v in rep.items()}


SEG_EMIT, SEG_COUNT = "(k_inflate_segments<true>)", "(k_inflate_segments<false>)"


# ---- a. the batch kernel ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("wrap", [zb.WRAP_RAW, zb.WRAP_ZLIB, zb.WRAP_GZIP])
def test_batch_kernel_catalogue(gpu_lib, oracle, wrap):
    """Every case in one call (more than 8 streams, so none leaves the batch kernel), at capacities exact, exact - 1,
    exact + 17 and 0; exact is what the oracle produces with room to spare (for invalid cases: up to the damage)."""
    zs = [wrapped(c.raw, c.plain, wrap, c.kind == "cut") for c in CATALOGUE]
    full = [len(oracle.inflate(z, (len(c.plain) if c.plain else 0) + (1 << 17), wrap)[1]) for z, c in zip(zs, CATALOGUE)]
    for name, caps in (("exact", full), ("minus1", [max(n - 1, 0) for n in full]), ("plus17", [n + 17 for n in full]),
                       ("zero", [0] * len(full))):
        want = [oracle.inflate(z, cap, wrap)[:2] for z, cap in zip(zs, caps)]
        (outs, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch(zs, caps, wrap=wrap))
        assert "k_inflate_batch" in rep and SEG_EMIT not in rep and SEG_COUNT not in rep, rep
        bad = [(c.name, s, w[0], len(o), len(w[1])) for c, s, o, w in zip(CATALOGUE, st, outs, want) if (s, o) != w]
        assert not bad, (name, bad[:20])
    # the valid cases decode to the writer's plaintext
    outs, st = gpu_lib.inflate_batch(zs, full, wrap=wrap)
    assert [c.name for c, o in zip(CATALOGUE, outs) if c.kind == "ok" and o != c.plain] == []


def test_batch_dev_unaligned(gpu_lib, oracle):
    """inflate_batch_dev on device buffers: every stream starts 1-3 bytes behind the end of the one in front (every
    residue mod 4), every output slot at an odd offset.  A stream's range runs to the next one's start, so the padding
    behind it is part of its input: the valid and invalid cases never read it (they end, or fail, before), the cut
    cases would, and are left to the batch test above."""
    import torch
    cases = [c for c in CATALOGUE if c.kind != "cut"]
    zs = [wrapped(c.raw, c.plain, zb.WRAP_ZLIB) for c in cases]
    want = [oracle.inflate(z, (len(c.plain) if c.plain else 0) + (1 << 17), zb.WRAP_ZLIB)[:2] for z, c in zip(zs, cases)]
    n = len(zs)
    src, so = bytearray(), []
    for i, z in enumerate(zs):
        src += b"\xa5" * (1 + i % 3)
        so.append(len(src))
        src += z
    so.append(len(src))
    caps = [len(w[1]) + 5 for w in want]
    do = np.zeros(n + 1, dtype=np.int64)
    do[0] = 3
    do[1:] = 3 + np.cumsum(caps)
    d_src = torch.from_numpy(np.frombuffer(bytes(src) + b"\0" * 8, dtype=np.uint8).copy()).cuda()
    d_so = torch.tensor(so, dtype=torch.int64).cuda()
    d_do = torch.from_numpy(do).cuda()
    d_dst = torch.zeros(int(do[-1]) + 8, dtype=torch.uint8, device="cuda")
    d_len = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_st = torch.full((n,), -99, dtype=torch.int32, device="cuda")
    _, rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_dev(d_src.data_ptr(), d_so.data_ptr(), n, d_dst.data_ptr(),
                                                                 d_do.data_ptr(), d_len.data_ptr(), d_st.data_ptr(),
                                                                 zb.WRAP_ZLIB, torch.cuda.current_stream()))
    torch.cuda.synchronize()
    assert "k_inflate_batch" in rep and SEG_EMIT not in rep, rep
    dst, lens, sts = d_dst.cpu().numpy(), d_len.cpu().numpy(), d_st.cpu().numpy()
    bad = []
    for i, (c, w) in enumerate(zip(cases, want)):
        got = (int(sts[i]), dst[int(do[i]):int(do[i]) + int(lens[i])].tobytes())
        if got != w:
            bad.append((c.name, got[0], w[0], len(got[1]), len(w[1])))
    assert not bad, bad[:20]


# ---- b. the streaming ABI --------------------------------------------------------------------------------------------
def _pieces(c, z):
    """(input piece, output piece) sizes for a case: big pieces always, byte-sized ones for the small cases."""
    ps = [(4096, 65536)]
    n = len(c.plain) if c.plain else 0
    if len(z) <= 1200 and n <= 2500:
        ps += [(1, 65536), (3, 5), (7, 1), (4096, 1)]
    return ps


def test_streaming_catalogue(gpu_lib, oracle):
    """inflate() fed in pieces of 1, 3, 7 and 4096 bytes with 1, 5 and 65536 bytes of room per call: valid cases end with
    Z_STREAM_END, the plaintext and all input used; invalid ones with Z_DATA_ERROR and the oracle's message; cut ones
    with the oracle's output and no end."""
    bad = []
    for k, c in enumerate(CATALOGUE):
        wrap = (zb.WRAP_ZLIB, zb.WRAP_RAW, zb.WRAP_GZIP)[k % 3]
        z = wrapped(c.raw, c.plain, wrap, c.kind == "cut")
        rc_o, out_o, _ = oracle.inflate(z, (len(c.plain) if c.plain else 0) + (1 << 17), wrap)
        msg_o = oracle.last_msg()
        for ip, op in _pieces(c, z):
            rc, out, msg, tin = gpu_lib.inflate_stream(z, wbits=WBITS[wrap], in_chunk=ip, out_chunk=op)
            if c.kind == "ok":
                good = (rc, out, msg, tin) == (zb.Z_STREAM_END, c.plain, None, len(z))
            elif c.kind == "bad":
                good = (rc, out, msg) == (zb.Z_DATA_ERROR, out_o, msg_o) and rc_o == zb.Z_DATA_ERROR
            else:
                good = rc in (zb.Z_OK, zb.Z_BUF_ERROR) and (out, msg) == (out_o, None)
            if not good:
                bad.append((c.name, wrap, ip, op, rc, msg, msg_o, len(out), len(out_o)))
    assert not bad, bad[:20]


def test_streaming_runs_the_stream_kernel(gpu_lib):
    c = next(c for c in CATALOGUE if c.name == "codes_15bit")
    (rc, out, msg, tin), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_stream(dw.zlib_wrap(c.raw, c.plain), in_chunk=7))
    assert rc == zb.Z_STREAM_END and out == c.plain
    assert "k_inflate_stream" in rep and "k_inflate_batch" not in rep and SEG_EMIT not in rep, rep


# ---- c. one long stream: uncompress() and the segment decoder -------------------------------------------------------------
def _sizes(seed, total, lo=40000, hi=250000):
    rng = random.Random(seed)
    out = []
    while total > hi + lo:                                      # every piece, the last one too, is lo bytes or more
        out.append(rng.randint(lo, hi))
        total -= out[-1]
    return out + [total]


@functools.lru_cache(maxsize=None)
def long_case(name):
    """(raw, plain) of the long streams."""
    if name == "marker_chunks_far":                             # markers every 128 KiB, each segment opens with dist 32768
        return dc.long_stream(11, dc.chunked_sizes((3 << 20) + 5555), lead="far")
    if name == "marker_chunks_run":                             # ... with a dist-1 run of 258 over the segment start
        return dc.long_stream(12, dc.chunked_sizes((2 << 20) + 77777), lead="run")
    if name == "marker_chunks_none":                            # no tail holds window symbols
        return dc.long_stream(13, dc.chunked_sizes((2 << 20) + 54321), lead="none")
    if name == "marker_irregular":                              # markers at irregular output sizes: the counting pass
        return dc.long_stream(14, _sizes(14, 3 << 20), lead="far")
    if name == "no_markers":                                    # non-final dynamic blocks only: the block finder
        return dc.long_stream(15, _sizes(15, 3 << 20, 20000, 90000), markers=False)
    # Window chains: every tail depends on the one in front (tests/test_deflate_writer_cpu.py counts them), so the
    # tails past the parallel rounds (4 for one stream, 64 in the planned decode) are left to the walk of
    # k_resolve_tails.  The chain streams have no 32 KiB period: a byte read from the wrong slot of its ring is wrong.
    if name == "period_32k":                                    # output with a period of 32 KiB
        return dc.long_stream(16, dc.chunked_sizes((6 << 20) + 1234), lead="period")
    if name == "period_32k_long":                               # longer than the planned decode's 64 tail rounds
        return dc.long_stream(17, dc.chunked_sizes((9 << 20) + 99), lead="period")
    if name == "chain_chunks":
        return dc.long_stream(18, dc.chunked_sizes((6 << 20) + 4321), lead="chain")
    if name == "chain_irregular":                               # the counting pass: segments not on 128 KiB bounds
        return dc.long_stream(19, _sizes(19, 4 << 20), lead="chain")
    if name == "chain_long":                                    # longer than the planned decode's 64 tail rounds
        return dc.long_stream(20, dc.chunked_sizes((9 << 20) + 77), lead="chain")
    raise KeyError(name)


# how each stream's segment starts are found: the assumed 128 KiB layout, the counting pass over sync markers, or the
# block finder
LONG = {"marker_chunks_far": "layout", "marker_chunks_run": "layout", "marker_chunks_none": "layout",
        "marker_irregular": "count", "no_markers": "finder", "period_32k": "layout", "chain_chunks": "layout",
        "chain_irregular": "count"}


@pytest.mark.parametrize("name", sorted(LONG))
def test_uncompress_long_stream(gpu_lib, oracle, name):
    raw, plain = long_case(name)
    z = dw.zlib_wrap(raw, plain)
    assert oracle.inflate(z, len(plain), 1)[:2] == (0, plain)
    (rc, out), rep = profiled(gpu_lib, lambda: gpu_lib.uncompress(z, len(plain)))
    assert rc == zb.Z_OK and out == plain
    assert rep.get(SEG_EMIT) and "k_inflate_batch" not in rep, rep
    if LONG[name] == "layout":
        assert rep[SEG_EMIT] == 1 and SEG_COUNT not in rep, rep  # the assumed layout held: no counting pass
    elif LONG[name] == "count":
        assert rep.get(SEG_COUNT) and "k_find_blocks_check" not in rep, rep
    else:
        assert rep.get("k_find_blocks_probe") and rep.get("k_find_blocks_check") and rep.get(SEG_COUNT), rep
    # k_tails_round and k_resolve_tails are launched for every stream (k_resolve_tails returns when the rounds left
    # nothing open): that the walk did its work for the chains shows in the output alone
    rc, _ = gpu_lib.uncompress(z, len(plain) - 1)
    assert rc == oracle.inflate(z, len(plain) - 1, 1)[0] == zb.Z_BUF_ERROR


@pytest.mark.parametrize("name", sorted(dc.long_invalid_blocks()))
def test_uncompress_invalid_in_later_segment(gpu_lib, oracle, name):
    """An invalid construct at the start of segment 2 of a stream with markers every 128 KiB: the segment decoder must
    refuse it, and the serial decoder then reports the oracle's code."""
    raw, plain = dc.long_stream(9, dc.chunked_sizes(4 * dc.CHUNK), bad_at=2, bad_block=dc.long_invalid_blocks()[name])
    z = dw.zlib_wrap(raw, plain)
    want = oracle.inflate(z, 4 * dc.CHUNK + 4096, 1)[0]
    (rc, out), rep = profiled(gpu_lib, lambda: gpu_lib.uncompress(z, 4 * dc.CHUNK + 4096))
    assert want == zb.Z_DATA_ERROR and rc == want, (rc, want)
    assert rep.get(SEG_EMIT) and rep.get("k_inflate_batch"), rep     # tried in segments, decided serially


def test_uncompress_too_far_in_first_segment(gpu_lib, oracle):
    """A distance past the output inside segment 0: the segment decoder's own rule for the first segment refuses it (the
    check value is that of a decoder that read zeros there), the serial decoder reports the oracle's code."""
    raw, plain = dc.long_stream(22, dc.chunked_sizes(4 * dc.CHUNK + 20000), bad_at=0, bad_block=dc.far_in_first_segment)
    z = dw.zlib_wrap(raw, plain)
    (rc, out), rep = profiled(gpu_lib, lambda: gpu_lib.uncompress(z, len(plain)))
    assert rc == oracle.inflate(z, len(plain), 1)[0] == zb.Z_DATA_ERROR
    assert rep.get(SEG_EMIT) and rep.get("k_inflate_batch"), rep


def test_uncompress_cut_in_later_segment(gpu_lib, oracle):
    raw, plain = long_case("marker_chunks_none")
    for keep in (len(raw) * 3 // 5, len(raw) - 1):
        z = dw.zlib_wrap(raw[:keep], plain, trailer=False)
        rc, _ = gpu_lib.uncompress(z, len(plain))
        assert rc == oracle.inflate(z, len(plain), 1)[0] == zb.Z_DATA_ERROR


# ---- d. zip_extract: the planned segment decode ---------------------------------------------------------------------------
ZIP_LONG = ["marker_chunks_far", "marker_chunks_run", "marker_chunks_none", "period_32k_long", "chain_long"]
ZIP_SHORT = ["codes_15bit", "hlit286_hdist30", "repeat_codes_min_max", "stored65535_phase5", "deferred_store_dist7"]


def _zip_members(damaged):
    by = {c.name: c for c in CATALOGUE}
    ms = [(n, *long_case(n)) for n in ZIP_LONG] + [(n, by[n].raw, by[n].plain) for n in ZIP_SHORT]
    if damaged:
        # a block of type 3 in segment 2, and a distance past the output in segment 0; the directory's CRC-32 is that of
        # the plaintext the writer meant (zeros in front of the output), so only the refusal of the data stops them
        for k, (at, block) in enumerate(((2, dc.long_invalid_blocks()["block_type_3"]), (0, dc.far_in_first_segment))):
            raw, plain = dc.long_stream(21 + k, dc.chunked_sizes(4 * dc.CHUNK + 20000), bad_at=at, bad_block=block)
            ms.insert(2 + 2 * k, ("damaged%d" % k, raw, plain))
    for n, raw, plain in ms:
        assert n.startswith("damaged") or raw.count(dc.MARKER) == (len(plain) + dc.CHUNK - 1) // dc.CHUNK - 1 or len(plain) <= dc.CHUNK
    return ms


def _extract(lib, archive, entries, dst, dst_off):
    n = len(entries)
    recs = np.zeros(n, dtype=zb._zip_entry_dtype())
    for i, e in enumerate(entries):
        recs[i] = e.raw
    off = np.array(dst_off, dtype=np.uint64)
    dlen = np.zeros(n, dtype=np.uint64)
    st = np.full(n, -99, dtype=np.int32)
    pa, keep = zb._ptr(archive)
    rc = lib.dll.zb200_zip_extract(pa, zb._nbytes(archive), recs.ctypes.data, n, C.c_void_p(dst), off.ctypes.data,
                                   dlen.ctypes.data, st.ctypes.data, None)
    assert rc == 0, lib.last_error()
    return [int(x) for x in dlen], [int(x) for x in st]


@pytest.mark.parametrize("where", ["host", "device"])
def test_zip_extract_planned(gpu_lib, oracle, where):
    """Members written by the deflate writer with exactly ceil(n / 128 KiB) - 1 markers take the planned segment decode,
    among them a chain of window references longer than its 64 tail rounds.  Output slots start at odd offsets (host) or
    behind an unaligned base (device), so the tails are stored byte by byte.  On the host a damaged member sits among the
    good ones: they fail alone, with the oracle's code, and the others stay on the plan (one emit launch for all of them;
    each damaged one adds one speculative and one counting attempt before the batch kernel decides it)."""
    import torch
    damaged = where == "host"
    ms = _zip_members(damaged)
    archive, _ = dw.zip_archive([(n, raw, plain) for n, raw, plain in ms])
    entries = gpu_lib.zip_list(archive)
    assert [e.name for e in entries] == [m[0] for m in ms]
    caps = [e.raw_len + 3 for e in entries]
    base = 7 if where == "host" else 0
    offs = [base]
    for c in caps:
        offs.append(offs[-1] + c)
    if where == "host":
        buf = np.zeros(offs[-1] + 16, dtype=np.uint8)
        (lens, st), rep = profiled(gpu_lib, lambda: _extract(gpu_lib, archive, entries, buf.ctypes.data, offs))
        get = lambda i: buf[offs[i]:offs[i] + lens[i]].tobytes()
    else:
        d_arc = torch.from_numpy(np.frombuffer(archive, dtype=np.uint8).copy()).cuda()
        d_buf = torch.zeros(offs[-1] + 16, dtype=torch.uint8, device="cuda")
        (lens, st), rep = profiled(gpu_lib, lambda: _extract(gpu_lib, d_arc, entries, d_buf.data_ptr() + 3, offs))
        torch.cuda.synchronize()
        host = d_buf.cpu().numpy()
        get = lambda i: host[3 + offs[i]:3 + offs[i] + lens[i]].tobytes()
    for i, (n, raw, plain) in enumerate(ms):
        if n.startswith("damaged"):
            assert st[i] == oracle.inflate(raw, len(plain), 0)[0] == zb.Z_DATA_ERROR, (n, st)
        else:
            assert st[i] == 0 and get(i) == plain, (n, st[i], lens[i], len(plain))
    assert rep.get(SEG_EMIT) == (3 if damaged else 1), rep
    assert rep.get(SEG_COUNT, 0) == (2 if damaged else 0), rep
    assert rep.get("k_inflate_batch"), rep                         # the short members
    # the chain members go past the 64 tail rounds: their last tails are resolved by the walk, which only the output shows


# ---- e. gunzip ----------------------------------------------------------------------------------------------------------------
def test_gunzip_members(gpu_lib):
    names = ["marker_chunks_far", "marker_chunks_run", "period_32k", "chain_chunks", "marker_chunks_none"]
    blob = b"".join(dw.gzip_wrap(*long_case(n)) for n in names)
    want = gzip.decompress(blob)
    assert want == b"".join(long_case(n)[1] for n in names)
    out, rep = profiled(gpu_lib, lambda: gpu_lib.gunzip(blob))
    assert out == want and gpu_lib.last_members == len(names)
    assert rep.get(SEG_EMIT) and "k_inflate_batch" not in rep, rep


# ---- f. a batch of a few long streams and short ones ------------------------------------------------------------------------
def test_batch_few_long_streams(gpu_lib, oracle):
    """Eight streams: three long ones take the one-stream segment decoder each, the short catalogue cases the batch
    kernel, all in one call; then the same with one long stream damaged in a later segment."""
    longs = [long_case(n) for n in ("marker_chunks_far", "marker_irregular", "no_markers")]
    shorts = [c for c in CATALOGUE if c.name in ("codes_15bit", "len284_extra31_dynamic", "dist_to_first_byte_32768",
                                                 "stored0_phase3", "straddle_phase17")]
    items = [longs[0], (shorts[0].raw, shorts[0].plain), longs[1], (shorts[1].raw, shorts[1].plain), longs[2]] + \
        [(c.raw, c.plain) for c in shorts[2:]]
    zs = [dw.zlib_wrap(r, p) for r, p in items]
    plains = [p for _, p in items]
    (outs, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch(zs, [len(p) for p in plains]))
    assert st == [0] * 8 and outs == plains
    # each long stream alone: the segment decoder and no batch kernel; in the call of eight, the segment launches are the
    # sum of those (so none of the three fell to the batch kernel), the block finder and the counting pass among them
    alone = {}
    for k in (0, 2, 4):
        (o1, s1), r1 = profiled(gpu_lib, lambda: gpu_lib.inflate_batch([zs[k]], [len(plains[k])]))
        assert s1 == [0] and o1 == [plains[k]] and r1.get(SEG_EMIT) and "k_inflate_batch" not in r1, r1
        for name in (SEG_EMIT, SEG_COUNT, "k_find_blocks_probe"):
            alone[name] = alone.get(name, 0) + r1.get(name, 0)
    assert {name: rep.get(name, 0) for name in alone} == alone, (rep, alone)
    assert alone[SEG_COUNT] >= 2 and alone["k_find_blocks_probe"] == 1 and rep.get("k_inflate_batch"), rep
    raw, plain = dc.long_stream(9, dc.chunked_sizes(4 * dc.CHUNK), bad_at=2, bad_block=dc.long_invalid_blocks()["repeat16_first"])
    zs[2] = dw.zlib_wrap(raw, plain)
    caps = [len(p) for p in plains]
    caps[2] = len(plain)
    outs, st = gpu_lib.inflate_batch(zs, caps)
    want2 = oracle.inflate(zs[2], caps[2], 1)[0]
    assert st[2] == want2 == zb.Z_DATA_ERROR
    assert [s for i, s in enumerate(st) if i != 2] == [0] * 7
    assert [o for i, o in enumerate(outs) if i != 2] == [p for i, p in enumerate(plains) if i != 2]
