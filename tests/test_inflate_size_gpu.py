"""GPU: zb200_inflate_batch_size and its device form -- the sizes, input spans and statuses that zb200_inflate_batch
would report, found without producing any output.  Every test asserts which kernels ran: the size calls never run the
emit pass of the segment decoder or the decoding batch kernel, and each stream's route (count kernel, sync markers, block
finder) is the one the routing rule gives it."""
import ctypes as C
import base64
import functools
import json
import os
import random
import zlib

import numpy as np
import pytest

import deflate_cases as dc
import deflate_writer as dw
from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

WRAP_AUTO = 3
CATALOGUE = dc.catalogue()
SEG_EMIT, SEG_COUNT = "(k_inflate_segments<true>)", "(k_inflate_segments<false>)"
COUNT, DECODE = "k_inflate_count", "k_inflate_batch"
HUGE = 1 << 40


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


def no_decode(rep):
    assert SEG_EMIT not in rep and DECODE not in rep, rep


def size_arena(lib, src, src_off, wrap, limit=0, used=True):
    """zb200_inflate_batch_size over an arena (numpy, pinned address or CUDA tensor) -> (out_len, src_used, status)."""
    n = len(src_off) - 1
    off = np.asarray(src_off, dtype=np.uint64)
    ol = np.zeros(max(n, 1), dtype=np.uint64)
    su = np.zeros(max(n, 1), dtype=np.uint64)
    st = np.full(max(n, 1), -99, dtype=np.int32)
    p, keep = zb._ptr(src)
    rc = lib.dll.zb200_inflate_batch_size(p, off.ctypes.data, n, ol.ctypes.data, su.ctypes.data if used else None,
                                          st.ctypes.data, wrap, limit, None)
    assert rc == 0, lib.last_error()
    return [int(x) for x in ol[:n]], [int(x) for x in su[:n]], [int(x) for x in st[:n]]


def oracle_want(oracle, z, cap, wrap):
    """(status, length) the size call must report: the oracle's, but a stream whose only fault is its check value is Z_OK."""
    rc, out, used = oracle.inflate(z, cap, wrap)
    if rc == zb.Z_DATA_ERROR and oracle.last_msg() == "incorrect data check":
        return (zb.Z_OK, len(out)), None
    return (rc, len(out)), used


# ---- catalogue: every hand-built case, all in the count kernel ------------------------------------------------------------
@pytest.mark.parametrize("wrap", [zb.WRAP_RAW, zb.WRAP_ZLIB, zb.WRAP_GZIP])
def test_catalogue(gpu_lib, oracle, wrap):
    zs = [wrapped(c.raw, c.plain, wrap, c.kind == "cut") for c in CATALOGUE]
    full = [len(oracle.inflate(z, (len(c.plain) if c.plain else 0) + (1 << 17), wrap)[1]) for z, c in zip(zs, CATALOGUE)]
    (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size(zs, wrap=wrap))
    assert rep.get(COUNT) and SEG_COUNT not in rep, rep
    no_decode(rep)
    bad = []
    for c, z, o, u, s in zip(CATALOGUE, zs, ol, su, st):
        want, used = oracle_want(oracle, z, HUGE >> 20, wrap)
        if (s, o) != want:
            bad.append((c.name, s, o, want))
        elif c.kind == "ok" and not (u == used == len(z)):
            bad.append((c.name, "src_used", u, used, len(z)))
    assert not bad, bad[:20]
    # the decode reproduces the lengths and statuses from slots of exactly these sizes
    outs, st2 = gpu_lib.inflate_batch(zs, ol, wrap=wrap)
    assert [len(o) for o in outs] == ol
    assert [c.name for c, a, b in zip(CATALOGUE, st, st2) if a != b and b != zb.Z_DATA_ERROR] == []
    # limits: exact - 1 and exact per stream (each in a call of nine copies: still the count kernel), 0 = none
    for name, lim in (("minus1", [n - 1 for n in full]), ("exact", full)):
        caps = [max(x, 0) for x in lim]
        dec_outs, dec_st = gpu_lib.inflate_batch(zs, caps, wrap=wrap)
        bad = []
        for k, (c, z, L) in enumerate(zip(CATALOGUE, zs, lim)):
            if L <= 0:
                continue                                           # limit 0 means none: the unlimited run above
            (ol9, _, st9), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size([z] * 9, wrap=wrap, limit=L))
            assert rep.get(COUNT) and DECODE not in rep, rep
            want, _ = oracle_want(oracle, z, L, wrap)
            got = (st9[0], ol9[0])
            dec = (dec_st[k], len(dec_outs[k]))
            if got != want or len(set(zip(ol9, st9))) != 1 or (dec != got and not (dec[0] == zb.Z_DATA_ERROR and got[0] == zb.Z_OK)):
                bad.append((c.name, name, L, got, want, dec))
        assert not bad, bad[:20]


# ---- corpus: system zlib at every setting, and this library's own deflate ---------------------------------------------------
def _plain(rng, n, base):
    kind = rng.randrange(4)
    if kind == 0:
        return rng.randbytes(n)
    if kind == 1:
        return bytes(n)
    out = bytearray()
    while len(out) < n:
        a = rng.randrange(len(base) - 4096)
        out += base[a:a + rng.randint(16, 4096)]
        if kind == 3:
            out += rng.randbytes(rng.randint(0, 64))
    return bytes(out[:n])


@functools.lru_cache(maxsize=None)
def corpus():
    """{wrap: [(stream, plaintext)]}: system zlib, levels 0-9, all strategies, windowBits 9-15, 0 B - 4 MiB."""
    rng = random.Random(2026)
    base = _base_text()
    out = {zb.WRAP_RAW: [], zb.WRAP_ZLIB: [], zb.WRAP_GZIP: [], WRAP_AUTO: []}
    sizes = [0, 1, 2, 3, 257, 258, 32768, 65535, 65536, 65537, 4 << 20]
    for k in range(2200):
        n = sizes[k] if k < len(sizes) else int(min(4 << 20, 2 ** rng.uniform(0, 17.5)))
        if k % 97 == 5:
            n = rng.randint(1 << 20, 4 << 20)
        plain = _plain(rng, n, base)
        wrap = (zb.WRAP_RAW, zb.WRAP_ZLIB, zb.WRAP_GZIP, WRAP_AUTO)[k % 4]
        level, strategy, wb = k % 10, (k // 10) % 5, 9 + (k // 50) % 7
        wbits = -wb if wrap == zb.WRAP_RAW else wb + 16 if (wrap == zb.WRAP_GZIP or (wrap == WRAP_AUTO and k % 8 == 3)) else wb
        co = zlib.compressobj(level, zlib.DEFLATED, wbits, 8, strategy)
        out[wrap].append((co.compress(plain) + co.flush(), plain))
    return out


@functools.lru_cache(maxsize=None)
def _base_text():
    import zhelpers
    return zhelpers.corpus(1, 1 << 20, 5)


def _with_tail(rng, z):
    return z + rng.randbytes(rng.randint(1, 40))


@pytest.mark.parametrize("wrap", [zb.WRAP_RAW, zb.WRAP_ZLIB, zb.WRAP_GZIP, WRAP_AUTO])
def test_corpus(gpu_lib, wrap):
    items = list(corpus()[wrap])
    if wrap == zb.WRAP_ZLIB:                                       # this library's own streams
        plains = [_plain(random.Random(i), 1000 * i * i, _base_text()) for i in range(40)]
        for lv in (1, 6, 9):
            zs, st, _, _ = gpu_lib.deflate_batch(plains, level=lv)
            assert st == [0] * len(plains)
            items += list(zip(zs, plains))
    assert len(items) >= 500
    rng = random.Random(wrap)
    spans = [_with_tail(rng, z) for z, _ in items]
    (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size(spans, wrap=wrap))
    assert rep.get(COUNT), rep
    no_decode(rep)
    bad = [(k, s, o, len(p), u, len(z)) for k, ((z, p), o, u, s) in enumerate(zip(items, ol, su, st))
           if (s, o, u) != (0, len(p), len(z))]
    assert not bad, bad[:20]
    outs, sts = gpu_lib.decompress_batch(spans, wrap=wrap)
    assert sts == [0] * len(items)
    assert [k for k, (o, (_, p)) in enumerate(zip(outs, items)) if o != p] == []


# ---- damaged streams -------------------------------------------------------------------------------------------------------------
def test_corrupt_golden(gpu_lib, oracle):
    es = json.load(open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "corrupt.json")))
    zs = [base64.b64decode(e["z"]) for e in es]
    (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size(zs))
    no_decode(rep)
    caps = [max(o, e["cap"]) + 4096 for o, e in zip(ol, es)]
    outs, dst = gpu_lib.inflate_batch(zs, caps)
    bad = []
    for k, (z, cap) in enumerate(zip(zs, caps)):
        dec = (dst[k], len(outs[k]))
        oracle.inflate(z, cap, 1)
        if oracle.last_msg() == "incorrect data check":
            ok = (st[k], ol[k]) == (zb.Z_OK, dec[1]) and dec[0] == zb.Z_DATA_ERROR
        else:
            ok = (st[k], ol[k]) == dec
        if not ok:
            bad.append((k, st[k], ol[k], dec, oracle.last_msg()))
    assert not bad, bad[:20]


# ---- long streams: the counting pass alone, or the count kernel -------------------------------------------------------------
@functools.lru_cache(maxsize=None)
def long_streams():
    """{name: (zlib stream, plain length, route)}."""
    import torch
    from zlib_b200 import load, synth
    lib = load()
    out = {}
    n = 1 << 30
    d_src = torch.from_numpy(synth.synth(n, 1, 3)).cuda()
    d_dst = torch.empty(lib.compress_bound(n) + 4096, dtype=torch.uint8, device="cuda")
    for lv in (1, 6):
        m = lib.deflate(d_src.data_ptr(), n, d_dst.data_ptr(), d_dst.numel(), lv, zb.WRAP_ZLIB)
        out[f"zb200_L{lv}_1GiB"] = (d_dst[:m].cpu().numpy().tobytes(), n, "markers")
    del d_src, d_dst
    text = synth.synth(64 << 20, 0, 7).tobytes()
    out["zlib_L6_text_64MiB"] = (zlib.compress(text, 6), len(text), "finder")
    out["zlib_L0_64MiB"] = (zlib.compress(text, 0), len(text), "declined")
    co = zlib.compressobj(6, zlib.DEFLATED, 15, 8, zlib.Z_FIXED)
    out["zlib_fixed_64MiB"] = (co.compress(text) + co.flush(), len(text), "declined")
    return out


LONG = ["zb200_L1_1GiB", "zb200_L6_1GiB", "zlib_L6_text_64MiB", "zlib_L0_64MiB", "zlib_fixed_64MiB"]


@pytest.mark.parametrize("name", LONG)
def test_long_stream(gpu_lib, name):
    z, n, route = long_streams()[name]
    shorts = [dw.zlib_wrap(c.raw, c.plain) for c in CATALOGUE if c.kind == "ok"][:8]
    for batch in ([z], [shorts[0], z, shorts[1]]):
        (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size(batch))
        k = batch.index(z)
        assert (st[k], ol[k], su[k]) == (0, n, len(z)), (name, st[k], ol[k], su[k], n, len(z))
        no_decode(rep)
        if route == "markers":
            assert rep.get(SEG_COUNT) and rep.get("k_find_markers") and "k_find_blocks_probe" not in rep, rep
        elif route == "finder":
            assert rep.get(SEG_COUNT) and rep.get("k_find_blocks_check"), rep
        else:
            assert rep.get(COUNT), rep
        if route != "declined":                                    # the count kernel only for the short streams around it
            assert bool(rep.get(COUNT)) == (len(batch) > 1), rep
    if len(z) < (32 << 20):                                        # in a call of more than eight: the count kernel
        batch = shorts + [z]
        (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size(batch))
        assert (st[-1], ol[-1], su[-1]) == (0, n, len(z))
        assert rep.get(COUNT) and SEG_COUNT not in rep, rep


@pytest.mark.parametrize("name", sorted(dc.long_invalid_blocks()))
def test_long_invalid(gpu_lib, name):
    raw, plain = dc.long_stream(9, dc.chunked_sizes(4 * dc.CHUNK), bad_at=2, bad_block=dc.long_invalid_blocks()[name])
    z = dw.zlib_wrap(raw, plain)
    outs, dst = gpu_lib.inflate_batch([z], [4 * dc.CHUNK + 4096])
    (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size([z]))
    assert (st[0], ol[0]) == (dst[0], len(outs[0])) and st[0] == zb.Z_DATA_ERROR, (st, ol, dst, len(outs[0]))
    assert rep.get(SEG_COUNT) and rep.get(COUNT), rep               # tried in segments, named by the count kernel
    no_decode(rep)


def test_past_4gib(gpu_lib):
    """5 GiB of zeros from system zlib: exact alone (segment counting pass) and among nine (count kernel)."""
    co = zlib.compressobj(1)
    block = bytes(64 << 20)
    z = b"".join(co.compress(block) for _ in range(80)) + co.flush()
    n = 5 << 30
    (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size([z]))
    assert (st, ol, su) == ([0], [n], [len(z)])
    assert rep.get(SEG_COUNT) and COUNT not in rep, rep
    no_decode(rep)
    shorts = [dw.zlib_wrap(c.raw, c.plain) for c in CATALOGUE if c.kind == "ok"][:8]
    (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size(shorts + [z]))
    assert (st[-1], ol[-1], su[-1]) == (0, n, len(z))
    assert rep.get(COUNT) and SEG_COUNT not in rep, rep
    (ol, su, st), rep = profiled(gpu_lib, lambda: gpu_lib.inflate_batch_size(shorts + [z], limit=(4 << 30) + 3))
    assert (st[-1], ol[-1]) == (zb.Z_BUF_ERROR, (4 << 30) + 3)


# ---- the device form -------------------------------------------------------------------------------------------------------------
def _dev_case(oracle):
    import torch
    cases = [c for c in CATALOGUE if c.kind != "cut"]
    zs = [wrapped(c.raw, c.plain, zb.WRAP_ZLIB) for c in cases]
    src, so = bytearray(), []
    for i, z in enumerate(zs):
        src += b"\xa5" * (1 + i % 3)
        so.append(len(src))
        src += z
    so.append(len(src))
    d_src = torch.from_numpy(np.frombuffer(bytes(src) + b"\0" * 8, dtype=np.uint8).copy()).cuda()
    d_so = torch.tensor(so, dtype=torch.int64).cuda()
    return cases, zs, src, so, d_src, d_so


def _size_dev(lib, d_src, d_so, n, wrap=zb.WRAP_ZLIB, limit=0, stream=None):
    import torch
    d_len = torch.full((n,), 7, dtype=torch.int64, device="cuda")
    d_used = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_st = torch.full((n,), -99, dtype=torch.int32, device="cuda")
    d_do = torch.full((n + 1,), -1, dtype=torch.int64, device="cuda")
    rc = lib.dll.zb200_inflate_batch_size_dev(C.c_void_p(d_src.data_ptr()), C.c_void_p(d_so.data_ptr()), n,
                                              C.c_void_p(d_len.data_ptr()), C.c_void_p(d_used.data_ptr()),
                                              C.c_void_p(d_st.data_ptr()), C.c_void_p(d_do.data_ptr()), wrap, limit,
                                              zb._stream(stream))
    assert rc == 0, lib.last_error()
    return d_len, d_used, d_st, d_do


def test_dev_unaligned(gpu_lib, oracle):
    import torch
    cases, zs, src, so, d_src, d_so = _dev_case(oracle)
    n = len(zs)
    (d_len, d_used, d_st, d_do), rep = profiled(gpu_lib, lambda: _size_dev(gpu_lib, d_src, d_so, n, stream=torch.cuda.current_stream()))
    torch.cuda.synchronize()
    assert rep.get(COUNT) and rep.get("k_size_scan") and SEG_COUNT not in rep, rep
    no_decode(rep)
    host = size_arena(gpu_lib, np.frombuffer(bytes(src) + b"\0" * 8, dtype=np.uint8), so, zb.WRAP_ZLIB)
    lens, used, sts = d_len.cpu().tolist(), d_used.cpu().tolist(), d_st.cpu().tolist()
    assert (lens, used, sts) == host
    do = d_do.cpu().tolist()
    assert do == [0] + list(np.cumsum(lens))
    # d_dst_off as it came out, straight into the decode
    d_dst = torch.zeros(do[-1] + 8, dtype=torch.uint8, device="cuda")
    d_len2 = torch.zeros(n, dtype=torch.int64, device="cuda")
    d_st2 = torch.full((n,), -99, dtype=torch.int32, device="cuda")
    gpu_lib.inflate_batch_dev(d_src.data_ptr(), d_so.data_ptr(), n, d_dst.data_ptr(), d_do.data_ptr(), d_len2.data_ptr(),
                              d_st2.data_ptr(), zb.WRAP_ZLIB, torch.cuda.current_stream())
    torch.cuda.synchronize()
    assert d_len2.cpu().tolist() == lens
    dst, st2 = d_dst.cpu().numpy(), d_st2.cpu().tolist()
    bad = []
    for i, (c, z) in enumerate(zip(cases, zs)):
        want, _ = oracle_want(oracle, z, HUGE >> 20, zb.WRAP_ZLIB)
        rc, out, _ = oracle.inflate(z, HUGE >> 20, zb.WRAP_ZLIB)
        if (sts[i], lens[i]) != want or dst[do[i]:do[i + 1]].tobytes() != out or (st2[i] != sts[i] and want[0] == zb.Z_DATA_ERROR):
            bad.append((c.name, sts[i], lens[i], want, st2[i]))
    assert not bad, bad[:20]


def test_dev_does_not_synchronise(gpu_lib, oracle):
    import torch
    cases, zs, src, so, d_src, d_so = _dev_case(oracle)
    n = len(zs)
    s = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s):
        torch.cuda._sleep(1 << 30)                                 # about half a second of spinning
        d_len, d_used, d_st, d_do = _size_dev(gpu_lib, d_src, d_so, n, stream=s)
        busy = not s.query()
    assert busy, "zb200_inflate_batch_size_dev waited for its stream"
    s.synchronize()
    host = size_arena(gpu_lib, np.frombuffer(bytes(src) + b"\0" * 8, dtype=np.uint8), so, zb.WRAP_ZLIB)
    assert (d_len.cpu().tolist(), d_used.cpu().tolist(), d_st.cpu().tolist()) == host
    assert d_do.cpu().tolist() == [0] + list(np.cumsum(host[0]))


# ---- arenas --------------------------------------------------------------------------------------------------------------------
def test_arenas(gpu_lib):
    """Pageable, pinned and device arenas give the same results; the pageable one of 64 MiB and more takes the staging
    threads, and its groups are copied while earlier ones are counted."""
    import torch
    rng = random.Random(77)
    base = _base_text()
    plains = [_plain(rng, rng.randint(64 << 10, 160 << 10), base) for _ in range(1500)]
    zs = [zlib.compress(p, 1) + rng.randbytes(rng.randint(0, 9)) for p in plains]
    arena = np.frombuffer(b"".join(zs) + b"\0" * 8, dtype=np.uint8).copy()
    so = [0] + list(np.cumsum([len(z) for z in zs]))
    assert so[-1] >= 64 << 20
    want = [len(p) for p in plains]
    pageable, rep = profiled(gpu_lib, lambda: size_arena(gpu_lib, arena, so, zb.WRAP_ZLIB))
    assert pageable[0] == want and pageable[2] == [0] * len(zs)
    assert rep.get(COUNT) and SEG_COUNT not in rep, rep
    no_decode(rep)
    pin = gpu_lib.dll.zb200_alloc_pinned(arena.nbytes)
    assert pin
    try:
        C.memmove(pin, arena.ctypes.data, arena.nbytes)
        assert size_arena(gpu_lib, pin, so, zb.WRAP_ZLIB) == pageable
    finally:
        gpu_lib.dll.zb200_free_pinned(C.c_void_p(pin))
    d_arena = torch.from_numpy(arena).cuda()
    assert size_arena(gpu_lib, d_arena, so, zb.WRAP_ZLIB) == pageable
    assert size_arena(gpu_lib, arena, so, zb.WRAP_ZLIB, used=False)[0::2] == pageable[0::2]
