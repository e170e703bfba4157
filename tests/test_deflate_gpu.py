"""GPU: K1-K3 deflate through the C-ABI.  Gate (a): the oracle and the compiled reference decode the
GPU's output to the original bytes; gate (d): size within 2 % of the reference at the same level."""
import random
import zlib

import numpy as np
import pytest

import zhelpers
from zlib_b200 import binding as zb

pytestmark = pytest.mark.gpu

SIZES = [0, 1, 2, 3, 4, 5, 100, 257, 258, 259, 1000, 32767, 32768, 32769, 65535, 65536, 131071, 131072, 131073,
         200000, 262144, 400000]


def _decode_everywhere(z, data, oracle, ref=None):
    rc, out, used = oracle.inflate(z, len(data))
    assert rc == 0 and out == data and used == len(z)
    assert zlib.decompress(z) == data                       # independent decoder (system zlib 1.3)
    if ref is not None:
        rc, out = ref.uncompress(z, len(data))
        assert rc == 0 and out == data


@pytest.mark.parametrize("level", [1, 6])
def test_round_trip_sizes_and_kinds(gpu_lib, oracle, level):
    for kind in range(5):
        for n in SIZES:
            data = zhelpers.corpus(kind, n, 7)
            rc, z = gpu_lib.compress2(data, level)
            assert rc == 0, (kind, n, rc, gpu_lib.last_error())
            assert len(z) <= gpu_lib.compress_bound(n)
            _decode_everywhere(z, data, oracle)


def test_all_levels(gpu_lib, oracle):
    data = zhelpers.corpus(1, 300000, 3) + zhelpers.corpus(3, 100000, 4) + zhelpers.corpus(0, 50000, 5)
    sizes = {}
    for level in range(10):
        rc, z = gpu_lib.compress2(data, level)
        assert rc == 0
        _decode_everywhere(z, data, oracle)
        sizes[level] = len(z)
        flevel = (z[1] >> 6) & 3
        assert flevel == (0 if level < 2 else 1 if level < 6 else 2 if level == 6 else 3)   # deflate.c:628-636
    assert sizes[0] > len(data) and sizes[0] <= gpu_lib.compress_bound(len(data))
    assert sizes[9] <= sizes[1]
    rc, z = gpu_lib.compress2(data, -1)
    assert rc == 0 and len(z) == sizes[6]


def test_level_ladder_against_the_reference(gpu_lib, reference_codec):
    """Every level: no larger than the reference's output at the SAME level (+2 %, gate (d)), sizes do not grow with the
    level (0.1 % slack: the budgets are knees of a sweep, not a proof), and the reference decodes each stream."""
    for kind, seed in ((0, 21), (1, 22)):
        data = gpu_lib.synth(16 << 20, kind=kind, seed=seed)
        raw = data.tobytes()
        prev = None
        for level in range(1, 10):
            rc, z = gpu_lib.compress2(data, level)
            assert rc == 0
            want = len(reference_codec.compress2(raw, level))
            assert len(z) <= 1.02 * want, (kind, level, len(z), want)
            if prev is not None:
                assert len(z) <= 1.001 * prev, (kind, level, len(z), prev)
            prev = len(z)
            rc, out = reference_codec.uncompress(z, len(raw))
            assert rc == 0 and out == raw


def test_reference_decodes_gpu_output(gpu_lib, oracle, reference_codec):
    rng = random.Random(3)
    for t in range(20):
        data = zhelpers.corpus(rng.randrange(5), rng.randint(0, 500000), 50 + t)
        for level in (1, 6):
            rc, z = gpu_lib.compress2(data, level)
            assert rc == 0
            _decode_everywhere(z, data, oracle, reference_codec)


@pytest.mark.parametrize("kind", [0, 1])
def test_ratio_gate_vs_reference(gpu_lib, oracle, kind):
    """<= 2 % larger than the reference compressing the WHOLE buffer as one stream (SURVEY 8(d))."""
    data = gpu_lib.synth(8 << 20, kind=kind, seed=11)
    for level in (1, 6):
        rc, z = gpu_lib.compress2(data, level)
        assert rc == 0
        want = len(oracle.deflate(data, level))
        assert len(z) <= 1.02 * want, (kind, level, len(z), want, len(z) / want)
        rc, out, _ = oracle.inflate(z, len(data))
        assert rc == 0 and out == data.tobytes()


def test_ratio_gate_at_config_one_shape(gpu_lib, reference_codec):
    """Gate (d) at BASELINE config 1's shape: 64 MiB of synthetic text, levels 1 and 6, against the unmodified reference
    build compressing the WHOLE buffer as one stream; and the reference decodes what we wrote (gate (a))."""
    n = 64 << 20
    text = gpu_lib.synth(n, kind=0, seed=7)
    for level in (1, 6):
        rc, z = gpu_lib.compress2(text, level)
        assert rc == 0
        want = len(reference_codec.compress2(text, level))
        assert len(z) <= 1.02 * want, (level, len(z), want, len(z) / want)
        rc, out = reference_codec.uncompress(z, n)
        assert rc == 0 and out == text.tobytes()


def test_huffman_length_limit(gpu_lib, oracle):
    """Fibonacci-weighted symbols push the optimal code past 15 bits and the code-length code past 7:
    the overflow repair of trees.c:527-545 must still give complete codes."""
    fib = [1, 1]
    while len(fib) < 25:
        fib.append(fib[-1] + fib[-2])
    buf = bytearray(b"".join(bytes([40 + i]) * f for i, f in enumerate(fib)))
    random.Random(5).shuffle(buf)
    data = bytes(buf)
    for level in (1, 6, 9):
        rc, z = gpu_lib.compress2(data, level)
        assert rc == 0
        _decode_everywhere(z, data, oracle)
    # many distinct code lengths in one header stress the 7-bit limit of the code-length code
    rng = random.Random(9)
    for t in range(6):
        weights = [rng.choice([1, 2, 3, 5, 8, 13, 40, 100, 400, 3000]) for _ in range(256)]
        data = bytes(rng.choices(range(256), weights=weights, k=150000))
        for level in (1, 6):
            rc, z = gpu_lib.compress2(data, level)
            assert rc == 0
            _decode_everywhere(z, data, oracle)


def test_multi_slab_host_pipeline(gpu_lib, oracle):
    """Inputs longer than one pipeline slab (888 chunks) take the overlapped copy/compute path and must still
    be one valid stream, from host memory and from device memory alike."""
    import ctypes as C
    n = (888 * 131072) * 2 + 777777
    data = gpu_lib.synth(n, kind=1, seed=21)
    rc, z = gpu_lib.compress2(data, 1)
    assert rc == 0
    assert zlib.decompress(z) == data.tobytes()
    assert z[-4:] == oracle.adler32(data).to_bytes(4, "big")
    rc, z2 = gpu_lib.compress2(data, 1, cap=len(z) - 1)
    assert rc == zb.Z_BUF_ERROR
    d_src = gpu_lib.dll.zb200_alloc_device(n)
    cap = gpu_lib.compress_bound(n)
    d_dst = gpu_lib.dll.zb200_alloc_device(cap)
    assert d_src and d_dst
    try:
        assert gpu_lib.dll.zb200_copy(d_src, data.ctypes.data, n, None) == 0
        m = gpu_lib.deflate(d_src, n, d_dst, cap, 1, zb.WRAP_ZLIB)
        out = C.create_string_buffer(m)
        assert gpu_lib.dll.zb200_copy(out, d_dst, m, None) == 0
        assert out.raw == z                                      # same bytes whichever memory the buffers live in
    finally:
        gpu_lib.dll.zb200_free_device(d_src)
        gpu_lib.dll.zb200_free_device(d_dst)


def test_buf_error_and_bad_level(gpu_lib):
    data = zhelpers.corpus(1, 50000, 1)
    rc, _ = gpu_lib.compress2(data, 6, cap=100)
    assert rc == zb.Z_BUF_ERROR
    rc, _ = gpu_lib.compress2(data, 10)
    assert rc == zb.Z_STREAM_ERROR
    rc, z = gpu_lib.compress2(zhelpers.corpus(0, 70000, 2), 6, cap=gpu_lib.compress_bound(70000))
    assert rc == 0                                              # incompressible input fits compressBound


def test_gpu_inflate_reads_gpu_deflate(gpu_lib):
    data = gpu_lib.synth(3 << 20, kind=1, seed=2)
    rc, z = gpu_lib.compress2(data, 6)
    assert rc == 0
    rc, out = gpu_lib.uncompress(z, len(data))
    assert rc == 0 and out == data.tobytes()


def test_raw_gzip_and_shards(gpu_lib, oracle):
    """Shards with a 32 KiB dictionary concatenate into one valid stream (multi-GPU assembly rule)."""
    import ctypes as C
    data = gpu_lib.synth((1 << 20) + 12345, kind=1, seed=4).tobytes()
    cuts = [0, 300000, 300000 + 131072 * 3, len(data)]
    parts, adl, crc = [], 1, 0
    for i, (a, b) in enumerate(zip(cuts, cuts[1:])):
        last = i == len(cuts) - 2
        flags = (0 if last else zb.ZB200_DEFLATE_NOT_LAST) | zb.ZB200_DEFLATE_NO_HEADER | zb.ZB200_DEFLATE_NO_TRAILER
        dict_ = data[max(0, a - 32768):a]
        cap = gpu_lib.compress_bound(b - a) + 64
        out = C.create_string_buffer(cap)
        n, c1, a1 = gpu_lib.deflate_shard(data[a:b], b - a, dict_ if dict_ else None, len(dict_), out, cap, 6, zb.WRAP_RAW, flags)
        parts.append(out.raw[:n])
        adl = gpu_lib.adler32_combine(adl, a1, b - a)
        crc = gpu_lib.crc32_combine(crc, c1, b - a)
    raw = b"".join(parts)
    assert zlib.decompress(raw, -15) == data
    z = b"\x78\x9c" + raw + adl.to_bytes(4, "big")
    rc, out, used = oracle.inflate(z, len(data))
    assert rc == 0 and out == data and used == len(z)
    assert crc == oracle.crc32(data)
    # gzip wrapper
    cap = gpu_lib.compress_bound(len(data)) + 32
    out = C.create_string_buffer(cap)
    n = gpu_lib.deflate(data, len(data), out, cap, 6, zb.WRAP_GZIP)
    assert zlib.decompress(out.raw[:n], 31) == data
    rc, o2, _ = oracle.inflate(out.raw[:n], len(data), 2)
    assert rc == 0 and o2 == data


def test_deflate_batch_independent_streams(gpu_lib, oracle):
    """zb200_deflate_batch: n inputs -> n streams (minizip-style per-file streams), each decodable by the reference,
    with the CRC-32 / Adler-32 of each input; a slot that is too small fails alone."""
    rng = random.Random(12)
    sizes = [0, 1, 2, 100, 4096, 65535, 65536, 70000, 131072, 131073, 300000, 1 << 20, (1 << 21) + 5] + \
            [rng.randint(1, 200000) for _ in range(27)]
    bufs = [zhelpers.corpus(rng.randrange(5), n, 300 + i) for i, n in enumerate(sizes)]
    for level, wrap, wbits in ((6, zb.WRAP_ZLIB, 15), (1, zb.WRAP_RAW, -15), (6, zb.WRAP_GZIP, 31)):
        outs, st, crcs, adls = gpu_lib.deflate_batch(bufs, level, wrap)
        assert st == [0] * len(bufs), st
        for d, z, c, a in zip(bufs, outs, crcs, adls):
            assert zlib.decompress(z, wbits) == d
            assert c == oracle.crc32(d) and a == oracle.adler32(d)
            if wrap == zb.WRAP_ZLIB:
                rc, out, used = oracle.inflate(z, len(d))
                assert rc == 0 and out == d and used == len(z)
    caps = [gpu_lib.compress_bound(len(b)) + 16 for b in bufs]
    caps[7] = 10                                               # 70000 random-ish bytes cannot fit
    outs, st, _, _ = gpu_lib.deflate_batch(bufs, 6, zb.WRAP_ZLIB, caps=caps)
    assert st[7] == zb.Z_BUF_ERROR and all(s == 0 for i, s in enumerate(st) if i != 7)
    assert zlib.decompress(outs[8]) == bufs[8]


def test_deflate_batch_many_slabs_and_big_jobs(gpu_lib, oracle):
    """Job mode of zb200_deflate_batch: more jobs than one slab holds (tiny files, empty ones in between), a job above the
    big-job threshold in the middle (single-stream pipeline), stored / greedy / lazy levels.  History never leaks from
    one job into the next: every stream decodes on its own."""
    rng = random.Random(77)
    base = zhelpers.corpus(1, 1 << 20, 5)
    bufs = []
    for i in range(2100):                                      # > 2 slabs by job count
        n = 0 if i % 97 == 0 else rng.randint(1, 3000)
        o = rng.randrange(len(base) - n)
        bufs.append(base[o:o + n])
    big = gpu_lib.synth((33 << 20) + 12345, kind=1, seed=9).tobytes()
    bufs.insert(1000, big)
    bufs.insert(1500, gpu_lib.synth((5 << 20) + 1, kind=0, seed=10).tobytes())
    for level, wrap, wbits in ((1, zb.WRAP_ZLIB, 15), (6, zb.WRAP_RAW, -15), (0, zb.WRAP_GZIP, 31), (9, zb.WRAP_ZLIB, 15)):
        sub = bufs if level in (1, 6) else bufs[900:1100]
        outs, st, crcs, adls = gpu_lib.deflate_batch(sub, level, wrap)
        assert st == [0] * len(sub)
        for d, z, c in zip(sub, outs, crcs):
            assert zlib.decompress(z, wbits) == d
            assert c == zlib.crc32(d)
        k = sub.index(big)
        if wrap == zb.WRAP_ZLIB:
            rc, out, used = oracle.inflate(outs[k], len(big))
            assert rc == 0 and out == big and used == len(outs[k])
            assert adls[k] == oracle.adler32(big)


def test_concurrent_host_threads(gpu_lib, oracle):
    """The library is re-entrant like the reference (qcsrc/readme.txt:3-4): different streams from different threads at
    once.  Contexts (stream + scratch) come from a pool, one per call in flight."""
    import threading
    datas = [gpu_lib.synth((3 << 20) + 1000 * i, kind=i % 2, seed=40 + i).tobytes() for i in range(6)]
    results = [None] * len(datas)

    def work(i):
        ok = True
        for rep in range(3):
            rc, z = gpu_lib.compress2(datas[i], 1 if (i + rep) % 2 else 6)
            ok = ok and rc == 0 and zlib.decompress(z) == datas[i]
            rc, out = gpu_lib.uncompress(z, len(datas[i]))
            ok = ok and rc == 0 and out == datas[i]
            ok = ok and gpu_lib.crc32(datas[i]) == oracle.crc32(datas[i])
        results[i] = ok

    threads = [threading.Thread(target=work, args=(i,)) for i in range(len(datas))]
    for th in threads:
        th.start()
    for th in threads:
        th.join()
    assert results == [True] * len(datas)


def test_large_pageable_source_goes_through_the_staging_threads(gpu_lib):
    """compress2() from a malloc'ed (pageable) buffer of 64 MiB or more: host threads copy pieces into pinned slots and
    send them on their own streams (HostStager); the stream is the same as from a pinned buffer and round-trips."""
    import ctypes as C
    n = (150 << 20) + 4321                                      # two slabs, a ragged last piece
    data = gpu_lib.synth(n, kind=1, seed=71)                    # numpy array: pageable
    rc, z = gpu_lib.compress2(data, 1)
    assert rc == zb.Z_OK
    pin = gpu_lib.dll.zb200_alloc_pinned(n)
    C.memmove(C.c_void_p(pin), C.c_void_p(data.ctypes.data), n)
    cap = gpu_lib.compress_bound(n)
    out = C.create_string_buffer(cap)
    ol = C.c_ulong(cap)
    assert gpu_lib.dll.compress2(out, C.byref(ol), C.c_void_p(pin), n, 1) == zb.Z_OK
    gpu_lib.dll.zb200_free_pinned(C.c_void_p(pin))
    assert out.raw[:ol.value] == z
    rc, back = gpu_lib.uncompress(z, n)
    assert rc == zb.Z_OK and back == data.tobytes()


def test_shard_in_two_halves_pipelines_pieces(gpu_lib, oracle):
    """zb200_deflate_shard_begin / _end: piece j + 1 is enqueued before piece j is read back (what the multi-GPU rounds
    do); the pieces, each primed with the 32 KiB in front of it, concatenate into one raw stream the oracle decodes."""
    import ctypes as C
    import numpy as np
    n = (9 << 20) + 4321
    data = gpu_lib.synth(n, kind=1, seed=33)
    cuts = [0, 3 << 20, (3 << 20) + 131072, 7 << 20, n]               # chunk-aligned piece boundaries
    cap = gpu_lib.compress_bound(4 << 20) + 64
    outs = [np.zeros(cap, dtype=np.uint8) for _ in range(4)]
    base = data.ctypes.data
    jobs, res = {}, []

    def begin(j):
        a, b = cuts[j], cuts[j + 1]
        dl = min(a, 32768)
        flags = zb.ZB200_DEFLATE_NO_HEADER | zb.ZB200_DEFLATE_NO_TRAILER | (0 if j == 3 else zb.ZB200_DEFLATE_NOT_LAST)
        return gpu_lib.deflate_shard_begin(base + a, b - a, (base + a - dl) if dl else None, dl, outs[j], cap, 6, zb.WRAP_RAW, flags)
    jobs[0] = begin(0)
    for j in range(4):
        if j + 1 < 4:
            jobs[j + 1] = begin(j + 1)
        res.append(gpu_lib.deflate_shard_end(jobs.pop(j)))
    raw = b"".join(bytes(outs[j][:res[j][0]]) for j in range(4))
    rc, out, used = oracle.inflate(raw, n, 0)
    assert rc == 0 and out == data.tobytes() and used == len(raw)
    crc = 0
    for j in range(4):
        crc = gpu_lib.crc32_combine(crc, res[j][1], cuts[j + 1] - cuts[j])
    assert crc == oracle.crc32(data)
    # device buffers, both halves on a caller's stream
    import torch
    d = torch.from_numpy(data).cuda()
    o = torch.empty(cap * 3, dtype=torch.uint8, device="cuda")
    s = torch.cuda.Stream()
    job = gpu_lib.deflate_shard_begin(d.data_ptr(), n, None, 0, o.data_ptr(), o.numel(), 1, zb.WRAP_ZLIB, 0, s)
    clen, c32, a32 = gpu_lib.deflate_shard_end(job)
    rc, out, _ = oracle.inflate(bytes(o[:clen].cpu().numpy()), n)
    assert rc == 0 and out == data.tobytes() and c32 == oracle.crc32(data) and a32 == oracle.adler32(data)
