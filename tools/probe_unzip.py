"""Reading the config-5 archive back: zb200_zip_extract against today's best path, on one GPU.

The archive is the one bench.py's config 5 writes: 10 000 members with the sizes of bench.zip_sizes(), member i holding
synth corpus bytes (T for even i, M for odd i) from its own 64 KiB-aligned offset, built by zb200_zip_build at levels 1
and 6.  For each level, timed after a warm-up (host clock behind the call's own synchronisation):
  (a) zb200_zip_extract, archive and outputs in device memory;
  (b) the same with pinned host buffers;
  (c) zb200_inflate_batch(WRAP_RAW) over the member data ranges plus zb200_checksum_batch, device memory;
  (d) Python zipfile on one host core over a seeded sample of members, extrapolated to the whole archive.
Every output of (a)-(c) is compared with the input in the same run.  Route counts: stored members, members with at most
one 128 KiB chunk of output (batch kernel), long members whose marker count fits the plan (planned segments), and the
rest (one-stream fallback; the profile's k_find_markers launches beyond the first count the members that reached it).

    python tools/probe_unzip.py [--reps 3] [--sample 200] [--out profiles/r3_unzip.json]
"""
import argparse
import ctypes as C
import io
import json
import os
import random
import subprocess
import sys
import time
import zipfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import zlib_b200  # noqa: E402
from zlib_b200 import binding as zb, synth  # noqa: E402
from bench import zip_sizes  # noqa: E402

CHUNK = 131072


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def build_inputs(sizes):
    nf = len(sizes)
    src_off = np.zeros(nf + 1, dtype=np.uint64)
    src_off[1:] = np.cumsum(sizes, dtype=np.uint64)
    starts = np.zeros(nf + 1, dtype=np.int64)
    starts[1:] = np.cumsum([(z + 65535) // 65536 * 65536 for z in sizes])
    src = np.empty(int(src_off[-1]) + 64, dtype=np.uint8)
    for i, z in enumerate(sizes):
        synth.fill(src.ctypes.data + int(src_off[i]), z, i & 1, 5, int(starts[i]))
    return src, src_off


def timed(fn, reps):
    fn()                                                        # warm-up
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts), float(np.median(ts))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--sample", type=int, default=200)
    ap.add_argument("--levels", default="1,6")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r3_unzip.json"))
    args = ap.parse_args()
    lib = zlib_b200.load()
    assert lib.dll.zb200_init(0) == 0, lib.last_error()
    dev = torch.device("cuda:0")
    sizes = zip_sizes()
    nf = len(sizes)
    src, src_off = build_inputs(sizes)
    total = int(src_off[-1])
    d_src = torch.from_numpy(src[:total]).to(dev)
    names = (C.c_char_p * nf)(*[b"f%05d.bin" % i for i in range(nf)])
    cap = lib.dll.zb200_zip_bound(names, C.c_void_p(src_off.ctypes.data), nf)
    p_arc = lib.dll.zb200_alloc_pinned(cap)
    p_out = lib.dll.zb200_alloc_pinned(total + 64)
    assert p_arc and p_out
    out_np = np.ctypeslib.as_array(C.cast(p_out, C.POINTER(C.c_uint8)), shape=(total + 64,))
    d_out = torch.empty(total + 64, dtype=torch.uint8, device=dev)
    dst_off = src_off.copy()                                    # member i decodes to the place it came from
    dst_len = np.zeros(nf, dtype=np.uint64)
    status = np.zeros(nf, dtype=np.int32)
    res = {"card": card(), "files": nf, "uncompressed_bytes": total, "levels": {}}
    for level in [int(x) for x in args.levels.split(",")]:
        ol = C.c_size_t(cap)
        t0 = time.perf_counter()
        rc = lib.dll.zb200_zip_build(names, C.c_void_p(src.ctypes.data), C.c_void_p(src_off.ctypes.data), nf, level,
                                     zb.DOS_DATETIME, C.c_void_p(p_arc), C.byref(ol))
        t_build = time.perf_counter() - t0
        assert rc == 0, lib.last_error()
        arc_len = ol.value
        arc_np = np.ctypeslib.as_array(C.cast(p_arc, C.POINTER(C.c_uint8)), shape=(arc_len,))
        ents = lib.zip_list(arc_np)
        assert [e.name for e in ents] == ["f%05d.bin" % i for i in range(nf)]
        recs = np.zeros(nf, dtype=zb._zip_entry_dtype())
        for i, e in enumerate(ents):
            recs[i] = e.raw
        d_arc = torch.from_numpy(arc_np.copy()).to(dev)
        rec = {"archive_bytes": arc_len, "zip_build_s": round(t_build, 3)}

        def extract(a_ptr, d_ptr):
            status[:] = -99
            r = lib.dll.zb200_zip_extract(C.c_void_p(a_ptr), arc_len, recs.ctypes.data, nf, C.c_void_p(d_ptr),
                                          dst_off.ctypes.data, dst_len.ctypes.data, status.ctypes.data, None)
            assert r == 0, lib.last_error()

        def verify(ok_out):
            return bool(ok_out and (status == 0).all() and (dst_len == np.array(sizes, dtype=np.uint64)).all())

        # (a) device memory
        t_min, t_med = timed(lambda: extract(d_arc.data_ptr(), d_out.data_ptr()), args.reps)
        ok = verify(torch.equal(d_out[:total], d_src))
        rec["a_extract_device"] = {"s": round(t_min, 4), "median_s": round(t_med, 4), "GBps": round(total / t_min / 1e9, 3),
                                   "verified": ok}
        # route counts: the plan's decision repeated on the host, and the profile of one more call
        lib.profile(True)
        extract(d_arc.data_ptr(), d_out.data_ptr())
        prof = lib.profile_report()
        lib.profile(False)
        stored = sum(1 for e in ents if e.method == 0)
        short = sum(1 for e in ents if e.method == 8 and e.raw_len <= CHUNK)
        planned = fallback = 0
        for e in ents:
            if e.method != 8 or e.raw_len <= CHUNK:
                continue
            a = e.local_off + 30 + len(e.name)
            marks = arc_np[a:a + e.comp_len - 1].tobytes().count(b"\x00\x00\xff\xff")
            if marks == (e.raw_len + CHUNK - 1) // CHUNK - 1:
                planned += 1
            else:
                fallback += 1
        reached = prof.get("k_find_markers", (0, 1))[1] - 1
        rec["routes"] = {"stored": stored, "batch": short, "planned_segments": planned, "one_stream_fallback": fallback,
                         "reached_one_stream_decoder": reached}
        rec["a_kernel_ms"] = {k: round(v[0], 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
        assert ok, "device extraction differs from the input"
        # (b) pinned host memory
        t_min, t_med = timed(lambda: extract(p_arc, p_out), args.reps)
        ok = verify(np.array_equal(out_np[:total], src[:total]))
        rec["b_extract_pinned_host"] = {"s": round(t_min, 4), "median_s": round(t_med, 4), "GBps": round(total / t_min / 1e9, 3),
                                        "verified": ok}
        assert ok, "pinned extraction differs from the input"
        # (c) today's best path: inflate_batch over the member data ranges (each range runs on into the next local header,
        # which the decoder never reaches) plus checksum_batch; device memory
        data_off = np.array([e.local_off + 30 + len(e.name) for e in ents] + [0], dtype=np.uint64)
        data_off[-1] = data_off[-2] + ents[-1].comp_len
        crc = np.zeros(nf, dtype=np.uint32)
        adl = np.zeros(nf, dtype=np.uint32)

        def batch():
            status[:] = -99
            r = lib.dll.zb200_inflate_batch(C.c_void_p(d_arc.data_ptr()), data_off.ctypes.data, nf, C.c_void_p(d_out.data_ptr()),
                                            dst_off.ctypes.data, dst_len.ctypes.data, status.ctypes.data, zb.WRAP_RAW, None)
            assert r == 0, lib.last_error()
            r = lib.dll.zb200_checksum_batch(C.c_void_p(d_out.data_ptr()), dst_off.ctypes.data, nf, crc.ctypes.data,
                                             adl.ctypes.data, None)
            assert r == 0, lib.last_error()
        d_out.zero_()
        t_min, t_med = timed(batch, args.reps)
        ok = verify(torch.equal(d_out[:total], d_src)) and bool((crc == np.array([e.crc32 for e in ents], dtype=np.uint32)).all())
        rec["c_inflate_batch_plus_checksum_device"] = {"s": round(t_min, 4), "median_s": round(t_med, 4),
                                                       "GBps": round(total / t_min / 1e9, 3), "verified": ok}
        assert ok, "inflate_batch path differs from the input"
        # (d) Python zipfile, one core, a seeded sample, extrapolated
        zf = zipfile.ZipFile(io.BytesIO(arc_np.tobytes()))
        pick = random.Random(level).sample(range(nf), min(nf, args.sample))
        got = 0
        t0 = time.perf_counter()
        for i in pick:
            d = zf.read("f%05d.bin" % i)
            got += len(d)
            assert d == src[int(src_off[i]):int(src_off[i + 1])].tobytes()
        t = time.perf_counter() - t0
        rec["d_python_zipfile_one_core"] = {"sampled_members": len(pick), "sampled_bytes": got, "sample_s": round(t, 3),
                                            "GBps": round(got / t / 1e9, 4), "extrapolated_s": round(total * t / got, 1),
                                            "note": "extrapolated from the sample"}
        res["levels"][str(level)] = rec
        print(json.dumps({level: rec}, indent=1), flush=True)
        del d_arc
    lib.dll.zb200_free_pinned(C.c_void_p(p_arc))
    lib.dll.zb200_free_pinned(C.c_void_p(p_out))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)
    print(f"wrote {args.out}")


if __name__ == "__main__":
    main()
