"""zb200_inflate_batch_size against the decode it sizes for, on one GPU -> profiles/r5_inflate_size.json.

  config 3   100 000 zlib streams of 64 KiB (bench.py's corpus and stream set: synthetic mixed data, level 6), device arena:
             zb200_inflate_batch_size (results to the host) against zb200_inflate_batch (device output), alternating;
             then the same with pinned host arenas (compressed in; for the decode, plain out as well).
  one 1 GiB stream from this library's compress2() at levels 1 and 6 (sync markers) and the 64 MiB system-zlib level-6
             text stream (block finder): the size call against uncompress() of the same host buffer.  With --parent, the
             uncompress() of the parent build's library is timed too, alternating with this one's in the same process.
Every timed call is a host clock around a call that synchronises.  Sizes are checked against the known plain lengths."""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import numpy as np                                                   # noqa: E402

import bench                                                         # noqa: E402
from zlib_b200 import binding as zb, synth                           # noqa: E402


def gpu_info():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip().splitlines()
        return q[0] if q else "unknown"
    except Exception as e:                                           # noqa: BLE001
        return f"unknown ({e})"


def stats(ts):
    ts = sorted(ts)
    return {"median_ms": round(ts[len(ts) // 2] * 1e3, 3), "min_ms": round(ts[0] * 1e3, 3), "runs": len(ts)}


def alternate(fns, runs):
    """{name: [seconds]} with the functions called in turn, `runs` rounds (after one warm-up round)."""
    out = {k: [] for k in fns}
    for r in range(runs + 1):
        for k, f in fns.items():
            t0 = time.perf_counter()
            f()
            if r:
                out[k].append(time.perf_counter() - t0)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r5_inflate_size.json"))
    ap.add_argument("--parent", default=None, help="libzb200.so of the parent build: its uncompress() is timed alongside")
    ap.add_argument("--streams", type=int, default=100000)
    ap.add_argument("--runs", type=int, default=5)
    a = ap.parse_args()
    import torch
    lib = zb.Lib()
    assert lib.dll.zb200_init(0) == 0, lib.last_error()
    par = zb.Lib(a.parent) if a.parent else None
    if par:
        assert par.dll.zb200_init(0) == 0, par.last_error()
    res = {"gpu": gpu_info(), "how": __doc__.strip()}
    dll = lib.dll

    # ---- config 3 ----
    sz, distinct, ns = 65536, 2048, a.streams
    host = synth.synth(distinct * sz, 1, 1)
    zs, kind = bench.make_stream_set(host, sz, distinct, False)
    zsn = (zs * ((ns + distinct - 1) // distinct))[:ns]
    so = np.zeros(ns + 1, dtype=np.uint64)
    so[1:] = np.cumsum([len(z) for z in zsn])
    zin = int(so[-1])
    arena = np.frombuffer(b"".join(zsn) + b"\0" * 8, dtype=np.uint8)
    do = (np.arange(ns + 1, dtype=np.uint64) * sz).astype(np.uint64)
    ol = np.zeros(ns, dtype=np.uint64); su = np.zeros(ns, dtype=np.uint64); st = np.zeros(ns, dtype=np.int32)
    dl = np.zeros(ns, dtype=np.uint64); dst_st = np.zeros(ns, dtype=np.int32)
    d_z = torch.from_numpy(arena.copy()).cuda()
    d_out = torch.empty(ns * sz + 16, dtype=torch.uint8, device="cuda")

    def size(src):
        assert dll.zb200_inflate_batch_size(src, so.ctypes.data, ns, ol.ctypes.data, su.ctypes.data, st.ctypes.data,
                                            zb.WRAP_ZLIB, 0, None) == 0, lib.last_error()

    def decode(src, dst):
        assert dll.zb200_inflate_batch(src, so.ctypes.data, ns, dst, do.ctypes.data, dl.ctypes.data, dst_st.ctypes.data,
                                       zb.WRAP_ZLIB, None) == 0, lib.last_error()

    t = alternate({"size": lambda: size(d_z.data_ptr()), "decode": lambda: decode(d_z.data_ptr(), d_out.data_ptr())}, a.runs)
    ok = bool((ol == sz).all() and (st == 0).all() and (su == np.diff(so)).all() and (dl == sz).all() and (dst_st == 0).all())
    res["config3_device"] = {"streams": ns, "stream_bytes": sz, "source": kind, "compressed_bytes": zin, "sizes_exact": ok,
                             "inflate_batch_size": stats(t["size"]), "inflate_batch": stats(t["decode"]),
                             "size_over_decode": round(np.median(t["size"]) / np.median(t["decode"]), 4)}
    print(json.dumps(res["config3_device"]), flush=True)
    del d_out
    pin_z = dll.zb200_alloc_pinned(zin + 64)
    pin_o = dll.zb200_alloc_pinned(ns * sz + 16)
    assert pin_z and pin_o
    C.memmove(pin_z, arena.ctypes.data, zin)
    ol[:] = 0
    t = alternate({"size": lambda: size(pin_z), "decode": lambda: decode(pin_z, pin_o)}, a.runs)
    ok = bool((ol == sz).all() and (st == 0).all() and (dl == sz).all())
    res["config3_pinned_host"] = {"streams": ns, "sizes_exact": ok, "inflate_batch_size": stats(t["size"]),
                                  "inflate_batch": stats(t["decode"]),
                                  "size_over_decode": round(np.median(t["size"]) / np.median(t["decode"]), 4)}
    print(json.dumps(res["config3_pinned_host"]), flush=True)
    dll.zb200_free_pinned(C.c_void_p(pin_o))
    dll.zb200_free_pinned(C.c_void_p(pin_z))
    del d_z, arena, zsn, zs

    # ---- long streams: size call against uncompress() of the same host buffer ----
    def long_row(name, z, n, route, runs):
        zarr = np.frombuffer(z, dtype=np.uint8)
        out = np.empty(n + 16, dtype=np.uint8)
        one = np.array([0, len(z)], dtype=np.uint64)
        o1, u1, s1 = np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.uint64), np.zeros(1, dtype=np.int32)

        def sz_call():
            assert dll.zb200_inflate_batch_size(zarr.ctypes.data, one.ctypes.data, 1, o1.ctypes.data, u1.ctypes.data,
                                                s1.ctypes.data, zb.WRAP_ZLIB, 0, None) == 0, lib.last_error()

        def unc(l):
            dlen = C.c_ulong(n)
            assert l.dll.uncompress(out.ctypes.data, C.byref(dlen), zarr.ctypes.data, len(z)) == 0 and dlen.value == n

        fns = {"size": sz_call, "uncompress": lambda: unc(lib)}
        if par:
            fns["uncompress_parent"] = lambda: unc(par)
        lib.profile(True)
        sz_call()
        rep = lib.profile_report()
        lib.profile(False)
        t = alternate(fns, runs)
        row = {"plain_bytes": n, "compressed_bytes": len(z), "route": route, "size_exact": bool((o1[0], u1[0], s1[0]) == (n, len(z), 0)),
               "kernels_of_size_call": {k: v[1] for k, v in rep.items()}}
        row.update({k: stats(v) for k, v in t.items()})
        row["size_over_uncompress"] = round(np.median(t["size"]) / np.median(t["uncompress"]), 4)
        if par:
            row["uncompress_over_parent"] = round(np.median(t["uncompress"]) / np.median(t["uncompress_parent"]), 4)
        res[name] = row
        print(name, json.dumps(row), flush=True)

    n = 1 << 30
    data = synth.synth(n, 1, 1)
    for lv in (1, 6):
        rc, z = lib.compress2(data, lv)
        assert rc == 0
        long_row(f"compress2_L{lv}_1GiB", z, n, "sync markers: counting pass", a.runs)
    del data
    text = synth.synth(64 << 20, 0, 7).tobytes()
    long_row("zlib_L6_text_64MiB", zlib.compress(text, 6), len(text), "block finder: counting pass", a.runs)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(res, f, indent=1)
    print("wrote", a.out)


if __name__ == "__main__":
    main()
