"""gzip files of several members on one GPU: zb200_bgzf_compress and zb200_gunzip against the nearest existing paths.

Input: 1 GiB of the mixed corpus (synth kind 1, seed 9).  Timed after a warm-up, host clock around calls that synchronise:
  (a) zb200_bgzf_compress at levels 1 and 6, device buffers and pinned host buffers;
  (b) zb200_gunzip of those BGZF files, device and pinned;
  (c) zb200_gunzip of 8 system-zlib members of 128 MiB each (level 1; long members, no sync markers: the block finder);
  (d) zb200_gunzip of a level-0 gzip of data that holds inner .gz members verbatim (every inner header is a candidate);
  (c') uncompress() of the first of those streams alone (zlib wrapper): whether the one-stream decoder takes it at all;
  (e) for comparison: Python gzip.decompress of a 64 MiB BGZF sample on one core (quadratic in the member count, not
      extrapolated) and one zlib.decompressobj per member of the same sample (extrapolated to 1 GiB); zb200_deflate of
      the whole input as one gzip stream (level 6); zb200_deflate_batch + zb200_inflate_batch over the same 65280-byte
      pieces as independent gzip streams (config 3's shape), device buffers.
Every output is compared with its input in the same run.  The card's name and power limit are recorded with the numbers.

    python tools/probe_gzip.py [--reps 3] [--out profiles/r4_gzip.json]
"""
import argparse
import ctypes as C
import gzip
import json
import os
import subprocess
import sys
import time
import zlib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import zlib_b200  # noqa: E402
from zlib_b200 import binding as zb  # noqa: E402

GIB, MIB = 1 << 30, 1 << 20
BLOCK = 65280


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    return {"name": torch.cuda.get_device_name(0), "nvidia_smi": q.stdout.strip()}


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return min(ts), float(np.median(ts))


def rate(nbytes, t):
    return round(nbytes / t / 1e9, 2)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--size", type=int, default=GIB)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r4_gzip.json"))
    args = ap.parse_args()
    lib = zlib_b200.load()
    assert lib.dll.zb200_init(0) == 0, lib.last_error()
    n = args.size
    host = np.asarray(lib.synth(n, kind=1, seed=9))
    d_src = torch.from_numpy(host).cuda()
    p_src = torch.from_numpy(host).pin_memory()
    res = {"card": card(), "input_bytes": n, "corpus": "synth kind 1 (mixed), seed 9", "reps": args.reps, "rows": {}}
    rows = res["rows"]

    def gunzip_call(src, src_len, dst, cap):
        ol, cnt = C.c_size_t(cap), C.c_size_t(0)
        rc = lib.dll.zb200_gunzip(src, src_len, dst, C.byref(ol), C.byref(cnt), None)
        assert rc == 0, (rc, lib.last_error())
        return ol.value, cnt.value

    def gunzip_rows(tag, blob_host, want_len, check):
        blob_host = np.frombuffer(blob_host, dtype=np.uint8) if isinstance(blob_host, bytes) else blob_host
        d_blob = torch.from_numpy(blob_host).cuda()
        p_blob = torch.from_numpy(blob_host).pin_memory()
        d_out = torch.empty(want_len + 64, dtype=torch.uint8, device="cuda")
        p_out = torch.empty(want_len + 64, dtype=torch.uint8).pin_memory()
        for kind, src, dst in (("device", d_blob, d_out), ("pinned", p_blob, p_out)):
            got = {}
            t = timed(lambda: got.update(r=gunzip_call(src.data_ptr(), len(blob_host), dst.data_ptr(), want_len + 64)), args.reps)
            assert got["r"][0] == want_len, (tag, got)
            assert check(dst[:want_len]), (tag, kind)
            rows[f"gunzip {tag} [{kind}]"] = {"s_min": round(t[0], 4), "s_median": round(t[1], 4), "members": got["r"][1],
                                              "compressed_bytes": len(blob_host), "GB_per_s_out": rate(want_len, t[0])}
            print(f"gunzip {tag} [{kind}]", rows[f"gunzip {tag} [{kind}]"], flush=True)

    same_as_input = lambda t: torch.equal(t.cuda() if not t.is_cuda else t, d_src)  # noqa: E731

    # ---- (a), (b): BGZF ----
    bound = lib.dll.zb200_bgzf_bound(n)
    d_bg = torch.empty(bound, dtype=torch.uint8, device="cuda")
    p_bg = torch.empty(bound, dtype=torch.uint8).pin_memory()
    bgzf6 = None
    for level in (1, 6):
        sizes = {}
        for kind, src, dst in (("device", d_src, d_bg), ("pinned", p_src, p_bg)):
            def run():
                ol = C.c_size_t(bound)
                assert lib.dll.zb200_bgzf_compress(src.data_ptr(), n, dst.data_ptr(), C.byref(ol), level, None) == 0, lib.last_error()
                sizes[kind] = ol.value
            t = timed(run, args.reps)
            rows[f"bgzf_compress L{level} [{kind}]"] = {"s_min": round(t[0], 4), "s_median": round(t[1], 4),
                                                        "out_bytes": sizes[kind], "GB_per_s_in": rate(n, t[0])}
            print(f"bgzf_compress L{level} [{kind}]", rows[f"bgzf_compress L{level} [{kind}]"], flush=True)
        assert sizes["device"] == sizes["pinned"]
        blob = d_bg[:sizes["device"]].cpu().numpy()
        assert np.array_equal(blob, p_bg[:sizes["pinned"]].numpy())
        if level == 6:
            bgzf6 = blob.copy()
        gunzip_rows(f"BGZF L{level}", blob, n, same_as_input)
    del d_bg, p_bg

    # ---- (c): long system-zlib members ----
    parts = []
    for k in range(8):
        co = zlib.compressobj(1, zlib.DEFLATED, 31)
        parts.append(co.compress(host[k * (n // 8):(k + 1) * (n // 8)].tobytes()) + co.flush())
    gunzip_rows("8 system-zlib members", b"".join(parts), n, same_as_input)
    # the first of them alone through uncompress() (zlib wrapper, pinned buffers): whether the one-stream decoder takes
    # such a stream at all, independent of zb200_gunzip
    co = zlib.compressobj(1, zlib.DEFLATED, 15)
    z1 = co.compress(host[:n // 8].tobytes()) + co.flush()
    p_z1 = torch.frombuffer(bytearray(z1), dtype=torch.uint8).pin_memory()
    p_o1 = torch.empty(n // 8 + 64, dtype=torch.uint8).pin_memory()
    ul = C.c_ulong(0)

    def unc():
        ul.value = n // 8 + 64
        assert lib.dll.uncompress(p_o1.data_ptr(), C.byref(ul), p_z1.data_ptr(), len(z1)) == 0
    t = timed(unc, 1)
    assert ul.value == n // 8 and torch.equal(p_o1[:n // 8], p_src[:n // 8])
    rows["uncompress() of one of the 8 system-zlib streams alone [pinned]"] = {"s_min": round(t[0], 4), "GB_per_s_out": rate(n // 8, t[0])}
    print(rows["uncompress() of one of the 8 system-zlib streams alone [pinned]"], flush=True)
    del parts, z1, p_z1, p_o1

    # ---- (d): a stored outer member full of inner .gz members ----
    inner = [gzip.compress(host[k * 50000:k * 50000 + 20000 + 97 * k].tobytes(), compresslevel=6, mtime=0) for k in range(64)]
    unit = b"".join(inner[k] + host[(k + 1) * 200000:(k + 1) * 200000 + 100000].tobytes() for k in range(64))
    payload = (unit * (n // len(unit) + 1))[:n]
    outer = gzip.compress(payload, compresslevel=0, mtime=0)
    d_payload = torch.frombuffer(bytearray(payload), dtype=torch.uint8).cuda()
    rows["level-0 outer: inner headers"] = {"inner_members": payload.count(b"\x1f\x8b\x08")}
    gunzip_rows("level-0 gzip holding .gz members", outer, n, lambda t: torch.equal(t.cuda() if not t.is_cuda else t, d_payload))
    del d_payload, outer, payload

    # ---- (e): comparisons ----
    sample = 64 * MIB
    cut, p = 0, 0
    while p < len(bgzf6) and cut < sample:                      # whole members covering the first 64 MiB of output
        bsize = int(bgzf6[p + 16]) | int(bgzf6[p + 17]) << 8
        cut += int.from_bytes(bgzf6[p + bsize - 3:p + bsize + 1].tobytes(), "little")
        p += bsize + 1
    sb = bgzf6[:p].tobytes()
    t0 = time.perf_counter()
    out = gzip.decompress(sb)
    tp = time.perf_counter() - t0
    assert out == host[:cut].tobytes()
    # Python 3.12's gzip.decompress copies the rest of the input after every member, so its time grows with the square
    # of the member count: a figure for that call on this sample, not a rate to extrapolate
    rows["python gzip.decompress BGZF L6, 1 core (64 MiB sample)"] = {"s_sample": round(tp, 3), "sample_out_bytes": cut,
                                                                      "GB_per_s_out": rate(cut, tp)}
    # one zlib.decompressobj per member, members located by their BSIZE: what one core does without the copies
    t0 = time.perf_counter()
    outs, q = [], 0
    while q < len(sb):
        bsize = sb[q + 16] | sb[q + 17] << 8
        outs.append(zlib.decompressobj(-15).decompress(sb[q + 18:q + bsize - 7]))
        q += bsize + 1
    tz = time.perf_counter() - t0
    assert b"".join(outs) == out
    rows["python zlib.decompressobj per BGZF member, 1 core (64 MiB sample)"] = {"s_sample": round(tz, 3), "sample_out_bytes": cut,
                                                                                 "s_extrapolated": round(tz * n / cut, 2), "GB_per_s_out": rate(cut, tz)}
    cap = lib.compress_bound(n) + 64
    d_z = torch.empty(cap, dtype=torch.uint8, device="cuda")
    zl = {}
    t = timed(lambda: zl.update(n=lib.deflate(d_src.data_ptr(), n, d_z.data_ptr(), cap, 6, zb.WRAP_GZIP)), args.reps)
    assert gzip.decompress(d_z[:zl["n"]].cpu().numpy().tobytes()) == host.tobytes()
    rows["zb200_deflate L6 gzip, one stream [device]"] = {"s_min": round(t[0], 4), "out_bytes": zl["n"], "GB_per_s_in": rate(n, t[0])}
    del d_z
    nb = (n + BLOCK - 1) // BLOCK
    src_off = np.minimum(np.arange(nb + 1, dtype=np.uint64) * BLOCK, n).astype(np.uint64)
    slot = np.arange(nb + 1, dtype=np.uint64) * (BLOCK + 1024)
    d_arena = torch.empty(int(slot[-1]) + 64, dtype=torch.uint8, device="cuda")
    clen = np.zeros(nb, dtype=np.uint64)
    st = np.zeros(nb, dtype=np.int32)

    def batch_deflate():
        assert lib.dll.zb200_deflate_batch(d_src.data_ptr(), src_off.ctypes.data, nb, d_arena.data_ptr(), slot.ctypes.data,
                                           clen.ctypes.data, None, None, st.ctypes.data, 6, zb.WRAP_GZIP, None) == 0
    t = timed(batch_deflate, args.reps)
    assert (st == 0).all()
    rows["zb200_deflate_batch L6 gzip, 65280-byte streams [device]"] = {"s_min": round(t[0], 4), "GB_per_s_in": rate(n, t[0])}
    # the streams packed back to back, decoded as config 3 does (device-resident zb200_inflate_batch)
    cl = clen.astype(np.int64)
    in_off = np.zeros(nb + 1, dtype=np.uint64)
    in_off[1:] = np.cumsum(cl)
    packed = torch.empty(int(in_off[-1]) + 64, dtype=torch.uint8, device="cuda")
    for k in range(nb):
        packed[int(in_off[k]):int(in_off[k + 1])] = d_arena[int(slot[k]):int(slot[k]) + int(cl[k])]
    d_out = torch.empty(n + 64, dtype=torch.uint8, device="cuda")
    dlen = np.zeros(nb, dtype=np.uint64)

    def batch_inflate():
        assert lib.dll.zb200_inflate_batch(packed.data_ptr(), in_off.ctypes.data, nb, d_out.data_ptr(), src_off.ctypes.data,
                                           dlen.ctypes.data, st.ctypes.data, zb.WRAP_GZIP, None) == 0
    t = timed(batch_inflate, args.reps)
    assert (st == 0).all() and torch.equal(d_out[:n], d_src)
    rows["zb200_inflate_batch gzip, 65280-byte streams [device]"] = {"s_min": round(t[0], 4), "GB_per_s_out": rate(n, t[0])}
    print(json.dumps(res, indent=1))
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
