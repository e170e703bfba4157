#!/usr/bin/env python
"""bench.py -- the driver-facing benchmark (one JSON line on stdout).

Workload = BASELINE.json configs[1]: 1 GiB of the synthetic mixed corpus (SURVEY.md 8(d)) PER GPU, deflate level 1 in
128 KiB chunks with 32 KiB dictionary priming.  A step = one pass of the hot path over that batch.

  N = 1   value     deflate level-1 throughput, GB/s of UNCOMPRESSED bytes, input and output resident in HBM, timed with
                    CUDA events on the launching stream.
          e2e       the same metric through the reference-facing call compress2(dest, &destLen, source, sourceLen, 1)
                    of libzb200.so with HOST (pinned) buffers: H2D + kernels + D2H inside the timed region.
  N > 1   ONE zlib stream over ONE N GiB corpus (same seed on every rank; the corpus is cut into N * P pieces dealt
          round robin, global piece g = round * N + rank, each compressed with the 32 KiB in front of it as dictionary).
          value     every rank compresses its pieces; after every round one NCCL all-gather of {len, n, crc32, adler32}
                    gives every piece its offset and the round's outputs travel to the ROOT GPU (NCCL send/recv over
                    NVLink) while the next round is compressed; the root adds header and trailer.  The timed region ends
                    when the assembled stream is complete on the root (max over ranks).
          e2e       the same with HOST buffers: pinned input per rank, ONE shared page-locked host buffer for the stream
                    (every rank copies its outputs D2H straight to their final place).
          Both assembled streams are decoded by the reference's own inflate and compared with the corpus
          (`verified_by_reference`, `assembled`).
  roofline  dominant kernel of a step (per-kernel CUDA events inside the library, zb200_profile): algorithmic bytes
            (n_in + n_out, SURVEY 8(d)) / that kernel's time, against the measured HBM peak.
  cpu_baseline / --impl reference
            the UNMODIFIED reference (oracle/_ref/libzref.so, built from /root/reference by oracle/Makefile) running
            compress2 level 1 on the host cores of this box, all threads, over the same number of bytes.  That process
            never loads libzb200.so (the corpus comes from libzbsynth.so).
"""
import argparse
import ctypes as C
import hashlib
import json
import re
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "deflate_level1_GBps_uncompressed"
UNIT = "GB/s"
ROUND_SHARES = (0.5, 0.375, 0.125)    # rounds of the multi-GPU run as shares of a rank's input: only the LAST round's transfer into rank 0 is exposed
                                      # (N = 2, same box: 13.39 ms / e2e 74.6 GB/s; 0.75,0.25: 13.34 / 74.0; 0.625,0.375: 13.25 / 72.7; one round: 13.47 / 65.8)
WINDOW = 32768
PRE = 65536                            # bytes generated in front of a piece (the corpus generator works in 64 KiB pages)


def log(*a):
    print(*a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:   # noqa: BLE001
            pass
    return {"hbm_gbs": 6650.0}, "fallback"


class ClockSampler(threading.Thread):
    """SM clock and throttle reasons DURING the timed region (B200_PROFILING.md).  NVML when importable (a sample
    every 2 ms: the timed region is ~0.1 s), else the nvidia-smi query of the profiling recipe."""

    NAMES = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()
        self.nvml = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[index]) if visible and visible.split(",")[index].isdigit() else index
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(phys)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.handle, pynvml.NVML_CLOCK_SM)
        except Exception:   # noqa: BLE001
            self.nvml = None

    def _nvml_row(self):
        n = self.nvml
        mhz = n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM)
        r = n.nvmlDeviceGetCurrentClocksThrottleReasons(self.handle)
        flags = [bool(r & n.nvmlClocksThrottleReasonHwSlowdown), bool(r & n.nvmlClocksThrottleReasonHwThermalSlowdown),
                 bool(r & n.nvmlClocksThrottleReasonSwThermalSlowdown), bool(r & n.nvmlClocksThrottleReasonSwPowerCap)]
        return [str(mhz), str(self.max_mhz)] + ["Active" if f else "Not Active" for f in flags]

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                if self.nvml is not None:
                    self.rows.append(self._nvml_row())
                else:
                    o = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i", str(self.index)],
                                       capture_output=True, text=True, timeout=5).stdout.strip()
                    if o:
                        self.rows.append([x.strip() for x in o.split(",")])
            except Exception:   # noqa: BLE001
                pass
            self.stop_flag.wait(0.002 if self.nvml is not None else 0.2)

    def summary(self):
        self.stop_flag.set()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        reasons = set()
        for r in self.rows:
            for i, nme in enumerate(self.NAMES):
                if len(r) > 2 + i and r[2 + i].lower().startswith("active"):
                    reasons.add(nme)
        mx = max((int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()), default=None)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(self.rows), "source": "nvml" if self.nvml is not None else "nvidia-smi"}


# ------------------------------------------------------------------------------------- the reference on the host cores
# Nothing in this block touches libzb200.so: the corpus comes from libzbsynth.so, the codec is oracle/_ref/libzref.so.
def _threads(fn, n):
    ths = [threading.Thread(target=fn, args=(i,)) for i in range(n)]
    t0 = time.perf_counter()
    [t.start() for t in ths]
    [t.join() for t in ths]
    return time.perf_counter() - t0


class RefBench:
    """compress2 of the unmodified reference over `total` bytes of the corpus, one slice per host thread."""

    def __init__(self, total, kind=1, seed=1):
        import zhelpers
        from zlib_b200 import synth
        self.ok = os.path.exists(zhelpers.REF_PATH)
        if not self.ok:
            return
        self.ref = zhelpers.Ref()
        self.cores = os.cpu_count() or 1
        self.per = max(131072, (total // self.cores) // 131072 * 131072)
        self.total = self.per * self.cores
        self.data = synth.synth(self.total, kind, seed)
        self.cap = self.ref.dll.compressBound(self.per)
        self.bufs = [C.create_string_buffer(self.cap) for _ in range(self.cores)]
        self.outs = [0] * self.cores

    def step(self, level):
        def work(i):
            ol = C.c_ulong(self.cap)
            rc = self.ref.dll.compress2(self.bufs[i], C.byref(ol), C.c_void_p(self.data.ctypes.data + i * self.per), self.per, level)
            assert rc == 0
            self.outs[i] = ol.value
        dt = _threads(work, self.cores)
        return self.total / dt / 1e9, self.total / max(1, sum(self.outs))


def reference_side_paths(sample_per_thread=16 << 20, kind=1, seed=1):
    """The other paths of the reference on all host cores, bounded samples (reported beside the GPU extras):
    compress2 level 6, uncompress of those streams, crc32 and adler32 -- every thread on its own slice."""
    import zhelpers
    from zlib_b200 import synth
    if not os.path.exists(zhelpers.REF_PATH):
        return None
    ref = zhelpers.Ref()
    cores = os.cpu_count() or 1
    per = sample_per_thread
    data = synth.synth(per * cores, kind, seed)
    cap = ref.dll.compressBound(per)
    zbufs = [C.create_string_buffer(cap) for _ in range(cores)]
    obufs = [C.create_string_buffer(per) for _ in range(cores)]
    zlen = [0] * cores
    sink = [0] * cores

    def f_comp(i):
        ol = C.c_ulong(cap)
        assert ref.dll.compress2(zbufs[i], C.byref(ol), C.c_void_p(data.ctypes.data + i * per), per, 6) == 0
        zlen[i] = ol.value

    def f_unc(i):
        ol = C.c_ulong(per)
        assert ref.dll.uncompress(obufs[i], C.byref(ol), zbufs[i], zlen[i]) == 0 and ol.value == per

    def f_crc(i):
        for _ in range(8):
            sink[i] = ref.dll.crc32(0, C.c_void_p(data.ctypes.data + i * per), per)

    def f_adl(i):
        for _ in range(8):
            sink[i] = ref.dll.adler32(1, C.c_void_p(data.ctypes.data + i * per), per)

    tot = per * cores
    out = {"cores": cores, "sample": f"{per >> 20} MiB of the mixed corpus per host thread"}
    out["compress2_level6_GBps"] = round(tot / _threads(f_comp, cores) / 1e9, 4)
    out["level6_ratio"] = round(tot / max(1, sum(zlen)), 4)
    out["uncompress_GBps"] = round(tot / _threads(f_unc, cores) / 1e9, 4)
    out["crc32_GBps"] = round(8 * tot / _threads(f_crc, cores) / 1e9, 3)
    out["adler32_GBps"] = round(8 * tot / _threads(f_adl, cores) / 1e9, 3)
    return out


def reference_stream_sizes(jobs):
    """jobs: {key: (numpy bytes, level)} -> {key: size of the reference's ONE-stream compress2 output} (threads in parallel;
    the whole buffer as one stream is the strict side of gate (d), SURVEY.md 8(d))."""
    import zhelpers
    ref = zhelpers.Ref()
    res = {}
    keys = list(jobs)

    def work(i):
        data, level = jobs[keys[i]]
        n = len(data)
        cap = ref.dll.compressBound(n)
        out = C.create_string_buffer(cap)
        ol = C.c_ulong(cap)
        assert ref.dll.compress2(out, C.byref(ol), C.c_void_p(data.ctypes.data), n, level) == 0
        res[keys[i]] = ol.value
    _threads(work, len(keys))
    return res


def reference_inflate_check(stream_ptr, stream_len, total, kind=1, seed=1, piece=64 << 20):
    """The reference's inflate() decodes the stream at `stream_ptr` piece by piece (its uncompress() takes 32-bit
    lengths); every piece is compared with the regenerated corpus.  Returns True when all `total` bytes agree and the
    stream ends with a good trailer exactly at stream_len."""
    import numpy as np
    import zhelpers
    from zlib_b200 import synth
    from zlib_b200.binding import z_stream, ZLIB_VERSION
    ref = zhelpers.Ref()
    d = ref.dll
    d.inflateInit_.restype, d.inflateInit_.argtypes = C.c_int, [C.POINTER(z_stream), C.c_char_p, C.c_int]
    d.inflate.restype, d.inflate.argtypes = C.c_int, [C.POINTER(z_stream), C.c_int]
    d.inflateEnd.restype, d.inflateEnd.argtypes = C.c_int, [C.POINTER(z_stream)]
    strm = z_stream()
    if d.inflateInit_(C.byref(strm), ZLIB_VERSION, C.sizeof(z_stream)) != 0:
        return False
    out = np.empty(piece, dtype=np.uint8)
    done, pos, ok, rc = 0, 0, True, 0
    while ok and rc == 0:
        if strm.avail_in == 0 and pos < stream_len:
            n = min(1 << 30, stream_len - pos)
            strm.next_in, strm.avail_in = stream_ptr + pos, n
            pos += n
        strm.next_out, strm.avail_out = out.ctypes.data, piece
        rc = d.inflate(C.byref(strm), 0)
        got = piece - strm.avail_out
        if rc not in (0, 1) or (rc == 0 and got == 0):
            ok = False
            break
        if got:
            if done + got > total:
                ok = False
                break
            want = synth.synth(got, kind, seed, done)
            ok = bool(np.array_equal(out[:got], want))
            done += got
    ok = ok and rc == 1 and done == total and strm.total_in == stream_len
    d.inflateEnd(C.byref(strm))
    return bool(ok)


def oracle_inflate_check(stream_ptr, stream_len, total, kind=1, seed=1):
    """reference_inflate_check where the reference is not built: the oracle (oracle/libzoracle.so, the reference's inflate
    restated in C) decodes the whole stream in one call; True when it ends exactly at stream_len with a good trailer and
    the output is the regenerated corpus."""
    import numpy as np
    import zhelpers
    from zlib_b200 import synth
    orc = zhelpers.Oracle()
    out = np.empty(max(total, 1), dtype=np.uint8)
    ol, used = C.c_size_t(0), C.c_size_t(0)
    rc = orc.dll.zo_inflate(C.c_void_p(stream_ptr), stream_len, C.c_void_p(out.ctypes.data), total, C.byref(ol), C.byref(used), 1)
    if rc != 0 or ol.value != total or used.value != stream_len:
        return False
    return bool(np.array_equal(out[:total], synth.synth(total, kind, seed)))


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    world = max(1, args.gpus)
    size = (args.size_mib << 20) * world                     # the same bytes our arm compresses at this N
    rb = RefBench(size)
    if not rb.ok:
        emit_line({"impl": "reference", "unavailable": "oracle/_ref/libzref.so not built on this box"})
        return 0
    vals, ratio = [], None
    for i in range(args.warmup + args.steps):
        v, ratio = rb.step(1)
        if i >= args.warmup:
            vals.append(v)
    v = sum(vals) / len(vals)
    line = {"impl": "reference", "metric": METRIC, "value": round(v, 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(rb.total / v / 1e6, 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic",
            "config": workload_config(args.size_mib, world),
            "cpu_baseline": {"value": round(v, 4), "unit": UNIT, "cores": rb.cores, "kind": "reference",
                             "sample": f"compress2 level 1 over all {rb.total >> 20} MiB of the corpus, one {rb.per >> 20} MiB slice per host thread"},
            "e2e": {"value": round(v, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "ratio": round(ratio, 4), "gpu_launches": 0}
    emit_line(line)
    return 0


def workload_config(size_mib, world):
    return {"workload": f"{size_mib} MiB synthetic mixed corpus per GPU (BASELINE.json configs[1]), deflate level 1, "
                        "128 KiB chunks with 32 KiB dictionary priming, one zlib stream",
            "level": 1, "chunk": 131072, "bytes_per_gpu": size_mib << 20, "total_bytes": (size_mib << 20) * world,
            "l2": "inputs (1 GiB per GPU) exceed the 126 MB L2; no flush needed",
            "parallelism": (f"one {world * size_mib} MiB corpus cut into rounds of {world} pieces dealt round robin over {world} GPUs "
                            "(2 equal rounds below 4 GPUs; shares of 1/2, 3/8, 1/8 from 4 GPUs on), assembled on rank 0") if world > 1 else "single GPU"}


# ------------------------------------------------------------------------------------- our arm
_REAL_STDOUT = None


def claim_stdout():
    """stdout carries ONE JSON line.  Libraries write there too (NCCL prints its version banner on the first communicator),
    so file descriptor 1 is pointed at stderr for the run and the line goes to a duplicate of the original."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit_line(obj):
    data = (json.dumps(obj) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


class SharedHost:
    """ONE host buffer that every rank (process) maps: POSIX shared memory.  Each rank page-locks only the byte ranges IT
    writes (pin(): cudaHostRegister of the whole buffer in every process ran into the box's locked-memory limit at 4 and 8
    ranks), so copies into it run at pinned speed and asynchronously.  `ptr` is None when /dev/shm cannot hold the buffer
    (then every rank falls back to a private pinned buffer)."""

    def __init__(self, lib, tag, size, rank, dist):
        from multiprocessing import shared_memory
        self.lib, self.rank, self.dist, self.size = lib, rank, dist, size
        self.shm, self.ptr, self.private, self.pinned = None, None, None, []
        st = os.statvfs("/dev/shm") if os.path.isdir("/dev/shm") else None
        fits = st is not None and st.f_bavail * st.f_frsize > size + (1 << 30)
        import torch
        flag = torch.tensor([1 if fits else 0], device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        if not bool(flag.item()):
            self.private = lib.dll.zb200_alloc_pinned(size)
            assert self.private
            return
        name = f"zb200_{tag}_{os.environ.get('MASTER_PORT', '0')}"
        if rank == 0:
            try:
                shared_memory.SharedMemory(name=name).unlink()
            except Exception:   # noqa: BLE001
                pass
            self.shm = shared_memory.SharedMemory(name=name, create=True, size=size)
        dist.barrier()
        if rank != 0:
            self.shm = shared_memory.SharedMemory(name=name)
        self.ptr = C.addressof(C.c_char.from_buffer(self.shm.buf))

    @property
    def where(self):
        return self.ptr if self.ptr is not None else self.private

    def pin(self, ranges):
        """Page-locks [off, off + n) for every (off, n) this rank writes.  True when all of them are locked."""
        if self.ptr is None:
            return True                                      # the private buffer is pinned memory already
        page = 4096
        spans = sorted((o // page * page, min(self.size, (o + n + page - 1) // page * page)) for o, n in ranges if n)
        merged = []
        for a, b in spans:
            if merged and a <= merged[-1][1]:
                merged[-1][1] = max(merged[-1][1], b)
            else:
                merged.append([a, b])
        for a, b in merged:
            if self.lib.dll.zb200_host_register(C.c_void_p(self.ptr + a), b - a) != 0:
                log(f"[rank {self.rank}] cudaHostRegister of {b - a} bytes failed: {self.lib.last_error()}")
                return False
            self.pinned.append(self.ptr + a)
        return True

    def close(self):
        if self.ptr is not None:
            for p in self.pinned:
                self.lib.dll.zb200_host_unregister(C.c_void_p(p))
            self.dist.barrier()
            self.shm.close()
            if self.rank == 0:
                self.shm.unlink()
        elif self.private:
            self.lib.dll.zb200_free_pinned(C.c_void_p(self.private))
        self.ptr = self.private = None


DUMP_SAMPLE = 1 << 22                  # stream bytes --dump-outputs keeps: 16 MiB of float32 values and 32 MiB of float64
                                       # positions, within 64 MB
DUMP_EDGE = 1 << 16                    # the stream's first and last bytes are always kept (header, last block, trailer)


def dump_stream(out_dir, lib, ptr, clen):
    """What the caller of the timed deflate receives, for comparing two builds output for output:
    deflate_level1_length.npy    the stream's length in bytes (float64, one element);
    deflate_level1_stream.npy    its bytes as float32: all of them when they fit DUMP_SAMPLE, else the first and last
                                 DUMP_EDGE bytes and positions drawn with a fixed seed, in stream order;
    deflate_level1_positions.npy where in the stream each of those bytes sits (float64)."""
    import numpy as np
    host = np.empty(clen, dtype=np.uint8)
    lib.dll.zb200_copy(C.c_void_p(host.ctypes.data), C.c_void_p(ptr), clen, None)
    if clen <= DUMP_SAMPLE:
        pos = np.arange(clen)
    else:
        drawn = np.random.default_rng(0).integers(DUMP_EDGE, clen - DUMP_EDGE, DUMP_SAMPLE - 2 * DUMP_EDGE)
        pos = np.unique(np.concatenate([np.arange(DUMP_EDGE), drawn, np.arange(clen - DUMP_EDGE, clen)]))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "deflate_level1_length.npy"), np.array([clen], dtype=np.float64))
    np.save(os.path.join(out_dir, "deflate_level1_stream.npy"), host[pos].astype(np.float32))
    np.save(os.path.join(out_dir, "deflate_level1_positions.npy"), pos.astype(np.float64))
    log(f"[rank 0] {len(pos)} of the {clen} stream bytes written to {out_dir}")


def traffic_of(kernel):
    """dram__bytes_read + dram__bytes_write per launch of `kernel` from the ncu capture summarised in profiles/traffic.json
    -- only when that capture was taken from the kernel sources as they are now (their hash is stored beside it)."""
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(tpath):
        return None, "no ncu capture committed"
    try:
        t = json.load(open(tpath))
    except Exception:   # noqa: BLE001
        return None, "unreadable"
    src = os.path.join(ROOT, "zlib_b200", "csrc", "zb_deflate.cu")
    sha = hashlib.sha256(open(src, "rb").read()).hexdigest()[:16]
    if t.get("_source_sha16") != sha:
        return None, "stale: zb_deflate.cu changed since the ncu capture in profiles/traffic.json"
    names = {re.sub(r"<.*>|[()]|zb::|^void ", "", k).strip(): v for k, v in t.items() if not k.startswith("_")}
    return names.get(kernel), "ncu --set full capture of this source (profiles/traffic.json)"


def main():
    claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5, help="timed steps of the headline and the end-to-end measurement (at "
                    "least 1); the side measurements of the extras keep their own counts")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="zb200", choices=["zb200", "reference"])
    ap.add_argument("--size-mib", type=int, default=1024)
    ap.add_argument("--pieces", default="", help="rounds per rank of the multi-GPU run: a count, or fractions of a rank's share "
                    "such as 0.5,0.375,0.125 (default: 0.5,0.375,0.125)")
    ap.add_argument("--no-extra", action="store_true", help="skip level 6 / inflate / checksum / zip side measurements")
    ap.add_argument("--no-verify", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the stream the last timed deflate step produced to DIR/*.npy (see dump_stream)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference" and args.dump_outputs:
        ap.error("--dump-outputs writes what the GPU path computed; --impl reference has no such output")
    if args.impl == "reference":
        return run_reference(args)

    import numpy as np
    import torch
    import torch.distributed as dist
    from zlib_b200 import load, binding as zb, dist as zdist, synth

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    lib = load()
    assert lib.dll.zb200_init(local) == 0, lib.last_error()
    s = torch.cuda.current_stream()
    peaks, peak_kind = measured_peaks()

    n = args.size_mib << 20                                  # bytes per GPU
    total = n * world                                        # bytes of the one corpus
    warm = max(3, args.warmup)
    if world == 1:
        rounds = 1
    elif args.pieces:
        rounds = tuple(float(x) for x in args.pieces.split(",")) if "," in args.pieces else max(1, int(args.pieces))
    else:                                                    # the last round's transfer to rank 0 is the exposed one: keep it small where it is large
        rounds = ROUND_SHARES
    ranges = zdist.piece_ranges(total, world, rounds)[rank]
    P = len(ranges)
    log(f"[rank {rank}] generating {args.size_mib} MiB of the {total >> 20} MiB mixed corpus ({len(ranges)} piece(s))")

    # ---- this rank's pieces: pinned host copy [PRE | piece] and the same on the device ----
    pin_src = lib.dll.zb200_alloc_pinned(n + P * PRE)
    assert pin_src
    d_src = torch.empty(n + P * PRE, dtype=torch.uint8, device=dev)
    pieces_dev, pieces_host, at = [], [], 0
    for a, b in ranges:
        lead = PRE if a > 0 else 0
        synth.fill(pin_src + at + (PRE - lead), (b - a) + lead, 1, 1, a - lead)
        dl = WINDOW if a > 0 else 0
        pieces_host.append((pin_src + at + PRE, b - a, pin_src + at + PRE - dl, dl))
        pieces_dev.append((d_src.data_ptr() + at + PRE, b - a, d_src.data_ptr() + at + PRE - dl, dl))
        at += PRE + (b - a)
    lib.dll.zb200_copy(C.c_void_p(d_src.data_ptr()), C.c_void_p(pin_src), n + P * PRE, None)
    host = np.ctypeslib.as_array(C.cast(pin_src + PRE, C.POINTER(C.c_uint8)), shape=(n,)) if world == 1 else None
    cap_piece = lib.compress_bound(max(b - a for a, b in ranges)) + 64
    cap = lib.compress_bound(n) + 64
    outs = [torch.empty(cap_piece, dtype=torch.uint8, device=dev) for _ in ranges] if world > 1 else None
    d_dst = torch.empty(cap, dtype=torch.uint8, device=dev) if world == 1 else None
    total_cap = lib.compress_bound(total) + 64
    # the assembled stream lives on rank 0: a buffer every rank can name (CUDA IPC) so that the copy engines carry the
    # pieces there; when IPC is not to be had, a torch tensor on rank 0 filled by NCCL send / recv
    d_final, final_ptr, final_close = None, None, None
    copy_dev = torch.cuda.Stream() if world > 1 else None
    if world > 1:
        final_ptr, final_close = zdist.share_device_buffer(lib, total_cap)
        if final_ptr is None and rank == 0:
            d_final = torch.empty(total_cap, dtype=torch.uint8, device=dev)
    pin_dst = lib.dll.zb200_alloc_pinned(cap) if world == 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    state = {}

    def step_deflate(level):
        if world == 1:
            state["clen"] = lib.deflate(d_src.data_ptr() + PRE, n, d_dst.data_ptr(), cap, level, zb.WRAP_ZLIB, s)
        else:
            state["clen"], state["crc"], state["adler"], _ = zdist.deflate_rounds(
                lib, pieces_dev, level, zb.WRAP_ZLIB, root=0, outs=outs, final=d_final, stream=s,
                peer_final=final_ptr, copy_stream=copy_dev)

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        l0 = lib.kernel_launches()
        e0.record(s)
        for _ in range(steps):
            fn()
        e1.record(s)
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms / steps, lib.kernel_launches() - l0

    # ---- headline: deflate level 1, device resident (N > 1: assembled on the root inside the timed region) ----
    sampler = ClockSampler(local)
    sampler.start()
    ms1, launches = timed(lambda: step_deflate(1), args.steps, warm)
    clocks = sampler.summary()
    clen1 = state["clen"]
    if args.dump_outputs and rank == 0:                      # before anything else reuses the output buffer
        dump_ptr = d_dst.data_ptr() if world == 1 else final_ptr if final_ptr is not None else d_final.data_ptr()
        dump_stream(args.dump_outputs, lib, dump_ptr, int(clen1))
    value = total / ms1 / 1e6
    log(f"[rank {rank}] deflate L1: {ms1:.2f} ms/step  {value:.2f} GB/s aggregate  ratio {total / clen1:.3f}")

    # ---- per-kernel times (separate pass; events add overhead, so not part of `value`) ----
    lib.profile(True)
    if world == 1:
        step_deflate(1)
    else:                                                    # one piece of this rank, no exchange
        a_ptr, a_n, a_d, a_dl = pieces_dev[0]
        lib.deflate_shard(a_ptr, a_n, a_d if a_dl else None, a_dl, outs[0].data_ptr(), cap_piece, 1, zb.WRAP_RAW,
                          zb.ZB200_DEFLATE_NOT_LAST | zb.ZB200_DEFLATE_NO_HEADER | zb.ZB200_DEFLATE_NO_TRAILER, s)
    prof = lib.profile_report()
    lib.profile(False)

    def kname(k):                                            # "(k_lz_walk<kWalkThreadsFast, false>)" -> "k_lz_walk"
        return re.sub(r"<.*>|[()]|zb::", "", k).strip()
    prof = {kname(k): v for k, v in prof.items()}
    prof_bytes = n if world == 1 else pieces_dev[0][1]       # input bytes the profiled pass covered
    dom = max(prof.items(), key=lambda kv: kv[1][0]) if prof else ("none", (0.0, 1))
    dom_launches = max(1, dom[1][1])                         # one launch per pipeline slab
    dom_ms = dom[1][0] / dom_launches                        # average launch duration of the dominant kernel
    algo_bytes = prof_bytes * (1.0 + clen1 / total)          # SURVEY 8(d): every input byte read once, every output byte written once
    launch_bytes = algo_bytes / dom_launches                 # algorithmic bytes one launch (one slab) accounts for
    achieved = launch_bytes / dom_ms / 1e6 if dom_ms > 0 else 0.0
    traffic, traffic_note = traffic_of(dom[0])
    kern_total = sum(v[0] for v in prof.values()) or 1.0
    roofline = {"bound": "hbm", "kernel": dom[0], "achieved": round(achieved, 2), "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": round(achieved / peaks["hbm_gbs"], 5), "traffic": traffic, "traffic_source": traffic_note,
                "peak_source": peak_kind, "algorithmic_bytes": round(algo_bytes), "algorithmic_bytes_per_launch": round(launch_bytes),
                "launches_per_step": dom_launches, "kernel_ms": round(dom_ms, 4),
                "kernel_share_of_step": round(dom[1][0] / kern_total, 4),
                "whole_step": {"achieved": round(total * (1.0 + clen1 / total) / ms1 / 1e6, 2),
                               "frac": round(total * (1.0 + clen1 / total) / ms1 / 1e6 / (peaks["hbm_gbs"] * world), 5)},
                "kernels_ms": {k.replace("zb::", ""): round(v[0], 4) for k, v in prof.items()},
                "profiled_bytes": prof_bytes}

    # ---- end to end with HOST buffers (H2D + kernels + D2H inside the timed region) ----
    shm = None
    if world == 1:
        def step_e2e():
            ol = C.c_ulong(cap)
            rc = lib.dll.compress2(C.c_void_p(pin_dst), C.byref(ol), C.c_void_p(pin_src + PRE), n, 1)
            assert rc == 0, (rc, lib.last_error())
            state["e2e_len"] = ol.value
        api = "compress2(dest,&destLen,source,sourceLen,1) on pinned host buffers"
    else:
        shm = SharedHost(lib, "bench", total_cap, rank, dist)
        shm_ptr = shm.where
        copy_stream = torch.cuda.Stream()
        placed = []

        def step_e2e(placed=None):
            state["e2e_len"], _, _, _ = zdist.deflate_rounds(lib, pieces_host, 1, zb.WRAP_ZLIB, root=0, outs=outs,
                                                             host_final=shm_ptr, stream=s, copy_stream=copy_stream, placed=placed)
        step_e2e(placed)                                     # where this rank's pieces land (the same every step: same data)
        pinned_ok = shm.pin(placed)
        t_ok = torch.tensor([1 if pinned_ok else 0], device=dev)
        dist.all_reduce(t_ok, op=dist.ReduceOp.MIN)
        pinned_ok = bool(t_ok.item())
        api = ("zb200_deflate_shard_begin/_end per piece from pinned host input, NCCL all-gather of {len,n,crc,adler} per round, "
               "D2H of every piece straight into ONE shared host buffer at its final offset "
               + ("(every rank page-locks the ranges it writes)" if shm.ptr is not None and pinned_ok else
                  "(NOT page-locked: cudaHostRegister refused)" if shm.ptr is not None else
                  "-- /dev/shm cannot hold the stream: every rank copies into a private pinned buffer"))
    step_e2e()
    step_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    barrier()
    e2e_s = (time.perf_counter() - t0) / args.steps
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e = {"value": round(total / e2e_s / 1e9, 4), "unit": UNIT, "h2d_bytes_per_step": total,
           "d2h_bytes_per_step": int(state["e2e_len"]) + 32 * world, "ms_per_step": round(e2e_s * 1e3, 3), "api": api}
    log(f"[rank {rank}] e2e: {e2e_s * 1e3:.1f} ms/step {e2e['value']} GB/s")

    extra, verified, assembled, cpu = {}, None, None, None
    import zhelpers
    have_ref = os.path.exists(zhelpers.REF_PATH)
    if rank == 0:
        # ---- correctness gate (a) on the measured outputs: the reference (else the oracle) decodes them bit-exact ----
        check = reference_inflate_check if have_ref else oracle_inflate_check
        verified_with = "reference inflate (oracle/_ref)" if have_ref else "oracle inflate (oracle/libzoracle.so)"
        if not args.no_verify:
            t0 = time.perf_counter()
            if world == 1:
                verified = check(pin_dst, int(state["e2e_len"]), total)
            else:
                h_final = np.empty(int(clen1), dtype=np.uint8)
                lib.dll.zb200_copy(C.c_void_p(h_final.ctypes.data), C.c_void_p(final_ptr if final_ptr is not None else d_final.data_ptr()), int(clen1), None)
                if shm.ptr is not None:                         # the stream in the shared host buffer is decoded by the reference;
                    ok_host = check(shm_ptr, int(state["e2e_len"]), total)
                    same = int(clen1) == int(state["e2e_len"]) and bool(np.array_equal(                    # the one on the root GPU must be the same bytes
                        h_final, np.ctypeslib.as_array(C.cast(shm_ptr, C.POINTER(C.c_uint8)), shape=(int(clen1),))))
                    ok_dev = same or check(h_final.ctypes.data, int(clen1), total)
                else:
                    ok_host, ok_dev = True, check(h_final.ctypes.data, int(clen1), total)
                verified = bool(ok_dev and ok_host)
                assembled = True
                del h_final
            log(f"[rank 0] assembled stream(s) decoded and compared by the {verified_with}: {verified} "
                f"({time.perf_counter() - t0:.1f} s)")
            assert verified, f"the {verified_with} could not decode the GPU deflate output"
        # ---- CPU baseline beside it: same number of bytes as one GPU's share ----
        if have_ref:
            rb = RefBench(n)
            v, r_ratio = rb.step(1)
            cpu = {"value": round(v, 4), "unit": UNIT, "cores": rb.cores, "kind": "reference",
                   "sample": f"reference compress2 level 1 over {rb.total >> 20} MiB of the same corpus, one {rb.per >> 20} MiB slice per host thread",
                   "ratio": round(r_ratio, 4)}
            log(f"[rank 0] reference compress2 L1 on {rb.cores} host threads: {v:.3f} GB/s ratio {r_ratio:.3f}")
            del rb

    if not args.no_extra:
        if world == 1:
            extras_single(args, lib, zb, synth, s, dev, n, cap, d_src, d_dst, pin_src, pin_dst, host, state, timed, peaks, extra, step_e2e, have_ref)
        else:
            extras_multi(args, lib, zb, zdist, synth, s, dev, n, world, rank, d_src, timed, peaks, extra, have_ref, barrier)
        if rank == 0:
            log(f"[rank 0] extras: {json.dumps(extra)}")

    if rank == 0:
        line = {"metric": METRIC, "value": round(value, 4), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                "warmup": warm, "ms_per_step": round(ms1, 3), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic",
                "config": workload_config(args.size_mib, world),
                "ratio": round(total / clen1, 4), "compressed_bytes": int(clen1),
                "roofline": roofline, "cpu_baseline": cpu, "e2e": e2e, "gpu_launches": int(launches),
                "clocks": clocks, "verified_by_reference": verified,
                "verified_with": None if verified is None else verified_with, "assembled": assembled if world > 1 else True,
                "gather": (None if world == 1 else "copy engines over NVLink into rank 0's buffer (CUDA IPC)" if final_ptr is not None
                           else "NCCL send / recv into rank 0's buffer"),
                "extra": extra}
        emit_line(line)
    if shm is not None:
        shm.close()
    if final_close is not None:
        final_close()
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------------- side measurements, one GPU
def make_stream_set(host_bytes, sz, distinct, have_ref):
    """`distinct` zlib streams of sz bytes each cut from host_bytes, level 6, produced by the reference when available."""
    import zhelpers
    if have_ref:
        ref = zhelpers.Ref()
        zs, kind = [None] * distinct, "reference compress2 level 6"

        def mk(t, nt=min(os.cpu_count() or 1, 32)):
            for i in range(distinct * t // nt, distinct * (t + 1) // nt):
                zs[i] = ref.compress2(host_bytes[i * sz:(i + 1) * sz], 6)
        _threads(mk, min(os.cpu_count() or 1, 32))
    else:
        import zlib as pyz
        zs, kind = [pyz.compress(host_bytes[i * sz:(i + 1) * sz].tobytes(), 6) for i in range(distinct)], "system zlib level 6"
    return zs, kind


def extras_single(args, lib, zb, synth, s, dev, n, cap, d_src, d_dst, pin_src, pin_dst, host, state, timed, peaks, extra, step_e2e, have_ref):
    import numpy as np
    import torch
    import zhelpers
    src_ptr = d_src.data_ptr() + PRE
    d_data = d_src[PRE:PRE + n]

    # ---- level 6 and the ratio gate (d) at the config shapes: C2 = this corpus, C1 = 64 MiB text ----
    def step6():
        state["clen6"] = lib.deflate(src_ptr, n, d_dst.data_ptr(), cap, 6, zb.WRAP_ZLIB, s)
    ms6, _ = timed(step6, max(1, args.steps // 2), 1)
    extra["deflate_level6"] = {"GBps": round(n / ms6 / 1e6, 3), "ratio": round(n / state["clen6"], 4), "ms": round(ms6, 2)}
    n1 = 64 << 20
    text = synth.synth(n1, 0, 7)
    d_text = torch.from_numpy(text).to(dev)
    gpu_sizes = {"C2_mixed_1GiB_L1": int(state["clen"]), "C2_mixed_1GiB_L6": int(state["clen6"])}
    for lv in (1, 6):
        gpu_sizes[f"C1_text_64MiB_L{lv}"] = int(lib.deflate(d_text.data_ptr(), n1, d_dst.data_ptr(), cap, lv, zb.WRAP_ZLIB, s))
    if have_ref and not args.no_verify:
        t0 = time.perf_counter()
        ref_sizes = reference_stream_sizes({"C2_mixed_1GiB_L1": (host, 1), "C2_mixed_1GiB_L6": (host, 6),
                                            "C1_text_64MiB_L1": (text, 1), "C1_text_64MiB_L6": (text, 6)})
        extra["ratio_vs_reference"] = {k: {"gpu_bytes": gpu_sizes[k], "reference_bytes": ref_sizes[k],
                                           "gpu_over_reference": round(gpu_sizes[k] / ref_sizes[k], 5),
                                           "within_2pct": bool(gpu_sizes[k] <= 1.02 * ref_sizes[k])} for k in gpu_sizes}
        extra["ratio_vs_reference"]["_how"] = ("the reference's compress2 over the WHOLE buffer as one stream at the same level "
                                               f"(4 host threads, {time.perf_counter() - t0:.0f} s); gate (d): gpu_bytes <= 1.02 x reference_bytes")
    del d_text

    # ---- fused checksum ----
    out2 = torch.zeros(2, dtype=torch.int32, device=dev)
    msc, _ = timed(lambda: lib.checksum_dev(src_ptr, n, out2.data_ptr(), s), 10, 3)
    extra["crc32_adler32_fused"] = {"GBps": round(n / msc / 1e6, 1), "ms": round(msc, 4),
                                    "frac_of_hbm_peak": round(n / msc / 1e6 / peaks["hbm_gbs"], 4)}

    # ---- batch inflate: 64 KiB zlib streams of the same corpus, level 6, produced by the reference when available ----
    sz, distinct = 65536, 2048
    ns = n // sz
    t0 = time.perf_counter()
    zs, src_kind = make_stream_set(host, sz, distinct, have_ref)
    zsn = (zs * ((ns + distinct - 1) // distinct))[:ns]
    src_off = np.zeros(ns + 1, dtype=np.int64)
    src_off[1:] = np.cumsum([len(z) for z in zsn])
    d_z = torch.from_numpy(np.frombuffer(b"".join(zsn) + b"\0" * 8, dtype=np.uint8).copy()).to(dev)
    d_so = torch.from_numpy(src_off).to(dev)
    d_do = torch.arange(ns + 1, dtype=torch.int64, device=dev) * sz
    d_len = torch.zeros(ns, dtype=torch.int64, device=dev)
    d_st = torch.zeros(ns, dtype=torch.int32, device=dev)
    d_inf = torch.empty(n, dtype=torch.uint8, device=dev)
    log(f"[rank 0] prepared {ns} streams ({src_kind}) in {time.perf_counter() - t0:.1f} s")
    msi, _ = timed(lambda: lib.inflate_batch_dev(d_z.data_ptr(), d_so.data_ptr(), ns, d_inf.data_ptr(), d_do.data_ptr(),
                                                 d_len.data_ptr(), d_st.data_ptr(), zb.WRAP_ZLIB, s), 3, 2)
    ok = int(d_st.abs().sum()) == 0 and bool((d_len == sz).all()) and bool(torch.equal(d_inf[:distinct * sz], d_data[:distinct * sz]))
    extra["inflate_batch"] = {"GBps": round(ns * sz / msi / 1e6, 3), "streams": ns, "stream_bytes": sz, "ms": round(msi, 2),
                              "source": src_kind, "all_ok": ok, "compressed_fraction": round(int(src_off[-1]) / (ns * sz), 4)}
    del d_inf
    # the same batch through zb200_inflate_batch with pinned HOST arenas: H2D + decode + D2H inside the timed region
    zin = int(src_off[-1])
    pin_z = lib.dll.zb200_alloc_pinned(zin + 64)
    assert pin_z
    z_host = d_z.cpu().numpy()                              # keep the array alive across the copy
    C.memmove(C.c_void_p(pin_z), C.c_void_p(z_host.ctypes.data), zin)
    del z_host
    h_so, h_do = src_off.astype(np.uint64), (np.arange(ns + 1, dtype=np.uint64) * sz)
    h_len, h_st = np.zeros(ns, dtype=np.uint64), np.zeros(ns, dtype=np.int32)
    th = []
    for _ in range(3):
        t0 = time.perf_counter()
        rc = lib.dll.zb200_inflate_batch(C.c_void_p(pin_z), C.c_void_p(h_so.ctypes.data), ns, C.c_void_p(pin_dst), C.c_void_p(h_do.ctypes.data),
                                         C.c_void_p(h_len.ctypes.data), C.c_void_p(h_st.ctypes.data), zb.WRAP_ZLIB, None)
        th.append(time.perf_counter() - t0)
        assert rc == 0 and not h_st.any() and bool((h_len == sz).all())
    okh = bool(np.array_equal(np.ctypeslib.as_array(C.cast(pin_dst, C.POINTER(C.c_uint8)), shape=(distinct * sz,)), host[:distinct * sz]))
    extra["inflate_batch_host_e2e"] = {"GBps": round(ns * sz / min(th) / 1e9, 3), "ms": round(min(th) * 1e3, 2), "host_buffers": "pinned",
                                       "h2d_bytes": zin, "d2h_bytes": ns * sz, "output_matches": okh}
    lib.dll.zb200_free_pinned(C.c_void_p(pin_z))
    del d_z
    # the e2e call again with malloc'ed (pageable) buffers -- what an unmodified caller of the reference passes
    pg_src = np.array(host, copy=True)
    pg_dst = np.empty(cap, dtype=np.uint8)
    pg_dst[:] = 0
    tp = []
    for _ in range(3):
        ol = C.c_ulong(cap)
        t0 = time.perf_counter()
        rc = lib.dll.compress2(C.c_void_p(pg_dst.ctypes.data), C.byref(ol), C.c_void_p(pg_src.ctypes.data), n, 1)
        tp.append(time.perf_counter() - t0)
        assert rc == 0 and ol.value == int(state["e2e_len"])
    extra["compress2_pageable_e2e"] = {"GBps": round(n / min(tp) / 1e9, 3), "ms": round(min(tp) * 1e3, 1), "host_buffers": "pageable (malloc)",
                                       "staging": "8 host threads, 4 MiB pieces through pinned slots"}
    del pg_src, pg_dst
    # uncompress() of ONE long stream: the compress2 output of the e2e leg (1 GiB in one zlib stream, pinned host
    # buffers); decoded in parallel at its chunk boundaries (BASELINE config 1's round trip, at config 2's size)
    step_e2e()                                             # pin_dst holds the level-1 stream again
    zlen1 = int(state["e2e_len"])
    pin_rt = lib.dll.zb200_alloc_pinned(n)
    assert pin_rt
    tu = []
    for _ in range(3):
        ul = C.c_ulong(n)
        t0 = time.perf_counter()
        rc = lib.dll.uncompress(C.c_void_p(pin_rt), C.byref(ul), C.c_void_p(pin_dst), zlen1)
        tu.append(time.perf_counter() - t0)
        assert rc == 0 and ul.value == n, (rc, lib.last_error())
    rt_ok = bool(np.array_equal(np.ctypeslib.as_array(C.cast(pin_rt, C.POINTER(C.c_uint8)), shape=(n,)), host))
    assert rt_ok, "uncompress(compress2(x)) != x"
    extra["uncompress_one_stream"] = {"GBps": round(n / min(tu) / 1e9, 3), "ms": round(min(tu) * 1e3, 1), "stream_bytes": zlen1,
                                      "host_buffers": "pinned", "round_trip_exact": rt_ok}
    lib.dll.zb200_free_pinned(C.c_void_p(pin_rt))
    # BASELINE config 1, direction (b): ONE 64 MiB text buffer compressed by the REFERENCE at level 6 (no flush points in
    # that stream: block starts are found), decoded by uncompress() of this library; the reference's own uncompress beside it
    if have_ref:
        refz = zhelpers.Ref()
        t0 = time.perf_counter()
        z1 = refz.compress2(text, 6)
        t_refc = time.perf_counter() - t0
        ob = C.create_string_buffer(n1)
        ul = C.c_ulong(n1)
        t0 = time.perf_counter()
        assert refz.dll.uncompress(ob, C.byref(ul), z1, len(z1)) == 0
        t_refu = time.perf_counter() - t0
        tz = []
        for _ in range(3):
            ul = C.c_ulong(n1)
            t0 = time.perf_counter()
            rc = lib.dll.uncompress(ob, C.byref(ul), z1, len(z1))
            tz.append(time.perf_counter() - t0)
            assert rc == 0 and ul.value == n1
        ok1 = ob.raw == text.tobytes()
        assert ok1, "uncompress(reference stream) differs"
        extra["uncompress_reference_stream_64MiB"] = {"GBps": round(n1 / min(tz) / 1e9, 3), "ms": round(min(tz) * 1e3, 1),
                                                      "stream_bytes": len(z1), "host_buffers": "pageable", "bit_exact": ok1,
                                                      "reference_uncompress_ms_one_core": round(t_refu * 1e3, 1),
                                                      "reference_compress2_level6_s_one_core": round(t_refc, 2)}
    # the full shape of BASELINE config 3: 100 000 streams of 64 KiB (the 2048 distinct ones repeated), 6.1 GiB out --
    # a structured sub-record with its own roofline and clocks (BASELINE's metric names deflate AND inflate GB/s)
    extra["inflate_batch_config3"] = inflate_config3(lib, zb, s, dev, zs, distinct, sz, d_data, timed, peaks, 0, 1, None)
    # checksum at the per-GPU size of BASELINE config 4 scaled to one call's uInt limit: 4 GiB - 64 KiB
    n4 = (4 << 30) - 65536
    d_big = torch.empty(n4, dtype=torch.uint8, device=dev)
    d_big.view(torch.int64).random_()
    msc4, _ = timed(lambda: lib.checksum_dev(d_big.data_ptr(), n4, out2.data_ptr(), s), 5, 2)
    extra["crc32_adler32_fused_4GiB"] = {"GBps": round(n4 / msc4 / 1e6, 1), "ms": round(msc4, 4),
                                         "frac_of_hbm_peak": round(n4 / msc4 / 1e6 / peaks["hbm_gbs"], 4)}
    del d_big
    # ZIP archive (config 5 shape): files of log-uniform size 4 KiB .. 16 MiB cut from the same corpus, one
    # zb200_zip_build call on pinned host buffers (H2D + batch deflate + device-side assembly + one D2H)
    import random as _r
    rng = _r.Random(5)
    offs = [0]
    while offs[-1] < n and len(offs) <= 65535:
        offs.append(min(n, offs[-1] + int(4096 * 2 ** rng.uniform(0, 12))))
    nf = len(offs) - 1
    zoff = np.array(offs, dtype=np.uint64)
    znames = (C.c_char_p * nf)(*[b"f%05d.bin" % i for i in range(nf)])
    zcap = lib.dll.zb200_zip_bound(znames, C.c_void_p(zoff.ctypes.data), nf)
    pin_zip = lib.dll.zb200_alloc_pinned(zcap)
    assert pin_zip
    zt = []
    for _ in range(3):
        ol = C.c_size_t(zcap)
        t0 = time.perf_counter()
        rc = lib.dll.zb200_zip_build(znames, C.c_void_p(pin_src + PRE), C.c_void_p(zoff.ctypes.data), nf, 1, zb.DOS_DATETIME,
                                     C.c_void_p(pin_zip), C.byref(ol))
        zt.append(time.perf_counter() - t0)
        assert rc == 0, (rc, lib.last_error())
    zok = None
    if not args.no_verify:
        import io
        import zipfile
        arc = bytes(np.ctypeslib.as_array(C.cast(pin_zip, C.POINTER(C.c_uint8)), shape=(ol.value,)))
        zf = zipfile.ZipFile(io.BytesIO(arc))
        pick = rng.sample(range(nf), min(nf, 25))
        zok = all(zf.read("f%05d.bin" % i) == host[offs[i]:offs[i + 1]].tobytes() for i in pick) and len(zf.namelist()) == nf
        assert zok, "zip members do not read back"
    extra["zip_build_level1"] = {"GBps": round(n / min(zt) / 1e9, 3), "files": nf, "archive_bytes": int(ol.value),
                                 "ms": round(min(zt) * 1e3, 1), "host_buffers": "pinned", "members_read_back": zok}
    lib.dll.zb200_free_pinned(C.c_void_p(pin_zip))
    extra["reference_cpu"] = reference_side_paths()        # the reference's other paths on this box's host cores


def inflate_config3(lib, zb, s, dev, zs, distinct, sz, d_expect, timed, peaks, rank, world, zdist):
    """BASELINE config 3: 100 000 independent 64 KiB zlib streams (the `distinct` reference-made ones repeated), device
    resident, sharded by stream over the ranks.  Returns the sub-record (rank 0's view after the all-reduce)."""
    import numpy as np
    import torch
    ns3 = 100000
    zs3 = (zs * ((ns3 + distinct - 1) // distinct))[:ns3]
    so3 = np.zeros(ns3 + 1, dtype=np.int64)
    so3[1:] = np.cumsum([len(z) for z in zs3])
    if world == 1:
        a, b = 0, ns3
    else:
        mine = zdist.balance_streams([len(z) for z in zs3], world)[rank]
        a, b = mine[0], mine[-1] + 1
    # every rank holds only its own range of streams and its own part of the output
    blob = b"".join(zs3[a:b]) + b"\0" * 8
    d_z3 = torch.from_numpy(np.frombuffer(blob, dtype=np.uint8).copy()).to(dev)
    d_so3 = torch.from_numpy(so3[a:b + 1] - so3[a]).to(dev)
    d_do3 = torch.arange(b - a + 1, dtype=torch.int64, device=dev) * sz
    d_out3 = torch.empty((b - a) * sz, dtype=torch.uint8, device=dev)
    d_len3 = torch.zeros(b - a, dtype=torch.int64, device=dev)
    d_st3 = torch.zeros(b - a, dtype=torch.int32, device=dev)
    sampler = ClockSampler(dev.index or 0)
    sampler.start()

    def step():
        lib.inflate_batch_dev(d_z3.data_ptr(), d_so3.data_ptr(), b - a, d_out3.data_ptr(), d_do3.data_ptr(),
                              d_len3.data_ptr(), d_st3.data_ptr(), zb.WRAP_ZLIB, s)
        if world > 1:                                       # the path's one exchange: {status, length} of every stream, everywhere
            import torch.distributed as dist
            res = torch.full((ns3, 2), -100, dtype=torch.int64, device=dev)
            res[a:b, 0] = d_st3.to(torch.int64)
            res[a:b, 1] = d_len3
            dist.all_reduce(res, op=dist.ReduceOp.MAX)
            step.res = res
    msi3, _ = timed(step, 3, 2)
    clocks = sampler.summary()
    # every stream decoded to its length, and every output equals the slice the reference compressed
    k0 = a % distinct
    ok_local = int(d_st3.abs().sum()) == 0 and bool((d_len3 == sz).all())
    cmp_n = min(b - a, distinct)
    for i in range(0, cmp_n, 256):                           # stream a + i is distinct stream (a + i) % distinct
        j = (k0 + i) % distinct
        m = min(256, cmp_n - i, distinct - j)
        ok_local = ok_local and bool(torch.equal(d_out3[i * sz:(i + m) * sz], d_expect[j * sz:(j + m) * sz]))
    if world > 1:
        import torch.distributed as dist
        res = step.res
        ok_all = bool((res[:, 0] == 0).all()) and bool((res[:, 1] == sz).all())
        flag = torch.tensor([1 if (ok_local and ok_all) else 0], device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        ok_local = bool(flag.item())
    comp = int(so3[-1])
    algo = ns3 * sz + comp
    gbps = ns3 * sz / msi3 / 1e6
    return {"metric": "inflate_batch_GBps_uncompressed", "value": round(gbps, 3), "unit": "GB/s", "GBps": round(gbps, 3),
            "streams": ns3, "stream_bytes": sz, "ms": round(msi3, 2), "all_ok": ok_local, "n_gpus": world,
            "source": "reference compress2 level 6 (2048 distinct streams repeated)", "compressed_bytes": comp,
            "roofline": {"bound": "hbm", "kernel": "k_inflate_batch", "achieved": round(algo / msi3 / 1e6, 2),
                         "peak": peaks["hbm_gbs"] * world, "unit": "GB/s", "frac": round(algo / msi3 / 1e6 / (peaks["hbm_gbs"] * world), 5),
                         "algorithmic_bytes": algo, "traffic": None},
            "clocks": clocks}


# ------------------------------------------------------------------------------------- side measurements, N GPUs
def extras_multi(args, lib, zb, zdist, synth, s, dev, n, world, rank, d_src, timed, peaks, extra, have_ref, barrier):
    """BASELINE configs 3, 4 and 5 across the ranks, each with its GB/s and a pass flag checked against the reference."""
    import numpy as np
    import torch
    import torch.distributed as dist
    import zhelpers
    sz, distinct = 65536, 2048
    # ---- C3: the first 128 MiB of the corpus is what the 2048 distinct streams hold (every rank builds the same set) ----
    base = synth.synth(distinct * sz, 1, 1)
    zs, src_kind = make_stream_set(base, sz, distinct, have_ref)
    d_base = torch.from_numpy(base).to(dev)
    rec = inflate_config3(lib, zb, s, dev, zs, distinct, sz, d_base, timed, peaks, rank, world, zdist)
    rec["source"] = src_kind + " (2048 distinct streams repeated), streams sharded by compressed size, all-reduce of {status, length}"
    if rank == 0:
        extra["inflate_batch_config3"] = rec
    del d_base, zs

    # ---- C4: crc32 + adler32 of ONE world GiB buffer, 1 GiB slice per rank, _combine fold across the ranks ----
    a0 = rank * n                                            # slice r = corpus bytes [r n, (r + 1) n) with seed 4
    h_slice = synth.synth(n, 1, 4, a0)
    d_slice = torch.from_numpy(h_slice).to(dev)
    st = {}

    def step_ck():
        st["crc"], st["adler"], st["len"] = zdist.checksum_sharded(lib, d_slice, stream=s)
    msck, _ = timed(step_ck, 5, 2)
    rec4 = {"GBps": round(world * n / msck / 1e6, 1), "ms": round(msck, 4), "bytes": world * n, "n_gpus": world,
            "frac_of_hbm_peak": round(world * n / msck / 1e6 / (peaks["hbm_gbs"] * world), 4),
            "exchange": "all-gather of {crc32, adler32, len} per rank, crc32_combine / adler32_combine fold in rank order on every rank"}
    if rank == 0 and have_ref and not args.no_verify:
        # the reference: crc32 / adler32 of every slice on host threads, folded with ITS crc32_combine / adler32_combine
        ref = zhelpers.Ref()
        part = [None] * world

        def work(r):
            hs = h_slice if r == 0 else synth.synth(n, 1, 4, r * n)
            part[r] = (ref.dll.crc32(0, C.c_void_p(hs.ctypes.data), n), ref.dll.adler32(1, C.c_void_p(hs.ctypes.data), n))
        _threads(work, world)
        crc, adl = part[0]
        for r in range(1, world):
            crc = ref.dll.crc32_combine(crc, part[r][0], n)
            adl = ref.dll.adler32_combine(adl, part[r][1], n)
        rec4["matches_reference"] = bool(crc == st["crc"] and adl == st["adler"] and st["len"] == world * n)
        assert rec4["matches_reference"], "sharded checksum differs from the reference's fold"
    if rank == 0:
        extra["crc32_adler32_sharded_config4"] = rec4
    del d_slice, h_slice

    # ---- C5: ONE ZIP32 archive of 10 000 files, members compressed on all ranks, extracted by the reference miniunz ----
    extra_zip = zip_config5(args, lib, zb, zdist, synth, dev, world, rank, have_ref, barrier)
    if rank == 0:
        extra["zip_sharded_config5"] = extra_zip


def zip_sizes(nfiles=10000, seed=5):
    """10 000 sizes in [4 KiB, 16 MiB]: 93 % log-uniform in [4 KiB, 256 KiB], 7 % log-uniform in [256 KiB, 16 MiB]
    (about 3 GiB in total).  A plain log-uniform law over the whole range averages 2 MiB per file, 20 GiB in all, and a
    ZIP32 archive (zip.c of the reference writes no ZIP64 records) holds sizes and offsets below 4 GiB -- so the choice
    here is ONE archive with the weight on small files rather than several archives."""
    import random
    rng = random.Random(seed)
    sizes = []
    for _ in range(nfiles):
        if rng.random() < 0.93:
            sizes.append(int(4096 * 64 ** rng.random()))
        else:
            sizes.append(int(262144 * 64 ** rng.random()))
    sizes[0], sizes[1] = 4096, 16 << 20                     # both ends of the range are present
    return sizes


def zip_config5(args, lib, zb, zdist, synth, dev, world, rank, have_ref, barrier):
    import numpy as np
    import torch
    import torch.distributed as dist
    sizes = zip_sizes()
    nf = len(sizes)
    names = [b"f%05d.bin" % i for i in range(nf)]
    shares = zdist.assign_files(sizes, world)
    mine = shares[rank]
    # file i holds corpus bytes starting at its own 64 KiB-aligned offset (content T/M alternating by file index)
    starts = np.zeros(nf + 1, dtype=np.int64)
    starts[1:] = np.cumsum([(z + 65535) // 65536 * 65536 for z in sizes])
    my_total = sum(sizes[i] for i in mine)
    pin_in = lib.dll.zb200_alloc_pinned(my_total + 64)
    assert pin_in
    off = np.zeros(len(mine) + 1, dtype=np.uint64)
    at = 0
    for k, i in enumerate(mine):
        synth.fill(pin_in + at, sizes[i], i & 1, 11, int(starts[i]))
        at += sizes[i]
        off[k + 1] = at
    cnames = (C.c_char_p * max(1, len(mine)))(*[names[i] for i in mine])
    seg_cap = lib.dll.zb200_zip_bound(cnames, C.c_void_p(off.ctypes.data), len(mine))
    d_seg = torch.empty(seg_cap, dtype=torch.uint8, device=dev)
    members = np.zeros((max(1, len(mine)), 4), dtype=np.uint64)
    # the archive is assembled in ONE shared page-locked host buffer: every rank copies its segment D2H to its place
    arc_cap = int(sum(sizes) * 1.01) + 200 * nf + 65536
    shm = SharedHost(lib, "zip", arc_cap, rank, dist)
    if shm.ptr is None:
        shm.close()
        lib.dll.zb200_free_pinned(C.c_void_p(pin_in))
        return {"skipped": "/dev/shm cannot hold the archive"} if rank == 0 else None
    shm_ptr = shm.ptr
    width = max(len(x) for x in shares)
    out = {}

    def step():
        ol = C.c_size_t(seg_cap)
        rc = lib.dll.zb200_zip_segment(cnames, C.c_void_p(pin_in), C.c_void_p(off.ctypes.data), len(mine), 1, zb.DOS_DATETIME,
                                       C.c_void_p(d_seg.data_ptr()), C.byref(ol), C.c_void_p(members.ctypes.data))
        assert rc == 0, (rc, lib.last_error())
        rec = torch.full((width + 1, 5), -1, dtype=torch.int64)
        rec[0, 0] = ol.value
        if mine:
            m = torch.from_numpy(members[:len(mine)].astype(np.int64))
            rec[1:len(mine) + 1, 0] = torch.tensor(mine, dtype=torch.int64)
            rec[1:len(mine) + 1, 1:4] = m[:, 0:3]
            rec[1:len(mine) + 1, 4] = m[:, 3] & 0xFFFFFFFF
        allrec = torch.empty(world * (width + 1) * 5, dtype=torch.int64, device=dev)
        dist.all_gather_into_tensor(allrec, rec.to(dev).view(-1))
        allrec = allrec.view(world, width + 1, 5).cpu().tolist()         # plain lists: 10 000 members are walked below
        seg_len = [int(allrec[r][0][0]) for r in range(world)]
        base = sum(seg_len[:rank])
        out["mine"] = (base, ol.value)
        lib._check(lib.dll.zb200_copy_async(shm_ptr + base, d_seg.data_ptr(), ol.value, None), "zb200_copy_async")
        lib._check(lib.dll.zb200_sync(None), "zb200_sync")
        out["total"] = sum(seg_len)
        if rank == 0:                                        # central directory over all members, in archive order
            order, glob, b0 = [], [], 0
            for r in range(world):
                for k in range(len(shares[r])):
                    i, lo, cl, rl, crc = allrec[r][k + 1]
                    order.append(names[i].decode())
                    glob.append((b0 + lo, cl, rl, crc))
                b0 += seg_len[r]
            cd = lib.zip_directory(order, glob, b0)
            C.memmove(shm_ptr + b0, cd, len(cd))
            out["arc_len"] = b0 + len(cd)
    step()
    barrier()
    shm.pin([out["mine"]])                                   # this rank's segment lands in the same place every time
    step()
    barrier()
    ts = []
    for _ in range(2):
        barrier()
        t0 = time.perf_counter()
        step()
        barrier()
        ts.append(time.perf_counter() - t0)
    t = torch.tensor([min(ts)], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    sec = float(t.item())
    res = None
    if rank == 0:
        res = {"GBps": round(sum(sizes) / sec / 1e9, 3), "ms": round(sec * 1e3, 1), "files": nf, "raw_bytes": int(sum(sizes)),
               "archive_bytes": int(out["arc_len"]), "n_gpus": world, "level": 1, "host_buffers": "pinned input per rank, shared page-locked archive",
               "sizes": "4 KiB .. 16 MiB: 93 % log-uniform below 256 KiB, 7 % log-uniform above, so that ONE archive stays inside ZIP32",
               "exchange": "all-gather of the member records, every rank's segment D2H to its place, directory written by rank 0"}
        if not args.no_verify:
            import tempfile
            import zipfile
            tmp = tempfile.mkdtemp(prefix="zb200_zip_")
            path = os.path.join(tmp, "c5.zip")
            with open(path, "wb") as f:
                f.write(shm.shm.buf[:out["arc_len"]])
            zf = zipfile.ZipFile(path)
            ok = len(zf.namelist()) == nf
            exe = os.path.join(ROOT, "oracle", "_ref", "miniunz")
            if os.path.exists(exe):
                xdir = os.path.join(tmp, "x")
                os.mkdir(xdir)
                p = subprocess.run([exe, "-o", path], cwd=xdir, capture_output=True, text=True, timeout=1200)
                ok = ok and p.returncode == 0 and len(os.listdir(xdir)) == nf
                for i in range(nf):                          # every member, bit-exact against the regenerated corpus
                    if not ok:
                        break
                    got = np.fromfile(os.path.join(xdir, names[i].decode()), dtype=np.uint8)
                    ok = len(got) == sizes[i] and bool(np.array_equal(got, synth.synth(sizes[i], i & 1, 11, int(starts[i]))))
                res["extracted_by"] = "reference miniunz (oracle/_ref), all members compared"
            else:
                ok = ok and zf.testzip() is None
                res["extracted_by"] = "python zipfile (oracle/_ref/miniunz not built)"
            import shutil
            shutil.rmtree(tmp, ignore_errors=True)
            res["extracted_bit_exact"] = bool(ok)
            assert ok, "ZIP members do not extract bit-exact"
    shm.close()
    lib.dll.zb200_free_pinned(C.c_void_p(pin_in))
    return res


if __name__ == "__main__":
    sys.exit(main())
