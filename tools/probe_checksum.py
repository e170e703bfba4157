"""Device-side timing of the fused checksum (development probe, not the bench): zb200_checksum_dev over a range of sizes,
CUDA events around ten launches each, results up to 256 MiB checked against zlib."""
import os, sys, zlib
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from zlib_b200 import load

L = load()
assert L.dll.zb200_init(0) == 0, L.last_error()
s = torch.cuda.current_stream()
for n in (1 << 20, (16 << 20) + 12345, 256 << 20, 1 << 30, (4 << 30) - 65536):
    x = torch.empty(n, dtype=torch.uint8, device="cuda")
    x[: n // 8 * 8].view(torch.int64).random_()
    out = torch.zeros(2, dtype=torch.int32, device="cuda")
    for _ in range(3):
        L.checksum_dev(x.data_ptr(), n, out.data_ptr(), s)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 10
    e0.record()
    for _ in range(reps):
        L.checksum_dev(x.data_ptr(), n, out.data_ptr(), s)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    ok = ""
    if n <= (256 << 20):
        h = x.cpu().numpy().tobytes()
        got = [v & 0xffffffff for v in out.tolist()]
        ok = "ok" if got == [zlib.crc32(h), zlib.adler32(h)] else "MISMATCH %s" % got
    print(f"n={n / 2**20:.1f} MiB  {ms:.4f} ms  {n/ms/1e6:.1f} GB/s  frac {n/ms/1e6/6553.9:.3f} {ok}", flush=True)
    del x
