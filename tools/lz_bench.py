"""f3 match stage: pbsgpu_blob_encode_batch_lz next to pbsgpu_blob_encode_batch_z on three 8 GiB device-resident images in
4 MiB chunks, into PINNED host memory through the raw C calls (the blocking call is the timed region; the two calls
alternate).  Images: (a) tools/blob_bench.py's half-zero image, (b) a text-like corpus (a 64 MiB seeded
oracle/zstd_lz.text_corpus tiled: K9's matches stay inside 128 KiB blocks, so tiling does not change its ratio),
(c) random bytes.  Also: libzstd level 1 (pyarrow) on a 64 MiB sample of each image (CPU, ratio only), and K9's kernel
time from a separate torch.profiler run of one _lz call per image."""
import subprocess
import sys
import time
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
import pbs_plus_b200 as pg  # noqa: E402
from oracle import zstd_lz  # noqa: E402

smi = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip()
print(f"device: {smi}")
e = pg.Engine(0)
L_ = e._L
n, CH = 8 << 30, 4 << 20
SAMPLE = 64 << 20
off = np.arange(0, n, CH, dtype=np.uint64)
ln = np.full(len(off), CH, dtype=np.uint64)
boff = np.arange(len(off), dtype=np.uint64) * np.uint64(CH + 12)
out = e.host_alloc(int(len(off)) * (CH + 12))
blen = np.zeros(len(off), dtype=np.uint64)
crc = np.zeros(len(off), dtype=np.uint32)
calls = {"_z": L_.pbsgpu_blob_encode_batch_z, "_lz": L_.pbsgpu_blob_encode_batch_lz}


def run(fn, d):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    rc = fn(e._h, d.data_ptr(), off.ctypes.data, ln.ctypes.data, len(off), out.ctypes.data, boff.ctypes.data,
            blen.ctypes.data, crc.ctypes.data)
    dt = time.perf_counter() - t0
    assert rc == 0, rc
    return dt, int(blen.sum())


def image(kind):
    if kind == "half-zero":
        d = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda")
        d[1 << 30: 5 << 30] = 0
    elif kind == "text":
        tile = torch.from_numpy(np.frombuffer(zstd_lz.text_corpus(1, SAMPLE), dtype=np.uint8).copy()).cuda()
        d = tile.repeat(n // SAMPLE)
    else:
        d = torch.randint(0, 256, (n,), dtype=torch.uint8, device="cuda")
    return d


import pyarrow as pa  # noqa: E402

lvl1 = pa.Codec("zstd", compression_level=1)
for kind in ("half-zero", "text", "random"):
    d = image(kind)
    res = {k: [] for k in calls}
    for rep in range(3):
        for k, fn in calls.items():
            res[k].append(run(fn, d))
    for k in calls:
        dts = [r[0] for r in res[k]]
        size = res[k][-1][1]
        print(f"({kind}) blob_encode_batch{k}: {n / min(dts) / 1e9:.1f} GB/s of input (best of 3; runs "
              f"{', '.join(f'{t * 1e3:.0f}' for t in dts)} ms), output {size / 2**30:.3f} GiB = ratio {n / size:.2f}")
    # a sample from the middle of the image (for half-zero: 32 MiB random + 32 MiB zeros)
    lo = (1 << 30) - SAMPLE // 2 if kind == "half-zero" else 0
    sample = d[lo: lo + SAMPLE].cpu().numpy().tobytes()
    print(f"({kind}) libzstd level 1 on a {SAMPLE >> 20} MiB sample (CPU): ratio {len(sample) / len(lvl1.compress(sample)):.2f}")
    with torch.profiler.profile(activities=[torch.profiler.ProfilerActivity.CUDA]) as prof:
        run(calls["_lz"], d)
        torch.cuda.synchronize()
    kern = [ev for ev in prof.key_averages() if ev.self_device_time_total > 0]
    k9 = [ev for ev in kern if "k_zlz" in ev.key]
    kt = sum(ev.self_device_time_total for ev in k9)   # microseconds
    other = sum(ev.self_device_time_total for ev in kern) - kt
    print(f"({kind}) K9 k_zlz kernel time (profiled run): {kt / 1e3:.1f} ms over {sum(ev.count for ev in k9)} launch(es) = "
          f"{n / (kt * 1e-6) / 1e9 if kt else float('nan'):.1f} GB/s of input; other device time in the call {other / 1e3:.1f} ms")
    del d
    torch.cuda.empty_cache()
e.host_free(out)
e.close()
