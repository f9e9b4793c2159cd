#!/usr/bin/env python
"""tools/gpu_entropy_devout_probe.py [n] -- zj_decode_batch_gpu_device on n 4K 4:2:0 JPEGs with one restart interval per MCU row:
pinned JPEG bytes in, pixels left in device memory; ZJ_GPU_ENTROPY_TRACE=1 prints phase times (adds synchronisation)."""
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np

import jpeg_util
from zune_jpeg_b200 import gpu
from zune_jpeg_b200.decoder import ZuneJpegOptions, decode_batch

w, h, n = 3840, 2160, int(sys.argv[1]) if len(sys.argv) > 1 else 256
jpegs = [jpeg_util.synth_jpeg(i, w, h, "420", 90, False, False, 1) for i in range(4)]
out_bytes = w * h * 3
pin = gpu.PinnedBuffer(sum(len(j) for j in jpegs))
ins, off = [], 0
for j in jpegs:
    pin.array[off:off + len(j)] = np.frombuffer(j, np.uint8)
    ins.append(pin.array[off:off + len(j)])
    off += len(j)
ins = [ins[i % 4] for i in range(n)]
dev = [gpu.DeviceBuffer(out_bytes) for _ in range(min(n, 64))]
targets = [(dev[i % len(dev)].ptr, out_bytes) for i in range(n)]
ref = decode_batch([jpegs[0]], ZuneJpegOptions(), threads=1)[0]
times = []
for rep in range(6):
    stats = {}
    t0 = time.perf_counter()
    decode_batch(ins, ZuneJpegOptions(), threads=0, device_out=targets, stats=stats)
    times.append(time.perf_counter() - t0)
assert dev[0].download().tobytes() == ref
best = min(times[1:])
print(f"{n} x {w}x{h}: best {1e3 * best:.1f} ms = {n * w * h / 1e6 / best:.0f} MP/s (all: {' '.join('%.1f' % (1e3 * t) for t in times)}), on GPU: {stats}")
