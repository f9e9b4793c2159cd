#!/usr/bin/env python
"""tools/orient_probe.py [n] -- EXIF orientation (ZJ_FLAG_ORIENT_*) on the bench's workload: n (256) 3840x2160 4:2:0 images,
resident coefficient planes (8 distinct images, as bench.py's pool), libjpeg output, RGB u8.  Prints the card and its power
limit, then:
  - zj_batch_run of the plan with o = 1 (no transform) and with o = 6 (ROTATE_270: the transposing kind), alternating, timed with
    CUDA events (medians); the difference is what orientation costs end to end;
  - orient_kernel's own time from torch.profiler (a separate pass after the timed one), and the pass's bytes moved (every output
    byte read once from the scratch and written once) over that time, against a device-to-device copy timed in the same run.
Before anything is timed, the o = 1 outputs of the 8 distinct images are checked against the statement
(tests/test_libjpeg_output.py) and the o = 6 outputs against their rotation."""
import ctypes as C
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import torch

import jpeg_util
from test_libjpeg_output import libjpeg_expected
from zune_jpeg_b200 import _ffi, gpu
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions

W, H, N = 3840, 2160, int(sys.argv[1]) if len(sys.argv) > 1 else 256
DISTINCT, REPS = 8, 10
ORIENTS = (1, 6)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b)


def main():
    torch.cuda.init()
    print(f"card: {card()}", flush=True)
    datas = [jpeg_util.synth_jpeg(i, W, H, "420", 90) for i in range(DISTINCT)]
    libjpeg = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    pools = {o: [] for o in ORIENTS}
    keep, wants = [], []
    for data in datas:
        img, planes = Decoder.new_with_options(libjpeg).decode_coefficients(data)
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b_, p in zip(bufs, planes):
            b_.upload(p)
        keep.append((planes, bufs))
        wants.append(libjpeg_expected(img, planes))
        for o in ORIENTS:
            di = _ffi.ZjImage()
            C.memmove(C.byref(di), C.byref(img), C.sizeof(di))
            di.flags |= (o - 1) << _ffi.FLAG_ORIENT_SHIFT
            for z, b_ in enumerate(bufs):
                di.comp[z].coeff = b_.ptr
            pools[o].append(di)
    size = W * H * 3
    outs = {o: gpu.DeviceBuffer(size * N) for o in ORIENTS}
    batches = {o: gpu.Batch([pools[o][i % DISTINCT] for i in range(N)], [outs[o].ptr + i * size for i in range(N)], [size] * N)
               for o in ORIENTS}
    for o, b in batches.items():
        outs[o].memset(0xAB)
        b.run()
        gpu.synchronize()
        for i in range(DISTINCT):
            got = outs[o].download(size, offset=i * size)
            want = wants[i] if o == 1 else np.ascontiguousarray(np.rot90(wants[i].reshape(H, W, 3), -1)).reshape(-1)
            assert np.array_equal(got, want), (o, i, int(np.count_nonzero(got != want)))
        every = gpu.DeviceArray(outs[o], (N, size), _ffi.DTYPE_U8).to_torch()   # (image i repeats image i % DISTINCT)
        assert all(torch.equal(every[i], every[i % DISTINCT]) for i in range(N)), o
    print("outputs checked: o = 1 = the statement, o = 6 = its rotation (all images)", flush=True)

    copy_src = torch.empty(size * N // 2, dtype=torch.uint8, device="cuda")
    copy_dst = torch.empty_like(copy_src)
    copy_dst.copy_(copy_src)
    torch.cuda.synchronize()
    t = {o: [] for o in ORIENTS}
    t["copy"] = []
    for _ in range(REPS):
        for o, b in batches.items():
            t[o].append(timed(b.run))
        t["copy"].append(timed(lambda: copy_dst.copy_(copy_src)))
    med = {k: float(np.median(v)) for k, v in t.items()}
    copy_rate = 2 * copy_src.numel() / (med["copy"] * 1e-3)           # bytes read + written per second

    # orient_kernel's own time, in a separate pass under the profiler
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(3):
            batches[6].run()
        torch.cuda.synchronize()
    kt = [e for e in prof.key_averages() if "orient_kernel" in e.key]
    orient_ms = sum(e.device_time_total for e in kt) / 1e3 / 3 if kt else float("nan")   # (us over 3 runs)
    pass_bytes = 2 * N * size
    res = {"card": card(), "images": N, "width": W, "height": H, "reps": REPS, "copy_GBps": copy_rate / 1e9,
           "batch_run_ms": {f"o={o}": med[o] for o in ORIENTS}, "spread_ms": {f"o={o}": [min(t[o]), max(t[o])] for o in ORIENTS},
           "orientation_cost_ms": med[6] - med[1], "orientation_cost_share": (med[6] - med[1]) / med[1],
           "orient_kernel_ms": orient_ms, "orient_pass_bytes": pass_bytes, "orient_pass_GBps": pass_bytes / (orient_ms * 1e-3) / 1e9,
           "orient_pass_share_of_copy_rate": pass_bytes / (orient_ms * 1e-3) / copy_rate,
           "orient_pass_share_of_copy_rate_from_difference": pass_bytes / ((med[6] - med[1]) * 1e-3) / copy_rate}
    for b in batches.values():
        b.destroy()
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
