#!/usr/bin/env python
"""tools/scaled_probe.py [n] -- DCT-scaled libjpeg output (ZJ_FLAG_SCALE_*) on the bench's workload: n (256) 3840x2160 4:2:0
images, resident coefficient planes (8 distinct images, as bench.py's pool), output RGB u8.  Prints the card and its power limit,
then:
  - zj_batch_run of the libjpeg plans at 1/1, 1/2, 1/4 and 1/8, alternating, timed with CUDA events (medians), in ms and in GP/s
    of source pixels and of output pixels;
  - a device-to-device copy in the same run, so that each plan's algorithmic bytes (coefficient bytes read -- the rows the reduced
    IDCTs use, one 32-byte sector per block at 1/8 -- plus output bytes written) can be stated as a share of the measured copy rate;
  - JPEG bytes -> one 224 x 224 f16 CHW batch tensor (Pillow bicubic, Resize(256) + CenterCrop(224)) through
    decode_batch_resized at 1/1 and 1/4, alternating, on 64 of the images.
Before anything is timed, the outputs of the 8 distinct images are checked against the statement (tests/test_scaled_output.py)."""
import ctypes as C
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import torch

import jpeg_util
from test_scaled_output import scaled_expected
from zune_jpeg_b200 import _ffi, gpu
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch_resized

W, H, N = 3840, 2160, int(sys.argv[1]) if len(sys.argv) > 1 else 256
DISTINCT, REPS, JPEG_N = 8, 10, 64
DENOMS = (1, 2, 4, 8)
MEAN = [255 * m for m in (0.485, 0.456, 0.406)] + [0.0]
INV = [1 / (255 * s) for s in (0.229, 0.224, 0.225)] + [1.0]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def coef_read_bytes(d, w, h):
    """coefficient bytes one w x h 4:2:0 image's plan reads: 128 per block at 1/1 (every row), the 16-byte rows the reduced
    IDCT uses otherwise (7 at 4x4, 5 at 2x2), 32 (one sector) at 1x1; luma blocks are 8/d samples a side, chroma 16/d"""
    per = {8: 128, 4: 7 * 16, 2: 5 * 16, 1: 32}
    mcu = -(-w // 16) * -(-h // 16)
    return mcu * (4 * per[8 // d] + 2 * per[min(16 // d, 8)])


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
    # the host stage is the same at every scale: one set of device planes, one descriptor per scale
    pools = {d: [] for d in DENOMS}
    keep = []
    wants = {d: [] for d in DENOMS}
    for data in datas:
        img, planes = Decoder.new_with_options(libjpeg).decode_coefficients(data)
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b_, p in zip(bufs, planes):
            b_.upload(p)
        keep.append((planes, bufs))
        for d in DENOMS:
            di = _ffi.ZjImage()
            C.memmove(C.byref(di), C.byref(img), C.sizeof(di))
            di.flags |= (d.bit_length() - 1) << _ffi.FLAG_SCALE_SHIFT
            wants[d].append(scaled_expected(di, planes))
            for z, b_ in enumerate(bufs):
                di.comp[z].coeff = b_.ptr
            pools[d].append(di)
    sizes = {d: int(np.prod(_ffi.scaled_size(W, H, d))) * 3 for d in DENOMS}
    outs = {d: gpu.DeviceBuffer(sizes[d] * N) for d in DENOMS}
    batches = {d: gpu.Batch([pools[d][i % DISTINCT] for i in range(N)], [outs[d].ptr + i * sizes[d] for i in range(N)], [sizes[d]] * N)
               for d in DENOMS}
    for d, b in batches.items():
        outs[d].memset(0xAB)
        b.run()
        gpu.synchronize()
        for i in range(DISTINCT):
            got = outs[d].download(sizes[d], offset=i * sizes[d])
            assert np.array_equal(got, wants[d][i]), (d, i, int(np.count_nonzero(got != wants[d][i])))
    print("outputs checked: every plan = its statement (8 distinct images)", flush=True)

    copy_src = torch.empty(sizes[1] * N // 2, dtype=torch.uint8, device="cuda")
    copy_dst = torch.empty_like(copy_src)
    for b in batches.values():
        b.run()
    copy_dst.copy_(copy_src)
    torch.cuda.synchronize()
    t = {d: [] for d in DENOMS}
    t["copy"] = []
    for _ in range(REPS):
        for d, b in batches.items():
            t[d].append(timed(b.run))
        t["copy"].append(timed(lambda: copy_dst.copy_(copy_src)))
    med = {k: float(np.median(v)) for k, v in t.items()}
    copy_rate = 2 * copy_src.numel() / (med["copy"] * 1e-3)           # bytes read + written per second
    res = {"card": card(), "images": N, "width": W, "height": H, "copy_GBps": copy_rate / 1e9, "reps": REPS}
    for d in DENOMS:
        ms = med[d]
        algo = N * (coef_read_bytes(d, W, H) + sizes[d])
        res[f"1/{d}"] = {"ms": ms, "source_GPps": N * W * H / (ms * 1e-3) / 1e9, "output_GPps": N * sizes[d] / 3 / (ms * 1e-3) / 1e9,
                         "algo_bytes": algo, "share_of_copy_rate": algo / (ms * 1e-3) / copy_rate, "spread_ms": [min(t[d]), max(t[d])]}
    for b in batches.values():
        b.destroy()
    del outs

    # ---- JPEG bytes -> one 224 x 224 f16 CHW batch tensor, at 1/1 and 1/4
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    rz = gpu.Resize((224, 224), "pil_bicubic", short_side=256)
    jdatas = [np.frombuffer(datas[i % DISTINCT], np.uint8) for i in range(JPEG_N)]
    jt = {1: [], 4: []}
    for rep in range(4):
        for d in jt:
            t0 = time.perf_counter()
            out, errs = decode_batch_resized(jdatas, rz, desc, None, libjpeg.set_scale_denom(d), threads=0)
            dt = time.perf_counter() - t0
            assert errs == [None] * JPEG_N, errs
            if rep == 0:
                want = rz.expected(wants[d][1], *_ffi.scaled_size(W, H, d), 3, desc)
                assert out.download()[1].tobytes() == want.tobytes(), d
            if rep > 0:
                jt[d].append(dt)
            del out
    for d in jt:
        s = float(np.median(jt[d]))
        res[f"jpeg_to_224_f16chw_1/{d}"] = {"s": s, "images_per_s": JPEG_N / s, "spread_s": [min(jt[d]), max(jt[d])]}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
