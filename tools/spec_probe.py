#!/usr/bin/env python
"""tools/spec_probe.py [n] -- spec-correct output (ZJ_VARIANT_SPEC) and libjpeg-turbo-exact output (ZJ_VARIANT_SPEC with
ZJ_FLAG_ISLOW) on the bench's workload: n (256) 3840x2160 4:2:0 images, resident coefficient planes (8 distinct images, as
bench.py's pool), output RGB u8.  Prints the card and its power limit, then:
  - zj_batch_run of the as-written plan, the spec plan and the islow plan, alternating, timed with CUDA events (medians), in GP/s;
  - a device-to-device copy in the same run, so that each rate can be stated as a share of the measured copy rate;
  - the bytes each plan reads and writes: the algorithmic 6 B/px, and for the spec kernel (both IDCTs) the bytes it reads
    counting the chroma context blocks it transforms again (computed from the shapes);
  - JPEG bytes -> f16 CHW (ImageNet mean / std) through decode_batch(device_out, desc), as written, spec and libjpeg,
    alternating: spec and libjpeg images take the host entropy route, so this shows what that costs.
Before anything is timed, the spec and islow outputs of the 8 distinct images are checked against their statements
(tests/test_spec_output.py, tests/test_libjpeg_output.py) and the as-written ones against the oracle."""
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
import oracle
from test_libjpeg_output import libjpeg_expected
from test_spec_output import spec_expected
from zune_jpeg_b200 import _ffi, gpu
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch

W, H, N = 3840, 2160, int(sys.argv[1]) if len(sys.argv) > 1 else 256
DISTINCT, REPS, JPEG_N = 8, 10, 64
MEAN = [255 * m for m in (0.485, 0.456, 0.406)] + [0.0]
INV = [1 / (255 * s) for s in (0.229, 0.224, 0.225)] + [1.0]
TM_HV = 20   # MCU columns per spec_kernel tile in 4:2:0 (zj_device.h: TM_HV)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def spec_read_bytes(w, h):
    """coefficient bytes spec_kernel<MODE_HV> reads for one w x h 4:2:0 image: every luma block once, every chroma block of a
    tile plus the context blocks it transforms again (one block column each side, one block row above and below)"""
    mcu_x, mcu_y = -(-w // 16), -(-h // 16)
    strips, cw, ch = (mcu_y + 1) // 2, -(-w // 2), -(-h // 2)
    blocks = strips * 4 * 2 * mcu_x
    for t in range(-(-mcu_x // TM_HV)):
        m0, m1 = t * TM_HV, min(t * TM_HV + TM_HV, mcu_x)
        cols = (m1 - m0) + (m0 > 0) + (m1 * 8 < cw)
        for s in range(strips):
            rows = 2 + (s > 0) + ((s + 1) * 16 < ch)
            blocks += 2 * rows * cols
    return blocks * 128


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
    spec_opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_spec_output(True)
    islow_opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    all_opts = (("as_written", ZuneJpegOptions()), ("spec", spec_opts), ("islow", islow_opts))
    statement = {"spec": spec_expected, "islow": libjpeg_expected,
                 "as_written": lambda img, planes: oracle.reconstruct(img, threads=os.cpu_count() or 4)}
    plans = {}
    keep = []
    wants = {name: [] for name, _ in all_opts}
    for name, opts in all_opts:
        pool = []
        for data in datas:
            img, planes = Decoder.new_with_options(opts).decode_coefficients(data)
            wants[name].append(statement[name](img, planes))
            bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
            for b_, p in zip(bufs, planes):
                b_.upload(p)
            keep.append((planes, bufs))
            d = _ffi.ZjImage()
            C.memmove(C.byref(d), C.byref(img), C.sizeof(d))
            for z, b_ in enumerate(bufs):
                d.comp[z].coeff = b_.ptr
            pool.append(d)
        plans[name] = [pool[i % DISTINCT] for i in range(N)]
    size = W * H * 3
    out = gpu.DeviceBuffer(size * N)
    ptrs = [out.ptr + i * size for i in range(N)]
    batches = {k: gpu.Batch(v, ptrs, [size] * N) for k, v in plans.items()}
    for name, b in batches.items():
        out.memset(0xAB)
        b.run()
        gpu.synchronize()
        for i in range(DISTINCT):
            got = out.download(size, offset=i * size)
            assert np.array_equal(got, wants[name][i]), (name, i, int(np.count_nonzero(got != wants[name][i])))
    print("outputs checked: spec and islow = their statements, as written = the oracle (8 distinct images)", flush=True)

    copy_src = torch.empty(size * N // 2, dtype=torch.uint8, device="cuda")
    copy_dst = torch.empty_like(copy_src)
    for b in batches.values():
        b.run()
    copy_dst.copy_(copy_src)
    torch.cuda.synchronize()
    t = {"as_written": [], "spec": [], "islow": [], "copy": []}
    for _ in range(REPS):
        for name, b in batches.items():
            t[name].append(timed(b.run))
        t["copy"].append(timed(lambda: copy_dst.copy_(copy_src)))
    med = {k: float(np.median(v)) for k, v in t.items()}
    copy_rate = 2 * copy_src.numel() / (med["copy"] * 1e-3)           # bytes read + written per second
    res = {"card": card(), "images": N, "width": W, "height": H, "copy_GBps": copy_rate / 1e9}
    coef = {k: sum(2 * p.size for p in keep[i * DISTINCT][0]) for i, (k, _) in enumerate(all_opts)}
    for name, _ in all_opts:
        ms = med[name]
        algo = N * (coef[name] + size)
        moved = N * (spec_read_bytes(W, H) + size) if name != "as_written" else algo
        res[name] = {"ms": ms, "GPps": N * W * H / (ms * 1e-3) / 1e9, "algo_B_per_px": algo / (N * W * H),
                     "moved_B_per_px": moved / (N * W * H), "share_of_copy_rate": algo / (ms * 1e-3) / copy_rate,
                     "moved_share_of_copy_rate": moved / (ms * 1e-3) / copy_rate, "spread_ms": [min(t[name]), max(t[name])]}
    del out
    for b in batches.values():
        b.destroy()

    # ---- JPEG bytes -> f16 CHW in device memory, as written, spec and libjpeg
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    jdatas = [np.frombuffer(datas[i % DISTINCT], np.uint8) for i in range(JPEG_N)]
    dst = gpu.DeviceBuffer(W * H * 3 * 2 * JPEG_N)
    dev_out = [(dst.ptr + i * W * H * 6, W * H * 6) for i in range(JPEG_N)]
    jt = {name: [] for name, _ in all_opts}
    for rep in range(4):
        for name, opts in all_opts:
            stats = {}
            t0 = time.perf_counter()
            r = decode_batch(jdatas, opts, threads=0, device_out=dev_out, desc=desc, stats=stats)
            dt = time.perf_counter() - t0
            assert all(x == W * H * 6 for x in r), r
            if rep == 0 and name != "as_written":
                want = desc.expected(wants[name][1], W, H, 3)
                assert dst.download(W * H * 6, offset=W * H * 6).tobytes() == want.tobytes()
            if rep > 0:
                jt[name].append(dt)
    for name in jt:
        s = float(np.median(jt[name]))
        res[f"jpeg_to_f16chw_{name}"] = {"s": s, "MPps": JPEG_N * W * H / s / 1e6, "spread_s": [min(jt[name]), max(jt[name])]}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
