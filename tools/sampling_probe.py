#!/usr/bin/env python
"""tools/sampling_probe.py [n] [width height] -- three-component JPEGs with the sampling factors of DESIGN.md section 4.6.5 against
4:2:0, libjpeg output.  Files (from tests/test_sampling_factors.py's encoder, quality 90, one seed per content, 3840x2160 by
default): 4:1:1, 4:1:0 and "Y 1x1, chroma 2x2", and 4:2:0 with the same seeds.
  1. resident planes: the host stage's planes of 8 images on the device, zj_batch_run to RGB, timed with CUDA events;
  2. JPEG bytes -> one f16 CHW 224 x 224 batch tensor (pil_bicubic, short_side = 256) through decode_batch_resized, n (64)
     images, median host time of calls that return once the tensor is in place;
  3. the CMYK files of tools/cmyk_probe.py on route 2, through the same kernel (raster_kernel).
Prints the card and its power limit first, and per set the time of raster_kernel and spec_kernel per call from torch.profiler
in a separate pass.  Every output is checked against Pillow (+ torchvision's Resize(256) + CenterCrop(224) on route 2) before
anything is timed."""
import io
import json
import os
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")]
import numpy as np
import torch
from PIL import Image

from cmyk_probe import card, content as cmyk_content, encode as cmyk_encode
from test_sampling_factors import jpeg
from zune_jpeg_b200 import gpu
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch_resized

N = int(sys.argv[1]) if len(sys.argv) > 1 else 64
W, H = (int(sys.argv[2]), int(sys.argv[3])) if len(sys.argv) > 3 else (3840, 2160)
DISTINCT, RESIDENT, REPS, S, OUT = 2, 8, 7, 256, 224
SETS = {"420": [(2, 2), (1, 1), (1, 1)], "411": [(4, 1), (1, 1), (1, 1)], "410": [(4, 2), (1, 1), (1, 1)],
        "chroma_2x2": [(1, 1), (2, 2), (2, 2)]}


def kernel_ms(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for e in prof.key_averages():
        for k in ("raster_kernel", "spec_kernel"):
            if k in e.key:
                out[k] = out.get(k, 0.0) + e.device_time_total / 1e3
    return out


def main():
    import torchvision.transforms as T
    torch.cuda.init()
    print(f"card: {card()}", flush=True)
    t0 = time.perf_counter()
    files = {k: [jpeg(s, W, H, seed=i, quality=90) for i in range(DISTINCT)] for k, s in SETS.items()}
    files["cmyk"] = [cmyk_encode(cmyk_content(i)) for i in range(DISTINCT)] if (W, H) == (3840, 2160) else []
    print(f"files written in {time.perf_counter() - t0:.1f} s", flush=True)
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    res = {"card": card(), "width": W, "height": H, "images": N, "resident_images": RESIDENT, "reps": REPS,
           "file_MB": {k: sum(map(len, v)) / max(len(v), 1) / 1e6 for k, v in files.items()}}

    # 1. resident planes -> RGB through zj_batch_run
    res["resident_ms"], res["resident_kernel_ms"] = {}, {}
    for name in SETS:
        keep, imgs, outs, wants = [], [], [], []
        for i in range(RESIDENT):
            data = files[name][i % DISTINCT]
            img, planes = Decoder.new_with_options(opts).decode_coefficients(data)
            bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
            for z, (b, p) in enumerate(zip(bufs, planes)):
                b.upload(p)
                img.comp[z].coeff = b.ptr
            keep.append((planes, bufs))
            imgs.append(img)
            outs.append(gpu.DeviceBuffer(W * H * 3))
            if i < DISTINCT:
                wants.append(np.asarray(Image.open(io.BytesIO(data)).convert("RGB")))
        gpu.synchronize()
        batch = gpu.Batch(imgs, [o.ptr for o in outs], [W * H * 3] * RESIDENT)
        batch.run()
        gpu.synchronize()
        for o, w in zip(outs, wants):
            assert o.download(W * H * 3).tobytes() == w.tobytes(), name
        start, stop = gpu.Event(), gpu.Event()
        times = []
        for _ in range(REPS):
            start.record()
            for _ in range(10):
                batch.run()
            stop.record()
            gpu.synchronize()
            times.append(start.elapsed_ms(stop) / 10)
        res["resident_ms"][name] = float(np.median(times))
        res["resident_kernel_ms"][name] = kernel_ms(batch.run)
        batch.destroy()
        del keep, outs
    print("resident planes checked against Pillow", flush=True)

    # 2. / 3. JPEG bytes -> one batch tensor
    resize = gpu.Resize((OUT, OUT), filter="pil_bicubic", short_side=S)
    desc = gpu.OutputDesc(layout="CHW", dtype="f16")
    tf = T.Compose([T.Resize(S, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(OUT)])
    names = [k for k in files if files[k]]

    def call(name):
        arr, errs = decode_batch_resized([files[name][i % DISTINCT] for i in range(N)], resize, desc, options=opts)
        assert errs == [None] * N, errs
        return arr

    for name in names:
        t = call(name).to_torch()
        for i in range(min(N, DISTINCT)):
            im = Image.open(io.BytesIO(files[name][i])).convert("RGB")
            want = torch.from_numpy(np.asarray(tf(im)).copy()).permute(2, 0, 1).half()
            assert torch.equal(t[i].cpu(), want), (name, i)
    print("batch tensors checked against Pillow + torchvision", flush=True)
    times = {k: [] for k in names}
    for _ in range(REPS):
        for name in names:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            call(name)
            times[name].append((time.perf_counter() - t0) * 1e3)
    res["tensor_call_ms"] = {k: float(np.median(v)) for k, v in times.items()}
    res["tensor_spread_ms"] = {k: [min(v), max(v)] for k, v in times.items()}
    res["tensor_images_per_s"] = {k: N / (v * 1e-3) for k, v in res["tensor_call_ms"].items()}
    res["tensor_kernel_ms"] = {k: kernel_ms(lambda: call(k)) for k in names}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
