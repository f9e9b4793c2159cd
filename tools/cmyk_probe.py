#!/usr/bin/env python
"""tools/cmyk_probe.py [n] -- four-component JPEGs (DESIGN.md section 4.6.4) on the batch-tensor route: n (64) 3840x2160 JPEGs
(8 distinct contents) -> one f16 CHW 224 x 224 batch tensor (pil_bicubic, short_side = 256), libjpeg output, through
decode_batch_resized.  The same contents are run twice, alternating: as Pillow-written CMYK JPEGs and as YCbCr 4:2:0 JPEGs.
Prints the card and its power limit, then the median call times (host clock around calls that return once the tensor is in
place), and, from torch.profiler in a separate pass, the time of cmyk_kernel and of spec_kernel per call.  Before anything is
timed, every slot is checked against Pillow's convert("RGB") followed by torchvision's Resize(256) + CenterCrop(224)."""
import io
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import torch
from PIL import Image

from zune_jpeg_b200 import gpu
from zune_jpeg_b200.decoder import ColorSpace, ZuneJpegOptions, decode_batch_resized

W, H, N = 3840, 2160, int(sys.argv[1]) if len(sys.argv) > 1 else 64
DISTINCT, REPS, S, OUT = 8, 7, 256, 224


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def content(seed):
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (H // 64 + 2, W // 64 + 2, 4), dtype=np.uint8)
    im = np.asarray(Image.fromarray(base, "CMYK").resize((W, H), Image.BICUBIC)).astype(np.int16)
    return Image.fromarray(np.clip(im + rng.integers(-12, 13, im.shape), 0, 255).astype(np.uint8), "CMYK")


def encode(im, **kw):
    b = io.BytesIO()
    im.save(b, "JPEG", quality=90, **kw)
    return b.getvalue()


def main():
    import torchvision.transforms as T
    torch.cuda.init()
    print(f"card: {card()}", flush=True)
    ims = [content(i) for i in range(DISTINCT)]
    sets = {"cmyk": [encode(im) for im in ims], "ycbcr": [encode(im.convert("RGB"), subsampling=2) for im in ims]}
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    resize = gpu.Resize((OUT, OUT), filter="pil_bicubic", short_side=S)
    desc = gpu.OutputDesc(layout="CHW", dtype="f16")
    tf = T.Compose([T.Resize(S, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(OUT)])

    def call(name):
        arr, errs = decode_batch_resized([sets[name][i % DISTINCT] for i in range(N)], resize, desc, options=opts)
        assert errs == [None] * N, errs
        return arr

    for name, datas in sets.items():
        t = call(name).to_torch()
        for i in range(DISTINCT):
            want = torch.from_numpy(np.asarray(tf(Image.open(io.BytesIO(datas[i])).convert("RGB"))).copy()).permute(2, 0, 1).half()
            assert torch.equal(t[i].cpu(), want), (name, i)
    print("outputs checked against Pillow + torchvision", flush=True)

    times = {k: [] for k in sets}
    for _ in range(REPS):
        for name in sets:
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            call(name)
            times[name].append((time.perf_counter() - t0) * 1e3)
    med = {k: float(np.median(v)) for k, v in times.items()}

    from torch.profiler import ProfilerActivity, profile
    kernel_ms = {}
    for name in sets:
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            call(name)
            torch.cuda.synchronize()
        for e in prof.key_averages():
            for k in ("cmyk_kernel", "spec_kernel"):
                if k in e.key:
                    kernel_ms[f"{name}:{k}"] = kernel_ms.get(f"{name}:{k}", 0.0) + e.device_time_total / 1e3
    res = {"card": card(), "images": N, "distinct": DISTINCT, "width": W, "height": H, "reps": REPS,
           "file_MB": {k: sum(len(d) for d in v) / DISTINCT / 1e6 for k, v in sets.items()},
           "call_ms": med, "spread_ms": {k: [min(v), max(v)] for k, v in times.items()},
           "images_per_s": {k: N / (v * 1e-3) for k, v in med.items()}, "kernel_ms_per_call": kernel_ms}
    print(json.dumps(res), flush=True)


if __name__ == "__main__":
    main()
