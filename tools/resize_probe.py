#!/usr/bin/env python
"""tools/resize_probe.py [n] -- the cropped, resized batch tensor on the bench's workload: n (256) 3840x2160 4:2:0 images, resident
coefficient planes (8 distinct images, as bench.py's pool), to an n x 3 x 224 x 224 f16 CHW tensor normalised with the ImageNet
mean / std.  Timed with CUDA events, the seven routes alternating:
  1 zj_gpu_reconstruct_device_resized, area, whole images
  2 the same with seeded RandomResizedCrop crops (scale 0.08-1, ratio 3/4-4/3)
  3 bilinear with the same crops
  4 what it replaces: zj_gpu_reconstruct_device_ex to full-size f16 CHW, then per image torch crop + interpolate + stack
  5 Pillow's bilinear (pil_bilinear) with the same crops: torchvision's RandomResizedCrop on PIL images
  6 pil_bilinear with short_side = 256, whole images: Resize(256) + CenterCrop(224)
  7 what a user would otherwise write for 5: route 4 with torch interpolate(antialias=True)
and the area kernel alone (zj_gpu_resize_device over resident u8; bytes read / time) against a device-to-device copy, and the
kernels of routes 5 and 6 (profiler): the table kernel's time, and the bytes each pass reads against the copy rate.  Every timed
output is checked against gpu.Resize.expected applied to the oracle's bytes before anything is printed (routes 1-3, 5, 6
bit-exact on a sample of slots, routes 4 and 7 within a tolerance: torch interpolates the f16 values).  Prints the card and its
power limit beside the numbers."""
import ctypes as C
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]
import numpy as np
import torch

import jpeg_util
import oracle
from zune_jpeg_b200 import _ffi, gpu
from zune_jpeg_b200.decoder import Decoder, ZuneJpegOptions

W, H, N = 3840, 2160, int(sys.argv[1]) if len(sys.argv) > 1 else 256
DISTINCT, OUT, REPS = 8, 224, 5
MEAN = [255 * m for m in (0.485, 0.456, 0.406)]
INV = [1 / (255 * s) for s in (0.229, 0.224, 0.225)]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = ""
    return q or torch.cuda.get_device_name(0)


def random_resized_crop(rng, width, height, scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3)):
    """torchvision RandomResizedCrop.get_params with a numpy generator"""
    area = width * height
    for _ in range(10):
        target = area * rng.uniform(*scale)
        aspect = math.exp(rng.uniform(math.log(ratio[0]), math.log(ratio[1])))
        w, h = int(round(math.sqrt(target * aspect))), int(round(math.sqrt(target / aspect)))
        if 0 < w <= width and 0 < h <= height:
            return int(rng.integers(0, width - w + 1)), int(rng.integers(0, height - h + 1)), w, h
    w, h = width, height     # (fallback of torchvision: the whole image at the clamped ratio; never reached at 16:9)
    return 0, 0, w, h


def timed(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    r = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), r


def main():
    torch.cuda.init()
    # ---- the pool: host stage once per distinct image, planes uploaded once; the oracle's bytes for the checks
    pool, u8s, keep = [], [], []
    for i in range(DISTINCT):
        data = jpeg_util.synth_jpeg(i, W, H, "420", 90)
        img, planes = Decoder.new_with_options(ZuneJpegOptions()).decode_coefficients(data)
        u8s.append(oracle.reconstruct(img, threads=os.cpu_count() or 4))
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b_, p in zip(bufs, planes):
            b_.upload(p)
        keep.append((planes, bufs))
        dimg = _ffi.ZjImage()
        C.memmove(C.byref(dimg), C.byref(img), C.sizeof(_ffi.ZjImage))
        for z, b_ in enumerate(bufs):
            dimg.comp[z].coeff = b_.ptr
        pool.append(dimg)
    imgs = [pool[i % DISTINCT] for i in range(N)]
    rng = np.random.default_rng(2024)
    crops = [random_resized_crop(rng, W, H) for _ in range(N)]
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    full = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    area, bil = gpu.Resize((OUT, OUT), "area"), gpu.Resize((OUT, OUT), "bilinear")
    big = torch.empty((N, 3, H, W), dtype=torch.float16, device="cuda")          # route 4's full-size tensor (12.7 GB)

    pil, pil_eval = gpu.Resize((OUT, OUT), "pil_bilinear"), gpu.Resize((OUT, OUT), "pil_bilinear", short_side=256)

    def route4(antialias=False):
        lib = _ffi.load()
        arr = (_ffi.ZjImage * N)(*imgs)
        ptrs = (C.c_void_p * N)(*[big[i].data_ptr() for i in range(N)])
        lens = (C.c_size_t * N)(*([3 * H * W * 2] * N))
        gpu._check(lib.zj_gpu_reconstruct_device_ex(0, None, arr, N, C.byref(full.c), ptrs, lens), "device_ex")
        outs = [torch.nn.functional.interpolate(big[i:i + 1, :, y:y + h, x:x + w], size=(OUT, OUT), mode="bilinear",
                                                align_corners=False, antialias=antialias) for i, (x, y, w, h) in enumerate(crops)]
        return torch.cat(outs)

    routes = {
        "1 area, whole images": lambda: gpu.reconstruct_device_resized(imgs, area, desc),
        "2 area, RandomResizedCrop": lambda: gpu.reconstruct_device_resized(imgs, area, desc, crops),
        "3 bilinear, RandomResizedCrop": lambda: gpu.reconstruct_device_resized(imgs, bil, desc, crops),
        "4 device_ex full f16 + torch crop/interpolate/stack": route4,
        "5 pil_bilinear, RandomResizedCrop": lambda: gpu.reconstruct_device_resized(imgs, pil, desc, crops),
        "6 pil_bilinear, short_side 256, whole images": lambda: gpu.reconstruct_device_resized(imgs, pil_eval, desc),
        "7 as 4, interpolate(antialias=True)": lambda: route4(True),
    }
    times = {k: [] for k in routes}
    last = {}
    for rep in range(REPS + 1):               # rep 0 warms every route up
        for k, fn in routes.items():
            ms, r = timed(fn)
            if rep:
                times[k].append(ms)
            last[k] = r
            del r
    # ---- checks (before printing): a seeded sample of slots per route against the specification on the oracle's bytes
    sample = sorted(set(np.random.default_rng(7).choice(N, 12, replace=False).tolist()) | set(range(DISTINCT)))
    spec = {"1 area, whole images": (area, None), "2 area, RandomResizedCrop": (area, crops), "3 bilinear, RandomResizedCrop": (bil, crops),
            "5 pil_bilinear, RandomResizedCrop": (pil, crops), "6 pil_bilinear, short_side 256, whole images": (pil_eval, None)}
    for k, (rz, rois) in spec.items():
        got = last[k].to_torch().cpu().numpy()
        for i in sample:
            exp = rz.expected(u8s[i % DISTINCT], W, H, 3, desc, rois[i] if rois else None)
            assert got[i].tobytes() == exp.tobytes(), f"{k}: slot {i} differs from the specification"
    got4 = last["4 device_ex full f16 + torch crop/interpolate/stack"].float().cpu().numpy()
    worst4 = 0.0
    for i in sample:
        exp = bil.expected(u8s[i % DISTINCT], W, H, 3, gpu.OutputDesc("CHW", "f32", False, 0, MEAN, INV), crops[i])
        worst4 = max(worst4, float(np.abs(got4[i] - exp).max()))
    assert worst4 < 0.02, worst4
    # route 7 against Pillow's bilinear: torch keeps floats where Pillow rounds the horizontal pass to u8 (about 1 u8 unit)
    got7 = last["7 as 4, interpolate(antialias=True)"].float().cpu().numpy()
    worst7 = 0.0
    for i in sample:
        exp = pil.expected(u8s[i % DISTINCT], W, H, 3, gpu.OutputDesc("CHW", "f32", False, 0, MEAN, INV), crops[i])
        worst7 = max(worst7, float(np.abs(got7[i] - exp).max()))
    assert worst7 < 0.05, worst7
    del last, got4, got7, big
    torch.cuda.empty_cache()

    # ---- the area kernel alone over resident u8 (more than the 126 MB L2: 32 distinct images), and a device-to-device copy
    n_src = 32
    srcs = [gpu.DeviceBuffer(W * H * 3) for _ in range(n_src)]
    for k, s_ in enumerate(srcs):
        s_.upload(u8s[k % DISTINCT])
    slots = torch.empty((N, 3, OUT, OUT), dtype=torch.float16, device="cuda")
    lib = _ffi.load()
    slot = area.slot_size(desc, 3)

    def alone():
        for i in range(N):
            gpu._check(lib.zj_gpu_resize_device(0, None, srcs[i % n_src].ptr, W, H, 3, None, C.byref(desc.c), C.byref(area.c),
                                                slots[i].data_ptr(), slot), "zj_gpu_resize_device")
    copy_src = torch.empty(n_src * W * H * 3, dtype=torch.uint8, device="cuda")
    copy_dst = torch.empty_like(copy_src)
    t_alone, t_copy = [], []
    for rep in range(REPS + 1):
        ms_a, _ = timed(alone)
        ms_c, _ = timed(lambda: copy_dst.copy_(copy_src))
        if rep:
            t_alone.append(ms_a)
            t_copy.append(ms_c)
    for i in sample:
        assert slots[i].cpu().numpy().tobytes() == area.expected(u8s[(i % n_src) % DISTINCT], W, H, 3, desc).tobytes(), i
    # kernel time of the same launches (profiler, a run of its own)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        alone()
        torch.cuda.synchronize()
    k_us = sum(e.device_time_total for e in prof.key_averages() if "resize_area_kernel" in e.key)
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        routes["1 area, whole images"]()
        torch.cuda.synchronize()
    ka = [(e.key, e.device_time_total, e.count) for e in prof.key_averages() if "resize_area_kernel" in e.key or "reconstruct" in e.key]
    # routes 5 and 6 per kernel; bytes each pass reads: the source span of the window's taps (rows x columns x 3), the intermediate
    pil_k = {}
    for name, rz, rois in (("5", pil, crops), ("6", pil_eval, None)):
        with profile(activities=[ProfilerActivity.CUDA]) as prof:
            routes[[k for k in routes if k.startswith(name)][0]]()
            torch.cuda.synchronize()
        kt = {t: sum(e.device_time_total for e in prof.key_averages() if f"pil_{t}_kernel" in e.key) for t in ("table", "horizontal", "vertical")}
        src_b = tmp_b = 0
        for i in range(N):
            cw, ch = (rois[i][2], rois[i][3]) if rois else (W, H)
            rw, rh, left, top = gpu.pil_geometry(cw, ch, OUT, OUT, rz.c.short_side)
            cx0, cx1 = gpu.pil_coefficients(cw, rw, False, left, 1)[0], gpu.pil_coefficients(cw, rw, False, left + OUT - 1, 1)[0]
            cy0, cy1 = gpu.pil_coefficients(ch, rh, False, top, 1)[0], gpu.pil_coefficients(ch, rh, False, top + OUT - 1, 1)[0]
            rows = cy1[0] + len(cy1[1]) - cy0[0]
            src_b += rows * (cx1[0] + len(cx1[1]) - cx0[0]) * 3
            tmp_b += rows * OUT * 3
        pil_k[name] = (kt, src_b, tmp_b)

    print(f"card: {card()}")
    print(f"workload: {N} x {W}x{H} 4:2:0, resident planes ({DISTINCT} distinct images) -> {N}x3x{OUT}x{OUT} f16 CHW, ImageNet mean/std")
    print(f"checks: routes 1-3, 5, 6 bit-exact vs Resize.expected on slots {sample}; route 4 within {worst4:.4f} of the bilinear spec, "
          f"route 7 within {worst7:.4f} of the pil_bilinear spec (f32)")
    for k, ts in times.items():
        med = float(np.median(ts))
        print(f"  {k:52s} median {med:8.2f} ms  (min {min(ts):.2f}, max {max(ts):.2f}; {N / med * 1e3:.0f} images/s)")
    read = N * W * H * 3
    med_a, med_c = float(np.median(t_alone)), float(np.median(t_copy))
    copy_rate = copy_src.numel() / (med_c * 1e-3)
    print(f"  area kernel alone, {N} zj_gpu_resize_device calls (one image each): median {med_a:.2f} ms = {read / (med_a * 1e-3) / 1e12:.2f} TB/s read")
    print(f"    kernel time (profiler): {k_us / 1e3:.2f} ms = {read / (k_us * 1e-6) / 1e12:.2f} TB/s read")
    print(f"  device-to-device copy of {copy_src.numel() / 1e6:.0f} MB: median {med_c:.3f} ms = {copy_rate / 1e12:.2f} TB/s copied "
          f"({2 * copy_rate / 1e12:.2f} TB/s read + written)")
    print(f"  area kernel alone / copy rate: {read / (k_us * 1e-6) / copy_rate:.2f} (kernel time), {read / (med_a * 1e-3) / copy_rate:.2f} (call time)")
    print("  route 1 kernels (profiler):")
    for key, us, cnt in ka:
        print(f"    {key[:90]:90s} {us / 1e3:8.2f} ms over {cnt} launches")
    for name, (kt, src_b, tmp_b) in pil_k.items():
        h_rate, v_rate = src_b / (kt["horizontal"] * 1e-6), tmp_b / (kt["vertical"] * 1e-6)
        print(f"  route {name} kernels (profiler): table {kt['table'] / 1e3:.3f} ms; horizontal {kt['horizontal'] / 1e3:.3f} ms reading "
              f"{src_b / 1e9:.2f} GB = {h_rate / 1e12:.2f} TB/s ({h_rate / copy_rate:.2f} of the copy rate); vertical "
              f"{kt['vertical'] / 1e3:.3f} ms reading {tmp_b / 1e9:.3f} GB = {v_rate / 1e12:.2f} TB/s ({v_rate / copy_rate:.2f})")


if __name__ == "__main__":
    main()
