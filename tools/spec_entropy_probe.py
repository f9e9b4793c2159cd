"""Probe: JPEG bytes -> pixels for libjpeg output with and without ZJ_USE_GPU_ENTROPY (DESIGN.md section 5.5).

256 x 3840x2160 4:2:0 files without DRI at q90, q95 and q90 with optimize=True, and the q90 set with one restart interval per
MCU row; for each, with and without the bit, alternating, medians of 5: device_out (u8 HWC in HBM) and decode_batch_resized
(pil_bicubic, short_side 256, 224^2 f16 CHW).  Every output is checked against the run without the bit before timing.  The
restart-marker set also runs through the as-written form of the interval kernel (default options).  One traced call per case
(ZJ_GPU_ENTROPY_TRACE) gives the images on the GPU route, the sync rounds (max, mean) and the turn-downs.
Prints one JSON line per case and the card's name and power limit.  Usage: python tools/spec_entropy_probe.py [--n 256]"""
import argparse
import hashlib
import re
import tempfile
import io
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import numpy as np  # noqa: E402
from PIL import Image  # noqa: E402

import jpeg_util  # noqa: E402
from zune_jpeg_b200 import gpu  # noqa: E402
from zune_jpeg_b200.decoder import ColorSpace, ZuneJpegOptions, decode_batch, decode_batch_resized  # noqa: E402


def files(n, w, h, q, optimize=False, rows=0):
    base = [jpeg_util.smooth_image(s, w, h, noise=6) for s in range(8)]
    out = []
    for k in range(n):
        bio = io.BytesIO()
        kw = dict(quality=q, optimize=optimize, subsampling=2)
        if rows:
            kw["restart_marker_rows"] = rows
        base[k % 8].save(bio, "JPEG", **kw)
        out.append(bio.getvalue())
    return out


def traced(fn):
    """run fn() with ZJ_GPU_ENTROPY_TRACE=1 and the library's stderr captured; returns the captured text"""
    os.environ["ZJ_GPU_ENTROPY_TRACE"] = "1"
    sys.stderr.flush()
    saved = os.dup(2)
    with tempfile.TemporaryFile() as f:
        os.dup2(f.fileno(), 2)
        try:
            fn()
        finally:
            os.dup2(saved, 2)
            os.close(saved)
            del os.environ["ZJ_GPU_ENTROPY_TRACE"]
        f.seek(0)
        return f.read().decode(errors="replace")


def digests(outs):
    return [hashlib.sha256(o.download().tobytes()).hexdigest() for o in outs]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--n", type=int, default=256)
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    import torch
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    W, H = 3840, 2160
    opts = {b: ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True).set_gpu_entropy(b) for b in (False, True)}
    rz = gpu.Resize((224, 224), "pil_bicubic", short_side=256)
    desc = gpu.OutputDesc("CHW", "f16", False, 0, (0.0,) * 4, (1.0,) * 4)
    for name, kw in (("q90", dict(q=90)), ("q95", dict(q=95)), ("q90_opt", dict(q=90, optimize=True)), ("q90_dri_row", dict(q=90, rows=1))):
        data = files(a.n, W, H, **kw)
        outs = [gpu.DeviceBuffer(W * H * 3) for _ in data]
        dev = [(o.ptr, o.nbytes) for o in outs]
        st = {}
        decode_batch(data, opts[False], device_out=dev)
        ref = digests(outs)
        decode_batch(data, opts[True], device_out=dev, stats=st)
        assert digests(outs) == ref, name
        r0, _ = decode_batch_resized(data, rz, desc, None, opts[False])
        r1, _ = decode_batch_resized(data, rz, desc, None, opts[True])
        assert r0.download().tobytes() == r1.download().tobytes(), name
        t = {(m, b): [] for m in ("device_out", "resized") for b in (False, True)}
        for _ in range(a.reps):
            for b in (False, True):
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                decode_batch(data, opts[b], device_out=dev)
                t[("device_out", b)].append(time.perf_counter() - t0)
                t0 = time.perf_counter()
                decode_batch_resized(data, rz, desc, None, opts[b])
                t[("resized", b)].append(time.perf_counter() - t0)
        if kw.get("rows"):   # the as-written form of the interval kernel on the same files (other pixels: as-written output)
            aw = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB)
            sa = {}
            decode_batch(data, aw, device_out=dev, stats=sa)
            ta = []
            for _ in range(a.reps):
                t0 = time.perf_counter()
                decode_batch(data, aw, device_out=dev)
                ta.append(time.perf_counter() - t0)
        log = traced(lambda: decode_batch(data, opts[True], device_out=dev))
        rounds = [tuple(map(float, m)) for m in re.findall(r"sync rounds: images \d+, max (\d+), mean ([\d.]+), turned down (\d+)", log)]
        mp = a.n * W * H / 1e9
        res = {"case": name, "images": a.n, "mb_per_file": round(statistics.mean(len(d) for d in data) / 1e6, 2), "gpu_entropy": st["gpu_entropy"]}
        if rounds:
            res["sync_rounds_max"] = max(r[0] for r in rounds)
            res["sync_rounds_mean_of_sub_batches"] = round(statistics.mean(r[1] for r in rounds), 2)
            res["sync_turned_down"] = int(sum(r[2] for r in rounds))
        if kw.get("rows"):
            res["as_written_interval_kernel_gpu_entropy"] = sa["gpu_entropy"]
            res["device_out_as_written_ms"] = round(statistics.median(ta) * 1e3, 1)
            res["device_out_as_written_gps"] = round(mp / statistics.median(ta), 2)
        for (m, b), v in t.items():
            res[f"{m}_{'bit' if b else 'host'}_ms"] = round(statistics.median(v) * 1e3, 1)
            res[f"{m}_{'bit' if b else 'host'}_gps"] = round(mp / statistics.median(v), 2)
        print(json.dumps(res), flush=True)
        del outs
    # kernel times of one call with the bit, separate run
    data = files(a.n, W, H, 90)
    outs = [gpu.DeviceBuffer(W * H * 3) for _ in data]
    dev = [(o.ptr, o.nbytes) for o in outs]
    decode_batch(data, opts[True], device_out=dev)
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        decode_batch(data, opts[True], device_out=dev)
        torch.cuda.synchronize()
    agg = {}
    for e in prof.events():
        if e.device_type.name == "CUDA":
            k = e.name.split("(")[0]
            agg.setdefault(k, [0, 0.0])
            agg[k][0] += 1
            agg[k][1] += e.device_time_total / 1e3 if hasattr(e, "device_time_total") else e.cuda_time_total / 1e3
    print(json.dumps({"kernels_ms": {k: [v[0], round(v[1], 2)] for k, v in sorted(agg.items(), key=lambda kv: -kv[1][1])[:12]}}), flush=True)


if __name__ == "__main__":
    main()
