"""Probe: progressive JPEG bytes -> pixels for libjpeg output with and without ZJ_USE_GPU_PROGRESSIVE (DESIGN.md section 5.6).

3840x2160 4:2:0 progressive files at q90, q95 and q90 with optimize=True, in batches of 256, 16 and 1 images.  For each case,
the host route (ZJ_USE_GPU_ENTROPY alone: progressive files take the host stage) and the bit, alternating, medians of --reps:
device_out (u8 HWC in HBM) and decode_batch_resized (pil_bicubic, short_side 256, 224^2 f16 CHW).  Every output of the bit's run
is checked against the host route's before timing.  One traced call per case (ZJ_GPU_ENTROPY_TRACE) gives the first scans' sync
rounds (max, mean), the turn-downs and the time of each phase.  Prints the card's name and power limit, then one JSON line per
case.  Usage: python tools/progressive_entropy_probe.py [--reps 5] [--sizes 256,16,1]"""
import argparse
import hashlib
import io
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

import jpeg_util  # noqa: E402
from zune_jpeg_b200 import gpu  # noqa: E402
from zune_jpeg_b200.decoder import ColorSpace, ZuneJpegOptions, decode_batch, decode_batch_resized  # noqa: E402


def files(n, w, h, q, optimize=False):
    out = []
    for s in range(min(n, 8)):
        bio = io.BytesIO()
        jpeg_util.smooth_image(s, w, h, noise=6).save(bio, "JPEG", quality=q, optimize=optimize, subsampling=2, progressive=True)
        out.append(bio.getvalue())
    return [out[k % len(out)] for k in range(n)]


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
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="256,16,1")
    a = ap.parse_args()
    import torch
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    W, H = 3840, 2160
    host = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True).set_gpu_entropy(True)
    opts = {False: host, True: host.set_gpu_progressive(True)}
    rz = gpu.Resize((224, 224), "pil_bicubic", short_side=256)
    desc = gpu.OutputDesc("CHW", "f16", False, 0, (0.0,) * 4, (1.0,) * 4)
    for n in (int(s) for s in a.sizes.split(",")):
        for name, kw in (("q90", dict(q=90)), ("q95", dict(q=95)), ("q90_opt", dict(q=90, optimize=True))):
            data = files(n, W, H, **kw)
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
            log = traced(lambda: decode_batch(data, opts[True], device_out=dev))
            prog = [m for m in re.findall(r"prog: images (\d+), scans (\d+), first-scan rounds max (\d+), mean ([\d.]+), turned down:(.*)", log)]
            phases = {}
            for what, ms in re.findall(r"\] (prog [A-Za-z ]+?|files \+ interval kernels|headers \+ marker scan|memset planes|status \+ reconstruct \(\+ d2h\))\s+([\d.]+) ms", log):
                phases[what] = round(phases.get(what, 0.0) + float(ms), 2)
            mp = n * W * H / 1e9
            res = {"case": name, "images": n, "mb_per_file": round(sum(len(d) for d in data) / n / 1e6, 2), "gpu_entropy": st["gpu_entropy"],
                   "rounds_max": max((int(p[2]) for p in prog), default=None),
                   "rounds_mean_of_sub_batches": round(statistics.mean(float(p[3]) for p in prog), 2) if prog else None,
                   "turned_down": " ".join(p[4].strip() for p in prog), "trace_ms": phases}
            for (m, b), v in t.items():
                res[f"{m}_{'bit' if b else 'host'}_ms"] = round(statistics.median(v) * 1e3, 1)
                res[f"{m}_{'bit' if b else 'host'}_gps"] = round(mp / statistics.median(v), 3)
            print(json.dumps(res), flush=True)
            del outs


if __name__ == "__main__":
    main()
