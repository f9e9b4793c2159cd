#!/usr/bin/env python
"""bench.py -- headline benchmark of the pixel-reconstruction path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config c1|c2|c3_444|c3_gray|c4|c5]
                    [--dump-outputs DIR]

A "step" is one pass of the hot path (dequant + IDCT + upsample + YCbCr->RGB, reference src/worker.rs:32)
over one batch of synthetic images.  Default workload = BASELINE.json configs[1]: a batch of 256 synthetic
3840x2160 baseline 4:2:0 JPEGs -> RGB on one B200.  The JPEGs are generated in-bench (seeded smooth random
images, quality 90), entropy-decoded by the host front-end into i16 coefficient planes, and then

  value  : whole-job MP/s with the planes ALREADY RESIDENT in HBM (CUDA events on the launching stream)
  e2e    : the same metric through the C-ABI call a host program makes (zj_gpu_reconstruct) with PINNED HOST
           buffers: H2D of every plane and D2H of every pixel inside the timed region
  roofline / cpu_baseline / clocks / gpu_launches: see DESIGN.md "Measurement".

`--impl reference` times the reference's CPU implementation of the same path on the host cores.  The reference
is Rust and cannot be built in this environment, so that arm runs the oracle port (oracle/, X86 variant = what
`use_unsafe=true` executes on an AVX2 host) with all host threads, strip-parallel like scoped_threadpool.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402

CONFIGS = {
    # name: (width, height, subsampling, progressive, gray, out_cs, default batch, description)
    "c1": (1920, 1080, "444", False, False, 0, 256, "tests/golden/ref/test-baseline.jpg (the reference's test-images/test-baseline.jpg: 1920x1080 baseline, really 4:4:4) batch of 256 copies -> RGB (BASELINE configs[0])"),
    "c2": (3840, 2160, "420", False, False, 0, 256, "3840x2160 baseline 4:2:0 JPEG batch of 256 -> RGB (BASELINE configs[1])"),
    "c3_444": (4096, 4096, "444", False, False, 0, 32, "4096x4096 baseline 4:4:4 JPEG batch -> RGB (BASELINE configs[2])"),
    "c3_gray": (4096, 4096, "444", False, True, 1, 64, "4096x4096 grayscale JPEG batch -> gray (BASELINE configs[2])"),
    "c4": (1920, 1080, "422", True, False, 0, 256, "1920x1080 progressive 4:2:2 JPEG batch -> RGB (BASELINE configs[3])"),
    "c5": (8192, 8192, "420", False, False, 5, 16, "8192x8192 baseline 4:2:0 + restart markers batch -> RGBA (BASELINE configs[4])"),
}
B_PER_PX = {"c1": 9, "c2": 6, "c3_444": 9, "c3_gray": 3, "c4": 7, "c5": 7}  # SURVEY 8(d): 2 B x samples/px + out B/px


KERNEL_OF = {"c1": "zj::reconstruct_fast_kernel<MODE_NONE>", "c2": "zj::reconstruct_fast_kernel<MODE_HV>", "c3_444": "zj::reconstruct_fast_kernel<MODE_NONE>",
             "c3_gray": "zj::gray_fast_kernel", "c4": "zj::reconstruct_fast_kernel<MODE_H>", "c5": "zj::reconstruct_fast_kernel<MODE_HV>"}


def kernel_sha16() -> str:
    """hash of the sources the reconstruction kernels are built from (profiles/traffic.json is keyed by it)"""
    import hashlib
    h = hashlib.sha256()
    for f in ("zj_kernels.cu", "zj_device.h"):
        with open(os.path.join(ROOT, "zune-jpeg_b200", "csrc", f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


def metric_name() -> str:
    try:
        return json.load(open(os.path.join(ROOT, "BASELINE.json")))["metric"]
    except Exception:
        return "decoded MP/s (dequant+IDCT+upsample+YCbCr→RGB), 4K 4:2:0 batch @1/2/4/8 B200"


def host_threads() -> int:
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:
        return os.cpu_count() or 1


def physical_cores() -> int:
    """distinct physical cores among the CPUs this process may run on (SMT siblings counted once)"""
    try:
        cpus = sorted(os.sched_getaffinity(0))
        seen = set()
        for c in cpus:
            with open(f"/sys/devices/system/cpu/cpu{c}/topology/thread_siblings_list") as f:
                seen.add(f.read().strip())
        return max(1, len(seen))
    except Exception:
        return host_threads()


def cpu_threads() -> int:
    """threads of the CPU port's persistent strip pool: one per physical core (more only oversubscribes the SIMD units and
    made the baseline move by 25 % from box to box)"""
    return max(1, min(host_threads(), physical_cores()))


IMAGENET_MEAN = (123.675, 116.28, 103.53, 0.0)
IMAGENET_INV_STD = (1 / 58.395, 1 / 57.12, 1 / 57.375, 1.0)
REF_FIXTURE = os.path.join(ROOT, "tests", "golden", "ref", "test-baseline.jpg")
DUMP_BYTES = 64_000_000    # --dump-outputs writes at most this much
DUMP_SEED = 2024


def dump_outputs(out_dir: str, n_images: int, out_bytes: int, pixels) -> None:
    """--dump-outputs: the pixel buffers the timed path wrote in its last step, as DIR/pixels.npy (float32, one row per
    image of the batch).  When the whole batch does not fit in DUMP_BYTES, a row holds the bytes at k sorted positions
    drawn from a generator seeded with (DUMP_SEED, image index): the same positions for the same arguments, so that the
    files of two builds compare element for element.  pixels(b) returns image b's output bytes (uint8)."""
    k = min(out_bytes, (DUMP_BYTES - 4096) // 4 // n_images)
    rows = np.empty((n_images, k), np.float32)
    for b in range(n_images):
        px = pixels(b)
        if k < out_bytes:
            px = px[np.sort(np.random.default_rng([DUMP_SEED, b]).integers(0, out_bytes, k))]
        rows[b] = px
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pixels.npy"), rows)


def make_pool(cfg: str, n_distinct: int, rank: int):
    """n_distinct synthetic JPEGs (c1: the reference's own file) -> host stage -> (descriptor, planes) per image."""
    import jpeg_util
    from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions
    w, h, sub, prog, gray, out_cs, _, _ = CONFIGS[cfg]
    from concurrent.futures import ThreadPoolExecutor

    def one(i):
        if cfg == "c1":
            data = open(REF_FIXTURE, "rb").read()
        else:
            data = jpeg_util.synth_jpeg(1000 * rank + i, w, h, sub, 90, prog, gray, restart_rows=1 if cfg == "c5" else 0)
        d = Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(ColorSpace(out_cs)))
        img, planes = d.decode_coefficients(data)
        return img, planes, data

    with ThreadPoolExecutor(max_workers=min(n_distinct, host_threads())) as ex:
        return list(ex.map(one, range(n_distinct)))


class ClockSampler:
    """SM clock / power / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  The region of the default run
    is only tens of milliseconds long, so the clocks are polled through NVML from a thread (every ~2 ms); nvidia-smi -lms is
    the fallback when the NVML binding is unavailable."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, device: int):
        self.device, self.proc, self.path = device, None, None
        self.thread, self.stop_flag, self.samples, self.h, self.nv = None, False, [], None, None
        self.t_mark = 0.0
        try:
            import pynvml
            pynvml.nvmlInit()
            import torch
            # NVML indexes physical devices; honour CUDA_VISIBLE_DEVICES through the PCI bus id of the CUDA device
            bus = torch.cuda.get_device_properties(device).pci_bus_id if hasattr(torch.cuda.get_device_properties(device), "pci_bus_id") else None
            self.h = pynvml.nvmlDeviceGetHandleByIndex(device)
            if bus is not None:
                for i in range(pynvml.nvmlDeviceGetCount()):
                    hh = pynvml.nvmlDeviceGetHandleByIndex(i)
                    if pynvml.nvmlDeviceGetPciInfo(hh).bus == bus:
                        self.h = hh
                        break
            self.nv = pynvml
        except Exception:
            self.nv = None

    def _poll(self):
        nv, h = self.nv, self.h
        while not self.stop_flag:
            try:
                t = time.perf_counter()
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((sm, t, rs))
            except Exception:
                break
            time.sleep(0.001)

    def mark(self):
        """start of the timed region (the thread is started before the warm-up steps so that it is up to speed)"""
        self.t_mark = time.perf_counter()

    def start(self):
        if self.nv is not None:
            import threading
            self.stop_flag, self.samples = False, []
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        try:
            f = tempfile.NamedTemporaryFile("w", suffix=".csv", delete=False)
            self.path = f.name
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100", "-i", str(self.device)],
                                         stdout=f, stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self) -> dict:
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            nv = self.nv
            inside = [x for x in self.samples if x[1] >= getattr(self, "t_mark", 0.0)]
            how = "NVML polled every ~1 ms during the timed region"
            if len(inside) < 3:   # a slow NVML call can straddle a region of a few tens of ms: fall back to the warm-up steps too
                inside, how = self.samples, "NVML polled every ~1 ms during the warm-up and timed steps (same workload)"
            if inside:
                sm = [x[0] for x in inside]
                out["sm_mhz"] = float(statistics.median(sm))
                try:
                    out["sm_max_mhz"] = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
                    out["power_w_end"] = round(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0, 2)
                except Exception:
                    pass
                out["samples"] = len(sm)
                bits = 0
                for x in inside:
                    bits |= int(x[2])
                names = {"hw_slowdown": 0x8, "hw_thermal_slowdown": 0x40, "sw_thermal_slowdown": 0x20, "sw_power_cap": 0x4}
                out["reasons"] = [n for n, b in names.items() if bits & b]
                out["how"] = how
            return out
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        try:
            rows = [r.strip().split(", ") for r in open(self.path) if r.strip()]
            os.unlink(self.path)
            sm = [float(r[1]) for r in rows if len(r) >= 8]
            if sm:
                out["sm_mhz"] = statistics.median(sm)
                out["sm_max_mhz"] = float(rows[0][2])
                out["power_w_max"] = max(float(r[3]) for r in rows if len(r) >= 8)
                out["samples"] = len(sm)
                names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
                out["reasons"] = [n for k, n in enumerate(names) if any(r[4 + k].strip() == "Active" for r in rows if len(r) >= 8)]
        except Exception:
            pass
        return out


def time_cpu_port(pool, seconds: float, threads: int):
    """oracle (X86 variant) strip-parallel on `threads` host threads; returns (MP/s, n images timed)."""
    import oracle
    imgs = []
    for (img, planes, _jpeg) in pool:
        for z in range(img.n_comp):
            img.comp[z].coeff = planes[z].ctypes.data
        imgs.append(img)
    mp = sum(i.width * i.height for i in imgs) / 1e6
    oracle.reconstruct(imgs[0], threads=threads)  # warm-up (page in, thread start)
    t0 = time.perf_counter()
    n = 0
    while True:
        for im in imgs:
            oracle.reconstruct(im, threads=threads)
        n += len(imgs)
        if time.perf_counter() - t0 >= seconds:
            break
    dt = time.perf_counter() - t0
    return mp * (n / len(imgs)) / dt, n


def run_reference(args):
    """--impl reference: the CPU port of the reference path on all host threads (rank 0 only)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    cfg = args.config
    w, h = CONFIGS[cfg][0], CONFIGS[cfg][1]
    threads = cpu_threads()
    n_sample = 8 if w * h <= 3840 * 2160 else 2
    pool = make_pool(cfg, n_sample, 0)
    import oracle
    imgs = []
    for (img, planes, _jpeg) in pool:
        for z in range(img.n_comp):
            img.comp[z].coeff = planes[z].ctypes.data
        imgs.append(img)
    mp_step = sum(i.width * i.height for i in imgs) / 1e6

    def step():
        for im in imgs:
            oracle.reconstruct(im, threads=threads)

    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps - bool(args.dump_outputs)):
        step()
    if args.dump_outputs:     # the last timed step keeps its outputs (only here: holding them slows the host allocator)
        last = [oracle.reconstruct(im, threads=threads) for im in imgs]
    dt = time.perf_counter() - t0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, len(last), last[0].size, last.__getitem__)
    value = mp_step * args.steps / dt
    sample = f"{n_sample} of the workload's images per step ({n_sample}x {w}x{h}), coefficient planes in RAM -> pixels in RAM"
    line = {
        "impl": "reference", "metric": metric_name(), "value": round(value, 2), "unit": "MP/s", "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": round(1e3 * dt / args.steps, 3), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "int32", "data": "synthetic",
        "config": {"workload": CONFIGS[cfg][7], "sample": sample, "threads": threads, "host_threads": host_threads(), "physical_cores": physical_cores(),
                   "note": "reference is Rust (no rustc/cargo here): this is the C oracle port of the same path, real AVX2/SSE4.1 intrinsics, strip-parallel"},
        "cpu_baseline": {"value": round(value, 2), "unit": "MP/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": round(value, 2), "unit": "MP/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))


def run_ours(args):
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200._ffi import ZjImage
    from zune_jpeg_b200.sharding import Plumbing
    import ctypes as C

    pl = Plumbing()  # torch.distributed only when WORLD_SIZE > 1
    rank, device, world = pl.rank, pl.local_rank, pl.world
    if gpu.device_count() == 0:
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    cfg = args.config
    w, h, sub, prog, gray, out_cs, def_batch, desc = CONFIGS[cfg]
    batch = args.batch or def_batch
    # --global-batch G (BASELINE configs[4] as written: "batch of 1024 sharded across 2/4/8"): STRONG scaling -- the G images are
    # cut into contiguous ranges, one per rank (zj_partition), and a rank streams its range through its resident sub-batch of
    # `batch` images (same buffers every time: a sub-batch touches gigabytes, far more than the L2 holds)
    reps = 1
    if args.global_batch:
        from zune_jpeg_b200.sharding import partition
        mine = len(partition(args.global_batch, world, rank))
        batch = min(batch, max(mine, 1))
        if mine % batch:
            raise SystemExit(f"bench.py: --global-batch {args.global_batch} over {world} rank(s) = {mine} images, not a multiple of the sub-batch {batch}")
        reps = mine // batch
    n_distinct = min(args.distinct, batch)
    t_setup = time.perf_counter()
    pool = make_pool(cfg, n_distinct, rank)

    # ---- device-resident batch: every batch entry owns its planes and its output in HBM
    stream = gpu.Stream(device)
    plane_bytes = [sum(p.nbytes for p in planes) for (_, planes, _) in pool]
    out_bytes = gpu.output_size(pool[0][0])
    dev_planes, dev_out, images = [], [], []
    for b in range(batch):
        img, planes, _ = pool[b % n_distinct]
        bufs = []
        for p in planes:
            if p.nbytes:
                d = gpu.DeviceBuffer(p.nbytes, device)
                d.upload(p, stream.ptr)
                bufs.append(d)
            else:
                bufs.append(None)
        dev_planes.append(bufs)
        o = gpu.DeviceBuffer(out_bytes, device)
        dev_out.append(o)
        di = ZjImage()
        C.memmove(C.byref(di), C.byref(img), C.sizeof(ZjImage))
        for z in range(img.n_comp):
            di.comp[z].coeff = bufs[z].ptr if bufs[z] is not None else None
        images.append(di)
    stream.synchronize()
    plan = gpu.Batch(images, [o.ptr for o in dev_out], [out_bytes] * batch, device)
    algo_bytes = plan.algorithmic_bytes
    mp_step = batch * w * h / 1e6

    # correctness spot check inside the bench: first image against the oracle (the checker, not the product)
    check = None
    if not args.no_check:
        import oracle
        plan.run(stream.ptr)
        stream.synchronize()
        got = dev_out[0].download(stream=stream.ptr)
        img0, planes0, _ = pool[0]
        for z in range(img0.n_comp):
            img0.comp[z].coeff = planes0[z].ctypes.data
        want = oracle.reconstruct(img0, threads=host_threads())
        check = bool(np.array_equal(got, want))
        if not check:
            raise SystemExit("bench.py: GPU output differs from the oracle -- refusing to report a number")

    # ---- timed region: W warm-up steps, then exactly K steps between barriers, CUDA events on the launching stream
    sampler = ClockSampler(device)
    sampler.start()
    for _ in range(args.warmup):
        plan.run(stream.ptr)
    stream.synchronize()
    pl.barrier()
    sampler.mark()
    ev0, ev1 = gpu.Event(device), gpu.Event(device)
    launches0 = gpu.launch_count()
    ev0.record(stream.ptr)
    for _ in range(args.steps * reps):
        plan.run(stream.ptr)
    ev1.record(stream.ptr)
    stream.synchronize()
    pl.barrier()
    ms = ev0.elapsed_ms(ev1)
    launches = gpu.launch_count() - launches0
    clocks = sampler.stop()
    ms_max = pl.max(ms)
    total_mp = pl.sum(mp_step * args.steps * reps)
    value = total_mp / (ms_max / 1e3)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, batch, out_bytes, lambda b: dev_out[b].download(stream=stream.ptr))

    # ---- sustained: the same launch back to back for >= args.sustain_seconds (the 20-step region above is a burst of ~70 ms;
    # this shows what the kernel holds once power / clocks have settled), clocks sampled during it
    sustained = None
    if args.sustain_seconds > 0 and rank == 0:
        n_s = max(args.steps, int(args.sustain_seconds * 1e3 / max(ms / args.steps, 1e-3)) + 1)
        s2 = ClockSampler(device)
        s2.start()
        s2.mark()
        e0, e1 = gpu.Event(device), gpu.Event(device)
        e0.record(stream.ptr)
        for _ in range(n_s):
            plan.run(stream.ptr)
        e1.record(stream.ptr)
        stream.synchronize()
        ms_s = e0.elapsed_ms(e1)
        ck = s2.stop()
        sustained = {"value": round(mp_step * n_s / (ms_s / 1e3), 2), "unit": "MP/s", "launches": n_s, "seconds": round(ms_s / 1e3, 3),
                     "ms_per_step": round(ms_s / n_s, 4), "roofline_frac": None, "clocks": ck}

    # ---- e2e: zj_gpu_reconstruct with pinned HOST planes and pinned HOST outputs (H2D + kernels + D2H timed)
    e2e = None
    if not args.no_e2e:
        # (an image's planes in ONE pinned block, each on a 256-byte boundary -- the layout the host stage decodes into:
        # zj_gpu_reconstruct uploads planes that follow each other with a single copy)
        class _Ptr:
            def __init__(self, ptr):
                self.ptr = ptr
        pinned_planes, pinned_blocks = [], []
        for (img, planes, _jpeg) in pool:
            offs, tot = [], 0
            for p in planes:
                offs.append(tot)
                tot += (p.nbytes + 255) & ~255
            blk = gpu.PinnedBuffer(max(tot, 1))
            pinned_blocks.append(blk)
            row = []
            for p, o in zip(planes, offs):
                if p.nbytes:
                    blk.array[o:o + p.nbytes] = p.view(np.uint8)
                    row.append(_Ptr(blk.ptr + o))
                else:
                    row.append(None)
            pinned_planes.append(row)
        pinned_out = gpu.PinnedBuffer(out_bytes * batch)
        himgs = (ZjImage * batch)()
        optrs = (C.c_void_p * batch)()
        olens = (C.c_size_t * batch)()
        for b in range(batch):
            img = pool[b % n_distinct][0]
            C.memmove(C.byref(himgs[b]), C.byref(img), C.sizeof(ZjImage))
            for z in range(img.n_comp):
                pb = pinned_planes[b % n_distinct][z]
                himgs[b].comp[z].coeff = pb.ptr if pb is not None else None
            optrs[b] = pinned_out.ptr + b * out_bytes
            olens[b] = out_bytes
        from zune_jpeg_b200 import _ffi
        lib = _ffi.load()
        k_e2e = max(1, min(args.steps, args.e2e_steps))

        def e2e_step():
            rc = lib.zj_gpu_reconstruct(device, stream.ptr, himgs, batch, optrs, olens)
            if rc != 0:
                raise SystemExit(f"zj_gpu_reconstruct failed: {rc} {lib.zj_gpu_last_cuda_error().decode()}")

        e2e_step()  # warm-up (stream-ordered allocator pools, page faults)
        pl.barrier()
        t0 = time.perf_counter()
        for _ in range(k_e2e * reps):
            e2e_step()
        stream.synchronize()
        dt = time.perf_counter() - t0
        pl.barrier()
        dt_max = pl.max(dt)
        e2e_value = pl.sum(mp_step * k_e2e * reps) / dt_max
        h2d = sum(plane_bytes[b % n_distinct] for b in range(batch)) * reps
        e2e = {"value": round(e2e_value, 2), "unit": "MP/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(out_bytes * batch * reps),
               "steps": k_e2e, "ms_per_step": round(1e3 * dt_max / k_e2e, 3),
               "how": "zj_gpu_reconstruct (C ABI), pinned host coefficient planes in, pinned host pixels out, wall clock around the synchronous call"}
        if not args.no_check:
            first = np.ctypeslib.as_array((C.c_uint8 * out_bytes).from_address(pinned_out.ptr))
            if not np.array_equal(first, want):
                raise SystemExit("bench.py: e2e output differs from the oracle")

    # ---- CPU baseline beside it (rank 0, N=1 only): the oracle port on the host cores, bounded sample
    cpu, cpu_4t = None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        threads = cpu_threads()
        v, n = time_cpu_port(pool, args.cpu_seconds, threads)
        cpu = {"value": round(v, 2), "unit": "MP/s", "cores": threads, "kind": "port", "host_threads": host_threads(), "physical_cores": physical_cores(),
               "sample": f"{n} images ({n_distinct} distinct {w}x{h}, repeated for >= {args.cpu_seconds:.0f} s), planes in RAM -> pixels in RAM, oracle X86 variant, strip-parallel (persistent pool, one thread per physical core)"}
        # the reference's default (ZuneJpegOptions::num_threads = 4, /root/reference/src/options.rs:33)
        v4, n4 = time_cpu_port(pool, max(3.0, args.cpu_seconds / 3), min(4, host_threads()))
        cpu_4t = {"value": round(v4, 2), "unit": "MP/s", "cores": min(4, host_threads()), "kind": "port",
                  "sample": f"{n4} images, same path, the reference's default of 4 threads (options.rs:33)"}

    # ---- whole decode (SURVEY 8(f) "next" row, informational): JPEG bytes -> pixels through zj_decode_batch, i.e. the
    # host threads entropy-decode different images while the GPU reconstructs the finished ones; beside it the CPU-only
    # equivalent (host stage + oracle path, one image per thread).  Rank 0, N=1 only.
    decode = None
    if rank == 0 and world == 1 and not args.no_decode:
        from concurrent.futures import ThreadPoolExecutor
        from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch
        threads = host_threads()
        nd = min(batch, args.decode_images)
        jpegs = [pool[b % n_distinct][2] for b in range(nd)]
        opts = ZuneJpegOptions().set_out_colorspace(ColorSpace(out_cs))
        # (the e2e leg's pinned output buffer is big enough and idle by now: page-locking another 6 GB takes seconds)
        pinned_dec = pinned_out if (e2e is not None and pinned_out.nbytes >= out_bytes * nd) else gpu.PinnedBuffer(out_bytes * nd)
        outs = [pinned_dec.array[b * out_bytes:(b + 1) * out_bytes] for b in range(nd)]
        nw = min(nd, 3 * threads)
        decode_batch(jpegs[:nw], opts, threads=threads, out=outs[:nw])      # warm-up: the workers' two sets of pinned planes, pools
        t0 = time.perf_counter()
        res = decode_batch(jpegs, opts, threads=threads, out=outs)
        dt = time.perf_counter() - t0
        if any(not isinstance(r, int) for r in res):
            raise SystemExit(f"bench.py: zj_decode_batch failed: {[r for r in res if not isinstance(r, int)][:1]}")
        if not args.no_check and not np.array_equal(outs[0], want):
            raise SystemExit("bench.py: zj_decode_batch output differs from the oracle")
        decode = {"value": round(nd * w * h / 1e6 / dt, 2), "unit": "MP/s", "threads": threads, "images": nd,
                  "jpeg_bytes": int(sum(len(j) for j in jpegs)), "seconds": round(dt, 3),
                  "how": "zj_decode_batch: JPEG bytes in host memory -> pixels in pinned host memory (headers + Huffman on the host threads, the rest on the GPU)"}
        if not args.no_cpu:
            import oracle

            import threading
            from zune_jpeg_b200 import _ffi
            lib = _ffi.load()
            tls = threading.local()

            def cpu_one(j):
                # one decoder per worker thread (its planes are reused), descriptor points straight at them: no copies in Python
                if not hasattr(tls, "d"):
                    tls.d = Decoder.new_with_options(opts)
                img = ZjImage()
                rc = lib.zj_decoder_decode_coefficients(tls.d._h, j, len(j), C.byref(img))
                if rc != 0:
                    raise SystemExit(f"host stage failed: {rc}")
                return len(oracle.reconstruct(img, threads=1))

            nc = min(nd, 4 * threads)
            with ThreadPoolExecutor(max_workers=threads) as ex:
                list(ex.map(cpu_one, jpegs[:threads]))
                t0 = time.perf_counter()
                list(ex.map(cpu_one, jpegs[:nc]))
                dtc = time.perf_counter() - t0
            decode["cpu"] = {"value": round(nc * w * h / 1e6 / dtc, 2), "unit": "MP/s", "threads": threads, "images": nc,
                             "how": "the same host stage + the oracle port of the pixel path, one image per thread"}

    # ---- one image at a time (SURVEY 8(f).1): when the JPEG carries restart markers its intervals are entropy-decoded side
    # by side on the host threads; latency of Decoder.decode_buffer-style calls with 1 thread (the reference's loop) and all
    if decode is not None and b"\xff\xdd" in jpegs[0][:4096]:
        from zune_jpeg_b200 import _ffi
        lib = _ffi.load()
        single = {}
        one_out = pinned_dec.ptr
        for label, nt in (("sequential", 1), ("parallel", threads)):
            d1 = Decoder.new_with_options(opts.set_num_threads(nt))
            img1 = ZjImage()
            best_h, best_t, seg = 1e9, 1e9, 0
            for _ in range(4):
                t0 = time.perf_counter()
                rc = lib.zj_decoder_decode_coefficients(d1._h, jpegs[0], len(jpegs[0]), C.byref(img1))
                t1 = time.perf_counter()
                if rc == 0:
                    o1, l1 = (C.c_void_p * 1)(one_out), (C.c_size_t * 1)(out_bytes)
                    rc = lib.zj_gpu_reconstruct(device, None, C.byref(img1), 1, o1, l1)
                t2 = time.perf_counter()
                if rc != 0:
                    raise SystemExit(f"bench.py: single-image decode failed: {rc}")
                best_h, best_t, seg = min(best_h, t1 - t0), min(best_t, t2 - t0), d1.entropy_segments()
            if not args.no_check and not np.array_equal(pinned_dec.array[:out_bytes], want):
                raise SystemExit("bench.py: single-image decode differs from the oracle")
            single[label] = {"threads": nt, "intervals_side_by_side": int(seg), "host_stage_ms": round(best_h * 1e3, 2),
                             "total_ms": round(best_t * 1e3, 2), "MP/s": round(w * h / 1e6 / best_t, 1)}
        # ... and as a strip pipeline (zj_decoder_decode_into, SURVEY 8(f).2): finished strip ranges go through the GPU while the
        # host is still entropy-decoding the rest of the image
        for label, nt in (("sequential_pipelined", 1), ("parallel_pipelined", threads)):
            d1 = Decoder.new_with_options(opts.set_num_threads(nt))
            best_t, seg = 1e9, 0
            for _ in range(4):
                l0 = gpu.launch_count()
                t0 = time.perf_counter()
                d1.decode_into(jpegs[0], pinned_dec.array[:out_bytes])
                best_t, seg = min(best_t, time.perf_counter() - t0), d1.entropy_segments()
                ranges = gpu.launch_count() - l0
            if not args.no_check and not np.array_equal(pinned_dec.array[:out_bytes], want):
                raise SystemExit("bench.py: pipelined single-image decode differs from the oracle")
            single[label] = {"threads": nt, "intervals_side_by_side": int(seg), "strip_ranges": int(ranges), "total_ms": round(best_t * 1e3, 2), "MP/s": round(w * h / 1e6 / best_t, 1)}
        decode["single_image"] = single
    # ---- the entropy stage on the GPU as well (zj_decode_batch_gpu: one restart interval per GPU thread).  Needs restart markers:
    # configs without them (c2) are measured on the same images encoded with one restart interval per MCU row, and say so.
    if decode is not None and not prog:
        import jpeg_util
        has_dri = b"\xff\xdd" in jpegs[0][:4096]
        if has_dri:
            gj = jpegs
        else:
            with ThreadPoolExecutor(max_workers=min(n_distinct, threads)) as ex:
                distinct = list(ex.map(lambda i: jpeg_util.synth_jpeg(1000 * rank + i, w, h, sub, 90, prog, gray, restart_rows=1), range(n_distinct)))
            gj = [distinct[b % n_distinct] for b in range(nd)]
        note = "" if has_dri else " (the config's images re-encoded with one restart interval per MCU row)"
        ref_px = decode_batch(gj[:1], opts, threads=1)[0]     # the host stage's pixels for image 0
        stats = {}
        # (warm-up = one untimed call of the same size: the call's two staging slots are sized by the batch and kept between calls;
        # growing a slot by gigabytes inside the timed call was measured at anything from 7 to 410 ms)
        decode_batch(gj, opts, threads=threads, out=outs, gpu_entropy=True, stats=stats)
        t0 = time.perf_counter()
        res = decode_batch(gj, opts, threads=threads, out=outs, gpu_entropy=True, stats=stats)
        dtg = time.perf_counter() - t0
        if any(not isinstance(r, int) for r in res):
            raise SystemExit("bench.py: zj_decode_batch_gpu failed")
        if not args.no_check and outs[0].tobytes() != ref_px:
            raise SystemExit("bench.py: zj_decode_batch_gpu output differs from the host stage's")
        decode["gpu_entropy"] = {"value": round(nd * w * h / 1e6 / dtg, 2), "unit": "MP/s", "images": nd, "images_entropy_decoded_on_gpu": stats.get("gpu_entropy"),
                                 "seconds": round(dtg, 3), "how": "zj_decode_batch_gpu: JPEG files uploaded, restart intervals entropy-decoded one per GPU thread into device planes, reconstructed, pixels downloaded to pinned host memory" + note}
        # ... and with pinned JPEG bytes in, pixels left in device memory (zj_decode_batch_gpu_device): no pixel traffic over PCIe
        pin_in = gpu.PinnedBuffer(sum(len(j) for j in gj[:n_distinct]))
        ins, o_in = [], 0
        for j in gj[:n_distinct]:
            pin_in.array[o_in:o_in + len(j)] = np.frombuffer(j, np.uint8)
            ins.append(pin_in.array[o_in:o_in + len(j)])
            o_in += len(j)
        ins = [ins[b % len(ins)] for b in range(nd)]
        dev_targets = [(dev_out[b % len(dev_out)].ptr, out_bytes) for b in range(nd)]   # the resident batch's output buffers
        decode_batch(ins, opts, threads=threads, device_out=dev_targets, stats=stats)   # warm-up (same size, see above)
        t0 = time.perf_counter()
        res = decode_batch(ins, opts, threads=threads, device_out=dev_targets, stats=stats)
        dtd = time.perf_counter() - t0
        if any(not isinstance(r, int) for r in res):
            raise SystemExit("bench.py: zj_decode_batch_gpu_device failed")
        if not args.no_check and dev_out[0].download(stream=stream.ptr).tobytes() != ref_px:
            raise SystemExit("bench.py: zj_decode_batch_gpu_device output differs from the host stage's")
        decode["gpu_entropy_device_out"] = {"value": round(nd * w * h / 1e6 / dtd, 2), "unit": "MP/s", "images": nd, "images_entropy_decoded_on_gpu": stats.get("gpu_entropy"),
                                            "seconds": round(dtd, 3), "h2d_bytes": int(sum(len(j) for j in gj)), "d2h_bytes": 0,
                                            "how": "zj_decode_batch_gpu_device: pinned JPEG bytes in, pixels left in device memory" + note}

        # ... and handed to a device-side consumer (SURVEY 8(f).4): normalised planar f16, the tensor a model reads
        if not gray:
            desc_f16 = gpu.OutputDesc("CHW", "f16", False, 3, IMAGENET_MEAN, IMAGENET_INV_STD)
            f16_bytes = w * h * 3 * 2
            f16_out = [gpu.DeviceBuffer(f16_bytes, device) for _ in range(min(nd, 64))]
            f16_targets = [(f16_out[b % len(f16_out)].ptr, f16_bytes) for b in range(nd)]
            decode_batch(ins, opts, threads=threads, device_out=f16_targets, desc=desc_f16, stats=stats)   # warm-up (same size)
            t0 = time.perf_counter()
            res = decode_batch(ins, opts, threads=threads, device_out=f16_targets, desc=desc_f16, stats=stats)
            dtf = time.perf_counter() - t0
            if any(not isinstance(r, int) for r in res):
                raise SystemExit("bench.py: zj_decode_batch_gpu_device_ex failed")
            if not args.no_check:
                got16 = f16_out[0].download(stream=stream.ptr).view(np.float16).reshape(3, h, w)
                if got16.tobytes() != desc_f16.expected(np.frombuffer(ref_px, np.uint8), w, h, len(ref_px) // (w * h)).tobytes():
                    raise SystemExit("bench.py: zj_decode_batch_gpu_device_ex output differs from the specification applied to the host stage's pixels")
            decode["gpu_entropy_device_out_f16chw"] = {"value": round(nd * w * h / 1e6 / dtf, 2), "unit": "MP/s", "images": nd, "seconds": round(dtf, 3),
                                                       "h2d_bytes": int(sum(len(j) for j in gj)), "d2h_bytes": 0,
                                                       "how": "zj_decode_batch_gpu_device_ex: pinned JPEG bytes in, (u8 - mean) * inv_std as planar f16 left in device memory" + note}
            for b_ in f16_out:
                b_.free()

    # ---- device-side consumer on the resident batch (SURVEY 8(f).4): coefficient planes in HBM -> normalised planar f16 in HBM
    # through zj_gpu_reconstruct_device_ex (reconstruction kernel + consumer kernel per sub-batch of at most 1 GB of u8)
    consumer = None
    if rank == 0 and world == 1 and not args.no_consumer and not gray:
        from zune_jpeg_b200 import _ffi
        lib = _ffi.load()
        desc_f16 = gpu.OutputDesc("CHW", "f16", False, 3, IMAGENET_MEAN, IMAGENET_INV_STD)
        f16_bytes = w * h * 3 * 2
        nb_c = min(batch, 128)
        f16_out = [gpu.DeviceBuffer(f16_bytes, device) for _ in range(nb_c)]
        cimgs = (ZjImage * nb_c)(*images[:nb_c])
        cptrs = (C.c_void_p * nb_c)(*[o.ptr for o in f16_out])
        clens = (C.c_size_t * nb_c)(*[f16_bytes] * nb_c)

        def consumer_step():
            rc = lib.zj_gpu_reconstruct_device_ex(device, stream.ptr, cimgs, nb_c, C.byref(desc_f16.c), cptrs, clens)
            if rc != 0:
                raise SystemExit(f"zj_gpu_reconstruct_device_ex failed: {rc} {lib.zj_gpu_last_cuda_error().decode()}")

        consumer_step()
        l0 = gpu.launch_count()
        e0, e1 = gpu.Event(device), gpu.Event(device)
        k_c = max(3, min(args.steps, 10))
        e0.record(stream.ptr)
        for _ in range(k_c):
            consumer_step()
        e1.record(stream.ptr)
        stream.synchronize()
        ms_c = e0.elapsed_ms(e1) / k_c
        if not args.no_check:
            got16 = f16_out[0].download(stream=stream.ptr).view(np.float16).reshape(3, h, w)
            if got16.tobytes() != desc_f16.expected(want, w, h, len(want) // (w * h)).tobytes():
                raise SystemExit("bench.py: consumer output differs from the specification applied to the oracle's pixels")
        c_algo = algo_bytes / batch * nb_c + out_bytes * nb_c + f16_bytes * nb_c      # coefficients in + u8 out and in again + f16 out (two kernels)
        consumer = {"value": round(nb_c * w * h / 1e6 / (ms_c / 1e3), 2), "unit": "MP/s", "images": nb_c, "ms_per_step": round(ms_c, 4),
                    "launches_per_step": int((gpu.launch_count() - l0) // k_c), "algorithmic_bytes_per_step": int(c_algo),
                    "hbm_frac": round(c_algo / (ms_c / 1e3) / 1e9 / float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("hbm_gbs", 6650.0)) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else c_algo / (ms_c / 1e3) / 1e9 / 6650.0, 4),
                    "how": "zj_gpu_reconstruct_device_ex: resident coefficient planes -> (u8 - mean) * inv_std, planar f16, resident; two kernels per sub-batch of at most 1 GB of interleaved u8 (written once, read once)"}
        for b_ in f16_out:
            b_.free()

    # ---- roofline of the dominant (only) kernel: algorithmic bytes per launch / mean launch time
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    kernel_ms = ms / max(launches, 1)
    achieved = algo_bytes / (kernel_ms / 1e3) / 1e9
    # measured DRAM bytes per launch (ncu --set full: dram__bytes_read.sum + dram__bytes_write.sum) are kept per config in
    # profiles/traffic.json TOGETHER WITH the hash of the kernel sources they were captured with: a figure taken from another
    # kernel is not reported
    traffic, traffic_note = None, None
    ksha = kernel_sha16()
    try:
        ent = json.load(open(os.path.join(ROOT, "profiles", "traffic.json"))).get(cfg)
        if ent is None:
            traffic_note = "no ncu capture for this config"
        elif ent.get("kernel_sha16") == ksha:
            traffic = ent["dram_bytes_per_launch"]
            traffic_note = ent.get("source")
        else:
            traffic_note = f"stale: profiles/traffic.json holds {ent.get('dram_bytes_per_launch')} B captured with kernel sources {ent.get('kernel_sha16')}, these are {ksha}"
    except Exception as e:
        traffic_note = f"profiles/traffic.json unreadable: {e}"
    if sustained is not None:
        sustained["roofline_frac"] = round(algo_bytes / (sustained["ms_per_step"] / 1e3) / 1e9 / peak, 4)
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s", "frac": round(achieved / peak, 4),
                "traffic": traffic, "traffic_note": traffic_note, "kernel_sha16": ksha, "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s (B200_PROFILING.md)",
                "algorithmic_bytes_per_launch": int(algo_bytes), "kernel_ms": round(kernel_ms, 4),
                "kernel": KERNEL_OF[cfg] + " (one launch per step covers the whole batch)"}

    if rank == 0:
        line = {
            "metric": metric_name(), "value": round(value, 2), "unit": "MP/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": round(ms_max / args.steps, 4), "higher_is_better": True, "scaling": "strong" if args.global_batch else "weak", "vs_baseline": None,
            "dtype": "int32", "data": "synthetic",
            "config": {"workload": desc, "batch_per_gpu": batch * reps, "resident_sub_batch": batch, "global_batch": args.global_batch or batch * world, "distinct_images": n_distinct, "jpeg_quality": 90,
                       "variant": "X86 (use_unsafe=true)", "bytes_per_px": B_PER_PX[cfg],
                       "l2": f"inputs {algo_bytes / 1e9:.2f} GB per step per GPU, far larger than the 126 MB L2 (no flush needed)",
                       "parallelism": f"images sharded over {world} GPU(s), no collective"},
            "e2e": e2e, "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu, "cpu_baseline_4t": cpu_4t, "sustained": sustained, "decode": decode, "consumer": consumer, "clocks": clocks,
            "checked_vs_oracle": check, "setup_s": round(time.perf_counter() - t_setup, 1),
        }
        print(json.dumps(line))
    pl.close()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="c2", choices=list(CONFIGS))
    ap.add_argument("--batch", type=int, default=0)
    ap.add_argument("--global-batch", type=int, default=0, help="strong scaling: this many images in total, sharded over the ranks and streamed through --batch resident images per rank")
    ap.add_argument("--distinct", type=int, default=8, help="distinct synthetic JPEGs cycled through the batch")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--sustain-seconds", type=float, default=2.0, help="length of the back-to-back `sustained` leg (0 = skip)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-decode", action="store_true", help="skip the whole-decode (JPEG bytes -> pixels) measurement")
    ap.add_argument("--decode-images", type=int, default=256,
                    help="images of the whole-decode leg: one per host thread is in its (ragged) last round, so few images under-report")
    ap.add_argument("--no-consumer", action="store_true", help="skip the device-side consumer leg (planes -> normalised planar f16)")
    ap.add_argument("--no-check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the pixels of the last step to DIR/pixels.npy "
                    "(float32, one row per image; a seeded sample of each image when the batch exceeds 64 MB; rank 0 only).  "
                    "--impl reference times and dumps a smaller sample of images, so its file has another shape than the GPU path's")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    args.warmup = max(args.warmup, 0)
    import __graft_entry__
    if not os.path.exists(__graft_entry__.LIB):
        __graft_entry__.build()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
