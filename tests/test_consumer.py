"""Device-side consumers (SURVEY.md 8(f).4): zj_gpu_reconstruct_device_ex / zj_gpu_convert_device / zj_decode_batch_gpu_device_ex
must produce exactly the specified function of the reference's bytes -- the oracle's u8 output pushed through
OutputDesc.expected (numpy: (float32(u8) - mean) * inv_std, 2x2 box sums, round-to-nearest-even f16).  Bit-exact for every
type: the float path is two IEEE fp32 operations, so numpy and the kernel must agree to the last bit (tolerance 0)."""
import ctypes as C

import numpy as np
import pytest

import oracle
import util

QTS = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]
MODES = {"444": (1, 1), "422": (2, 1), "440": (1, 2), "420": (2, 2)}
MEAN, INV = (123.675, 116.28, 103.53, 7.0), (1 / 58.395, 1 / 57.12, 1 / 57.375, 0.5)


def test_expected_spec_on_cpu():
    """The numpy statement of the specification itself (no GPU): shapes, channel drop, box average, normalisation."""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(1)
    u8 = rng.integers(0, 256, size=5 * 7 * 4, dtype=np.uint8)
    d = gpu.OutputDesc("CHW", "f32", half=True, channels=3, mean=MEAN, inv_std=INV)
    e = d.expected(u8, 7, 5, 4)
    assert e.shape == (3, 2, 3) and e.dtype == np.float32
    a = u8.reshape(5, 7, 4).astype(np.float64)
    box = (a[0:2, 0:2, 1].sum()) * 0.25
    assert e[1, 0, 0] == np.float32((np.float32(box) - np.float32(MEAN[1])) * np.float32(INV[1]))
    d8 = gpu.OutputDesc("HWC", "u8", half=True)
    e8 = d8.expected(u8, 7, 5, 4)
    assert e8.shape == (2, 3, 4) and e8[0, 0, 2] == (int(a[0:2, 0:2, 2].sum()) + 2) >> 2
    assert gpu.OutputDesc().expected(u8, 7, 5, 4).tobytes() == u8.tobytes()


def test_desc_default_and_validation():
    from zune_jpeg_b200 import _ffi
    lib = _ffi.load()
    d = _ffi.ZjOutputDesc()
    lib.zj_output_desc_default(C.byref(d))
    assert lib.zj_output_desc_is_default(C.byref(d)) == 1 and list(d.inv_std) == [1.0] * 4 and list(d.mean) == [0.0] * 4
    d.dtype = 7
    planes = util.random_planes(np.random.default_rng(0), 32, 32, 3, 1, 1)
    img = util.make_image(32, 32, planes, QTS, 1, 1, 0, 0)
    assert lib.zj_consumer_output_size(C.byref(img), C.byref(d)) == 0
    d.dtype, d.layout, d.scale_log2 = _ffi.DTYPE_F16, _ffi.LAYOUT_CHW, 1
    assert lib.zj_consumer_output_size(C.byref(img), C.byref(d)) == 16 * 16 * 3 * 2


def _device_images(gpu, rng, cases):
    imgs, wants, keep = [], [], []
    for (w, h, mode, out_cs) in cases:
        hs, vs = MODES[mode]
        planes = util.random_planes(rng, w, h, 3, hs, vs)
        host = util.make_image(w, h, planes, QTS, hs, vs, out_cs, 0)
        wants.append(oracle.reconstruct(host))
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b, p in zip(bufs, planes):
            b.upload(p)
        keep.append((planes, bufs))
        imgs.append(util.make_image(w, h, planes, QTS, hs, vs, out_cs, 0, ptrs=[b.ptr for b in bufs]))
    return imgs, wants, keep


DESCS = [("CHW", "f16", False, 0), ("CHW", "f32", False, 0), ("HWC", "f32", False, 0), ("HWC", "f16", True, 0), ("CHW", "u8", False, 0),
         ("CHW", "u8", True, 0), ("HWC", "u8", True, 0), ("CHW", "f32", True, 3), ("HWC", "f16", False, 3), ("HWC", "u8", False, 0)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout,dtype,half,channels", DESCS)
def test_reconstruct_device_ex_matches_spec(layout, dtype, half, channels):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(hash((layout, dtype, half, channels)) & 0xFFFF)
    # widths that are / are not multiples of 8 and 16, odd heights, RGB / "RGBA" (4 bytes per pixel) / luma-only outputs
    cases = [(640, 96, "420", 0), (333, 131, "444", 0), (1000, 64, "422", 5), (72, 40, "440", 1), (2500, 48, "420", 0), (17, 33, "444", 5)]
    imgs, wants, keep = _device_images(gpu, rng, cases)
    desc = gpu.OutputDesc(layout, dtype, half, channels, MEAN, INV)
    before = gpu.launch_count()
    outs = gpu.reconstruct_device_ex(imgs, desc)
    assert gpu.launch_count() > before
    for (w, h, mode, out_cs), img, want, out in zip(cases, imgs, wants, outs):
        nc = len(want) // (w * h)
        exp = desc.expected(want, w, h, nc)
        got = out.download()
        assert got.shape == exp.shape == desc.shape_of(img)
        assert got.tobytes() == exp.tobytes(), f"{w}x{h} {mode} out_cs={out_cs} {layout}/{dtype}/half={half}: {np.count_nonzero(got != exp)} values differ"


@pytest.mark.gpu
def test_consumer_sub_batches():
    """More images than one sub-batch holds (ZJ_CONSUMER_CHUNK_MB): every sub-batch reuses the same scratch buffer."""
    import os
    import subprocess
    import sys
    if os.environ.get("ZJ_CONSUMER_CHUNK_MB") != "48":      # the budget is read once per process: run this test in a child
        env = dict(os.environ, ZJ_CONSUMER_CHUNK_MB="48")
        r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", __file__ + "::test_consumer_sub_batches"], env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(5)
    cases = [(1920, 1088, "420", 0)] * 12        # 6.3 MB of u8 each: 48 MB sub-batches hold 7
    imgs, wants, keep = _device_images(gpu, rng, cases[:3])
    imgs, wants = imgs * 4, wants * 4
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    before = gpu.launch_count()
    outs = gpu.reconstruct_device_ex(imgs, desc)
    assert gpu.launch_count() - before == 4      # two sub-batches x (reconstruction + consumer)
    for want, out in zip(wants, outs):
        assert out.download().tobytes() == desc.expected(want, 1920, 1088, 3).tobytes()


@pytest.mark.gpu
@pytest.mark.parametrize("entry", ["zj_gpu_reconstruct_device_ex", "zj_gpu_reconstruct_device_resized"])
def test_more_than_65535_images_of_one_format(entry):
    """65537 small images of one pixel format fit one sub-batch, but a launch takes at most 65535 (the image index is gridDim.z):
    the reconstruction and the second pass each run in two launches."""
    from zune_jpeg_b200 import _ffi, gpu
    lib = _ffi.load()
    n = 65537
    imgs, wants, keep = _device_images(gpu, np.random.default_rng(17), [(17, 33, "444", 0)])
    arr = (_ffi.ZjImage * n).from_buffer_copy(bytes(imgs[0]) * n)      # every descriptor names the same device planes
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    if entry == "zj_gpu_reconstruct_device_ex":
        exp = desc.expected(wants[0], 17, 33, 3)
        out = gpu.DeviceBuffer(exp.nbytes * n)
        ptrs = (C.c_void_p * n)(*range(out.ptr, out.ptr + exp.nbytes * n, exp.nbytes))
        lens = (C.c_size_t * n)(*[exp.nbytes] * n)
        call = lambda: lib.zj_gpu_reconstruct_device_ex(0, None, arr, n, C.byref(desc.c), ptrs, lens)
    else:
        rz = gpu.Resize((8, 16), "area")
        exp = rz.expected(wants[0], 17, 33, 3, desc)
        out = gpu.DeviceBuffer(exp.nbytes * n)
        call = lambda: lib.zj_gpu_reconstruct_device_resized(0, None, arr, n, None, C.byref(desc.c), C.byref(rz.c), out.ptr, exp.nbytes * n)
    before = gpu.launch_count()
    assert call() == 0
    assert gpu.launch_count() - before == 4      # (65535 + 2 images) x (reconstruction + second pass)
    got = out.download().reshape(n, exp.nbytes)
    bad = np.nonzero((got != np.frombuffer(exp.tobytes(), np.uint8)).any(axis=1))[0]
    assert bad.size == 0, f"{bad.size} slots differ, first {bad[:8]}"


@pytest.mark.gpu
def test_cuda_array_interface_and_dlpack():
    """The hand-off: torch reads the consumer's output in place through __cuda_array_interface__ / DLPack."""
    import torch
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(9)
    imgs, wants, keep = _device_images(gpu, rng, [(256, 64, "420", 0)])
    desc = gpu.OutputDesc("CHW", "f32", False, 0, MEAN, INV)
    out = gpu.reconstruct_device_ex(imgs, desc)[0]
    t = out.to_torch()
    assert t.is_cuda and t.dtype == torch.float32 and tuple(t.shape) == (3, 64, 256) and t.data_ptr() == out.buf.ptr
    t2 = torch.from_dlpack(out)
    assert t2.data_ptr() == out.buf.ptr
    exp = desc.expected(wants[0], 256, 64, 3)
    assert np.array_equal(t.cpu().numpy(), exp)


@pytest.mark.gpu
def test_convert_alone_and_decode_batch_ex():
    """zj_gpu_convert_device over bytes already on the device, and the JPEG-bytes front door with a consumer descriptor."""
    import jpeg_util
    from zune_jpeg_b200 import _ffi, gpu
    from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions
    rng = np.random.default_rng(3)
    u8 = rng.integers(0, 256, size=77 * 45 * 3, dtype=np.uint8)
    src = gpu.DeviceBuffer(u8.nbytes)
    src.upload(u8)
    for desc in (gpu.OutputDesc("CHW", "f16", True, 0, MEAN, INV), gpu.OutputDesc("HWC", "f32", False, 0, MEAN, INV)):
        assert gpu.convert_device(src, 77, 45, 3, desc).download().tobytes() == desc.expected(u8, 77, 45, 3).tobytes()
    # JPEG bytes -> normalised planar f16 in device memory; one image with restart markers (GPU entropy), one without (host route)
    datas = [jpeg_util.synth_jpeg(1, 640, 352, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(2, 333, 200, "444", 90)]
    sizes = [(640, 352), (333, 200)]
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    lib = _ffi.load()
    n = len(datas)
    opt = _ffi.ZjOptions()
    lib.zj_options_default(C.byref(opt))
    bufs = (C.c_void_p * n)(*[C.cast(C.c_char_p(d), C.c_void_p).value for d in datas])
    lens = (C.c_size_t * n)(*[len(d) for d in datas])
    outs = [gpu.DeviceBuffer(w * h * 3 * 2) for (w, h) in sizes]
    optrs = (C.c_void_p * n)(*[o.ptr for o in outs])
    olens = (C.c_size_t * n)(*[o.nbytes for o in outs])
    status = (C.c_int * n)()
    ngpu = C.c_size_t()
    rc = lib.zj_decode_batch_gpu_device_ex(C.byref(opt), bufs, lens, n, C.byref(desc.c), optrs, olens, status, C.byref(ngpu))
    assert rc == 0 and list(status) == [0, 0] and ngpu.value == 1
    for data, (w, h), o, ol in zip(datas, sizes, outs, olens):
        assert ol == w * h * 3 * 2
        d = Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB))
        img, planes = d.decode_coefficients(data)
        want = oracle.reconstruct(img)
        got = o.download(ol).view(np.float16).reshape(3, h, w)
        assert got.tobytes() == desc.expected(want, w, h, 3).tobytes()
