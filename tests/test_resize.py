"""Cropped, resized batch tensors (DESIGN.md section 4.5.1): zj_gpu_reconstruct_device_resized / zj_gpu_resize_device /
zj_decode_batch_gpu_device_resized must produce exactly Resize.expected -- the numpy statement of the specification -- applied to
the oracle's u8 bytes, bit for bit (tolerance 0).  On the CPU: the statement itself (half size, identity, edge cases, torch),
zj_image_rows against the oracle, and the argument checks that run before any device is touched."""
import ctypes as C
import types

import numpy as np
import pytest

import oracle
import util
from zune_jpeg_b200 import _ffi

QTS = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]
MODES = {"444": (1, 1), "422": (2, 1), "440": (1, 2), "420": (2, 2)}
MEAN, INV = (123.675, 116.28, 103.53, 7.0), (1 / 58.395, 1 / 57.12, 1 / 57.375, 0.5)
DTYPES = ("u8", "f16", "f32")


# ------------------------------------------------------------------ the specification on the CPU
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("layout", ["CHW", "HWC"])
def test_area_at_half_size_is_the_half_size_consumer(dtype, layout):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(11)
    for (w, h, nc) in [(64, 48, 3), (18, 6, 4), (2, 2, 1), (130, 34, 3)]:
        u8 = rng.integers(0, 256, size=w * h * nc, dtype=np.uint8)
        desc = gpu.OutputDesc(layout, dtype, False, 0, MEAN, INV)
        half = gpu.OutputDesc(layout, dtype, True, 0, MEAN, INV)
        got = gpu.Resize((h // 2, w // 2), "area").expected(u8, w, h, nc, desc)
        assert got.tobytes() == half.expected(u8, w, h, nc).tobytes(), (w, h, nc)


@pytest.mark.parametrize("filt", ["area", "bilinear"])
def test_identity_size_returns_the_crop(filt):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(12)
    w, h, nc = 37, 23, 3
    u8 = rng.integers(0, 256, size=w * h * nc, dtype=np.uint8)
    a = u8.reshape(h, w, nc)
    for (x, y, cw, ch) in [(0, 0, w, h), (5, 3, 20, 11), (36, 0, 1, 23), (0, 22, 37, 1)]:
        crop = np.ascontiguousarray(a[y:y + ch, x:x + cw])
        for desc in (gpu.OutputDesc(), gpu.OutputDesc("CHW", "f32", False, 0, MEAN, INV), gpu.OutputDesc("HWC", "f16", False, 0, MEAN, INV)):
            got = gpu.Resize((ch, cw), filt).expected(u8, w, h, nc, desc, (x, y, cw, ch))
            assert got.tobytes() == desc.expected(crop, cw, ch, nc).tobytes(), (filt, x, y, cw, ch)


def test_edge_cases():
    """1x1 outputs, 1-pixel-wide crops, up-scales, RGBA with the 4th byte dropped."""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(13)
    w, h = 29, 17
    u8 = rng.integers(0, 256, size=w * h * 4, dtype=np.uint8)
    a = u8.reshape(h, w, 4).astype(np.int64)
    u8d = gpu.OutputDesc()
    # 1x1 area: the rounded mean of the crop; 1x1 bilinear: the crop's centre sample pair
    s = a[2:13, 4:25, :].sum(axis=(0, 1))
    n = 11 * 21
    assert np.array_equal(gpu.Resize((1, 1), "area").expected(u8, w, h, 4, u8d, (4, 2, 21, 11)).reshape(4), (s + n // 2) // n)
    assert np.array_equal(gpu.Resize((1, 1), "bilinear").expected(u8, w, h, 4, u8d, (4, 2, 21, 11)).reshape(4), a[2 + 5, 4 + 10])
    # a 1-pixel-wide crop: every output column is the same; a 1-pixel crop fills the slot with that pixel
    for filt in ("area", "bilinear"):
        col = gpu.Resize((9, 5), filt).expected(u8, w, h, 4, u8d, (7, 0, 1, h))
        assert (col == col[:, :1]).all()
        one = gpu.Resize((3, 6), filt).expected(u8, w, h, 4, u8d, (28, 16, 1, 1))
        assert (one == a[16, 28]).all()
    # integer up-scale by area = pixel replication; channels=3 drops the 4th byte
    d3 = gpu.OutputDesc("HWC", "u8", False, 3)
    up = gpu.Resize((3 * h, 2 * w), "area").expected(u8, w, h, 4, d3)
    assert np.array_equal(up, np.repeat(np.repeat(a[:, :, :3], 3, axis=0), 2, axis=1))


@pytest.mark.parametrize("filt", ["area", "bilinear"])
def test_close_to_torch(filt):
    """Within 0.01 u8 units of torch's CPU interpolate (bilinear) / adaptive_avg_pool2d (area): same definition, other rounding."""
    import torch
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(14)
    f32 = gpu.OutputDesc("CHW", "f32")
    for (w, h, ow, oh) in [(517, 333, 300, 224), (9, 17, 224, 224), (700, 1000, 701, 999), (1, 5, 7, 3), (64, 64, 32, 32), (640, 480, 224, 224)]:
        u8 = rng.integers(0, 256, size=w * h * 3, dtype=np.uint8)
        t = torch.from_numpy(u8.reshape(h, w, 3)).permute(2, 0, 1)[None].float()
        if filt == "bilinear":
            ref = torch.nn.functional.interpolate(t, size=(oh, ow), mode="bilinear", align_corners=False, antialias=False)[0].numpy()
        else:
            ref = torch.nn.functional.adaptive_avg_pool2d(t, (oh, ow))[0].numpy()
        got = gpu.Resize((oh, ow), filt).expected(u8, w, h, 3, f32)
        assert got.shape == ref.shape and np.abs(got - ref).max() <= 0.01, (w, h, ow, oh)


# ------------------------------------------------------------------ zj_image_rows against the oracle
def _strip_geometry(lib, img, hs, vs):
    ns = C.c_uint32()
    assert lib.zj_image_strip_range(C.byref(img), 0, 0, None, None, None, C.byref(ns)) == 0
    return ns.value, 8 * hs * vs


@pytest.mark.parametrize("mode", list(MODES))
def test_image_rows_against_the_oracle(mode):
    lib = _ffi.load()
    rng = np.random.default_rng(list(MODES).index(mode))
    hs, vs = MODES[mode]
    checked = widened = 0
    for (w, h) in [(200, 203), (64, 41), (130, 69), (48, 33), (96, 100)]:
        for out_cs, variant, progressive, n_comp in [(0, 0, False, 3), (1, 1, True, 3), (5, 1, False, 3), (1, 0, False, 1)]:
            if n_comp == 1 and mode != "444":
                continue
            planes = util.random_planes(rng, w, h, n_comp, hs, vs)
            img = util.make_image(w, h, planes, QTS[:n_comp], hs, vs, out_cs, variant, progressive)
            try:
                whole = oracle.reconstruct(img)
            except RuntimeError:
                continue        # a geometry the reference panics on
            nc = len(whole) // (w * h)
            rows = whole.reshape(h, w * nc)
            ns, srows = _strip_geometry(lib, img, hs if n_comp == 3 else 1, vs if n_comp == 3 else 1)
            ranges = [(0, h), (0, 1), (h - 1, h), (srows - 1, srows + 1)]
            if ns * srows < h:
                ranges.append((ns * srows, h))                              # inside the rows the reference never writes
            ranges += [tuple(sorted(rng.choice(h + 1, 2, replace=False))) for _ in range(4)]
            for rb, re_ in ranges:
                rb, re_ = int(rb), int(re_)
                if not 0 <= rb < re_ <= h:
                    continue
                sub, row0 = util.ZjImage(), C.c_uint32()
                assert lib.zj_image_rows(C.byref(img), rb, re_, C.byref(sub), C.byref(row0)) == 0
                piece = oracle.reconstruct(sub).reshape(sub.height, w * nc)
                assert np.array_equal(piece[row0.value:row0.value + re_ - rb], rows[rb:re_]), (w, h, mode, out_cs, rb, re_)
                # no more strips than the rows need (a range inside the never-written rows takes the last strip), unless that
                # range cannot be planned as an image of its own
                touched = [k for k in range(ns) if k * srows < re_ and rb < (k + 1) * srows] or ([ns - 1] if ns else [])
                sub_ns, _ = _strip_geometry(lib, sub, hs if n_comp == 3 else 1, vs if n_comp == 3 else 1)
                if touched and sub_ns > len(touched):
                    probe = util.ZjImage()
                    rc = lib.zj_image_strip_range(C.byref(img), touched[0], touched[-1] + 1, C.byref(probe), None, None, None)
                    assert rc != 0, (w, h, mode, rb, re_, sub_ns, touched)
                    widened += 1
                checked += 1
    assert checked > 20 and widened < checked // 4


def test_image_rows_rejects_bad_ranges():
    lib = _ffi.load()
    planes = util.random_planes(np.random.default_rng(3), 64, 40, 3, 2, 2)
    img = util.make_image(64, 40, planes, QTS, 2, 2, 0, 0)
    sub, row0 = util.ZjImage(), C.c_uint32()
    for rb, re_ in [(5, 5), (6, 5), (0, 41)]:
        assert lib.zj_image_rows(C.byref(img), rb, re_, C.byref(sub), C.byref(row0)) == _ffi.ERR_INVALID_ARG
    assert lib.zj_image_rows(C.byref(img), 0, 40, None, C.byref(row0)) == _ffi.ERR_INVALID_ARG


# ------------------------------------------------------------------ argument checks (before any device is touched)
def _resize(ow, oh, filt=0):
    r = _ffi.ZjResize()
    r.out_w, r.out_h, r.filter = ow, oh, filt
    return r


def _roi(x, y, w, h):
    r = _ffi.ZjRoi()
    r.x, r.y, r.w, r.h = x, y, w, h
    return r


def test_slot_size():
    from zune_jpeg_b200 import gpu
    lib = _ffi.load()
    r = _resize(7, 5)
    for dtype, es in zip(DTYPES, (1, 2, 4)):
        for channels in (0, 3):
            d = gpu.OutputDesc("CHW", dtype, False, channels)
            for nc in (1, 3, 4):
                oc = 3 if (channels == 3 and nc == 4) else nc
                assert lib.zj_resize_slot_size(C.byref(d.c), C.byref(r), nc) == 7 * 5 * oc * es
            assert lib.zj_resize_slot_size(C.byref(d.c), C.byref(r), 2) == 0
    d = gpu.OutputDesc()
    for bad in (_resize(0, 5), _resize(7, 0), _resize(7, 5, 2), _resize(65536, 5)):
        assert lib.zj_resize_slot_size(C.byref(d.c), C.byref(bad), 3) == 0
    r.reserved = 1
    assert lib.zj_resize_slot_size(C.byref(d.c), C.byref(r), 3) == 0
    assert lib.zj_resize_slot_size(C.byref(gpu.OutputDesc(half=True).c), C.byref(_resize(7, 5)), 3) == 0
    assert lib.zj_resize_slot_size(None, C.byref(_resize(7, 5)), 3) == 0


def test_argument_validation_without_a_device():
    from zune_jpeg_b200 import gpu
    lib = _ffi.load()
    no_dev = lib.zj_gpu_device_count() == 0
    rng = np.random.default_rng(4)
    planes = util.random_planes(rng, 64, 40, 3, 2, 2)
    rgb = util.make_image(64, 40, planes, QTS, 2, 2, 0, 0)
    gray = util.make_image(64, 40, planes, QTS, 2, 2, 1, 0)
    fake = 0x100000      # never dereferenced: every call below fails before a device is touched, or runs only without one
    d, r = gpu.OutputDesc("CHW", "f16"), _resize(16, 8)
    slot = 16 * 8 * 3 * 2

    def planes_call(imgs, rois, desc=d, rz=r, out_len=None):
        arr = (_ffi.ZjImage * len(imgs))(*imgs)
        ra = (_ffi.ZjRoi * len(rois))(*rois) if rois is not None else None
        n_len = slot * len(imgs) if out_len is None else out_len
        return lib.zj_gpu_reconstruct_device_resized(0, None, arr, len(imgs), ra, C.byref(desc.c), C.byref(rz), fake, n_len)

    bad = _ffi.ERR_INVALID_ARG
    assert planes_call([rgb], [_roi(60, 0, 5, 8)]) == bad               # x + w > width
    assert planes_call([rgb], [_roi(0, 35, 8, 6)]) == bad               # y + h > height
    assert planes_call([rgb], [_roi(0, 0, 0, 8)]) == bad                # empty crop
    assert planes_call([rgb], [_roi(0, 0, 8, 0)]) == bad
    assert planes_call([rgb], None, rz=_resize(0, 8)) == bad            # empty output
    assert planes_call([rgb], None, rz=_resize(16, 8, 7)) == bad        # unknown filter
    assert planes_call([rgb], None, desc=gpu.OutputDesc("CHW", "f16", True)) == bad   # scale_log2 != 0
    assert planes_call([rgb, gray], None) == bad                        # two channel counts in one tensor
    assert planes_call([rgb, rgb], None, out_len=2 * slot - 1) == _ffi.ERR_SHORT_OUTPUT
    if no_dev:
        assert planes_call([rgb, rgb], [_roi(3, 5, 40, 30), _roi(63, 39, 1, 1)]) == _ffi.ERR_NO_DEVICE

    def alone(w, h, nc, roi, desc=d, rz=r, dst_len=slot):
        return lib.zj_gpu_resize_device(0, None, fake, w, h, nc, C.byref(roi) if roi is not None else None, C.byref(desc.c), C.byref(rz), fake, dst_len)

    assert alone(64, 40, 3, _roi(1, 1, 64, 1)) == bad
    assert alone(64, 40, 2, None) == bad
    assert alone(0, 40, 3, None) == bad
    assert alone(65536, 1, 1, None) == bad
    assert alone(64, 40, 3, None, rz=_resize(16, 8, 2)) == bad
    assert alone(64, 40, 3, None, dst_len=slot - 1) == _ffi.ERR_SHORT_OUTPUT
    if no_dev:
        assert alone(64, 40, 3, _roi(7, 3, 9, 9)) == _ffi.ERR_NO_DEVICE

    # the JPEG-bytes front door: descriptor and size checks come before the device
    data = b"\xff\xd8\xff\xd9"
    bufs = (C.c_void_p * 1)(C.cast(C.c_char_p(data), C.c_void_p).value)
    lens = (C.c_size_t * 1)(len(data))
    status = (C.c_int * 1)()
    opt = _ffi.ZjOptions()
    lib.zj_options_default(C.byref(opt))

    def front(desc=d, rz=r, out_len=slot):
        return lib.zj_decode_batch_gpu_device_resized(C.byref(opt), bufs, lens, 1, None, C.byref(desc.c), C.byref(rz), fake, out_len, status, None)

    assert front(rz=_resize(16, 0)) == bad
    assert front(desc=gpu.OutputDesc("HWC", "u8", True)) == bad
    assert front(out_len=slot - 1) == _ffi.ERR_SHORT_OUTPUT
    if no_dev:
        assert front() == _ffi.ERR_NO_DEVICE


# ------------------------------------------------------------------ on the GPU: bit-exact against the specification
_ORACLE_CACHE = {}


def _device_images(gpu, cases):
    """cases: (w, h, mode, out_cs, seed) -> device images, the oracle's bytes, buffers to keep alive"""
    imgs, wants, keep = [], [], []
    for (w, h, mode, out_cs, seed) in cases:
        hs, vs = MODES[mode]
        planes = util.random_planes(np.random.default_rng(seed), w, h, 3, hs, vs)
        host = util.make_image(w, h, planes, QTS, hs, vs, out_cs, 0)
        key = (w, h, mode, out_cs, seed)
        if key not in _ORACLE_CACHE:
            _ORACLE_CACHE[key] = oracle.reconstruct(host)
        wants.append(_ORACLE_CACHE[key])
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b, p in zip(bufs, planes):
            b.upload(p)
        keep.append((planes, bufs))
        imgs.append(util.make_image(w, h, planes, QTS, hs, vs, out_cs, 0, ptrs=[b.ptr for b in bufs]))
    return imgs, wants, keep


def _crops(lib, img, w, h, mode):
    """whole image, interior, touching each edge, 1x1, across strip boundaries, inside the never-written rows"""
    hs, vs = MODES[mode]
    ns, srows = _strip_geometry(lib, img, hs, vs)
    out = [None, (w // 4, h // 4, w // 2, max(h // 3, 1)), (0, h // 3, w // 3 + 1, h // 3 + 1), (w - w // 3, 0, w // 3, h // 2 + 1),
           (w // 5, h - h // 4, w // 2, h // 4), (w - 1, h - 1, 1, 1), (1, min(srows - 3, h - 7) if h > 7 else 0, w - 2, min(7, h))]
    if ns * srows < h:
        out.append((3, ns * srows, w - 5, h - ns * srows))
    return out


# widths that are / are not multiples of 8 and 16, odd heights, the Q1 tail (420 203 rows, 422 69 rows), RGB / RGBA / gray
GEOMS = [(640, 96, "420", 0), (333, 131, "444", 0), (1000, 64, "422", 5), (72, 40, "440", 1), (200, 203, "420", 0), (520, 69, "422", 5),
         (17, 33, "444", 5), (136, 69, "422", 1)]
SIZES = [(24, 40), (150, 90), (7, 31)]      # (OH, OW): down, up, non-uniform aspect


@pytest.mark.gpu
@pytest.mark.parametrize("channels", [0, 3])
@pytest.mark.parametrize("layout", ["CHW", "HWC"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("filt", ["area", "bilinear"])
def test_reconstruct_device_resized_matches_spec(filt, dtype, layout, channels):
    from zune_jpeg_b200 import gpu
    lib = _ffi.load()
    desc = gpu.OutputDesc(layout, dtype, False, channels, MEAN, INV)
    oc_of = lambda out_cs: {0: 3, 1: 1}.get(out_cs, 3 if channels == 3 else 4)
    for oc in sorted({oc_of(g[3]) for g in GEOMS}):
        geoms = [g for g in GEOMS if oc_of(g[3]) == oc]
        imgs, wants, keep = _device_images(gpu, [(*g, 100 + k) for k, g in enumerate(geoms)])
        batch, expect_args = [], []
        for (w, h, mode, out_cs), img, want in zip(geoms, imgs, wants):
            for roi in _crops(lib, img, w, h, mode):
                batch.append((img, roi))
                expect_args.append((want, w, h, len(want) // (w * h), roi))
        for size in SIZES:
            rz = gpu.Resize(size, filt)
            out = gpu.reconstruct_device_resized([b[0] for b in batch], rz, desc, [b[1] for b in batch])
            got = out.download()
            assert got.shape == (len(batch), *rz.slot_shape(desc, expect_args[0][3]))
            for k, (want, w, h, nc, roi) in enumerate(expect_args):
                exp = rz.expected(want, w, h, nc, desc, roi)
                assert got[k].tobytes() == exp.tobytes(), f"{w}x{h} nc={nc} roi={roi} size={size}: {np.count_nonzero(got[k] != exp)} differ"


@pytest.mark.gpu
@pytest.mark.parametrize("filt", ["area", "bilinear"])
def test_resize_alone_unaligned_crops(filt):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(21)
    for (w, h, nc, channels, offset) in [(77, 45, 3, 0, 0), (77, 45, 3, 0, 1), (131, 29, 4, 3, 2), (95, 61, 1, 0, 3), (64, 64, 4, 0, 0)]:
        # the pixels start `offset` bytes into the allocation: an unaligned source of exactly w * h * nc bytes
        u8 = rng.integers(0, 256, size=w * h * nc, dtype=np.uint8)
        buf = gpu.DeviceBuffer(u8.nbytes + offset)
        buf.upload(u8, offset=offset)
        src = types.SimpleNamespace(ptr=buf.ptr + offset)
        for roi in [None, (1, 3, w - 2, h - 5), (3, 0, 5, h), (w - 7, h - 2, 7, 2), (5, 7, 1, 1)]:
            for dtype, layout, size in [("u8", "HWC", (13, 21)), ("f16", "CHW", (40, 150)), ("f32", "HWC", (1, 1)), ("u8", "CHW", (h, w))]:
                desc = gpu.OutputDesc(layout, dtype, False, channels, MEAN, INV)
                rz = gpu.Resize(size, filt)
                got = gpu.resize_device(src, w, h, nc, rz, desc, roi).download()
                exp = rz.expected(u8, w, h, nc, desc, roi)
                assert got.tobytes() == exp.tobytes(), (w, h, nc, roi, dtype, layout, size)


@pytest.mark.gpu
def test_resized_sub_batches():
    """More images than one sub-batch holds (ZJ_CONSUMER_CHUNK_MB): every sub-batch reuses the same scratch buffer."""
    import os
    import subprocess
    import sys
    if os.environ.get("ZJ_CONSUMER_CHUNK_MB") != "48":      # the budget is read once per process: run this test in a child
        env = dict(os.environ, ZJ_CONSUMER_CHUNK_MB="48")
        r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", __file__ + "::test_resized_sub_batches"], env=env,
                           capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return
    from zune_jpeg_b200 import gpu
    imgs, wants, keep = _device_images(gpu, [(1920, 1088, "420", 0, 5 + k) for k in range(3)])
    imgs, wants = imgs * 4, wants * 4        # 6.3 MB of u8 each: 48 MB sub-batches hold 7
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    rz = gpu.Resize((224, 224), "area")
    before = gpu.launch_count()
    got = gpu.reconstruct_device_resized(imgs, rz, desc).download()
    assert gpu.launch_count() - before == 4      # two sub-batches x (reconstruction + resize)
    for k, want in enumerate(wants):
        assert got[k].tobytes() == rz.expected(want, 1920, 1088, 3, desc).tobytes()
    # crops: only their strips are reconstructed, so more images fit a sub-batch
    rois = [(k * 70, 37 * k, 1000, 300) for k in range(12)]
    got = gpu.reconstruct_device_resized(imgs, rz, desc, rois).download()
    for k, want in enumerate(wants):
        assert got[k].tobytes() == rz.expected(want, 1920, 1088, 3, desc, rois[k]).tobytes()


@pytest.mark.gpu
def test_decode_batch_resized_front_door():
    """JPEG bytes -> one batch tensor: restart-marker (GPU entropy) and plain files, a damaged file, a crop that does not fit.
    Statuses and errors are decode_batch's; good slots are the specification applied to the host stage's bytes; failed slots
    are not written."""
    import jpeg_util
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import ColorSpace, DecodeErrors, Decoder, ZuneJpegOptions, decode_batch, decode_batch_resized
    datas = [jpeg_util.synth_jpeg(1, 640, 352, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(2, 333, 200, "444", 90),
             jpeg_util.synth_jpeg(3, 500, 301, "422", 85, restart_rows=2), None, jpeg_util.synth_jpeg(4, 256, 128, "420", 90),
             bytes([0xff, 0xd8, 0xa4])]                                                     # a header error
    cut = bytearray(datas[0]); del cut[len(cut) // 2:]
    datas[3] = bytes(cut)                                                                   # truncated entropy data
    rois = [(10, 20, 300, 200), None, (0, 0, 500, 301), None, (200, 0, 100, 128), None]      # [4] does not fit (200 + 100 > 256)
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB)
    want = decode_batch(datas, opts, threads=4)
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    for filt in ("area", "bilinear"):
        rz = gpu.Resize((96, 128), filt)
        # run once into a sentinel-filled tensor: allocate, fill, decode into the same buffer through the C ABI
        out, errs = decode_batch_resized(datas, rz, desc, rois, opts, threads=4)
        out.buf.memset(0xAB)
        lib = _ffi.load()
        n = len(datas)
        raw = opts._raw()
        raw.num_threads = 4
        bufs = (C.c_void_p * n)(*[C.cast(C.c_char_p(d), C.c_void_p).value for d in datas])
        lens = (C.c_size_t * n)(*[len(d) for d in datas])
        sizes = [(640, 352), (333, 200), (500, 301), (640, 352), (256, 128), (1, 1)]
        status = (C.c_int * n)()
        slot = rz.slot_size(desc, 3)
        rc = lib.zj_decode_batch_gpu_device_resized(C.byref(raw), bufs, lens, n, gpu._roi_array(rois, sizes), C.byref(desc.c), C.byref(rz.c),
                                                    out.buf.ptr, slot * n, status, None)
        assert rc == sum(1 for st in status if st != 0) and status[4] != 0 and status[5] != 0
        got = out.download()
        for k, (data, w_, e) in enumerate(zip(datas, want, errs)):
            if k == 4:      # decoded, but its crop does not fit
                assert isinstance(w_, bytes) and isinstance(e, DecodeErrors) and e.status == _ffi.ERR_INVALID_ARG and status[k] == _ffi.ERR_INVALID_ARG
            elif isinstance(w_, DecodeErrors):
                assert isinstance(e, DecodeErrors) and e.status == w_.status == status[k] and str(e) == str(w_) and e.kind == w_.kind
            else:
                assert e is None and status[k] == 0
            if status[k] != 0:
                assert (got[k].view(np.uint8) == 0xAB).all(), k
                continue
            d = Decoder.new_with_options(opts)
            img, planes = d.decode_coefficients(data)
            host = oracle.reconstruct(img)
            assert got[k].tobytes() == rz.expected(host, img.width, img.height, 3, desc, rois[k]).tobytes(), (filt, k)


@pytest.mark.gpu
def test_torch_hand_off():
    import torch
    from zune_jpeg_b200 import gpu
    imgs, wants, keep = _device_images(gpu, [(256, 64, "420", 0, 9), (200, 203, "420", 0, 10)])
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    rz = gpu.Resize((32, 48), "bilinear")
    out = gpu.reconstruct_device_resized(imgs, rz, desc, [(5, 6, 100, 50), None])
    t = out.to_torch()
    assert t.is_cuda and t.dtype == torch.float16 and tuple(t.shape) == (2, 3, 32, 48) and t.data_ptr() == out.buf.ptr
    assert t[1].cpu().numpy().tobytes() == rz.expected(wants[1], 200, 203, 3, desc).tobytes()
