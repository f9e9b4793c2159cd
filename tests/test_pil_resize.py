"""Pillow-exact resizing into the batch tensors (ZJ_FILTER_PIL_BILINEAR / _BICUBIC, DESIGN.md section 4.5.2).  On the CPU:
Resize.expected -- the numpy statement of the header's rules -- equals Pillow's Image.resize and torchvision's PIL-backend
resized_crop / Resize + CenterCrop byte for byte; the argument checks; the rows the planes route reconstructs.  On the GPU:
every entry point equals Resize.expected bit for bit, and JPEG bytes in libjpeg output mode give torchvision's own bytes."""
import ctypes as C
import io
import types

import numpy as np
import pytest
from PIL import Image

import jpeg_util
import oracle
import ref_files
import util
from zune_jpeg_b200 import _ffi

QTS = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]
MODES = {"444": (1, 1), "422": (2, 1), "440": (1, 2), "420": (2, 2)}
MEAN, INV = (123.675, 116.28, 103.53, 7.0), (1 / 58.395, 1 / 57.12, 1 / 57.375, 0.5)
DTYPES = ("u8", "f16", "f32")
FILTERS = ("pil_bilinear", "pil_bicubic")
PIL = {"pil_bilinear": Image.BILINEAR, "pil_bicubic": Image.BICUBIC}
MODE_OF = {1: "L", 3: "RGB", 4: "RGBX"}


def _pillow_resize(a, roi, size, filt):
    """Pillow itself: a = h x w x nc u8, roi = (x, y, w, h) or None, size = (OH, OW)"""
    h, w, nc = a.shape
    x, y, cw, ch = roi if roi is not None else (0, 0, w, h)
    im = Image.fromarray(a[:, :, 0] if nc == 1 else a, MODE_OF[nc])
    out = np.asarray(im.crop((x, y, x + cw, y + ch)).resize((size[1], size[0]), PIL[filt]))
    return out.reshape(size[0], size[1], nc)


def _structured(rng, w, h, nc):
    """random bytes over a gradient: edges and flat areas, so that negative bicubic lobes clip at both ends"""
    base = rng.integers(0, 256, (h, w, nc), dtype=np.uint8) // 2
    return (base + np.linspace(0, 127, w, dtype=np.uint8)[None, :, None]).astype(np.uint8)


# ------------------------------------------------------------------ the statement against Pillow and torchvision
@pytest.mark.parametrize("filt", FILTERS)
@pytest.mark.parametrize("nc", [1, 3, 4])
def test_expected_equals_pillow(filt, nc):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(100 + nc)
    cases = []
    for _ in range(12):                                                   # random crops and sizes, up and down
        w, h = (int(v) for v in rng.integers(2, 400, 2))
        x, y = int(rng.integers(0, w)), int(rng.integers(0, h))
        cw, ch = int(rng.integers(1, w - x + 1)), int(rng.integers(1, h - y + 1))
        cases.append((w, h, (x, y, cw, ch), (int(rng.integers(1, 300)), int(rng.integers(1, 300)))))
    cases += [(37, 23, (0, 0, 37, 23), (23, 37)),                         # identity
              (37, 23, None, (1, 1)), (37, 23, (36, 22, 1, 1), (5, 7)), (37, 23, (5, 0, 1, 23), (9, 4)),   # 1x1 out, 1-pixel crops
              (37, 23, (0, 0, 10, 23), (40, 3)), (37, 23, (27, 13, 10, 10), (10, 31)),                    # crops at every edge
              (1200, 7, None, (3, 2)), (12, 1100, (0, 3, 12, 1097), (1, 2)), (640, 480, None, (1000, 700))]  # > 500x down, up
    # (Pillow resizes a crop more than 100 times taller than wide vertically first: the statement does not follow it there)
    for (w, h, roi, size) in cases:
        a = _structured(rng, w, h, nc)
        for desc in (gpu.OutputDesc(), gpu.OutputDesc("CHW", "f32", False, 0, MEAN, INV)):
            got = gpu.Resize(size, filt).expected(a.reshape(-1), w, h, nc, desc, roi)
            want = _pillow_resize(a, roi, size, filt)
            if desc.c.dtype != _ffi.DTYPE_U8:                         # floats are the consumer rule of Pillow's bytes
                want = desc.expected(want.reshape(-1), size[1], size[0], nc).reshape(got.shape)
            assert got.tobytes() == want.tobytes(), (filt, nc, w, h, roi, size)


# portrait, landscape, square; (RH - 224) / 2 and (RW - 224) / 2 landing on x.5 (round half to even) and on integers
SHORT = [(300, 451, (224, 224), 256), (451, 300, (224, 224), 256), (300, 300, (224, 224), 256), (257, 513, (224, 224), 256),
         (513, 257, (224, 224), 256), (640, 427, (224, 224), 256), (97, 1000, (100, 40), 41), (333, 333, (5, 5), 10)]


@pytest.mark.parametrize("filt", FILTERS)
def test_short_side_equals_pillow_and_torchvision(filt):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(7)
    try:
        import torchvision  # noqa: F401
        from torchvision.transforms import InterpolationMode, v2
    except Exception:
        v2 = None
    halves = set()
    for (w, h, size, s) in SHORT:
        a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        rz = gpu.Resize(size, filt, short_side=s)
        got = rz.expected(a.reshape(-1), w, h, 3)
        rw, rh, left, top = gpu.pil_geometry(w, h, size[1], size[0], s)
        halves.add(((rw - size[1]) % 2, (rh - size[0]) % 2))
        im = Image.fromarray(a)
        want = np.asarray(im.resize((rw, rh), PIL[filt]).crop((left, top, left + size[1], top + size[0])))
        assert got.tobytes() == want.tobytes(), (w, h, size, s)
        if v2 is not None:
            mode = InterpolationMode.BILINEAR if filt == "pil_bilinear" else InterpolationMode.BICUBIC
            tv = np.asarray(v2.Compose([v2.Resize(s, interpolation=mode), v2.CenterCrop(size)])(im))
            assert got.tobytes() == tv.tobytes(), (w, h, size, s)
    assert (1, 1) in halves and (0, 0) in halves


@pytest.mark.parametrize("filt", FILTERS)
def test_resized_crop_equals_torchvision(filt):
    from zune_jpeg_b200 import gpu
    v2 = pytest.importorskip("torchvision.transforms.v2")
    from torchvision.transforms import InterpolationMode
    mode = InterpolationMode.BILINEAR if filt == "pil_bilinear" else InterpolationMode.BICUBIC
    rng = np.random.default_rng(8)
    for _ in range(8):
        w, h = (int(v) for v in rng.integers(230, 900, 2))
        a = rng.integers(0, 256, (h, w, 3), dtype=np.uint8)
        y, x = int(rng.integers(0, h // 2)), int(rng.integers(0, w // 2))
        ch, cw = int(rng.integers(1, h - y)), int(rng.integers(1, w - x))
        want = np.asarray(v2.functional.resized_crop(Image.fromarray(a), y, x, ch, cw, [224, 224], interpolation=mode))
        got = gpu.Resize((224, 224), filt).expected(a.reshape(-1), w, h, 3, roi=(x, y, cw, ch))
        assert got.tobytes() == want.tobytes(), (w, h, x, y, cw, ch)


# ------------------------------------------------------------------ argument checks (before any device is touched)
def _resize(ow, oh, filt, short_side=0):
    r = _ffi.ZjResize()
    r.out_w, r.out_h, r.filter, r.short_side = ow, oh, filt, short_side
    return r


def test_filter_values_and_slot_size():
    from zune_jpeg_b200 import gpu
    lib = _ffi.load()
    for filt in (18, 19):
        for short_side in (0, 256):
            for dtype, es in zip(DTYPES, (1, 2, 4)):
                for channels in (0, 3):
                    d = gpu.OutputDesc("CHW", dtype, False, channels)
                    for nc in (1, 3, 4):
                        oc = 3 if (channels == 3 and nc == 4) else nc
                        assert lib.zj_resize_slot_size(C.byref(d.c), C.byref(_resize(7, 5, filt, short_side)), nc) == 7 * 5 * oc * es
    d = gpu.OutputDesc()
    for filt in (2, 7, 16, 17, 20, 21):                                  # Pillow's NEAREST, LANCZOS, BOX, HAMMING are not offered
        assert lib.zj_resize_slot_size(C.byref(d.c), C.byref(_resize(7, 5, filt)), 3) == 0, filt
    for filt in (_ffi.FILTER_AREA, _ffi.FILTER_BILINEAR):                # short_side belongs to the PIL filters
        assert lib.zj_resize_slot_size(C.byref(d.c), C.byref(_resize(7, 5, filt, 256)), 3) == 0
    assert C.sizeof(_ffi.ZjResize) == 16
    with pytest.raises(ValueError):
        gpu.Resize((224, 224), "area", short_side=256)


def test_resized_size_checks_without_a_device():
    from zune_jpeg_b200 import gpu
    lib = _ffi.load()
    no_dev = lib.zj_gpu_device_count() == 0
    planes = util.random_planes(np.random.default_rng(4), 64, 40, 3, 2, 2)
    img = util.make_image(64, 40, planes, QTS, 2, 2, 0, 0)
    fake = 0x100000      # never dereferenced
    d = gpu.OutputDesc("CHW", "f16")
    bad = _ffi.ERR_INVALID_ARG

    def planes_call(rz, roi=None):
        arr = (_ffi.ZjImage * 1)(img)
        ra = (_ffi.ZjRoi * 1)(_ffi.ZjRoi(*roi)) if roi else None
        return lib.zj_gpu_reconstruct_device_resized(0, None, arr, 1, ra, C.byref(d.c), C.byref(rz), fake, 1 << 20)

    def alone(rz, w=64, h=40):
        return lib.zj_gpu_resize_device(0, None, fake, w, h, 3, None, C.byref(d.c), C.byref(rz), fake, 1 << 20)

    for filt in (18, 19):
        assert planes_call(_resize(32, 32, filt, 31)) == bad               # 64x40 -> 51x31: narrower than the window
        assert planes_call(_resize(40, 32, filt, 32), (0, 0, 20, 40)) == bad   # the crop's resized size (32 x 64), not the image's
        assert planes_call(_resize(1, 1, filt, 65536)) == bad              # resized size over 65535
        assert planes_call(_resize(1, 1, filt, 2000), (0, 0, 64, 1)) == bad   # 64 x 1 -> RW = 128000: over 65535
        assert alone(_resize(52, 32, filt, 32)) == bad                     # 64x40 -> 51x32
        assert alone(_resize(1, 1, filt, 2000), 65535, 40) == bad          # RW = int(2000 * 65535 / 40) > 65535
        if no_dev:
            assert planes_call(_resize(51, 32, filt, 32)) == _ffi.ERR_NO_DEVICE
            assert planes_call(_resize(8, 8, filt), (3, 5, 1, 1)) == _ffi.ERR_NO_DEVICE
            assert alone(_resize(51, 32, filt, 32)) == _ffi.ERR_NO_DEVICE


def _strip_geometry(lib, img, hs, vs):
    ns = C.c_uint32()
    assert lib.zj_image_strip_range(C.byref(img), 0, 0, None, None, None, C.byref(ns)) == 0
    return ns.value, 8 * hs * vs


@pytest.mark.parametrize("mode", list(MODES))
def test_window_rows_against_the_oracle(mode):
    """The planes route reconstructs zj_image_rows(crop.y + y0, crop.y + y1): the rows the window's vertical taps read.  The
    resize of those rows alone equals the resize of the whole image, and for the evaluation preset they are fewer than the crop's."""
    from zune_jpeg_b200 import gpu
    lib = _ffi.load()
    rng = np.random.default_rng(40 + list(MODES).index(mode))
    hs, vs = MODES[mode]
    fewer = 0
    for (w, h) in [(200, 203), (130, 69), (96, 300)]:
        planes = util.random_planes(rng, w, h, 3, hs, vs)
        img = util.make_image(w, h, planes, QTS, hs, vs, 0, 0)
        whole = oracle.reconstruct(img)
        for filt in FILTERS:
            for (roi, size, s) in [(None, (24, 24), 32), ((3, 7, w - 10, h - 20), (9, 16), 0), ((0, h // 2, w // 2, h - h // 2), (5, 5), 6),
                                   ((w - 1, h - 1, 1, 1), (3, 3), 0), (None, (h, w), 0)]:
                x, y, cw, ch = roi if roi else (0, 0, w, h)
                rz = gpu.Resize(size, filt, short_side=s or None)
                rw, rh, left, top = gpu.pil_geometry(cw, ch, size[1], size[0], s)
                cy = gpu.pil_coefficients(ch, rh, filt == "pil_bicubic", top, size[0])
                y0, y1 = cy[0][0], cy[-1][0] + len(cy[-1][1])
                fewer += y1 - y0 < ch
                sub, row0 = util.ZjImage(), C.c_uint32()
                assert lib.zj_image_rows(C.byref(img), y + y0, y + y1, C.byref(sub), C.byref(row0)) == 0
                piece = oracle.reconstruct(sub)
                # the piece's rows stand in for crop rows [y0, y1): place them in an image whose other rows are garbage
                fake = rng.integers(0, 256, (h, w * 3), dtype=np.uint8)
                fake[y + y0:y + y1] = piece.reshape(sub.height, w * 3)[row0.value:row0.value + y1 - y0]
                want = rz.expected(whole, w, h, 3, None, roi)
                assert rz.expected(fake.reshape(-1), w, h, 3, None, roi).tobytes() == want.tobytes(), (w, h, filt, roi, size, s)
    assert fewer > 0


# ------------------------------------------------------------------ on the GPU: bit-exact against the statement
def _device_images(gpu, cases):
    """cases: (w, h, mode, out_cs, variant, flags, seed) -> device images, their reference bytes, buffers to keep alive"""
    from test_libjpeg_output import libjpeg_expected
    from test_spec_output import spec_expected, spec_planes
    imgs, wants, keep = [], [], []
    for (w, h, mode, out_cs, variant, flags, seed) in cases:
        hs, vs = MODES[mode]
        rng = np.random.default_rng(seed)
        planes = spec_planes(rng, w, h, 3, hs, vs) if variant == _ffi.VARIANT_SPEC else util.random_planes(rng, w, h, 3, hs, vs)
        host = util.make_image(w, h, planes, QTS, hs, vs, out_cs, variant)
        host.flags = flags
        if variant == _ffi.VARIANT_SPEC:
            wants.append((libjpeg_expected if flags else spec_expected)(host, planes))
        else:
            wants.append(oracle.reconstruct(host))
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b, p in zip(bufs, planes):
            b.upload(p)
        keep.append((planes, bufs))
        img = util.make_image(w, h, planes, QTS, hs, vs, out_cs, variant, ptrs=[b.ptr for b in bufs])
        img.flags = flags
        imgs.append(img)
    return imgs, wants, keep


SPEC, ISLOW = _ffi.VARIANT_SPEC, _ffi.FLAG_ISLOW
# as-written, spec and libjpeg images; RGB (nc 3), gray (nc 1), RGBX (nc 4); 4:2:0 / 4:2:2 / 4:4:4 / 4:4:0
GEOMS = [(640, 96, "420", 0, 0, 0), (333, 131, "444", 0, SPEC, 0), (1000, 64, "422", 5, SPEC, ISLOW), (72, 40, "440", 1, 0, 0),
         (200, 203, "420", 0, SPEC, ISLOW), (520, 69, "422", 5, 0, 0), (17, 33, "444", 5, SPEC, 0), (136, 69, "422", 1, SPEC, ISLOW)]


def _crops(w, h):
    return [None, (w // 4, h // 4, w // 2, max(h // 3, 1)), (0, h // 3, w // 3 + 1, h // 3 + 1), (w - w // 3, 0, w // 3, h // 2 + 1),
            (w - 1, h - 1, 1, 1), (1, 0, w - 2, h)]


@pytest.mark.gpu
@pytest.mark.parametrize("layout", ["CHW", "HWC"])
@pytest.mark.parametrize("dtype", DTYPES)
@pytest.mark.parametrize("filt", FILTERS)
def test_reconstruct_device_resized_matches_statement(filt, dtype, layout):
    """3 dtypes x 2 layouts x the (NC, OC) pairs (1, 1), (3, 3), (4, 4), (4, 3) x both filters x both short_side modes"""
    from zune_jpeg_b200 import gpu
    for channels in (0, 3):
        desc = gpu.OutputDesc(layout, dtype, False, channels, MEAN, INV)
        oc_of = lambda out_cs: {0: 3, 1: 1}.get(out_cs, 3 if channels == 3 else 4)
        for oc in sorted({oc_of(g[3]) for g in GEOMS}):
            geoms = [g for g in GEOMS if oc_of(g[3]) == oc]
            imgs, wants, keep = _device_images(gpu, [(*g, 200 + k) for k, g in enumerate(geoms)])
            for size, s in [((24, 40), None), ((150, 90), None), ((7, 31), None), ((16, 16), 16), ((1, 1), 1)]:
                batch = [(img, want, g, roi) for g, img, want in zip(geoms, imgs, wants) for roi in _crops(g[0], g[1])]
                if s:       # crops whose resized size covers the window
                    batch = [b for b in batch if gpu.pil_geometry(*(b[3] or (0, 0, b[2][0], b[2][1]))[2:], size[1], size[0], s)]
                rz = gpu.Resize(size, filt, short_side=s)
                got = gpu.reconstruct_device_resized([b[0] for b in batch], rz, desc, [b[3] for b in batch]).download()
                for k, (img, want, g, roi) in enumerate(batch):
                    nc = len(want) // (g[0] * g[1])
                    exp = rz.expected(want, g[0], g[1], nc, desc, roi)
                    assert got[k].tobytes() == exp.tobytes(), f"{g} roi={roi} size={size} s={s}: {np.count_nonzero(got[k] != exp)} differ"


@pytest.mark.gpu
@pytest.mark.parametrize("filt", FILTERS)
def test_resize_alone_exact_size_sources(filt):
    """zj_gpu_resize_device over sources of exactly w * h * nc bytes at offsets 0-3 into their allocation"""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(21)
    for (w, h, nc, channels, offset) in [(77, 45, 3, 0, 0), (77, 45, 3, 0, 1), (131, 29, 4, 3, 2), (95, 61, 1, 0, 3), (64, 64, 4, 0, 1)]:
        u8 = _structured(rng, w, h, nc).reshape(-1)
        buf = gpu.DeviceBuffer(u8.nbytes + offset)
        buf.upload(u8, offset=offset)
        src = types.SimpleNamespace(ptr=buf.ptr + offset)
        for roi in [None, (1, 3, w - 2, h - 5), (3, 0, 5, h), (w - 7, h - 2, 7, 2), (5, 7, 1, 1)]:
            for dtype, layout, size, s in [("u8", "HWC", (13, 21), None), ("f16", "CHW", (40, 150), None), ("f32", "HWC", (1, 1), None),
                                           ("u8", "CHW", (h, w), None), ("u8", "HWC", (2, 2), 2), ("f16", "HWC", (5, 3), 7)]:
                x, y, cw, ch = roi or (0, 0, w, h)
                if s and gpu.pil_geometry(cw, ch, size[1], size[0], s) is None:
                    continue
                desc = gpu.OutputDesc(layout, dtype, False, channels, MEAN, INV)
                rz = gpu.Resize(size, filt, short_side=s)
                got = gpu.resize_device(src, w, h, nc, rz, desc, roi).download()
                exp = rz.expected(u8, w, h, nc, desc, roi)
                assert got.tobytes() == exp.tobytes(), (w, h, nc, offset, roi, dtype, layout, size, s)


@pytest.mark.gpu
def test_mixed_batch_and_strong_down_scales():
    """One call with crops of different sizes and aspect ratios, down-scales to 1 and 2 pixels (thousands of taps per output)"""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(31)
    w, h = 3840, 2160
    u8 = rng.integers(0, 256, w * h * 3, dtype=np.uint8)
    buf = gpu.DeviceBuffer(u8.nbytes)
    buf.upload(u8)
    for filt in FILTERS:
        for size, s in [((1, 1), None), ((2, 7), None), ((224, 224), 256)]:
            rz = gpu.Resize(size, filt, short_side=s)
            desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
            got = gpu.resize_device(buf, w, h, 3, rz, desc).download()
            assert got.tobytes() == rz.expected(u8, w, h, 3, desc).tobytes(), (filt, size, s)
    imgs, wants, keep = _device_images(gpu, [(640, 480, "420", 0, SPEC, ISLOW, 1), (480, 640, "422", 0, 0, 0, 2),
                                             (301, 299, "444", 0, SPEC, 0, 3), (1000, 96, "420", 0, SPEC, ISLOW, 4)])
    rois = [(10, 20, 600, 300), (0, 0, 480, 640), (5, 5, 250, 290), (100, 0, 800, 96)]
    desc = gpu.OutputDesc("HWC", "u8")
    for filt in FILTERS:
        for s in (None, 96):
            rz = gpu.Resize((96, 96), filt, short_side=s)
            got = gpu.reconstruct_device_resized(imgs, rz, desc, rois).download()
            for k, (img, want) in enumerate(zip(imgs, wants)):
                assert got[k].tobytes() == rz.expected(want, img.width, img.height, 3, desc, rois[k]).tobytes(), (filt, s, k)


def _pillow_decode(data):
    return Image.open(io.BytesIO(data)).convert("RGB")


@pytest.mark.gpu
def test_jpeg_bytes_equal_torchvision_on_pillow():
    """The headline: JPEG bytes in libjpeg output mode through decode_batch_resized, u8 HWC, equal Pillow's decode followed by
    torchvision's resized_crop, and by Resize(256) + CenterCrop(224); f16 CHW equals OutputDesc.expected of those bytes."""
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import ColorSpace, ZuneJpegOptions, decode_batch_resized
    try:
        from torchvision.transforms import InterpolationMode, v2
    except Exception:
        v2 = None
    datas = [ref_files.read(n) for n in ref_files.NAMES]
    datas += [jpeg_util.synth_jpeg(1, 640, 362, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(2, 333, 250, "422", 90),
              jpeg_util.synth_jpeg(3, 500, 301, "444", 85), jpeg_util.synth_jpeg(4, 257, 299, gray=True)]
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    pil = [_pillow_decode(d) for d in datas]
    rng = np.random.default_rng(5)
    rois = []
    for im in pil:
        w, h = im.size
        x, y = int(rng.integers(0, w // 3 + 1)), int(rng.integers(0, h // 3 + 1))
        rois.append((x, y, int(rng.integers(max(1, w // 4), w - x + 1)), int(rng.integers(max(1, h // 4), h - y + 1))))
    u8 = gpu.OutputDesc("HWC", "u8")
    f16 = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    for filt in FILTERS:
        mode = PIL[filt]
        for short_side, use_rois in ((None, True), (256, False)):
            rz = gpu.Resize((224, 224), filt, short_side=short_side)
            ok = [short_side is None or gpu.pil_geometry(*im.size, 224, 224, short_side) is not None for im in pil]
            outs = {}
            for desc in (u8, f16):
                out, errs = decode_batch_resized(datas, rz, desc, rois if use_rois else None, opts, threads=4)
                assert [e is None for e in errs] == ok, errs
                outs[desc.c.dtype] = out.download()
            for k, im in enumerate(pil):
                if not ok[k]:
                    continue
                if use_rois:
                    x, y, cw, ch = rois[k]
                    want = np.asarray(im.crop((x, y, x + cw, y + ch)).resize((224, 224), mode))
                else:
                    rw, rh, left, top = gpu.pil_geometry(*im.size, 224, 224, short_side)
                    want = np.asarray(im.resize((rw, rh), mode).crop((left, top, left + 224, top + 224)))
                if v2 is not None:
                    ip = InterpolationMode.BILINEAR if filt == "pil_bilinear" else InterpolationMode.BICUBIC
                    tv = (v2.functional.resized_crop(im, rois[k][1], rois[k][0], rois[k][3], rois[k][2], [224, 224], interpolation=ip)
                          if use_rois else v2.Compose([v2.Resize(256, interpolation=ip), v2.CenterCrop(224)])(im))
                    assert np.asarray(tv).tobytes() == want.tobytes(), (filt, k)
                assert outs[_ffi.DTYPE_U8][k].tobytes() == want.tobytes(), (filt, short_side, k)
                assert outs[_ffi.DTYPE_F16][k].tobytes() == f16.expected(want.reshape(-1), 224, 224, 3).tobytes(), (filt, short_side, k)
