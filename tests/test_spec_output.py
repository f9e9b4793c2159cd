"""Spec-correct output mode (ZJ_VARIANT_SPEC, ZuneJpegOptions.set_spec_output): every row decoded, libjpeg-style chroma
up-sampling, JFIF colour, opaque alpha.  The statement is in include/zune_jpeg_b200.h; spec_expected() below restates it in
numpy (with the X86 IDCT of ref_model), and every GPU result is compared with it bit for bit.  The CPU part checks the statement
on the host stage's spec-mode planes against libjpeg-turbo (Pillow), the host stage itself and the C ABI; it launches nothing."""
import ctypes as C
import io

import numpy as np
import pytest
from PIL import Image

import jpeg_util
import oracle
import ref_files
import ref_model
import util
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch

SPEC = _ffi.VARIANT_SPEC
NC = {_ffi.CS_RGB: 3, _ffi.CS_RGBA: 4, _ffi.CS_RGBX: 4, _ffi.CS_YCBCR: 3, _ffi.CS_GRAYSCALE: 1}
MODES = {"none": (1, 1), "h": (2, 1), "v": (1, 2), "hv": (2, 2)}
QTS = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]


# ------------------------------------------------------------------------------------------------ the statement in numpy
def _component(img, planes, z):
    c = img.comp[z]
    s = ref_model.idct_blocks(planes[z].reshape(-1, 64), np.array(c.qt, np.int32), ref_model.X86)
    return ref_model.plane_from_blocks(s, c.width_stride // 8).astype(np.int32)


def _clamped(a, axis, d):
    """a shifted by d (-1: the previous sample, +1: the next one) along axis, the index clamped to the array"""
    n = a.shape[axis]
    idx = np.clip(np.arange(n) + d, 0, n - 1)
    return np.take(a, idx, axis=axis)


def _interleave(even, odd, axis):
    out = np.stack([even, odd], axis=axis + 1)
    shape = list(even.shape)
    shape[axis] *= 2
    return out.reshape(shape)


def _upsample(c, hs, vs):
    """libjpeg-turbo jdsample.c integer fancy up-sampling of a cw x ch chroma plane, neighbours clamped to it"""
    if vs == 2:
        s_even = 3 * c + _clamped(c, 0, -1)       # column sums for output rows 2j (j' = j - 1) and 2j + 1 (j' = j + 1)
        s_odd = 3 * c + _clamped(c, 0, +1)
        if hs == 2:
            rows = []
            for s in (s_even, s_odd):
                rows.append(_interleave((3 * s + _clamped(s, 1, -1) + 8) >> 4, (3 * s + _clamped(s, 1, +1) + 7) >> 4, 1))
            return _interleave(rows[0], rows[1], 0)
        return _interleave((s_even + 1) >> 2, (s_odd + 2) >> 2, 0)
    if hs == 2:
        return _interleave((3 * c + _clamped(c, 1, -1) + 1) >> 2, (3 * c + _clamped(c, 1, +1) + 2) >> 2, 1)
    return c


def spec_expected(img, planes) -> np.ndarray:
    """The statement of ZJ_VARIANT_SPEC: the width * height * nc bytes the output must hold."""
    w, h = img.width, img.height
    y = _component(img, planes, 0)[:h, :w]
    cs = img.out_cs
    if cs == _ffi.CS_GRAYSCALE:
        px = y[:, :, None]
    elif img.n_comp == 1:
        px = np.stack([y, y, y], -1)
    else:
        hs, vs = img.comp[0].h_samp, img.comp[0].v_samp
        cw, ch = -(-w // hs), -(-h // vs)
        cb, cr = (_upsample(_component(img, planes, z)[:ch, :cw], hs, vs)[:h, :w] for z in (1, 2))
        if cs == _ffi.CS_YCBCR:
            px = np.stack([y, cb, cr], -1)
        else:
            cb, cr = cb - 128, cr - 128
            px = np.stack([y + ((91881 * cr + 32768) >> 16), y + ((-22554 * cb - 46802 * cr + 32768) >> 16),
                           y + ((116130 * cb + 32768) >> 16)], -1)
    px = np.clip(px, 0, 255).astype(np.uint8)
    if cs in (_ffi.CS_RGBA, _ffi.CS_RGBX):
        px = np.concatenate([px, np.full(px.shape[:2] + (1,), 255, np.uint8)], -1)
    return px.reshape(-1)


def spec_planes(rng, w, h, n_comp, hs, vs, **kw):
    """util.random_planes, padded with zero blocks to whole strips: 4:2:2 / 4:2:0 strips hold two MCU rows"""
    planes = util.random_planes(rng, w, h, n_comp, hs, vs, **kw)
    mcu_x, mcu_y = util.geometry(w, h, hs, vs)
    if hs == 2 and mcu_y % 2:
        planes = [np.concatenate([p, np.zeros(mcu_x * (hs * vs if z == 0 else 1) * 64, np.int16)]) for z, p in enumerate(planes)]
    return planes


def spec_decoder(cs=ColorSpace.RGB, threads=4):
    return Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(cs).set_spec_output(True).set_num_threads(threads))


def _pillow(data, gray=False):
    im = Image.open(io.BytesIO(data))
    return np.asarray(im.convert("L" if gray else "RGB")).astype(np.int16)


def _deviation(data, gray=False):
    """max |delta| over the whole image between the statement on spec-mode host-stage planes and libjpeg-turbo"""
    img, planes = spec_decoder(ColorSpace.GRAYSCALE if gray else ColorSpace.RGB).decode_coefficients(data)
    assert img.variant == SPEC
    ref = _pillow(data, gray)
    got = spec_expected(img, planes).reshape(ref.shape).astype(np.int16)
    d = np.abs(got - ref)
    return int(d.max()), float(d.mean())


# ------------------------------------------------------------------------------------------------ CPU
def test_spec_expected_matches_the_idct_and_filters_on_small_cases():
    """The numpy statement on hand-checkable inputs: flat planes give flat pixels, a 2-sample H row gives the libjpeg values."""
    c = np.array([[10, 50]], np.int32)
    assert _upsample(c, 2, 1).tolist() == [[10, 20, 40, 50]]                # (3*10+10+1)>>2, (30+50+2)>>2, (150+10+1)>>2, (150+50+2)>>2
    c = np.array([[10], [50]], np.int32)
    assert _upsample(c, 1, 2)[:, 0].tolist() == [10, 20, 40, 50]
    c = np.array([[16, 16], [16, 16]], np.int32)
    assert (_upsample(c, 2, 2) == 16).all()
    rng = np.random.default_rng(1)
    planes = spec_planes(rng, 17, 9, 3, 2, 2, dc_only_frac=1.0)
    for p in planes:
        p[0::64] = 0                                                           # DC 0 everywhere: every sample is 128
    img = util.make_image(17, 9, planes, QTS, 2, 2, _ffi.CS_RGBA, SPEC)
    assert (spec_expected(img, planes).reshape(9, 17, 4) == [128, 128, 128, 255]).all()


SYNTH = [  # (seed, width, height, subsampling, quality, progressive, gray)
    (1, 637, 480, "420", 75, False, False), (2, 640, 362, "420", 90, False, False), (3, 1023, 770, "420", 95, False, False),
    (4, 333, 250, "422", 85, False, False), (5, 301, 203, "444", 60, False, False), (6, 640, 362, "420", 100, False, False),
    (7, 555, 333, "420", 90, True, False), (8, 321, 199, "444", 90, False, True), (9, 350, 201, "422", 100, False, False),
]


@pytest.mark.parametrize("seed,w,h,sub,q,prog,gray", SYNTH)
def test_statement_against_libjpeg_on_synthetic_images(seed, w, h, sub, q, prog, gray):
    mx, mean = _deviation(jpeg_util.synth_jpeg(seed, w, h, sub, q, prog, gray), gray)
    assert mx <= 4 and mean < 0.2, (mx, mean)


@pytest.mark.parametrize("name", ref_files.NAMES)
def test_statement_against_libjpeg_on_reference_fixtures(name):
    """As written these files are 21-255 off libjpeg (DESIGN.md section 2); under the statement every pixel is within 4."""
    mx, mean = _deviation(ref_files.read(name))
    assert mx <= 4 and mean < 0.5, (name, mx, mean)


def _as_written_and_spec(data, threads=4):
    a_img, a_planes = Decoder.new_with_options(ZuneJpegOptions().set_num_threads(threads)).decode_coefficients(data)
    s_img, s_planes = spec_decoder(threads=threads).decode_coefficients(data)
    return (a_img, a_planes), (s_img, s_planes)


@pytest.mark.parametrize("restart,prog", [(0, False), (1, False), (0, True)])
def test_host_stage_planes_cover_every_row(restart, prog):
    """1280 x 738 4:2:0 has 47 MCU rows.  As written the last one is never decoded (Q1) and its planes are one MCU row short;
    spec output decodes it, in a last strip whose lower half stays zero -- sequential, interval-parallel and progressive."""
    data = jpeg_util.synth_jpeg(11, 1280, 738, "420", 90, progressive=prog, restart_rows=restart)
    (a_img, a_planes), (s_img, s_planes) = _as_written_and_spec(data)
    lib = _ffi.load()
    assert s_img.variant == SPEC and lib.zj_validate_image(C.byref(s_img)) == 0
    strip_y, strip_c = 160 * 4 * 64, 80 * 2 * 64                                 # i16 per strip of 32 rows
    assert s_planes[0].size == 24 * strip_y and s_planes[1].size == 24 * strip_c
    mcu_row_y = strip_y // 2
    assert np.any(s_planes[0][46 * mcu_row_y:47 * mcu_row_y] != 0)            # MCU row 46 is there ...
    assert not np.any(s_planes[0][47 * mcu_row_y:])                            # ... the half strip below it is not
    if not prog:
        assert a_planes[0].size == 23 * strip_y                               # (as written: 23 strips)
        # the spec planes' first 23 strips are the as-written planes (Q9-Q11 do not fire on this file)
        assert np.array_equal(s_planes[0][:a_planes[0].size], a_planes[0])
        a_img.variant = SPEC
        assert lib.zj_validate_image(C.byref(a_img)) == _ffi.ERR_SHORT_PLANE  # as-written planes cannot feed spec output
    if restart:
        d = spec_decoder()
        d.decode_coefficients(data)
        assert d.entropy_segments() > 1                                        # the intervals ran side by side


def test_spec_decodes_ignore_the_quirk_switch_and_leave_it_alone():
    """huffman_third_index.jpg trips Q9 as written: the spec decode is libjpeg-close with every quirk switched on, and an
    as-written decode after it still shows the quirk (the switch is process-wide, a spec decode does not change it)."""
    data = ref_files.read("huffman_third_index.jpg")
    lib = _ffi.load()
    assert lib.zj_host_get_quirks() == _ffi.QUIRK_ALL
    mx_spec, _ = _deviation(data)
    assert mx_spec <= 4
    img, planes = Decoder.new_with_options(ZuneJpegOptions()).decode_coefficients(data)
    spec_img, spec_planes_ = spec_decoder().decode_coefficients(data)
    assert not np.array_equal(planes[0][:spec_planes_[0].size], spec_planes_[0][:planes[0].size])
    try:
        lib.zj_host_set_quirks(0)
        img2, planes2 = Decoder.new_with_options(ZuneJpegOptions()).decode_coefficients(data)
        assert np.array_equal(planes2[0], spec_planes_[0][:planes2[0].size])   # the switch off == the spec decode's planes
        spec_img3, spec_planes3 = spec_decoder().decode_coefficients(data)
        assert np.array_equal(spec_planes3[0], spec_planes_[0])
    finally:
        lib.zj_host_set_quirks(_ffi.QUIRK_ALL)
    assert lib.zj_host_get_quirks() == _ffi.QUIRK_ALL


def test_gray_jpeg_keeps_the_requested_colourspace():
    data = jpeg_util.synth_jpeg(3, 99, 45, gray=True)
    for cs in (ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.RGBX, ColorSpace.GRAYSCALE):
        img, _ = spec_decoder(cs).decode_coefficients(data)
        assert img.n_comp == 1 and img.out_cs == int(cs)
    img, _ = spec_decoder(ColorSpace.YCbCr).decode_coefficients(data)
    assert img.out_cs == _ffi.CS_GRAYSCALE                                      # no stated output: GRAYSCALE as before
    img, _ = Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB)).decode_coefficients(data)
    assert img.out_cs == _ffi.CS_GRAYSCALE                                      # as written: forced to GRAYSCALE


def test_abi_validation_and_strip_ranges():
    lib = _ffi.load()
    rng = np.random.default_rng(2)
    # geometries the reference panics on as written (the output-capacity rule, Q7) and tiny ones
    written = []
    for (w, h, mode, cs) in [(9, 40, "hv", _ffi.CS_RGB), (1, 1, "hv", _ffi.CS_RGB), (65535, 9, "h", _ffi.CS_RGB),
                             (17, 40, "hv", _ffi.CS_GRAYSCALE), (15, 33, "h", _ffi.CS_YCBCR)]:
        hs, vs = MODES[mode]
        planes = spec_planes(rng, w, h, 3, hs, vs, density=0.0)
        img = util.make_image(w, h, planes, QTS, hs, vs, cs, _ffi.VARIANT_X86)
        written.append(lib.zj_validate_image(C.byref(img)))
        img.variant = SPEC
        assert lib.zj_validate_image(C.byref(img)) == 0, (w, h, mode, cs, written)
        assert lib.zj_output_size(C.byref(img)) == w * h * NC[cs]
    assert written.count(_ffi.ERR_REF_PANIC) >= 2, written
    # unsupported pairs
    planes = spec_planes(rng, 40, 24, 3, 2, 2)
    for cs in (_ffi.CS_CMYK, _ffi.CS_YCCK):
        assert lib.zj_validate_image(C.byref(util.make_image(40, 24, planes, QTS, 2, 2, cs, SPEC))) == _ffi.ERR_UNSUPPORTED
    g = spec_planes(rng, 40, 24, 1, 1, 1)
    for cs, rc in ((_ffi.CS_YCBCR, _ffi.ERR_UNSUPPORTED), (_ffi.CS_CMYK, _ffi.ERR_UNSUPPORTED), (_ffi.CS_RGB, 0),
                   (_ffi.CS_RGBA, 0), (_ffi.CS_RGBX, 0), (_ffi.CS_GRAYSCALE, 0)):
        assert lib.zj_validate_image(C.byref(util.make_image(40, 24, g, QTS[:1], 1, 1, cs, SPEC))) == rc, cs
    assert lib.zj_validate_image(C.byref(util.make_image(40, 24, planes, QTS, 2, 2, 0, 3))) == _ffi.ERR_INVALID_ARG
    # planes one MCU row short (what an as-written host stage leaves for an odd MCU-row count)
    short = util.random_planes(rng, 640, 362, 3, 2, 2)
    assert lib.zj_validate_image(C.byref(util.make_image(640, 362, short, QTS, 2, 2, 0, SPEC))) == _ffi.ERR_SHORT_PLANE
    # strip ranges: the query form works, every cut is refused
    planes = spec_planes(rng, 640, 362, 3, 2, 2)
    img = util.make_image(640, 362, planes, QTS, 2, 2, _ffi.CS_RGB, SPEC)
    ns = C.c_uint32()
    assert lib.zj_image_strip_range(C.byref(img), 0, 0, None, None, None, C.byref(ns)) == 0 and ns.value == 12
    sub = _ffi.ZjImage()
    off, nb = C.c_size_t(), C.c_size_t()
    for s0, s1 in ((0, 12), (0, 6), (6, 12)):
        assert lib.zj_image_strip_range(C.byref(img), s0, s1, C.byref(sub), C.byref(off), C.byref(nb), None) == _ffi.ERR_UNSUPPORTED
    row0 = C.c_uint32()
    assert lib.zj_image_rows(C.byref(img), 100, 200, C.byref(sub), C.byref(row0)) == 0
    assert sub.height == 362 and row0.value == 100                             # returned whole


def test_option_reaches_the_descriptor():
    o = ZuneJpegOptions()
    assert o.get_spec_output() is False and o._raw().use_unsafe == 1
    s = o.set_spec_output(True)
    assert s.get_spec_output() is True and o.get_spec_output() is False
    assert s._raw().use_unsafe == _ffi.USE_SPEC_OUTPUT == 2
    assert s.set_use_unsafe(False)._raw().use_unsafe == 2
    data = jpeg_util.synth_jpeg(1, 64, 48)
    for opts, variant in ((ZuneJpegOptions(), _ffi.VARIANT_X86), (ZuneJpegOptions().set_use_unsafe(False), _ffi.VARIANT_SCALAR), (s, SPEC)):
        img, _ = Decoder.new_with_options(opts).decode_coefficients(data)
        assert img.variant == variant


# ------------------------------------------------------------------------------------------------ GPU
WIDTHS = [1, 2, 7, 15, 16, 17, 33, 255, 637, 3840]
HEIGHTS = [1, 7, 9, 17, 33, 362, 2160]
COLOR_CS = [_ffi.CS_RGB, _ffi.CS_RGBA, _ffi.CS_RGBX, _ffi.CS_YCBCR, _ffi.CS_GRAYSCALE]


def _cases(mode, seed):
    """(w, h) pairs covering every width and every height, plus a few small squares, without the full cross product"""
    rng = np.random.default_rng(seed)
    out = [(w, HEIGHTS[(i + seed) % len(HEIGHTS)]) for i, w in enumerate(WIDTHS)]
    out += [(WIDTHS[(i + seed) % 8], hh) for i, hh in enumerate(HEIGHTS)]
    out += [(int(rng.integers(1, 80)), int(rng.integers(1, 80))) for _ in range(3)]
    return [(w, h) for (w, h) in out if w * h <= 3840 * 362 or (w, h) == (3840, 2160)]


def _host_images(rng, cases, mode, cs_list, n_comp=3, extreme_every=3):
    hs, vs = MODES[mode]
    imgs, keep, wants = [], [], []
    for k, (w, h) in enumerate(cases):
        cs = cs_list[k % len(cs_list)]
        planes = spec_planes(rng, w, h, n_comp, hs, vs, extreme=(k % extreme_every == 0))
        img = util.make_image(w, h, planes, QTS[:n_comp], hs, vs, cs, SPEC)
        imgs.append(img); keep.append(planes); wants.append(spec_expected(img, planes))
    return imgs, keep, wants


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_reconstruct_host_entry_matches_statement(mode):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(100 + list(MODES).index(mode))
    cases = _cases(mode, list(MODES).index(mode))
    for cs in COLOR_CS:
        imgs, keep, wants = _host_images(rng, cases, mode, [cs])
        got = gpu.reconstruct(imgs, device=0)
        for (w, h), g, want in zip(cases, got, wants):
            assert np.array_equal(g, want), (mode, cs, w, h, int(np.count_nonzero(g != want)))


def _device_run(imgs, keep, use_batch, out_offset=0):
    from zune_jpeg_b200 import gpu
    bufs, dimgs, outs = [], [], []
    for img, planes in zip(imgs, keep):
        b = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for bb, p in zip(b, planes):
            bb.upload(p)
        bufs.append(b)
        d = _ffi.ZjImage()
        C.memmove(C.byref(d), C.byref(img), C.sizeof(d))
        for z, bb in enumerate(b):
            d.comp[z].coeff = bb.ptr
        dimgs.append(d)
        n = gpu.output_size(img)
        o = gpu.DeviceBuffer(n + out_offset + 16)
        o.memset(0xAB)
        outs.append(o)
    gpu.synchronize()
    ptrs = [o.ptr + out_offset for o in outs]
    lens = [gpu.output_size(i) for i in imgs]
    lib = _ffi.load()
    if use_batch:
        batch = gpu.Batch(dimgs, ptrs, lens)
        batch.run()
        gpu.synchronize()
        batch.destroy()
    else:
        arr = gpu._img_array(dimgs)
        n = len(dimgs)
        rc = lib.zj_gpu_reconstruct_device(0, None, arr, n, (C.c_void_p * n)(*ptrs), (C.c_size_t * n)(*lens))
        assert rc == 0, rc
    res = []
    for o, ln in zip(outs, lens):
        full = o.download()
        assert (full[:out_offset] == 0xAB).all() and (full[out_offset + ln:] == 0xAB).all()   # nothing outside the image
        res.append(full[out_offset:out_offset + ln])
    return res


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("use_batch", [False, True])
def test_reconstruct_device_and_batch_match_statement(mode, use_batch):
    rng = np.random.default_rng(200 + list(MODES).index(mode))
    cases = [c for c in _cases(mode, 3 + list(MODES).index(mode)) if c[0] * c[1] <= 640 * 2160]
    imgs, keep, wants = _host_images(rng, cases, mode, COLOR_CS, extreme_every=2)
    for off in (0, 1):                                                          # 16-byte and byte-aligned outputs
        got = _device_run(imgs, keep, use_batch, off)
        for (w, h), img, g, want in zip(cases, imgs, got, wants):
            assert np.array_equal(g, want), (mode, use_batch, off, w, h, img.out_cs)


@pytest.mark.gpu
def test_gray_input():
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(300)
    cases = _cases("none", 5)
    imgs, keep, wants = _host_images(rng, cases, "none", [_ffi.CS_GRAYSCALE, _ffi.CS_RGB, _ffi.CS_RGBA, _ffi.CS_RGBX], n_comp=1)
    for (w, h), img, g, want in zip(cases, imgs, gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want), (w, h, img.out_cs)


@pytest.mark.gpu
def test_mixed_as_written_and_spec_images_in_one_call():
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(400)
    imgs, keep, wants = [], [], []
    for k, (w, h, mode, cs) in enumerate([(640, 362, "hv", 0), (333, 250, "h", 0), (255, 33, "v", 2), (100, 17, "none", 5),
                                          (640, 362, "hv", 5), (17, 9, "hv", 1), (637, 480, "hv", 0), (99, 45, "none", 1)]):
        hs, vs = MODES[mode]
        spec = k % 2 == 0
        planes = spec_planes(rng, w, h, 3, hs, vs)
        img = util.make_image(w, h, planes, QTS, hs, vs, cs, SPEC if spec else _ffi.VARIANT_X86)
        imgs.append(img); keep.append(planes)
        wants.append(spec_expected(img, planes) if spec else oracle.reconstruct(img))
    for use_batch in (False, True):
        for g, want, img in zip(_device_run(imgs, keep, use_batch), wants, imgs):
            assert np.array_equal(g, want), (img.width, img.height, img.variant)
    for g, want in zip(gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want)


def _want_from_bytes(data, cs=ColorSpace.RGB):
    img, planes = spec_decoder(cs).decode_coefficients(data)
    return img, spec_expected(img, planes)


@pytest.mark.gpu
def test_jpeg_bytes_routes():
    from zune_jpeg_b200 import gpu
    datas = [jpeg_util.synth_jpeg(1, 640, 362, "420", 90), jpeg_util.synth_jpeg(2, 333, 250, "422", 95, restart_rows=1),
             jpeg_util.synth_jpeg(3, 301, 203, "444", 90, progressive=True), jpeg_util.synth_jpeg(4, 99, 45, gray=True),
             ref_files.read("medium_vertical_samp_2500x1786.jpg")]
    wants = [_want_from_bytes(d)[1] for d in datas]
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_spec_output(True)
    for d, want in zip(datas, wants):
        assert np.frombuffer(Decoder.new_with_options(opts).decode_buffer(d), np.uint8).tobytes() == want.tobytes()
    got = decode_batch(datas, opts, threads=4)
    assert [g == w.tobytes() for g, w in zip(got, wants)] == [True] * len(datas)
    got = decode_batch(datas, opts, threads=4, devices=[0, 0])
    assert [g == w.tobytes() for g, w in zip(got, wants)] == [True] * len(datas)
    one = decode_batch(datas[:1], opts, threads=4, devices=[0, 0])             # fewer images than devices: whole images
    assert one[0] == wants[0].tobytes()
    # restart-marker files, which the GPU entropy route would take as written, go through the host stage
    dri = [jpeg_util.synth_jpeg(5, 640, 352, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(6, 640, 362, "420", 90, restart_rows=2)]
    stats = {}
    got = decode_batch(dri, opts, threads=4, gpu_entropy=True, stats=stats)
    assert stats["gpu_entropy"] == 0
    assert [g == _want_from_bytes(d)[1].tobytes() for g, d in zip(got, dri)] == [True, True]


@pytest.mark.gpu
def test_decode_into_large_baseline_image():
    """>= 4 MP baseline into pinned memory: the strip pipeline stays off (a spec image cannot be cut), the bytes are right."""
    from zune_jpeg_b200 import gpu
    data = jpeg_util.synth_jpeg(7, 2560, 1610, "420", 90, restart_rows=4)     # 4.1 MP, odd MCU-row count (101)
    img, want = _want_from_bytes(data)
    buf = gpu.PinnedBuffer(want.size)
    view = buf.array if hasattr(buf, "array") else np.ctypeslib.as_array((C.c_uint8 * want.size).from_address(buf.ptr))
    view[:] = 0xAB
    n = spec_decoder().decode_into(data, view)
    assert n == want.size and view.tobytes() == want.tobytes()


MEAN = (0.485 * 255, 0.456 * 255, 0.406 * 255, 0.0)
INV = (1 / (0.229 * 255), 1 / (0.224 * 255), 1 / (0.225 * 255), 1.0)


@pytest.mark.gpu
def test_consumers():
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import decode_batch_resized
    datas = [jpeg_util.synth_jpeg(1, 640, 362, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(2, 333, 250, "422", 90),
             jpeg_util.synth_jpeg(3, 257, 199, gray=True), jpeg_util.synth_jpeg(4, 500, 301, "444", 85)]
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_spec_output(True)
    wants = [_want_from_bytes(d) for d in datas]
    # device_out + desc: f16 CHW, ImageNet normalisation
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    outs = [gpu.DeviceBuffer(img.width * img.height * 3 * 2) for img, _ in wants]
    stats = {}
    res = decode_batch(datas, opts, threads=4, device_out=[(o.ptr, o.nbytes) for o in outs], desc=desc, stats=stats)
    assert stats["gpu_entropy"] == 0
    for (img, want), o, r in zip(wants, outs, res):
        assert r == o.nbytes
        assert o.download().tobytes() == desc.expected(want, img.width, img.height, 3).tobytes()
    # one batch tensor from a mix of gray and colour JPEGs, RGB
    rz = gpu.Resize((96, 128), "area")
    rois = [(10, 20, 300, 200), None, (0, 0, 257, 199), (100, 1, 400, 300)]
    out, errs = decode_batch_resized(datas, rz, desc, rois, opts, threads=4)
    assert errs == [None] * 4
    got = out.download()
    for k, (img, want) in enumerate(wants):
        assert got[k].tobytes() == rz.expected(want, img.width, img.height, 3, desc, rois[k]).tobytes(), k
