"""DCT-scaled decoding of libjpeg output (ZJ_FLAG_SCALE_*, ZuneJpegOptions.set_scale_denom): libjpeg-turbo's decode to 1/2, 1/4
or 1/8 with the reduced IDCTs of jidctred.c, which is what Pillow's Image.draft gives.  The statement is in
include/zune_jpeg_b200.h; scaled_expected() below restates it in numpy and every GPU result is compared with it bit for bit.
The CPU part checks the statement on the host stage's planes against Pillow's draft at tolerance 0, the reduced IDCTs against an
independent transcription at 64 and 32 bits, and the C ABI; it launches nothing."""
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
from test_libjpeg_output import INPUTS, _input, islow_blocks, libjpeg_decoder, libjpeg_expected, range_limit
from test_spec_output import _cases, _device_run, _upsample, spec_expected, spec_planes
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch, draft_scale

SPEC, ISLOW = _ffi.VARIANT_SPEC, _ffi.FLAG_ISLOW
MODES = {"none": (1, 1), "h": (2, 1), "v": (1, 2), "hv": (2, 2)}
QTS = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]
COLOR_CS = [_ffi.CS_RGB, _ffi.CS_RGBA, _ffi.CS_RGBX, _ffi.CS_YCBCR, _ffi.CS_GRAYSCALE]
DENOMS = (2, 4, 8)


def _flags(d):
    return ISLOW | (d.bit_length() - 1) << _ffi.FLAG_SCALE_SHIFT


# ------------------------------------------------------------------------------------------------ the statement in numpy
def _descale(x, n):
    return (x + np.int32(1 << (n - 1))) >> np.int32(n)


def _red_1d(v, s):
    """one 1-D pass of jpeg_idct_4x4 (s = 4) or jpeg_idct_2x2 (s = 2) along the last axis, before the DESCALE"""
    i32 = np.int32
    if s == 4:
        t0 = v[..., 0] << i32(14)
        t2 = v[..., 2] * i32(15137) + v[..., 6] * i32(-6270)
        t10, t12 = t0 + t2, t0 - t2
        z1, z2, z3, z4 = v[..., 7], v[..., 5], v[..., 3], v[..., 1]
        a = z1 * i32(-1730) + z2 * i32(11893) + z3 * i32(-17799) + z4 * i32(8697)
        b = z1 * i32(-4176) + z2 * i32(-4926) + z3 * i32(7373) + z4 * i32(20995)
        return np.stack([t10 + b, t12 + a, t12 - a, t10 - b], -1)
    t10 = v[..., 0] << i32(15)
    t0 = v[..., 7] * i32(-5906) + v[..., 5] * i32(6967) + v[..., 3] * i32(-10426) + v[..., 1] * i32(29692)
    return np.stack([t10 + t0, t10 - t0], -1)


def scaled_blocks(coef, qt, s):
    """coef int16 [N, 64], qt [64] -> uint8 [N, s, s]: rule 2'' in 32-bit wrapping arithmetic (s = 8: islow_blocks)"""
    if s == 8:
        return islow_blocks(coef, qt)
    with np.errstate(over="ignore"):
        c = coef.reshape(-1, 8, 8).astype(np.int32)
        d = c * np.asarray(qt, np.int32).reshape(8, 8)
        if s == 1:
            return range_limit(_descale(d[:, 0, 0], 3))[:, None, None]
        odd = [1, 2, 3, 5, 6, 7] if s == 4 else [1, 3, 5, 7]
        cols = d.transpose(0, 2, 1)                                               # [N, column, row]
        ws = _descale(_red_1d(cols, s), 12 if s == 4 else 13)                     # [N, column, s]
        ws = np.where(~np.any(c[:, odd, :] != 0, axis=1)[..., None], cols[..., :1] << np.int32(2), ws)
        ws = ws.transpose(0, 2, 1)                                                # [N, s rows, 8 columns]
        out = range_limit(_descale(_red_1d(ws, s), 19 if s == 4 else 20))
        return np.where(~np.any(ws[..., odd] != 0, axis=-1)[..., None], range_limit(_descale(ws[..., :1], 5)), out)


def reduced_blocks_ref(coef, qt, s, bits=None):
    """an independent transcription of jpeg_idct_4x4 / 2x2 / 1x1 (jidctred.c), block by block with Python integers, both zero
    shortcuts as jidctred.c takes them.  bits=None: a JLONG wide enough for every intermediate; bits=32: JLONG and int of 32
    bits, wrapping."""
    def wrap(x):
        if bits is None:
            return x
        x &= (1 << bits) - 1
        return x - (1 << bits) if x >> (bits - 1) else x

    def descale(x, n):
        return wrap(x + (1 << (n - 1))) >> n

    def rl(x):
        return int(range_limit(x))

    def one_d(z, p):   # z: the 8 inputs of a column or row
        if s == 4:
            tmp0 = wrap(z[0] << 14)
            tmp2 = wrap(z[2] * 15137 + z[6] * -6270)
            tmp10, tmp12 = wrap(tmp0 + tmp2), wrap(tmp0 - tmp2)
            t0 = wrap(z[7] * -1730 + z[5] * 11893 + z[3] * -17799 + z[1] * 8697)
            t2 = wrap(z[7] * -4176 + z[5] * -4926 + z[3] * 7373 + z[1] * 20995)
            return [descale(tmp10 + t2, p), descale(tmp12 + t0, p), descale(tmp12 - t0, p), descale(tmp10 - t2, p)]
        tmp10 = wrap(z[0] << 15)
        tmp0 = wrap(z[7] * -5906 + z[5] * 6967 + z[3] * -10426 + z[1] * 29692)
        return [descale(tmp10 + tmp0, p), descale(tmp10 - tmp0, p)]

    out = np.zeros((coef.shape[0], s, s), np.uint8)
    q = [int(x) for x in np.asarray(qt).reshape(64)]
    skip = {4: (4,), 2: (2, 4, 6), 1: ()}[s]
    odd = {4: (1, 2, 3, 5, 6, 7), 2: (1, 3, 5, 7), 1: ()}[s]
    for n, blk in enumerate(coef.reshape(-1, 64)):
        b = [int(x) for x in blk]
        if s == 1:
            out[n, 0, 0] = rl(descale(wrap(b[0] * q[0]), 3))
            continue
        ws = [[0] * 8 for _ in range(s)]
        for col in range(8):
            if col in skip:
                continue
            if all(b[8 * r + col] == 0 for r in odd):
                for r in range(s):
                    ws[r][col] = wrap((b[col] * q[col]) << 2)
                continue
            res = one_d([wrap(b[8 * r + col] * q[8 * r + col]) for r in range(8)], 12 if s == 4 else 13)
            for r in range(s):
                ws[r][col] = res[r]
        for r in range(s):
            if all(ws[r][k] == 0 for k in odd):
                out[n, r, :] = rl(descale(ws[r][0], 5))
            else:
                out[n, r, :] = [rl(v) for v in one_d(ws[r], 19 if s == 4 else 20)]
    return out


def _block_size(img, z, d):
    """rule 1'': jdmaster.c's DCT_scaled_size of component z"""
    s0 = 8 // d
    hmax, vmax = img.comp[0].h_samp, img.comp[0].v_samp
    hz, vz = img.comp[z].h_samp, img.comp[z].v_samp
    ss = s0
    while ss < 8 and (hmax * s0) % (hz * ss * 2) == 0 and (vmax * s0) % (vz * ss * 2) == 0:
        ss *= 2
    return ss


def _plane(img, planes, z, ss):
    c = img.comp[z]
    b = scaled_blocks(planes[z].reshape(-1, 64), np.array(c.qt, np.int32), ss)
    bpr = c.width_stride // 8
    rows = b.shape[0] // bpr
    return b[: rows * bpr].reshape(rows, bpr, ss, ss).transpose(0, 2, 1, 3).reshape(rows * ss, bpr * ss).astype(np.int32)


def scaled_expected(img, planes) -> np.ndarray:
    """The statement of a DCT-scaled image: the W' * H' * nc bytes its output must hold (rules 1''-5''); scale 0 is
    libjpeg_expected"""
    k = (img.flags & _ffi.FLAG_SCALE_MASK) >> _ffi.FLAG_SCALE_SHIFT
    if k == 0:
        return libjpeg_expected(img, planes)
    d = 1 << k
    s0 = 8 // d
    W, H = img.width, img.height
    ow, oh = -(-W // d), -(-H // d)
    y = _plane(img, planes, 0, s0)[:oh, :ow]
    cs = img.out_cs
    if cs == _ffi.CS_GRAYSCALE:
        px = y[:, :, None]
    elif img.n_comp == 1:
        px = np.stack([y, y, y], -1)
    else:
        hmax, vmax = img.comp[0].h_samp, img.comp[0].v_samp
        cc = []
        for z in (1, 2):
            ss = _block_size(img, z, d)
            dw = -(-W * img.comp[z].h_samp * ss // (hmax * 8))
            dh = -(-H * img.comp[z].v_samp * ss // (vmax * 8))
            c = _plane(img, planes, z, ss)[:dh, :dw]
            hf, vf = hmax * s0 // (img.comp[z].h_samp * ss), vmax * s0 // (img.comp[z].v_samp * ss)
            fancy = s0 > 1
            if (hf, vf) == (1, 1):
                u = c
            elif (hf, vf) == (2, 1) and fancy and dw > 2 or (hf, vf) == (1, 2) and fancy:
                u = _upsample(c, hf, vf)
            else:
                u = np.repeat(np.repeat(c, vf, 0), hf, 1)
            cc.append(u[:oh, :ow])
        cb, cr = cc
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


def scaled_decoder(d, cs=ColorSpace.RGB, threads=4):
    return Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(cs).set_libjpeg_output(True).set_scale_denom(d)
                                    .set_num_threads(threads))


def _pillow_draft(data, d, gray=False):
    """Pillow's draft to 1/d (Image.thumbnail's first step), or None where Pillow does not draft that far"""
    im = Image.open(io.BytesIO(data))
    w, h = im.size
    mode = "L" if gray else "RGB"
    im.draft(mode, (max(w // d, 1), max(h // d, 1)))
    if im.size != _ffi.scaled_size(w, h, d):
        return None
    return np.asarray(im.convert(mode))


TINY = [(10, 37, 29, "420"), (11, 19, 13, "422"), (12, 9, 7, "420"), (13, 5, 3, "422"), (14, 3, 9, "422"), (15, 70, 45, "444")]


def _tiny(case):
    seed, w, h, sub = case
    return jpeg_util.synth_jpeg(seed, w, h, sub, 90), False


DRAFT_INPUTS = INPUTS + [pytest.param(("tiny",) + c, id="tiny%dx%d_%s" % c[1:]) for c in TINY]


def _draft_input(case):
    return _tiny(case[1:]) if isinstance(case, tuple) and case[0] == "tiny" else _input(case)


# ------------------------------------------------------------------------------------------------ CPU
def _test_blocks(rng, n, lo, hi):
    """random blocks in [lo, hi) of four kinds: dense, sparse, some columns with AC only (the pass-1 shortcut), DC only"""
    coef = np.zeros((n, 64), np.int16)
    for k in range(n):
        kind = k % 4
        if kind == 0:
            coef[k] = rng.integers(lo // 8, hi // 8, 64)
        elif kind == 1:
            m = rng.random(64) < 0.2
            coef[k][m] = rng.integers(lo // 4, hi // 4, int(m.sum()))
        elif kind == 2:
            b = np.zeros((8, 8), np.int16)
            b[0] = rng.integers(lo, hi, 8)
            for col in rng.choice(8, 3, replace=False):
                b[1:, col] = rng.integers(lo // 16, hi // 16, 7)
            coef[k] = b.reshape(64)
        coef[k, 0] = rng.integers(lo, hi)
    return coef


@pytest.mark.parametrize("s", [4, 2, 1])
def test_reduced_idct_matches_a_64_bit_transcription_on_valid_range_blocks(s):
    rng = np.random.default_rng(10 + s)
    coef = _test_blocks(rng, 400, -1024, 1024)
    qt = rng.integers(1, 16, 64).astype(np.int32)
    for q in (qt, util.std_qt(False, 50)):
        want = reduced_blocks_ref(coef, q, s)
        assert np.array_equal(scaled_blocks(coef, q, s), want)
        assert np.array_equal(reduced_blocks_ref(coef, q, s, bits=32), want)


@pytest.mark.parametrize("s", [4, 2, 1])
def test_reduced_idct_dc_only_and_shortcut_blocks(s):
    """DC-only blocks are one value, range_limit[DESCALE(DC q, 3)] (= DESCALE(4 DC q, 5)); a coefficient in a row the transform
    never reads (row 4 at 1/2, rows 2, 4, 6 at 1/4) changes nothing, not even which shortcut is taken"""
    qt = np.full(64, 3, np.int32)
    qt[0] = 8
    for dc, want in [(0, 128), (1, 129), (-1, 127), (127, 255), (-128, 0), (4000, 32), (-4000, 224)]:
        blk = np.zeros((1, 64), np.int16)
        blk[0, 0] = dc
        assert (scaled_blocks(blk, qt, s) == want).all() and (reduced_blocks_ref(blk, qt, s) == want).all(), (s, dc)
    if s > 1:
        rng = np.random.default_rng(30 + s)
        coef = rng.integers(-200, 200, (50, 64)).astype(np.int16)
        unread = [4] if s == 4 else [2, 4, 6]
        moved = coef.reshape(-1, 8, 8).copy()
        moved[:, unread, :] = rng.integers(-200, 200, (50, len(unread), 8))
        moved[:, :, unread] = 0
        base = coef.reshape(-1, 8, 8).copy()
        base[:, :, unread] = 0
        assert np.array_equal(scaled_blocks(base.reshape(-1, 64), qt, s), scaled_blocks(moved.reshape(-1, 64), qt, s))


@pytest.mark.parametrize("s", [4, 2, 1])
def test_reduced_idct_wraps_like_jidctred_with_32_bit_jlong(s):
    """The whole int16 range with every table entry up to 255, many columns and rows without AC: the 32-bit statement is
    jidctred.c with a 32-bit JLONG, both shortcuts included"""
    rng = np.random.default_rng(40 + s)
    coef = rng.integers(-32768, 32768, (300, 64)).astype(np.int16).reshape(-1, 8, 8)
    coef[:, 1:, :] *= (rng.random((300, 1, 8)) < 0.5).astype(np.int16)
    coef[:, :, 1:] *= (rng.random((300, 8, 1)) < 0.7).astype(np.int16)
    coef = coef.reshape(-1, 64)
    qt = rng.integers(0, 256, 64)
    assert np.array_equal(scaled_blocks(coef, qt, s), reduced_blocks_ref(coef, qt, s, bits=32))


@pytest.mark.parametrize("case", DRAFT_INPUTS)
def test_statement_equals_pillow_draft(case):
    """The claim of the scaled mode: the statement on the host stage's planes is Pillow's draft, byte for byte, RGB and L"""
    data, gray = _draft_input(case)
    compared = 0
    for out_gray in ((True,) if gray else (False, True)):
        for d in DENOMS:
            want = _pillow_draft(data, d, out_gray)
            if want is None:
                continue
            img, planes = scaled_decoder(d, ColorSpace.GRAYSCALE if out_gray else ColorSpace.RGB).decode_coefficients(data)
            assert img.flags & _ffi.FLAG_SCALE_MASK == (d.bit_length() - 1) << _ffi.FLAG_SCALE_SHIFT
            got = scaled_expected(img, planes).reshape(want.shape)
            assert int(np.abs(got.astype(np.int16) - want).max()) == 0, (d, out_gray, int(np.count_nonzero(got != want)))
            compared += 1
    assert compared >= 1


def test_draft_scale_restates_pillow():
    for (w, h, size) in [(4000, 3000, (224, 224)), (4000, 3000, (500, 500)), (4000, 3000, (1000, 1000)), (4000, 3000, (2000, 2000)),
                         (4000, 3000, (3000, 3000)), (100, 7, (50, 1)), (37, 29, (4, 4))]:
        d, size_d = draft_scale(w, h, size)
        im = Image.new("RGB", (w, h))
        buf = io.BytesIO()
        im.save(buf, "JPEG")
        p = Image.open(io.BytesIO(buf.getvalue()))
        p.draft("RGB", size)
        assert p.size == size_d == _ffi.scaled_size(w, h, d), (w, h, size, d)


def _scaled_image(w, h, planes, hs, vs, cs, d, n_comp=3, qts=QTS):
    img = util.make_image(w, h, planes, qts[:n_comp], hs, vs, cs, SPEC)
    img.flags = _flags(d)
    return img


def test_abi_flags_sizes_and_shapes():
    lib = _ffi.load()
    rng = np.random.default_rng(2)
    planes = spec_planes(rng, 41, 23, 3, 2, 2)
    img = _scaled_image(41, 23, planes, 2, 2, _ffi.CS_RGBA, 4)
    assert lib.zj_validate_image(C.byref(img)) == 0
    assert lib.zj_output_size(C.byref(img)) == 11 * 6 * 4
    desc = _ffi.ZjOutputDesc()
    lib.zj_output_desc_default(C.byref(desc))
    desc.channels, desc.dtype = 3, _ffi.DTYPE_F32
    ow, oh, oc = C.c_uint32(), C.c_uint32(), C.c_uint32()
    assert lib.zj_consumer_output_shape(C.byref(img), C.byref(desc), C.byref(ow), C.byref(oh), C.byref(oc)) == 0
    assert (ow.value, oh.value, oc.value) == (11, 6, 3)
    assert lib.zj_consumer_output_size(C.byref(img), C.byref(desc)) == 11 * 6 * 3 * 4
    for d, size in ((2, (21, 12)), (8, (6, 3))):
        img.flags = _flags(d)
        assert lib.zj_output_size(C.byref(img)) == size[0] * size[1] * 4
    # rows are the scaled image's: the whole image comes back for any rows inside it
    sub, row0 = _ffi.ZjImage(), C.c_uint32()
    assert lib.zj_image_rows(C.byref(img), 1, 3, C.byref(sub), C.byref(row0)) == 0 and row0.value == 1 and sub.height == 23
    assert lib.zj_image_rows(C.byref(img), 1, 4, C.byref(sub), C.byref(row0)) == _ffi.ERR_INVALID_ARG
    # a scale needs ZJ_VARIANT_SPEC | ZJ_FLAG_ISLOW
    img.flags = 1 << _ffi.FLAG_SCALE_SHIFT
    assert lib.zj_validate_image(C.byref(img)) == _ffi.ERR_INVALID_ARG and lib.zj_output_size(C.byref(img)) == 0
    for variant in (_ffi.VARIANT_X86, _ffi.VARIANT_SCALAR):
        img.variant = variant
        img.flags = 3 << _ffi.FLAG_SCALE_SHIFT
        assert lib.zj_validate_image(C.byref(img)) == _ffi.ERR_INVALID_ARG
        img.flags = 0
        assert lib.zj_validate_image(C.byref(img)) == 0
    # strip cuts are refused, as for every spec image
    img.variant, img.flags = SPEC, _flags(2)
    off, nb = C.c_size_t(), C.c_size_t()
    assert lib.zj_image_strip_range(C.byref(img), 0, 1, C.byref(sub), C.byref(off), C.byref(nb), None) == _ffi.ERR_UNSUPPORTED


@pytest.mark.parametrize("data", [jpeg_util.synth_jpeg(1, 637, 480, "420", 90), jpeg_util.synth_jpeg(2, 333, 250, "422", 95, restart_rows=1),
                                  jpeg_util.synth_jpeg(3, 301, 203, "444", 90, progressive=True), jpeg_util.synth_jpeg(4, 99, 45, gray=True)],
                         ids=["420", "422_restart", "444_progressive", "gray"])
def test_host_stage_is_the_libjpeg_host_stage(data):
    """use_unsafe = 3 | k << 4 gives the libjpeg decode's descriptor and planes, with the scale bits set"""
    l_img, l_planes = libjpeg_decoder().decode_coefficients(data)
    for d in DENOMS:
        s_img, s_planes = scaled_decoder(d).decode_coefficients(data)
        assert s_img.variant == l_img.variant == SPEC
        assert s_img.flags == l_img.flags | (d.bit_length() - 1) << _ffi.FLAG_SCALE_SHIFT
        assert (s_img.width, s_img.height, s_img.n_comp, s_img.out_cs) == (l_img.width, l_img.height, l_img.n_comp, l_img.out_cs)
        assert len(l_planes) == len(s_planes) and all(np.array_equal(a, b) for a, b in zip(l_planes, s_planes))
    # every other use_unsafe value keeps its meaning: 0x12 and 0x43 are truthy, i.e. the X86 variant, without a scale
    for v in (0x12, 0x43, 0x03 | 4 << 4):
        o = _ffi.ZjOptions()
        _ffi.load().zj_options_default(C.byref(o))
        o.use_unsafe = v
        dec = Decoder.new_with_options(ZuneJpegOptions())
        _ffi.load().zj_decoder_free(dec._h)
        dec._h = _ffi.load().zj_decoder_new(C.byref(o))
        img, _ = dec.decode_coefficients(data)
        assert img.variant == _ffi.VARIANT_X86 and img.flags & (_ffi.FLAG_SCALE_MASK | ISLOW) == 0, hex(v)


def test_options_builder():
    o = ZuneJpegOptions()
    assert o.get_scale_denom() == 1
    lj = o.set_libjpeg_output(True)
    for d in (1, 2, 4, 8):
        s = lj.set_scale_denom(d)
        assert s.get_scale_denom() == d and lj.get_scale_denom() == 1
        assert s._raw().use_unsafe == _ffi.USE_LIBJPEG_OUTPUT | (d.bit_length() - 1) << 4
    assert [lj.set_scale_denom(d)._raw().use_unsafe for d in (2, 4, 8)] == [0x13, 0x23, 0x33]
    for bad in (0, 3, 16, -2, 1.5):
        with pytest.raises(ValueError):
            o.set_scale_denom(bad)
    with pytest.raises(ValueError):                           # d > 1 without libjpeg output: refused when the options are used
        o.set_scale_denom(4)._raw()
    with pytest.raises(ValueError):
        Decoder.new_with_options(o.set_spec_output(True).set_scale_denom(2))
    assert o.set_scale_denom(1)._raw().use_unsafe == 1


# ------------------------------------------------------------------------------------------------ GPU
def _host_images(rng, cases, mode, cs_list, d, n_comp=3, extreme_every=3):
    hs, vs = MODES[mode]
    imgs, keep, wants = [], [], []
    for k, (w, h) in enumerate(cases):
        planes = spec_planes(rng, w, h, n_comp, hs, vs, extreme=(k % extreme_every == 0))
        img = _scaled_image(w, h, planes, hs, vs, cs_list[k % len(cs_list)], d, n_comp)
        imgs.append(img); keep.append(planes); wants.append(scaled_expected(img, planes))
    return imgs, keep, wants


@pytest.mark.gpu
@pytest.mark.parametrize("d", DENOMS)
@pytest.mark.parametrize("mode", list(MODES))
def test_reconstruct_host_entry_matches_statement(mode, d):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(1000 + 10 * list(MODES).index(mode) + d)
    cases = _cases(mode, list(MODES).index(mode) + d)
    for cs in COLOR_CS:
        imgs, keep, wants = _host_images(rng, cases, mode, [cs], d)
        for (w, h), g, want in zip(cases, gpu.reconstruct(imgs, device=0), wants):
            assert np.array_equal(g, want), (mode, d, cs, w, h, int(np.count_nonzero(g != want)))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("use_batch", [False, True])
def test_reconstruct_device_and_batch_match_statement(mode, use_batch):
    rng = np.random.default_rng(1100 + list(MODES).index(mode))
    for d in DENOMS:
        cases = [c for c in _cases(mode, 3 + d) if c[0] * c[1] <= 640 * 2160]
        imgs, keep, wants = _host_images(rng, cases, mode, COLOR_CS, d, extreme_every=2)
        for off in (0, 1):
            for (w, h), img, g, want in zip(cases, imgs, _device_run(imgs, keep, use_batch, off), wants):
                assert np.array_equal(g, want), (mode, d, use_batch, off, w, h, img.out_cs)


@pytest.mark.gpu
def test_gray_input():
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(1200)
    for d in DENOMS:
        cases = _cases("none", 5 + d)
        imgs, keep, wants = _host_images(rng, cases, "none", [_ffi.CS_GRAYSCALE, _ffi.CS_RGB, _ffi.CS_RGBA, _ffi.CS_RGBX], d, n_comp=1)
        for (w, h), img, g, want in zip(cases, imgs, gpu.reconstruct(imgs), wants):
            assert np.array_equal(g, want), (d, w, h, img.out_cs)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_wrapping_coefficients(mode):
    """the whole int16 range, table entries up to 255 and many columns and rows without AC, at every scale"""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(1300 + list(MODES).index(mode))
    hs, vs = MODES[mode]
    qts = [rng.integers(0, 256, 64).astype(np.int32) for _ in range(3)]
    imgs, keep, wants = [], [], []
    for k, (w, h) in enumerate([(333, 97), (64, 64), (17, 130), (5, 3)]):
        planes = spec_planes(rng, w, h, 3, hs, vs, extreme=True, dc_only_frac=0.1)
        for p in planes:
            b = p.reshape(-1, 8, 8)
            b[:, 1:, :] *= (rng.random((b.shape[0], 1, 8)) < 0.5).astype(np.int16)
            b[:, :, 1:] *= (rng.random((b.shape[0], 8, 1)) < 0.7).astype(np.int16)
        for d in DENOMS:
            img = _scaled_image(w, h, planes, hs, vs, COLOR_CS[(k + d) % len(COLOR_CS)], d, qts=qts)
            imgs.append(img); keep.append(planes); wants.append(scaled_expected(img, planes))
    for img, g, want in zip(imgs, gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want), (mode, img.width, img.height, img.flags)


@pytest.mark.gpu
def test_mixed_call_with_every_kind_of_image():
    """One call with X86, spec, spec + islow and all three scales, colour and grey output: each launch group its own kernel"""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(1400)
    imgs, keep, wants = [], [], []
    shapes = [(640, 362, "hv", 0), (333, 250, "h", 0), (255, 33, "v", 2), (100, 17, "none", 5), (640, 362, "hv", 5), (17, 9, "hv", 1),
              (637, 480, "hv", 0), (99, 45, "none", 1), (321, 40, "h", 1), (256, 64, "hv", 1), (31, 200, "v", 0), (1023, 77, "hv", 6)]
    for k, (w, h, mode, cs) in enumerate(shapes * 2):
        hs, vs = MODES[mode]
        kind = k % 6                      # 0: X86, 1: spec, 2: spec + islow, 3-5: scaled 1/2, 1/4, 1/8
        planes = spec_planes(rng, w, h, 3, hs, vs)
        img = util.make_image(w, h, planes, QTS, hs, vs, cs, SPEC if kind else _ffi.VARIANT_X86)
        img.flags = 0 if kind < 2 else (ISLOW if kind == 2 else _flags(1 << (kind - 2)))
        imgs.append(img); keep.append(planes)
        wants.append(oracle.reconstruct(img) if kind == 0 else (spec_expected if kind == 1 else scaled_expected)(img, planes))
    for use_batch in (False, True):
        for g, want, img in zip(_device_run(imgs, keep, use_batch), wants, imgs):
            assert np.array_equal(g, want), (img.width, img.height, img.variant, img.flags)
    for g, want in zip(gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want)
    if gpu.device_count() >= 2:
        # one scaled image on two devices (it cannot be cut into strip ranges: whole), then the whole call
        for g, want in zip(gpu.reconstruct_multi(imgs[4:5], [0, 1]) + gpu.reconstruct_multi(imgs, [0, 1]), wants[4:5] + wants):
            assert np.array_equal(g, want)


def _draft_datas():
    return [_draft_input(p.values[0]) for p in DRAFT_INPUTS]


@pytest.mark.gpu
@pytest.mark.parametrize("d", DENOMS)
def test_jpeg_bytes_equal_pillow_draft(d):
    """JPEG bytes in, Pillow's draft bytes out, through decode_buffer, decode_into and decode_batch (one and two devices)"""
    from zune_jpeg_b200 import gpu
    datas = _draft_datas()
    rgb = ZuneJpegOptions().set_libjpeg_output(True).set_scale_denom(d)
    n = 0
    for data, gray in datas:
        want = _pillow_draft(data, d, gray)
        if want is None:
            continue
        o = rgb.set_out_colorspace(ColorSpace.GRAYSCALE if gray else ColorSpace.RGB)
        assert Decoder.new_with_options(o).decode_buffer(data) == want.tobytes()
        buf = np.full(want.size + 7, 0xAB, np.uint8)
        assert Decoder.new_with_options(o).decode_into(data, buf) == want.size and buf[:want.size].tobytes() == want.tobytes()
        assert (buf[want.size:] == 0xAB).all()
        n += 1
    assert n >= 16
    blobs = [data for data, _ in datas]
    wants = [_pillow_draft(data, d) for data in blobs]
    for devices in (None, [0, 0]) if gpu.device_count() < 2 else (None, [0, 1]):
        got = decode_batch(blobs, rgb, threads=4, devices=devices)
        for g, w in zip(got, wants):
            if w is not None:
                assert g == w.tobytes(), devices


@pytest.mark.gpu
def test_device_plane_routes():
    """gpu.reconstruct_device_ex (f16 CHW) and gpu.reconstruct_device_resized on device planes of scaled images: sizes and rois
    are the scaled image's"""
    from zune_jpeg_b200 import gpu
    datas = [jpeg_util.synth_jpeg(1, 637, 480, "420", 90), jpeg_util.synth_jpeg(9, 350, 201, "422", 100),
             jpeg_util.synth_jpeg(8, 321, 199, "444", 90, gray=True)]
    keep, dimgs, wants = [], [], []
    for d, data in zip((2, 4, 8), datas):
        img, planes = scaled_decoder(d).decode_coefficients(data)
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b, p in zip(bufs, planes):
            b.upload(p)
        di = _ffi.ZjImage()
        C.memmove(C.byref(di), C.byref(img), C.sizeof(di))
        for z, b in enumerate(bufs):
            di.comp[z].coeff = b.ptr
        keep.append(bufs); dimgs.append(di)
        wants.append(_pillow_draft(data, d))
    gpu.synchronize()
    desc = gpu.OutputDesc("CHW", "f16", False, 0, (120.0, 110.0, 100.0, 0.0), (1 / 60, 1 / 57, 1 / 58, 1.0))
    for a, p in zip(gpu.reconstruct_device_ex(dimgs, desc), wants):
        gpu.synchronize()
        assert a.shape == (3, p.shape[0], p.shape[1])
        assert a.download().tobytes() == desc.expected(p.reshape(-1), p.shape[1], p.shape[0], 3).tobytes()
    for rz, rois in ((gpu.Resize((32, 40), "bilinear"), [(5, 100, 300, 140), None, (1, 2, 30, 20)]),
                     (gpu.Resize((24, 24), "pil_bicubic", short_side=24), None)):
        out = gpu.reconstruct_device_resized(dimgs, rz, desc, rois)
        gpu.synchronize()
        got = out.download()
        for k, p in enumerate(wants):
            roi = rois[k] if rois else None
            assert got[k].tobytes() == rz.expected(p.reshape(-1), p.shape[1], p.shape[0], 3, desc, roi).tobytes(), k


@pytest.mark.gpu
def test_batch_resized_equals_pillow_draft_then_torchvision():
    """The headline: decode_batch_resized with libjpeg output at 1/4 and pil_bicubic with short_side gives Pillow's draft followed
    by torchvision's Resize(S) + CenterCrop, byte for byte, on the same files"""
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import decode_batch_resized
    datas = [jpeg_util.synth_jpeg(1, 1280, 960, "420", 90), jpeg_util.synth_jpeg(2, 1111, 1500, "422", 85),
             jpeg_util.synth_jpeg(3, 1023, 770, "444", 95, progressive=True), ref_files.read(ref_files.NAMES[0])]
    datas = [d for d in datas if min(Image.open(io.BytesIO(d)).size) >= 4 * 64]
    S, size = 64, (56, 56)
    opts = ZuneJpegOptions().set_libjpeg_output(True).set_scale_denom(4)
    rz = gpu.Resize(size, "pil_bicubic", short_side=S)
    out, errs = decode_batch_resized(datas, rz, gpu.OutputDesc(), None, opts, threads=4)
    assert errs == [None] * len(datas)
    got = out.download()
    try:
        from torchvision.transforms import InterpolationMode, v2
    except Exception:
        v2 = None
    for k, data in enumerate(datas):
        im = Image.open(io.BytesIO(data))
        im.draft("RGB", (im.size[0] // 4, im.size[1] // 4))
        im = im.convert("RGB")
        w, h = im.size
        rw, rh, left, top = gpu.pil_geometry(w, h, size[1], size[0], S)
        want = np.asarray(im.resize((rw, rh), Image.BICUBIC).crop((left, top, left + size[1], top + size[0])))
        assert got[k].tobytes() == want.tobytes(), k
        if v2 is not None:
            tv = np.asarray(v2.Compose([v2.Resize(S, interpolation=InterpolationMode.BICUBIC), v2.CenterCrop(size)])(im))
            assert got[k].tobytes() == tv.tobytes(), k
