"""libjpeg-turbo-exact output (ZJ_VARIANT_SPEC with ZJ_FLAG_ISLOW, ZuneJpegOptions.set_libjpeg_output): the spec-correct output
of tests/test_spec_output.py with libjpeg-turbo's islow IDCT (jidctint.c) in place of the X86 IDCT.  The statement is in
include/zune_jpeg_b200.h; libjpeg_expected() below restates it in numpy, and every GPU result is compared with it bit for bit.
The CPU part checks the statement on the host stage's planes against Pillow at tolerance 0, the IDCT against an independent
64-bit transcription, and the C ABI; it launches nothing."""
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
from test_spec_output import SYNTH, _cases, _device_run, _upsample, spec_expected, spec_planes
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch

SPEC, ISLOW = _ffi.VARIANT_SPEC, _ffi.FLAG_ISLOW
MODES = {"none": (1, 1), "h": (2, 1), "v": (1, 2), "hv": (2, 2)}
QTS = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]
COLOR_CS = [_ffi.CS_RGB, _ffi.CS_RGBA, _ffi.CS_RGBX, _ffi.CS_YCBCR, _ffi.CS_GRAYSCALE]


# ------------------------------------------------------------------------------------------------ the statement in numpy
def _islow_1d(s, bias, sh):
    """one 1-D pass of jpeg_idct_islow (jidctint.c, CONST_BITS 13) along the last axis of an int32 array, wrapping; the
    DESCALE rounding `bias` is added before the arithmetic shift by `sh`"""
    i32 = np.int32
    s0, s1, s2, s3, s4, s5, s6, s7 = (s[..., k] for k in range(8))
    z1 = (s2 + s6) * i32(4433)                                  # FIX_0_541196100
    tmp2 = z1 + s6 * i32(-15137)                                # - FIX_1_847759065
    tmp3 = z1 + s2 * i32(6270)                                  # FIX_0_765366865
    tmp0 = (s0 + s4) << i32(13)
    tmp1 = (s0 - s4) << i32(13)
    tmp10, tmp13, tmp11, tmp12 = tmp0 + tmp3, tmp0 - tmp3, tmp1 + tmp2, tmp1 - tmp2
    o0, o1, o2, o3 = s7, s5, s3, s1
    z1, z2, z3, z4 = o0 + o3, o1 + o2, o0 + o2, o1 + o3
    z5 = (z3 + z4) * i32(9633)                                  # FIX_1_175875602
    o0, o1, o2, o3 = o0 * i32(2446), o1 * i32(16819), o2 * i32(25172), o3 * i32(12299)
    z1, z2 = z1 * i32(-7373), z2 * i32(-20995)
    z3, z4 = z3 * i32(-16069) + z5, z4 * i32(-3196) + z5
    o0, o1, o2, o3 = o0 + z1 + z3, o1 + z2 + z4, o2 + z2 + z3, o3 + z1 + z4
    out = np.stack([tmp10 + o3, tmp11 + o2, tmp12 + o1, tmp13 + o0, tmp13 - o0, tmp12 - o1, tmp11 - o2, tmp10 - o3], -1)
    return (out + bias) >> i32(sh)


def range_limit(v):
    """jdmaster.c's range_limit[v & 1023] (the level shift included)"""
    v = np.asarray(v) & 1023
    return np.where(v < 128, v + 128, np.where(v < 512, 255, np.where(v < 896, 0, v - 896))).astype(np.uint8)


def islow_blocks(coef, qt):
    """coef int16 [N, 64] natural order, qt [64] -> uint8 [N, 8, 8]: jpeg_idct_islow in 32-bit wrapping arithmetic, the
    pass-1 shortcut for columns whose AC coefficients are zero as jidctint.c takes it"""
    with np.errstate(over="ignore"):
        c = coef.reshape(-1, 8, 8)
        d = c.astype(np.int32) * np.asarray(qt, np.int32).reshape(8, 8)
        cols = d.transpose(0, 2, 1)                                             # [N, column, row]
        ws = _islow_1d(cols, np.int32(1 << 10), 11)                             # DESCALE(x, CONST_BITS - PASS1_BITS)
        dc_only = ~np.any(c[:, 1:, :] != 0, axis=1)                             # [N, column]
        ws = np.where(dc_only[..., None], (cols[..., :1] << np.int32(2)), ws)  # dcval = DEQUANTIZE(...) << PASS1_BITS
        out = _islow_1d(ws.transpose(0, 2, 1), np.int32(1 << 17), 18)          # DESCALE(x, CONST_BITS + PASS1_BITS + 3)
        return range_limit(out)                                                 # (the row shortcut gives the same values)


def islow_blocks_ref(coef, qt, bits=None):
    """an independent transcription of jpeg_idct_islow, block by block with Python integers, both zero-AC shortcuts taken as
    jidctint.c takes them.  bits=None: JLONG wide enough for every intermediate (64 bits, for 8-bit JPEG data); bits=32: JLONG
    and int of 32 bits, wrapping (only the shifts see the wrap: +, - and * are exact modulo 2^32)."""
    def wrap(x):
        if bits is None:
            return x
        x &= (1 << bits) - 1
        return x - (1 << bits) if x >> (bits - 1) else x

    def descale(x, n):
        return wrap(x + (1 << (n - 1))) >> n

    def one_d(s, p):
        z1 = (s[2] + s[6]) * 4433
        t2, t3 = z1 - s[6] * 15137, z1 + s[2] * 6270
        t0, t1 = (s[0] + s[4]) << 13, (s[0] - s[4]) << 13
        t10, t13, t11, t12 = t0 + t3, t0 - t3, t1 + t2, t1 - t2
        a0, a1, a2, a3 = s[7], s[5], s[3], s[1]
        z1, z2, z3, z4 = a0 + a3, a1 + a2, a0 + a2, a1 + a3
        z5 = (z3 + z4) * 9633
        a0, a1, a2, a3 = a0 * 2446, a1 * 16819, a2 * 25172, a3 * 12299
        z1, z2, z3, z4 = -z1 * 7373, -z2 * 20995, -z3 * 16069 + z5, -z4 * 3196 + z5
        a0 += z1 + z3
        a1 += z2 + z4
        a2 += z2 + z3
        a3 += z1 + z4
        return [descale(v, p) for v in (t10 + a3, t11 + a2, t12 + a1, t13 + a0, t13 - a0, t12 - a1, t11 - a2, t10 - a3)]

    out = np.zeros((coef.shape[0], 8, 8), np.uint8)
    q = [int(x) for x in np.asarray(qt).reshape(64)]
    for n, blk in enumerate(coef.reshape(-1, 64)):
        b = [int(x) for x in blk]
        ws = [[0] * 8 for _ in range(8)]
        for col in range(8):
            if all(b[8 * r + col] == 0 for r in range(1, 8)):
                for r in range(8):
                    ws[r][col] = wrap((b[col] * q[col]) << 2)
                continue
            res = one_d([b[8 * r + col] * q[8 * r + col] for r in range(8)], 11)
            for r in range(8):
                ws[r][col] = res[r]
        for r in range(8):
            if all(ws[r][k] == 0 for k in range(1, 8)):
                out[n, r, :] = range_limit(descale(ws[r][0], 5))
            else:
                out[n, r, :] = range_limit(one_d(ws[r], 18))
    return out


def _component(img, planes, z):
    c = img.comp[z]
    s = islow_blocks(planes[z].reshape(-1, 64), np.array(c.qt, np.int32))
    return ref_model.plane_from_blocks(s, c.width_stride // 8).astype(np.int32)


def libjpeg_expected(img, planes) -> np.ndarray:
    """The statement of ZJ_VARIANT_SPEC | ZJ_FLAG_ISLOW: the width * height * nc bytes the output must hold.  Steps 2-5 are
    spec_expected's (test_spec_output.py); step 1 is islow_blocks."""
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


def libjpeg_decoder(cs=ColorSpace.RGB, threads=4):
    return Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(cs).set_libjpeg_output(True).set_num_threads(threads))


def _pillow(data, gray=False):
    return np.asarray(Image.open(io.BytesIO(data)).convert("L" if gray else "RGB"))


def _synth(case):
    seed, w, h, sub, q, prog, gray = case
    return jpeg_util.synth_jpeg(seed, w, h, sub, q, prog, gray), gray


INPUTS = [pytest.param(c, id="synth%d" % c[0]) for c in SYNTH] + [pytest.param(n, id=n) for n in ref_files.NAMES]


def _input(case):
    return _synth(case) if isinstance(case, tuple) else (ref_files.read(case), False)


# ------------------------------------------------------------------------------------------------ CPU
def test_range_limit_table():
    assert range_limit([0, 127, 128, 511, 512, 895, 896, 1023, 1024, -1]).tolist() == [128, 255, 255, 255, 0, 0, 0, 127, 128, 127]


def test_islow_dc_only_blocks_by_hand():
    """All AC zero: every sample is range_limit[(4 * DC * q + 16) >> 5], i.e. DC * q / 8 + 128 rounded half up, then clipped."""
    qt = np.full(64, 1, np.int32)
    qt[0] = 8                                        # DC * 8 / 8 = DC
    # beyond +-128 the 10-bit table index wraps: 4000 & 1023 = 928 -> 928 - 896 = 32
    for dc, want in [(0, 128), (1, 129), (-1, 127), (3, 131), (16, 144), (127, 255), (128, 255), (-16, 112), (-128, 0),
                     (-200, 0), (4000, 32), (-4000, 224)]:
        blk = np.zeros((1, 64), np.int16)
        blk[0, 0] = dc
        assert (islow_blocks(blk, qt) == want).all() and (islow_blocks_ref(blk, qt) == want).all(), dc


def test_islow_matches_a_64_bit_transcription_on_valid_range_blocks():
    """Blocks of an 8-bit JPEG (dequantised values within +-2^14, where no intermediate leaves 32 bits): the 32-bit wrapping
    form equals jidctint.c with a 64-bit JLONG, and both shortcuts are exercised (DC-only blocks, columns and rows)."""
    rng = np.random.default_rng(5)
    n = 600
    coef = np.zeros((n, 64), np.int16)
    for k in range(n):
        kind = k % 4
        if kind == 0:
            coef[k] = rng.integers(-64, 64, 64)
        elif kind == 1:                              # sparse low frequencies
            m = rng.random(64) < 0.2
            coef[k][m] = rng.integers(-200, 200, int(m.sum()))
        elif kind == 2:                              # some columns with AC, the rest DC-only columns
            b = np.zeros((8, 8), np.int16)
            b[0] = rng.integers(-1000, 1000, 8)
            for col in rng.choice(8, 3, replace=False):
                b[1:, col] = rng.integers(-30, 30, 7)
            coef[k] = b.reshape(64)
        coef[k, 0] = rng.integers(-1024, 1024)
    qt = rng.integers(1, 16, 64).astype(np.int32)
    assert np.abs(coef.astype(np.int64) * qt).max() < (1 << 15)
    for q in (qt, util.std_qt(False, 50)):
        want = islow_blocks_ref(coef, q)
        assert np.array_equal(islow_blocks(coef, q), want) and np.array_equal(islow_blocks_ref(coef, q, bits=32), want)


def test_islow_wraps_like_jidctint_with_32_bit_jlong():
    """Outside the range of 8-bit JPEG data the statement is jidctint.c with a 32-bit JLONG, wrapping.  A column whose AC is
    zero takes the pass-1 shortcut: with a dequantised DC of 2^18 or more the full 32-bit pass would wrap where the shortcut
    does not, so the shortcut is part of the statement (the pass-2 shortcut never differs from the full pass)."""
    blk = np.zeros((1, 64), np.int16)
    blk[0, 0:8] = [32000, -32000, 30000, 1200, -1500, 2000, 31000, -29000]
    blk[0, 8 + 1] = 5                                # column 1 has AC, every other column is DC-only
    qt = np.full(64, 255, np.int32)
    d = blk.reshape(8, 8).astype(np.int32) * qt.reshape(8, 8)
    with np.errstate(over="ignore"):
        full = _islow_1d(d.T[None].astype(np.int32), np.int32(1 << 10), 11)[0]   # [column, row], no shortcut
    assert full[2, 0] != d[0, 2] << 2                  # the full form wraps ...
    assert np.array_equal(islow_blocks(blk, qt), islow_blocks_ref(blk, qt, bits=32))   # ... the shortcut is taken as in jidctint.c
    rng = np.random.default_rng(6)                      # whole int16 range, any table entry, columns and rows without AC
    coef = rng.integers(-32768, 32768, (300, 64)).astype(np.int16).reshape(-1, 8, 8)
    coef[:, 1:, :] *= (rng.random((300, 1, 8)) < 0.5).astype(np.int16)
    coef[:, :, 1:] *= (rng.random((300, 8, 1)) < 0.7).astype(np.int16)
    coef = coef.reshape(-1, 64)
    qt = rng.integers(0, 256, 64)
    assert np.array_equal(islow_blocks(coef, qt), islow_blocks_ref(coef, qt, bits=32))


@pytest.mark.parametrize("case", INPUTS)
def test_statement_equals_pillow(case):
    """The claim of the mode: the statement on the host stage's libjpeg-mode planes is Pillow's decode, byte for byte."""
    data, gray = _input(case)
    img, planes = libjpeg_decoder(ColorSpace.GRAYSCALE if gray else ColorSpace.RGB).decode_coefficients(data)
    assert img.variant == SPEC and img.flags & ISLOW
    ref = _pillow(data, gray)
    got = libjpeg_expected(img, planes).reshape(ref.shape)
    assert int(np.abs(got.astype(np.int16) - ref).max()) == 0, int(np.count_nonzero(got != ref))


def test_abi_flag_and_options():
    lib = _ffi.load()
    rng = np.random.default_rng(2)
    planes = spec_planes(rng, 40, 24, 3, 2, 2)
    img = util.make_image(40, 24, planes, QTS, 2, 2, _ffi.CS_RGB, SPEC)
    img.flags = ISLOW
    assert lib.zj_validate_image(C.byref(img)) == 0
    img.flags = ISLOW | _ffi.FLAG_PROGRESSIVE
    assert lib.zj_validate_image(C.byref(img)) == 0
    for variant in (_ffi.VARIANT_X86, _ffi.VARIANT_SCALAR):           # the flag belongs to the spec statement only
        img.variant = variant
        img.flags = ISLOW
        assert lib.zj_validate_image(C.byref(img)) == _ffi.ERR_INVALID_ARG
        img.flags = 0
        assert lib.zj_validate_image(C.byref(img)) == 0
    # strip ranges: the query form works, every cut is refused, as for spec images
    planes = spec_planes(rng, 640, 362, 3, 2, 2)
    img = util.make_image(640, 362, planes, QTS, 2, 2, _ffi.CS_RGB, SPEC)
    img.flags = ISLOW
    ns = C.c_uint32()
    assert lib.zj_image_strip_range(C.byref(img), 0, 0, None, None, None, C.byref(ns)) == 0 and ns.value == 12
    sub = _ffi.ZjImage()
    off, nb = C.c_size_t(), C.c_size_t()
    for s0, s1 in ((0, 12), (0, 6), (6, 12)):
        assert lib.zj_image_strip_range(C.byref(img), s0, s1, C.byref(sub), C.byref(off), C.byref(nb), None) == _ffi.ERR_UNSUPPORTED
    # the options: by value, use_unsafe = ZJ_USE_LIBJPEG_OUTPUT, whatever else is set
    o = ZuneJpegOptions()
    assert o.get_libjpeg_output() is False
    s = o.set_libjpeg_output(True)
    assert s.get_libjpeg_output() is True and o.get_libjpeg_output() is False
    assert s._raw().use_unsafe == _ffi.USE_LIBJPEG_OUTPUT == 3
    assert s.set_use_unsafe(False)._raw().use_unsafe == 3 and s.set_spec_output(True)._raw().use_unsafe == 3
    assert s.set_libjpeg_output(False)._raw().use_unsafe == 1
    assert s.set_spec_output(True).set_libjpeg_output(False)._raw().use_unsafe == _ffi.USE_SPEC_OUTPUT


@pytest.mark.parametrize("data", [jpeg_util.synth_jpeg(1, 637, 480, "420", 90), jpeg_util.synth_jpeg(2, 333, 250, "422", 95, restart_rows=1),
                                  jpeg_util.synth_jpeg(3, 301, 203, "444", 90, progressive=True), jpeg_util.synth_jpeg(4, 99, 45, gray=True)],
                         ids=["420", "422_restart", "444_progressive", "gray"])
def test_host_stage_is_the_spec_host_stage(data):
    """use_unsafe = 3 gives the spec decode's descriptor and planes, with ZJ_FLAG_ISLOW set"""
    s_img, s_planes = Decoder.new_with_options(ZuneJpegOptions().set_spec_output(True)).decode_coefficients(data)
    l_img, l_planes = libjpeg_decoder().decode_coefficients(data)
    assert l_img.variant == s_img.variant == SPEC
    assert l_img.flags == s_img.flags | ISLOW and not s_img.flags & ISLOW
    assert (l_img.width, l_img.height, l_img.n_comp, l_img.out_cs) == (s_img.width, s_img.height, s_img.n_comp, s_img.out_cs)
    assert len(l_planes) == len(s_planes) and all(np.array_equal(a, b) for a, b in zip(l_planes, s_planes))


# ------------------------------------------------------------------------------------------------ GPU
def _islow_image(w, h, planes, hs, vs, cs, n_comp=3):
    img = util.make_image(w, h, planes, QTS[:n_comp], hs, vs, cs, SPEC)
    img.flags = ISLOW
    return img


def _host_images(rng, cases, mode, cs_list, n_comp=3, extreme_every=3):
    hs, vs = MODES[mode]
    imgs, keep, wants = [], [], []
    for k, (w, h) in enumerate(cases):
        planes = spec_planes(rng, w, h, n_comp, hs, vs, extreme=(k % extreme_every == 0))
        img = _islow_image(w, h, planes, hs, vs, cs_list[k % len(cs_list)], n_comp)
        imgs.append(img); keep.append(planes); wants.append(libjpeg_expected(img, planes))
    return imgs, keep, wants


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_reconstruct_host_entry_matches_statement(mode):
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(500 + list(MODES).index(mode))
    cases = _cases(mode, list(MODES).index(mode))
    for cs in COLOR_CS:
        imgs, keep, wants = _host_images(rng, cases, mode, [cs])
        for (w, h), g, want in zip(cases, gpu.reconstruct(imgs, device=0), wants):
            assert np.array_equal(g, want), (mode, cs, w, h, int(np.count_nonzero(g != want)))


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("use_batch", [False, True])
def test_reconstruct_device_and_batch_match_statement(mode, use_batch):
    rng = np.random.default_rng(600 + list(MODES).index(mode))
    cases = [c for c in _cases(mode, 3 + list(MODES).index(mode)) if c[0] * c[1] <= 640 * 2160]
    imgs, keep, wants = _host_images(rng, cases, mode, COLOR_CS, extreme_every=2)
    for off in (0, 1):                                                          # 16-byte and byte-aligned outputs
        for (w, h), img, g, want in zip(cases, imgs, _device_run(imgs, keep, use_batch, off), wants):
            assert np.array_equal(g, want), (mode, use_batch, off, w, h, img.out_cs)


@pytest.mark.gpu
def test_gray_input():
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(700)
    cases = _cases("none", 5)
    imgs, keep, wants = _host_images(rng, cases, "none", [_ffi.CS_GRAYSCALE, _ffi.CS_RGB, _ffi.CS_RGBA, _ffi.CS_RGBX], n_comp=1)
    for (w, h), img, g, want in zip(cases, imgs, gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want), (w, h, img.out_cs)


@pytest.mark.gpu
@pytest.mark.parametrize("mode", list(MODES))
def test_wrapping_coefficients(mode):
    """The whole int16 range with every table entry up to 255, many columns and rows without AC: the 32-bit wrap and the pass-1
    shortcut for dequantised DCs beyond 2^18 (test_islow_wraps_like_jidctint_with_32_bit_jlong), on the GPU."""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(800 + list(MODES).index(mode))
    hs, vs = MODES[mode]
    qts = [rng.integers(0, 256, 64).astype(np.int32) for _ in range(3)]
    imgs, keep, wants = [], [], []
    for k, (w, h) in enumerate([(333, 97), (64, 64), (17, 130)]):
        planes = spec_planes(rng, w, h, 3, hs, vs, extreme=True, dc_only_frac=0.1)
        for p in planes:
            b = p.reshape(-1, 8, 8)
            b[:, 1:, :] *= (rng.random((b.shape[0], 1, 8)) < 0.5).astype(np.int16)
            b[:, :, 1:] *= (rng.random((b.shape[0], 8, 1)) < 0.7).astype(np.int16)
        img = util.make_image(w, h, planes, qts, hs, vs, COLOR_CS[k % len(COLOR_CS)] if k else _ffi.CS_GRAYSCALE, SPEC)
        img.flags = ISLOW
        imgs.append(img); keep.append(planes); wants.append(libjpeg_expected(img, planes))
    for (w, h), g, want in zip([(i.width, i.height) for i in imgs], gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want), (mode, w, h)


@pytest.mark.gpu
def test_mixed_x86_spec_and_islow_images_in_one_call():
    """One call with as-written, spec and libjpeg images, colour and grey output: each launch group gets its own IDCT."""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(900)
    imgs, keep, wants = [], [], []
    for k, (w, h, mode, cs) in enumerate([(640, 362, "hv", 0), (333, 250, "h", 0), (255, 33, "v", 2), (100, 17, "none", 5),
                                          (640, 362, "hv", 5), (17, 9, "hv", 1), (637, 480, "hv", 0), (99, 45, "none", 1),
                                          (640, 362, "hv", 0), (321, 40, "h", 1), (256, 64, "hv", 1)]):
        hs, vs = MODES[mode]
        kind = k % 3                                                          # 0: X86, 1: spec, 2: spec + islow
        planes = spec_planes(rng, w, h, 3, hs, vs)
        img = util.make_image(w, h, planes, QTS, hs, vs, cs, SPEC if kind else _ffi.VARIANT_X86)
        img.flags = ISLOW if kind == 2 else 0
        imgs.append(img); keep.append(planes)
        wants.append(oracle.reconstruct(img) if kind == 0 else (spec_expected if kind == 1 else libjpeg_expected)(img, planes))
    assert {(i.variant, i.flags, i.out_cs == 1) for i in imgs} >= {(SPEC, ISLOW, True), (SPEC, 0, True), (SPEC, ISLOW, False)}
    for use_batch in (False, True):
        for g, want, img in zip(_device_run(imgs, keep, use_batch), wants, imgs):
            assert np.array_equal(g, want), (img.width, img.height, img.variant, img.flags)
    for g, want in zip(gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want)


def _datas():
    return [_input(p.values[0]) for p in INPUTS]


@pytest.mark.gpu
def test_jpeg_bytes_equal_pillow():
    """All 16 inputs of the Pillow tests, JPEG bytes in, Pillow's bytes out, through every JPEG-bytes entry point."""
    datas = _datas()
    pil = [_pillow(d, gray) for d, gray in datas]
    rgb = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    opts = [rgb.set_out_colorspace(ColorSpace.GRAYSCALE) if gray else rgb for _, gray in datas]
    for (d, _), o, want in zip(datas, opts, pil):
        assert Decoder.new_with_options(o).decode_buffer(d) == want.tobytes()
        buf = np.full(want.size, 0xAB, np.uint8)
        assert Decoder.new_with_options(o).decode_into(d, buf) == want.size and buf.tobytes() == want.tobytes()
    # decode_batch: one options object for the batch; the grey JPEG of SYNTH keeps RGB = Y, Y, Y (Pillow's convert("RGB"))
    pil_rgb = [_pillow(d) for d, _ in datas]
    blobs = [d for d, _ in datas]
    for devices in (None, [0, 0]):
        got = decode_batch(blobs, rgb, threads=4, devices=devices)
        assert [g == w.tobytes() for g, w in zip(got, pil_rgb)] == [True] * len(blobs), devices


@pytest.mark.gpu
def test_decode_into_large_image_and_gpu_entropy_route():
    from zune_jpeg_b200 import gpu
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    data = jpeg_util.synth_jpeg(7, 2560, 1610, "420", 90, restart_rows=4)     # 4.1 MP, odd MCU-row count (101)
    want = _pillow(data)
    buf = gpu.PinnedBuffer(want.size)
    view = buf.array if hasattr(buf, "array") else np.ctypeslib.as_array((C.c_uint8 * want.size).from_address(buf.ptr))
    view[:] = 0xAB
    assert Decoder.new_with_options(opts).decode_into(data, view) == want.size and view.tobytes() == want.tobytes()
    # restart-marker files, which the GPU entropy route would take as written, go through the host stage
    dri = [jpeg_util.synth_jpeg(5, 640, 352, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(6, 640, 362, "420", 90, restart_rows=2)]
    stats = {}
    got = decode_batch(dri, opts, threads=4, gpu_entropy=True, stats=stats)
    assert stats["gpu_entropy"] == 0
    assert [g == _pillow(d).tobytes() for g, d in zip(got, dri)] == [True, True]


MEAN = (0.485 * 255, 0.456 * 255, 0.406 * 255, 0.0)
INV = (1 / (0.229 * 255), 1 / (0.224 * 255), 1 / (0.225 * 255), 1.0)


@pytest.mark.gpu
def test_consumers_equal_the_specification_on_pillow_pixels():
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import decode_batch_resized
    datas = [jpeg_util.synth_jpeg(1, 640, 362, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(2, 333, 250, "422", 90),
             jpeg_util.synth_jpeg(3, 257, 199, gray=True), jpeg_util.synth_jpeg(4, 500, 301, "444", 85)]
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True)
    pil = [_pillow(d) for d in datas]
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    outs = [gpu.DeviceBuffer(p.size * 2) for p in pil]
    stats = {}
    res = decode_batch(datas, opts, threads=4, device_out=[(o.ptr, o.nbytes) for o in outs], desc=desc, stats=stats)
    assert stats["gpu_entropy"] == 0
    for p, o, r in zip(pil, outs, res):
        assert r == o.nbytes
        assert o.download().tobytes() == desc.expected(p.reshape(-1), p.shape[1], p.shape[0], 3).tobytes()
    rz = gpu.Resize((96, 128), "area")
    rois = [(10, 20, 300, 200), None, (0, 0, 257, 199), (100, 1, 400, 300)]
    out, errs = decode_batch_resized(datas, rz, desc, rois, opts, threads=4)
    assert errs == [None] * 4
    got = out.download()
    for k, p in enumerate(pil):
        assert got[k].tobytes() == rz.expected(p.reshape(-1), p.shape[1], p.shape[0], 3, desc, rois[k]).tobytes(), k


@pytest.mark.gpu
def test_device_plane_routes():
    """gpu.reconstruct_device_ex (f16 CHW) and gpu.reconstruct_device_resized on device planes of libjpeg-mode images"""
    from zune_jpeg_b200 import gpu
    datas = [jpeg_util.synth_jpeg(1, 637, 480, "420", 90), jpeg_util.synth_jpeg(9, 350, 201, "422", 100),
             jpeg_util.synth_jpeg(8, 321, 199, "444", 90, gray=True)]
    keep, dimgs, pil = [], [], []
    for d in datas:
        img, planes = libjpeg_decoder().decode_coefficients(d)
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b, p in zip(bufs, planes):
            b.upload(p)
        di = _ffi.ZjImage()
        C.memmove(C.byref(di), C.byref(img), C.sizeof(di))
        for z, b in enumerate(bufs):
            di.comp[z].coeff = b.ptr
        keep.append(bufs); dimgs.append(di); pil.append(_pillow(d))
    gpu.synchronize()
    desc = gpu.OutputDesc("CHW", "f16", False, 0, MEAN, INV)
    for a, p in zip(gpu.reconstruct_device_ex(dimgs, desc), pil):
        gpu.synchronize()
        assert a.download().tobytes() == desc.expected(p.reshape(-1), p.shape[1], p.shape[0], 3).tobytes()
    rz = gpu.Resize((64, 80), "bilinear")
    rois = [(5, 300, 600, 170), None, (1, 2, 100, 100)]                           # a crop of the last rows, whole, the first
    out = gpu.reconstruct_device_resized(dimgs, rz, desc, rois)
    gpu.synchronize()
    got = out.download()
    for k, p in enumerate(pil):
        assert got[k].tobytes() == rz.expected(p.reshape(-1), p.shape[1], p.shape[0], 3, desc, rois[k]).tobytes(), k
