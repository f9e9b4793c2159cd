"""Three-component JPEGs with any sampling factors libjpeg accepts -- 4:1:1, 4:1:0, factors of 3, chroma above luma, chroma factors
that differ -- in spec and libjpeg output (DESIGN.md section 4.6.5): the statement of include/zune_jpeg_b200.h (next to
zj_decoder_jpeg_colorspace) restated in numpy, checked against Pillow 12.2 on the host stage's planes, and the GPU routes checked
against the statement and Pillow bit for bit.  Pillow cannot write these factors, so the file has its own small encoder."""
from __future__ import annotations

import ctypes as C
import io
import struct

import numpy as np
import pytest
from PIL import Image, ImageOps
from scipy.fft import dctn

import ref_model
from test_cmyk_output import cmyk_jpeg, pillow
from test_libjpeg_output import islow_blocks
from test_scaled_output import scaled_blocks
from test_spec_output import _upsample
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, DecodeErrors, Decoder, ZuneJpegOptions, decode_batch


# ------------------------------------------------------------------------------------------------ a small encoder
def _segments(data):
    """(marker byte, payload) of every marker segment before the first SOS"""
    out, p = [], 2
    while p + 4 <= len(data) and data[p] == 0xFF:
        m, n = data[p + 1], struct.unpack(">H", data[p + 2:p + 4])[0]
        out.append((m, data[p + 4:p + 2 + n]))
        if m == 0xDA:
            break
        p += 2 + n
    return out


def _tables(quality):
    """the quantisation tables (zigzag order) and Huffman tables ((class, id) -> (counts, symbols)) Pillow writes: Annex K's"""
    b = io.BytesIO()
    Image.new("RGB", (16, 16)).save(b, "JPEG", quality=quality)
    qt, huff = {}, {}
    for m, p in _segments(b.getvalue()):
        while m == 0xDB and p:
            qt[p[0] & 15], p = list(p[1:65]), p[65:]
        while m == 0xC4 and p:
            counts = list(p[1:17])
            n = sum(counts)
            huff[(p[0] >> 4, p[0] & 15)], p = (counts, list(p[17:17 + n])), p[17 + n:]
    return qt, huff


def _codes(counts, syms):
    code, k, out = 0, 0, {}
    for length in range(1, 17):
        for _ in range(counts[length - 1]):
            out[syms[k]] = (code, length)
            k += 1
            code += 1
        code <<= 1
    return out


ZIGZAG = [r * 8 + c for r, c in sorted(((r, c) for r in range(8) for c in range(8)),
                                       key=lambda p: (p[0] + p[1], p[0] if (p[0] + p[1]) % 2 else -p[0]))]


class _Bits:
    def __init__(self):
        self.out, self.acc, self.n = bytearray(), 0, 0

    def put(self, v, n):
        self.acc = (self.acc << n) | (v & ((1 << n) - 1))
        self.n += n
        while self.n >= 8:
            self.n -= 8
            byte = (self.acc >> self.n) & 0xFF
            self.out.append(byte)
            if byte == 0xFF:
                self.out.append(0)
        self.acc &= (1 << self.n) - 1

    def code(self, table, sym):
        self.put(*table[sym])

    def value(self, v):
        if v:
            self.put(v if v > 0 else v - 1, abs(v).bit_length())

    def flush(self):
        if self.n:
            self.put(0x7F, 8 - self.n)


def _ac(bits, table, zz):
    last = 0
    for k in np.flatnonzero(zz[1:]) + 1:
        v, run = int(zz[k]), int(k) - last - 1
        while run > 15:
            bits.code(table, 0xF0)
            run -= 16
        bits.code(table, run << 4 | abs(v).bit_length())
        bits.value(v)
        last = int(k)
    if last < 63:
        bits.code(table, 0x00)


def _component_blocks(seed, w, h, samp, quality):
    """smooth content with some texture per component at its own resolution, padded to the MCU grid, forward-DCT'd and quantised:
    [block rows, block columns, 64] in zigzag order per component"""
    rng = np.random.default_rng(seed)
    qt, _ = _tables(quality)
    hmax, vmax = max(s[0] for s in samp), max(s[1] for s in samp)
    mcu_x, mcu_y = -(-w // (8 * hmax)), -(-h // (8 * vmax))
    out = []
    for z, (hs, vs) in enumerate(samp):
        cw, ch = -(-w * hs // hmax), -(-h * vs // vmax)
        base = rng.integers(40, 216, (ch // 5 + 2, cw // 5 + 2), dtype=np.uint8)
        a = np.asarray(Image.fromarray(base).resize((cw, ch), Image.BILINEAR), np.float64)
        a = a + rng.integers(-10, 11, a.shape) + np.linspace(-20, 20, cw)[None, :]
        a = np.pad(a, ((0, mcu_y * vs * 8 - ch), (0, mcu_x * hs * 8 - cw)), mode="edge") - 128
        br, bc = a.shape[0] // 8, a.shape[1] // 8
        f = dctn(a.reshape(br, 8, bc, 8).transpose(0, 2, 1, 3), axes=(2, 3), norm="ortho").reshape(br, bc, 64)
        q = np.zeros(64)
        q[ZIGZAG] = qt[0 if z == 0 else 1]
        out.append(np.clip(np.rint(f / q), -1023, 1023).astype(np.int64)[..., ZIGZAG])
    return out


def jpeg(samp, w, h, seed=0, restart=0, progressive=False, quality=90, app=b""):
    """a JPEG with sampling factors samp = [(h, v)] per component, ids 1, 2, ...: YCbCr for three components, CMYK (no Adobe
    marker) for four.  Baseline: one interleaved scan, restart markers every `restart` MCUs.  Progressive: an interleaved DC
    scan, then one spectral-selection AC scan per component."""
    qt, huff = _tables(quality)
    codes = {k: _codes(*v) for k, v in huff.items()}
    blocks = _component_blocks(seed, w, h, samp, quality)
    hmax, vmax = max(s[0] for s in samp), max(s[1] for s in samp)
    mcu_x, mcu_y = -(-w // (8 * hmax)), -(-h // (8 * vmax))
    hdr = bytearray(b"\xff\xd8") + app
    for t in (0, 1):
        hdr += b"\xff\xdb" + struct.pack(">H", 67) + bytes([t]) + bytes(qt[t])
    n = len(samp)
    sof = bytes([8]) + struct.pack(">HH", h, w) + bytes([n])
    for z, (hs, vs) in enumerate(samp):
        sof += bytes([z + 1, hs << 4 | vs, 0 if z == 0 else 1])
    hdr += (b"\xff\xc2" if progressive else b"\xff\xc0") + struct.pack(">H", len(sof) + 2) + sof
    for (cls, t), (counts, syms) in sorted(huff.items()):
        body = bytes([cls << 4 | t]) + bytes(counts) + bytes(syms)
        hdr += b"\xff\xc4" + struct.pack(">H", len(body) + 2) + body
    if restart:
        hdr += b"\xff\xdd" + struct.pack(">HH", 4, restart)

    def sos(comps, ss, se):
        return b"\xff\xda" + struct.pack(">H", 6 + 2 * len(comps)) + bytes([len(comps)]) + \
            b"".join(bytes([z + 1, 0x00 if z == 0 else 0x11]) for z in comps) + bytes([ss, se, 0])

    def interleaved(dc_only):
        bits, pred = _Bits(), [0] * n
        for m in range(mcu_x * mcu_y):
            if restart and m and m % restart == 0:
                bits.flush()
                bits.out += bytes([0xFF, 0xD0 + (m // restart - 1) % 8])
                pred = [0] * n
            my, mx = divmod(m, mcu_x)
            for z, (hs, vs) in enumerate(samp):
                t = 0 if z == 0 else 1
                for v in range(vs):
                    for hh in range(hs):
                        zz = blocks[z][my * vs + v, mx * hs + hh]
                        bits.code(codes[(0, t)], abs(int(zz[0]) - pred[z]).bit_length())
                        bits.value(int(zz[0]) - pred[z])
                        pred[z] = int(zz[0])
                        if not dc_only:
                            _ac(bits, codes[(1, t)], zz)
        bits.flush()
        return bytes(bits.out)

    body = bytearray()
    if not progressive:
        body += sos(list(range(n)), 0, 63) + interleaved(False)
    else:
        body += sos(list(range(n)), 0, 0) + interleaved(True)
        for z, (hs, vs) in enumerate(samp):
            bw, bh = -(-(-(-w * hs // hmax)) // 8), -(-(-(-h * vs // vmax)) // 8)
            bits = _Bits()
            for by in range(bh):
                for bx in range(bw):
                    _ac(bits, codes[(1, 0 if z == 0 else 1)], blocks[z][by, bx])
            bits.flush()
            body += sos([z], 1, 63) + bytes(bits.out)
    return bytes(hdr) + bytes(body) + b"\xff\xd9"


def exif_app1(o):
    ex = Image.Exif()
    ex[0x0112] = o
    payload = ex.tobytes()
    if not payload.startswith(b"Exif"):
        payload = b"Exif\x00\x00" + payload
    return b"\xff\xe1" + struct.pack(">H", len(payload) + 2) + payload


# ------------------------------------------------------------------------------------------------ the statement in numpy
def block_size(hmax, vmax, h, v, s0):
    ss = s0
    while ss < 8 and (hmax * s0) % (2 * h * ss) == 0 and (vmax * s0) % (2 * v * ss) == 0:
        ss *= 2
    return ss


def upsampled(img, planes, d=1, islow=True, comps=None):
    """steps 1-3 on the host stage's planes: the up-sampled component planes (int) of the W' x H' image (comps: the components,
    img.comp[0..2] by default)"""
    comps = comps or [img.comp[z] for z in range(3)]
    hmax, vmax = max(c.h_samp for c in comps), max(c.v_samp for c in comps)
    s0 = 8 // d
    W, H = -(-img.width // d), -(-img.height // d)
    up = []
    for c, plane in zip(comps, planes):
        h, v = c.h_samp, c.v_samp
        ss = block_size(hmax, vmax, h, v, s0)
        bpr = c.width_stride // 8
        blocks = plane.reshape(-1, 64)
        qt = np.asarray(c.qt, np.int32)
        if ss == 8 and not islow:
            smp = np.clip(ref_model.idct_blocks(blocks, qt, ref_model.X86), 0, 255)
        else:
            smp = scaled_blocks(blocks, qt, ss) if ss < 8 else islow_blocks(blocks, qt)
        rows = blocks.shape[0] // bpr
        smp = np.asarray(smp).reshape(rows, bpr, ss, ss).transpose(0, 2, 1, 3).reshape(rows * ss, bpr * ss).astype(np.int32)
        dw, dh = -(-img.width * h * ss // (hmax * 8)), -(-img.height * v * ss // (vmax * 8))
        a = smp[:dh, :dw]
        assert (hmax * s0) % (h * ss) == 0 and (vmax * s0) % (v * ss) == 0
        rh, rv = hmax * s0 // (h * ss), vmax * s0 // (v * ss)
        fancy = s0 > 1
        if (rh, rv) == (2, 1) and fancy and dw > 2:
            a = _upsample(a, 2, 1)
        elif (rh, rv) == (1, 2) and fancy:
            a = _upsample(a, 1, 2)
        elif (rh, rv) == (2, 2) and fancy and dw > 2:
            a = _upsample(a, 2, 2)
        else:                                       # int_upsample: each sample rh x rv times
            a = np.repeat(np.repeat(a, rv, 0), rh, 1)
        up.append(a[:H, :W])
    return up


def _clip(x):
    return np.clip(x, 0, 255)


def statement(img, planes, cs, d=1, islow=True):
    """steps 4-5: the output pixels [H', W', nc] for colourspace cs"""
    y, cb, cr = (np.asarray(p, np.int64) for p in upsampled(img, planes, d, islow))
    if cs == ColorSpace.GRAYSCALE:
        return y.astype(np.uint8)[..., None]
    if cs == ColorSpace.YCbCr:
        return np.stack([y, cb, cr], -1).astype(np.uint8)
    cb, cr = cb - 128, cr - 128
    rgb = [_clip(y + ((91881 * cr + 32768) >> 16)), _clip(y + ((-22554 * cb - 46802 * cr + 32768) >> 16)),
           _clip(y + ((116130 * cb + 32768) >> 16))]
    if cs in (ColorSpace.RGBA, ColorSpace.RGBX):
        rgb.append(np.full_like(y, 255))
    return np.stack(rgb, -1).astype(np.uint8)


def pil(data, cs, d=1):
    """Pillow's pixels (after its draft to 1/d; None where it does not draft that far); YCbCr: libjpeg's YCbCr output"""
    if cs != ColorSpace.YCbCr:
        return pillow(data, cs, d)
    im = Image.open(io.BytesIO(data))
    w, h = im.size
    im.draft("YCbCr", (max(w // d, 1), max(h // d, 1)))
    if im.mode != "YCbCr" or im.size != _ffi.scaled_size(w, h, d):
        return None
    return np.asarray(im)


def options(cs=ColorSpace.RGB, mode="libjpeg", d=1, orient=False):
    o = ZuneJpegOptions().set_out_colorspace(cs).set_num_threads(4)
    o = o.set_spec_output(True) if mode == "spec" else o.set_libjpeg_output(True)
    if d > 1:
        o = o.set_scale_denom(d)
    return o.set_exif_orientation(True) if orient else o


# ------------------------------------------------------------------------------------------------ the files
# every factor set of three components that libjpeg decodes and the fused kernels do not take ...
SAMPLINGS = {
    "411": [(4, 1), (1, 1), (1, 1)],
    "410": [(4, 2), (1, 1), (1, 1)],
    "1x4": [(1, 4), (1, 1), (1, 1)],
    "2x4": [(2, 4), (1, 1), (1, 1)],
    "3x1": [(3, 1), (1, 1), (1, 1)],
    "3x2": [(3, 2), (1, 1), (1, 1)],
    "chroma_up": [(1, 1), (2, 2), (2, 2)],
    "22_21": [(2, 2), (2, 1), (2, 1)],
    "22_12": [(2, 2), (1, 2), (1, 2)],
    "mixed": [(2, 1), (1, 2), (1, 1)],
    "mixed22": [(2, 2), (2, 1), (1, 2)],
    "mixed41": [(4, 1), (2, 1), (1, 1)],
}
# ... and two that it refuses: more than 10 blocks in an interleaved MCU, and a ratio that is not an integer
REFUSED = {
    "4x4": ([(4, 4), (1, 1), (1, 1)], "blocks in an MCU of an interleaved scan, more than 10"),
    "3x3": ([(3, 3), (1, 1), (1, 1)], "blocks in an MCU of an interleaved scan, more than 10"),
    "all22": ([(2, 2), (2, 2), (2, 2)], "blocks in an MCU of an interleaved scan, more than 10"),
    "3_over_2": ([(3, 1), (2, 1), (2, 1)], "non-integer up-sampling ratio"),
}
SIZES = [(37, 29), (64, 48), (1, 1), (5, 3), (70, 9)]


def _files():
    out = {}
    for k, (name, samp) in enumerate(sorted(SAMPLINGS.items())):
        for j, (w, h) in enumerate(SIZES):
            out[f"{name}_{w}x{h}"] = (samp, dict(seed=100 * k + j, w=w, h=h))
        out[f"{name}_dri"] = (samp, dict(seed=100 * k + 7, w=45, h=38, restart=2))
        out[f"{name}_prog"] = (samp, dict(seed=100 * k + 8, w=41, h=35, progressive=True))
    return out


FILES = _files()


def make(name):
    samp, kw = FILES[name]
    kw = dict(kw)
    return jpeg(samp, kw.pop("w"), kw.pop("h"), **kw)


# ------------------------------------------------------------------------------------------------ CPU
@pytest.mark.parametrize("name", sorted(FILES))
def test_statement_on_host_planes_equals_pillow(name):
    data = make(name)
    samp = FILES[name][0]
    for mode, d in (("spec", 1), ("libjpeg", 1), ("libjpeg", 2), ("libjpeg", 4), ("libjpeg", 8)):
        dec = Decoder.new_with_options(options(ColorSpace.RGB, mode, d))
        img, planes = dec.decode_coefficients(data)
        assert img.n_comp == 3 and [(img.comp[z].h_samp, img.comp[z].v_samp) for z in range(3)] == samp
        if mode == "spec":
            # spec output differs from libjpeg output only in its IDCT (the GPU tests check it against the statement)
            _, lplanes = Decoder.new_with_options(options(ColorSpace.RGB, "libjpeg")).decode_coefficients(data)
            assert all(np.array_equal(a, b) for a, b in zip(planes, lplanes))
            continue
        for cs in (ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.GRAYSCALE, ColorSpace.YCbCr):
            want = pil(data, cs, d)
            if want is None:
                continue
            got = statement(img, planes, cs, d)
            assert got.shape == want.shape, (cs, d, got.shape, want.shape)
            assert np.array_equal(got, want), (cs, d, int(np.abs(got.astype(int) - want.astype(int)).max()))


def test_rgb_equals_torchvision():
    """(every set but "mixed", whose luma is up-sampled 1 x 2: there the libjpeg torchvision bundles differs from Pillow's by 1)"""
    torch = pytest.importorskip("torch")
    tv_io = pytest.importorskip("torchvision.io")
    for name in ("411_37x29", "410_64x48", "3x2_70x9", "chroma_up_dri", "22_12_prog", "mixed41_37x29", "1x4_dri"):
        data = make(name)
        img, planes = Decoder.new_with_options(options()).decode_coefficients(data)
        tv = tv_io.decode_jpeg(torch.frombuffer(bytearray(data), dtype=torch.uint8), mode=tv_io.ImageReadMode.RGB)
        assert np.array_equal(statement(img, planes, ColorSpace.RGB), tv.permute(1, 2, 0).numpy()), name


@pytest.mark.parametrize("name", sorted(REFUSED))
@pytest.mark.parametrize("progressive", [False, True])
def test_refused_by_libjpeg_and_here(name, progressive):
    samp, msg = REFUSED[name]
    data = jpeg(samp, 40, 33, seed=5, progressive=progressive)
    with pytest.raises(Exception):
        im = Image.open(io.BytesIO(data))
        im.load()
    for d in (1, 8):
        dec = Decoder.new_with_options(options(ColorSpace.RGB, "libjpeg", d))
        with pytest.raises(DecodeErrors) as e:
            dec.decode_coefficients(data)
        assert e.value.kind == 1 and msg in e.value.display
    with pytest.raises(DecodeErrors) as e:
        Decoder.new_with_options(options(ColorSpace.RGB, "spec")).decode_coefficients(data)
    assert msg in e.value.display
    # (the headers alone are fine, as for jpeg_read_header)
    Decoder.new_with_options(options()).read_headers(data)


# What the as-written host stage says about each new factor set (37 x 29 baseline files): the reference's errors, unchanged
AS_WRITTEN = {
    "411": "Unknown down-sampling method, cannot continue",
    "410": "Unknown down-sampling method, cannot continue",
    "1x4": "Unknown down-sampling method, cannot continue",
    "2x4": "Unknown down-sampling method, cannot continue",
    "3x1": "Horizontal sample is not a power of two(3) cannot decode",
    "3x2": "Horizontal sample is not a power of two(3) cannot decode",
    "chroma_up": "Invalid image width and height stride for component Cb, expected 20, but found 48",
    "22_21": "Invalid image width and height stride for component Cb, expected 24, but found 48",
    "22_12": "Invalid component sample for component Cb, expected (1,1), found (2,1)",
    "mixed": "Invalid component sample for component Cb, expected (1,1), found (2,1)",
    "mixed22": "Invalid image width and height stride for component Cb, expected 24, but found 48",
    "mixed41": "Invalid image width and height stride for component Cb, expected 16, but found 32",
}


@pytest.mark.parametrize("unsafe", [0, 1])
def test_as_written_options_keep_their_errors(unsafe):
    for name, want in AS_WRITTEN.items():
        dec = Decoder.new_with_options(ZuneJpegOptions().set_use_unsafe(bool(unsafe)))
        with pytest.raises(DecodeErrors) as e:
            dec.decode_coefficients(make(f"{name}_37x29"))
        assert (e.value.kind, e.value.display) == (1, want), name


def test_abi():
    lib = _ffi.load()
    dec = Decoder.new_with_options(options())
    img, planes = dec.decode_coefficients(make("411_37x29"))
    assert [img.comp[z].width_stride for z in range(3)] == [4 * 2 * 8, 2 * 8, 2 * 8]
    assert lib.zj_validate_image(C.byref(img)) == 0
    assert lib.zj_output_size(C.byref(img)) == 37 * 29 * 3
    # spec images are never cut into strips; zj_image_rows returns them whole
    sub = _ffi.ZjImage()
    assert lib.zj_image_strip_range(C.byref(img), 0, 1, C.byref(sub), None, None, None) == _ffi.ERR_UNSUPPORTED
    row0 = C.c_uint32(99)
    assert lib.zj_image_rows(C.byref(img), 10, 20, C.byref(sub), C.byref(row0)) == 0
    assert row0.value == 10 and sub.height == img.height and sub.comp[0].coeff == img.comp[0].coeff
    # the as-written variants have no statement for these factors
    for variant in (_ffi.VARIANT_X86, _ffi.VARIANT_SCALAR):
        x = _ffi.ZjImage()
        C.memmove(C.byref(x), C.byref(img), C.sizeof(x))
        x.variant, x.flags = variant, 0
        assert lib.zj_validate_image(C.byref(x)) == _ffi.ERR_UNSUPPORTED
        assert lib.zj_output_size(C.byref(x)) == 0
    # factors outside 1..4, and a ratio that is not an integer
    for comp, hs, stride in ((1, 5, 5 * 2 * 8), (1, 3, 3 * 2 * 8)):
        x = _ffi.ZjImage()
        C.memmove(C.byref(x), C.byref(img), C.sizeof(x))
        x.comp[0].h_samp, x.comp[0].width_stride = 2, 2 * 2 * 8
        x.comp[comp].h_samp, x.comp[comp].width_stride = hs, stride
        assert lib.zj_validate_image(C.byref(x)) in (_ffi.ERR_UNSUPPORTED, _ffi.ERR_INVALID_ARG)
    # a scaled, oriented descriptor: the displayed size
    dec = Decoder.new_with_options(options(ColorSpace.RGBA, "libjpeg", 4, orient=True))
    img, _ = dec.decode_coefficients(make("3x2_70x9")[:2] + exif_app1(6) + make("3x2_70x9")[2:])
    assert lib.zj_validate_image(C.byref(img)) == 0
    assert lib.zj_output_size(C.byref(img)) == 3 * 18 * 4


@pytest.mark.parametrize("samp", [[(4, 1), (1, 1), (1, 1), (4, 1)], [(3, 1), (1, 1), (1, 1), (3, 1)], [(1, 1), (2, 2), (2, 2), (1, 1)],
                                  [(4, 1), (1, 1), (2, 1), (1, 1)]])
def test_four_components_take_factors_up_to_4(samp):
    """the four-component statement with factors 1..4 (CMYK, no Adobe marker) against Pillow"""
    from test_cmyk_output import cmyk_to_pillow, to_output
    for kw in (dict(w=37, h=29), dict(w=45, h=38, restart=3), dict(w=41, h=35, progressive=True)):
        data = jpeg(samp, kw.pop("w"), kw.pop("h"), seed=len(kw), **kw)
        for d in (1, 2, 8):
            dec = Decoder.new_with_options(options(ColorSpace.RGB, "libjpeg", d))
            img, planes = dec.decode_coefficients(data)
            assert dec.jpeg_colorspace() == ColorSpace.CMYK
            comps = [dec.component(z) for z in range(4)]
            cmyk, rgb = cmyk_to_pillow(upsampled(img, planes, d, comps=comps), False)
            for cs in (ColorSpace.RGB, ColorSpace.CMYK):
                want = pillow(data, cs, d)
                if want is not None:
                    assert np.array_equal(to_output(cmyk, rgb, cs), want), (samp, kw, d, cs)


def test_existing_factor_sets_keep_their_route():
    """luma (1|2) x (1|2) with chroma 1 x 1 keeps the fused kernels' planes (strips of two MCU rows for 4:2:0 spec output)"""
    b = io.BytesIO()
    Image.new("RGB", (40, 40)).save(b, "JPEG", subsampling=2)
    img, planes = Decoder.new_with_options(options()).decode_coefficients(b.getvalue())
    assert (img.comp[0].h_samp, img.comp[0].v_samp, img.comp[1].h_samp) == (2, 2, 1)
    assert planes[0].size == img.comp[0].width_stride * 16 * 4   # 3 MCU rows, decoded as two strips of two (raster planes: 3)


# ------------------------------------------------------------------------------------------------ GPU
CS_ALL = [ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.RGBX, ColorSpace.GRAYSCALE, ColorSpace.YCbCr]
GPU_FILES = [n for n in sorted(FILES) if n.endswith(("_37x29", "_1x1", "_5x3", "_dri", "_prog"))]


def _want(data, cs, d=1):
    """Pillow's pixels where it gives them for this d, else the statement (checked against Pillow by the CPU tests)"""
    w = pil(data, cs, d)
    if w is None:
        dec = Decoder.new_with_options(options(ColorSpace.RGB, "libjpeg", d))
        img, planes = dec.decode_coefficients(data)
        w = statement(img, planes, cs, d)
    return w


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 4, 8])
def test_decode_buffer_and_into_equal_pillow(d):
    from zune_jpeg_b200.gpu import PinnedBuffer
    for name in GPU_FILES:
        data = make(name)
        for cs in CS_ALL:
            want = _want(data, cs, d)
            got = Decoder.new_with_options(options(cs, "libjpeg", d)).decode_buffer(data)
            assert np.array_equal(np.frombuffer(got, np.uint8), want.reshape(-1)), (name, cs, d)
            pb = PinnedBuffer(want.size + 13)
            n = Decoder.new_with_options(options(cs, "libjpeg", d)).decode_into(data, pb.array[5:])
            assert n == want.size and np.array_equal(pb.array[5:5 + n], want.reshape(-1)), (name, cs, d, "into")


@pytest.mark.gpu
def test_spec_output_equals_statement():
    for name in GPU_FILES:
        data = make(name)
        img, planes = Decoder.new_with_options(options(ColorSpace.RGB, "spec")).decode_coefficients(data)
        for cs in CS_ALL:
            got = Decoder.new_with_options(options(cs, "spec")).decode_buffer(data)
            assert np.array_equal(np.frombuffer(got, np.uint8), statement(img, planes, cs, islow=False).reshape(-1)), (name, cs)


def _mixed_inputs():
    """new factor sets with standard YCbCr, gray and CMYK neighbours, a CMYK file with factors above 2, and one oriented file:
    (data, exif orientation)"""
    out = []
    for i, name in enumerate(sorted(SAMPLINGS)):
        out.append((make(f"{name}_37x29" if i % 2 else f"{name}_prog"), 1))
        b = io.BytesIO()
        if i % 3 == 0:
            Image.fromarray(np.full((23, 37, 3), 40 * (i % 6), np.uint8)).save(b, "JPEG", quality=85, subsampling=i % 3)
        elif i % 3 == 1:
            Image.fromarray(np.full((31, 29), 30 * (i % 8), np.uint8)).save(b, "JPEG", quality=85)
        else:
            b.write(cmyk_jpeg(i, 33, 21, sub=2 if i % 2 else 0))
        out.append((b.getvalue(), 1))
    out.append((jpeg([(4, 1), (1, 1), (2, 1), (1, 1)], 37, 21, seed=91), 1))   # CMYK with factors 4 and 2
    raw = jpeg(SAMPLINGS["410"], 45, 27, seed=77)
    out.append((raw[:2] + exif_app1(6) + raw[2:], 6))
    return out


def _oriented(want, o):
    ops = {3: Image.Transpose.ROTATE_180, 6: Image.Transpose.ROTATE_270, 8: Image.Transpose.ROTATE_90}
    if o not in ops:
        return want
    return np.stack([np.asarray(Image.fromarray(np.ascontiguousarray(want[..., k])).transpose(ops[o])) for k in range(want.shape[-1])], -1)


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 4])
@pytest.mark.parametrize("cs", [ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.GRAYSCALE])
def test_decode_batch_mixed(d, cs):
    inputs = _mixed_inputs()
    res = decode_batch([x[0] for x in inputs], options(cs, "libjpeg", d, orient=True), threads=3)
    for (data, o), r in zip(inputs, res):
        assert not isinstance(r, Exception), r
        want = pil(data, cs, d)
        if want is None:   # (Pillow does not draft that far)
            continue
        assert np.array_equal(np.frombuffer(r, np.uint8), _oriented(want, o).reshape(-1))


@pytest.mark.gpu
def test_decode_batch_device_out_and_multi():
    torch = pytest.importorskip("torch")
    inputs = _mixed_inputs()
    datas = [x[0] for x in inputs]
    opts = options(ColorSpace.RGB, "libjpeg", 1, orient=True)
    wants = [_oriented(pil(data, ColorSpace.RGB), o) for data, o in inputs]
    bufs = [torch.empty(w.size, dtype=torch.uint8, device="cuda:0") for w in wants]
    res = decode_batch(datas, opts, device_out=[(b.data_ptr(), b.numel()) for b in bufs])
    for r, b, w in zip(res, bufs, wants):
        assert not isinstance(r, Exception), r
        assert np.array_equal(b.cpu().numpy(), w.reshape(-1))
    for devs in ([0], [0, 0]):
        res = decode_batch(datas, opts, devices=devs)
        for r, w in zip(res, wants):
            assert np.array_equal(np.frombuffer(r, np.uint8), w.reshape(-1))
        res = decode_batch(datas[:1], opts, devices=devs)
        assert np.array_equal(np.frombuffer(res[0], np.uint8), wants[0].reshape(-1))


@pytest.mark.gpu
def test_device_out_f16_chw():
    torch = pytest.importorskip("torch")
    from zune_jpeg_b200 import gpu
    datas = [make(n) for n in ("411_37x29", "chroma_up_prog", "mixed22_dri")]
    mean, std = [120.0, 110.0, 100.0], [60.0, 61.0, 62.0]
    desc = gpu.OutputDesc(layout="CHW", dtype="f16", mean=mean, inv_std=[1.0 / v for v in std])
    wants = [pil(d, ColorSpace.RGB) for d in datas]
    bufs = [torch.empty((3,) + w.shape[:2], dtype=torch.float16, device="cuda:0") for w in wants]
    res = decode_batch(datas, options(), device_out=[(b.data_ptr(), b.numel() * 2) for b in bufs], desc=desc)
    for r, b, w in zip(res, bufs, wants):
        assert not isinstance(r, Exception), r
        inv = torch.tensor([1.0 / v for v in std], dtype=torch.float32)
        ref = ((torch.from_numpy(w).float() - torch.tensor(mean)) * inv).permute(2, 0, 1).half()
        assert torch.equal(b.cpu(), ref)


@pytest.mark.gpu
def test_decode_batch_resized_equals_pillow_then_torchvision():
    torch = pytest.importorskip("torch")
    T = pytest.importorskip("torchvision.transforms")
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import decode_batch_resized
    raw = jpeg(SAMPLINGS["3x2"], 310, 240, seed=43)
    datas = [jpeg(SAMPLINGS["411"], 300, 200, seed=40), jpeg(SAMPLINGS["chroma_up"], 260, 330, seed=41, progressive=True),
             jpeg(SAMPLINGS["mixed"], 280, 250, seed=42, restart=5), raw[:2] + exif_app1(6) + raw[2:], cmyk_jpeg(44, 270, 260)]
    S, out = 256, 224
    tf = T.Compose([T.Resize(S, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(out)])
    opts = options(ColorSpace.RGB, "libjpeg", 1, orient=True)
    arr, errs = decode_batch_resized(datas, gpu.Resize((out, out), filter="pil_bicubic", short_side=S), options=opts)
    assert errs == [None] * len(datas)
    t = arr.to_torch().cpu().numpy()
    for i, data in enumerate(datas):
        im = ImageOps.exif_transpose(Image.open(io.BytesIO(data)).convert("RGB"))
        got = t[i]
        if got.shape[0] == 3:
            got = got.transpose(1, 2, 0)
        assert np.array_equal(got, np.asarray(tf(im))), i


@pytest.mark.gpu
def test_planes_in_batch():
    """zj_batch over device-resident planes of the host stage: new factor sets mixed with a standard 4:2:0 image"""
    from zune_jpeg_b200 import gpu
    b = io.BytesIO()
    Image.fromarray(np.random.default_rng(3).integers(0, 256, (40, 50, 3), dtype=np.uint8)).save(b, "JPEG", subsampling=2)
    datas = [make("410_37x29"), make("3x1_64x48"), b.getvalue(), make("mixed_prog")]
    keep, imgs, wants, outs = [], [], [], []
    for k, data in enumerate(datas):
        cs = ColorSpace.RGBA if k % 2 else ColorSpace.RGB
        img, planes = Decoder.new_with_options(options(cs, "libjpeg", 2 if k == 3 else 1)).decode_coefficients(data)
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for z, (buf, p) in enumerate(zip(bufs, planes)):
            buf.upload(p)
            img.comp[z].coeff = buf.ptr
        want = pil(data, cs, 2 if k == 3 else 1)
        out = gpu.DeviceBuffer(want.size)
        keep.append((planes, bufs)); imgs.append(img); wants.append(want); outs.append(out)
    gpu.synchronize()
    batch = gpu.Batch(imgs, [o.ptr for o in outs], [w.size for w in wants])
    batch.run()
    gpu.synchronize()
    for o, w in zip(outs, wants):
        assert o.download(w.size).tobytes() == w.tobytes()
    batch.destroy()
