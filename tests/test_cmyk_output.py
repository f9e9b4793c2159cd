"""Four-component JPEGs -- CMYK, and YCCK as Photoshop writes it -- in spec and libjpeg output (DESIGN.md section 4.6.4): the
statement of include/zune_jpeg_b200.h (next to zj_decoder_jpeg_colorspace) restated in numpy, checked against Pillow 12.2 on the
host stage's planes, and the GPU routes checked against the statement and Pillow bit for bit."""
from __future__ import annotations

import ctypes as C
import io
import struct

import numpy as np
import pytest
from PIL import Image, ImageOps

import ref_model
from test_libjpeg_output import islow_blocks
from test_scaled_output import scaled_blocks
from test_spec_output import _upsample
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, DecodeErrors, Decoder, ZuneJpegOptions, decode_batch


# ------------------------------------------------------------------------------------------------ test files
def _content(seed, w, h):
    """smooth CMYK content with some texture (photographic enough that every coefficient range is exercised)"""
    rng = np.random.default_rng(seed)
    base = rng.integers(0, 256, (h // 6 + 2, w // 6 + 2, 4), dtype=np.uint8)
    im = np.asarray(Image.fromarray(base, "CMYK").resize((w, h), Image.BILINEAR)).astype(np.int16)
    im = im + rng.integers(-24, 25, im.shape)
    return Image.fromarray(np.clip(im, 0, 255).astype(np.uint8), "CMYK")


def cmyk_jpeg(seed, w, h, sub=0, progressive=False, restart=0, exif=None, quality=90):
    """a CMYK JPEG as Pillow writes it: Adobe transform 0, ids C M Y K; sub = 2: C at 2x2"""
    kw = dict(quality=quality, subsampling=sub, progressive=progressive)
    if restart:
        kw["restart_marker_rows"] = restart
    if exif is not None:
        kw["exif"] = exif
    b = io.BytesIO()
    _content(seed, w, h).save(b, "JPEG", **kw)
    return b.getvalue()


def _header_segments(data):
    """(offset of the 0xFF, marker byte, segment length) of every marker segment before the first SOS"""
    out, p = [], 2
    while p + 4 <= len(data) and data[p] == 0xFF:
        m, n = data[p + 1], struct.unpack(">H", data[p + 2:p + 4])[0]
        out.append((p, m, n))
        if m == 0xDA:
            break
        p += 2 + n
    return out


def set_transform(data, t):
    """every Adobe APP14 segment's transform byte (payload byte 11) set to t"""
    b = bytearray(data)
    for p, m, n in _header_segments(data):
        if m == 0xEE and b[p + 4:p + 9] == b"Adobe":
            b[p + 4 + 11] = t
    return bytes(b)


def drop_app14(data):
    for p, m, n in _header_segments(data):
        if m == 0xEE:
            return drop_app14(data[:p] + data[p + 2 + n:])
    return data


def insert_app14(data, payload):
    """an APP14 segment with this payload right after SOI"""
    return data[:2] + b"\xff\xee" + struct.pack(">H", len(payload) + 2) + payload + data[2:]


def adobe(t):
    return b"Adobe" + bytes([0, 100, 0, 0, 0, 0, t])


def rewrite_ids(data, ids):
    """the SOF's component ids and every SOS's selectors replaced by ids (in SOF order)"""
    b = bytearray(data)
    old = []
    for p, m, n in _header_segments(data):
        if m in (0xC0, 0xC1, 0xC2):
            for z in range(b[p + 9]):
                old.append(b[p + 10 + 3 * z])
                b[p + 10 + 3 * z] = ids[z]
    p = 0
    while True:
        p = data.find(b"\xff\xda", p)
        if p < 0:
            break
        for k in range(b[p + 4]):
            b[p + 5 + 2 * k] = ids[old.index(data[p + 5 + 2 * k])]
        p += 2
    return bytes(b)


# ------------------------------------------------------------------------------------------------ a small baseline encoder
# Y and K at 2x2 with Cb and Cr at 1x1 (libjpeg's and Photoshop's YCCK layout) is not something Pillow writes: DC-only blocks
# whose values come from the content, coded with one fixed Huffman table pair.
def _bits(out, acc, v, n):
    acc[0] = (acc[0] << n) | (v & ((1 << n) - 1))
    acc[1] += n
    while acc[1] >= 8:
        acc[1] -= 8
        byte = (acc[0] >> acc[1]) & 0xFF
        out.append(byte)
        if byte == 0xFF:
            out.append(0)


def ycck_2211_jpeg(seed, w, h, transform=2, restart=0):
    rng = np.random.default_rng(seed)
    samp = [(2, 2), (1, 1), (1, 1), (2, 2)]
    mcu_x, mcu_y = -(-w // 16), -(-h // 16)
    qt = np.ones(64, np.uint8) * 4
    # DC category k code: k as a 4-bit code (a complete table of 16 codes of length 4 for categories 0-11); AC: EOB only, 1 bit
    dc_counts, dc_syms = [0, 0, 0, 12] + [0] * 12, list(range(12))
    ac_counts, ac_syms = [1] + [0] * 15, [0]
    hdr = bytearray(b"\xff\xd8")
    hdr += insert_app14(b"\xff\xd8", adobe(transform))[2:] if transform is not None else b""
    hdr += b"\xff\xdb" + struct.pack(">H", 67) + b"\x00" + bytes(qt)
    sof = bytes([8]) + struct.pack(">HH", h, w) + bytes([4])
    for z, (hs, vs) in enumerate(samp):
        sof += bytes([z + 1, hs << 4 | vs, 0])
    hdr += b"\xff\xc0" + struct.pack(">H", len(sof) + 2) + sof
    for cls, counts, syms in ((0x00, dc_counts, dc_syms), (0x10, ac_counts, ac_syms)):
        body = bytes([cls]) + bytes(counts) + bytes(syms)
        hdr += b"\xff\xc4" + struct.pack(">H", len(body) + 2) + body
    if restart:
        hdr += b"\xff\xdd" + struct.pack(">HH", 4, restart)
    hdr += b"\xff\xda" + struct.pack(">H", 14) + bytes([4, 1, 0, 2, 0, 3, 0, 4, 0, 0, 63, 0])
    out, acc = bytearray(), [0, 0]
    pred = [0, 0, 0, 0]
    dc = rng.integers(-100, 100, (4, 2 * mcu_y, 2 * mcu_x))
    for m in range(mcu_x * mcu_y):
        if restart and m and m % restart == 0:
            if acc[1]:
                _bits(out, acc, 0x7F, 8 - acc[1])
            out += bytes([0xFF, 0xD0 + (m // restart - 1) % 8])
            pred = [0, 0, 0, 0]
        my, mx = divmod(m, mcu_x)
        for z, (hs, vs) in enumerate(samp):
            for v in range(vs):
                for hh in range(hs):
                    val = int(dc[z, my * vs + v, mx * hs + hh])
                    diff = val - pred[z]
                    pred[z] = val
                    k = abs(diff).bit_length()
                    _bits(out, acc, k, 4)
                    if k:
                        _bits(out, acc, diff if diff > 0 else diff - 1, k)
                    _bits(out, acc, 0, 1)   # EOB
    if acc[1]:
        _bits(out, acc, 0x7F, 8 - acc[1])
    return bytes(hdr) + bytes(out) + b"\xff\xd9"


# ------------------------------------------------------------------------------------------------ the statement in numpy
def _clip(x):
    return np.clip(x, 0, 255)


def cmyk_to_pillow(s, ycck):
    """steps 3-4: the four up-sampled sample planes (int) -> Pillow's c, m, y, k and R, G, B"""
    s = [np.asarray(p, np.int64) for p in s]
    if ycck:
        y, cb, cr = s[0], s[1] - 128, s[2] - 128
        c0 = _clip(255 - (y + ((91881 * cr + 32768) >> 16)))
        m0 = _clip(255 - (y + ((-22554 * cb - 46802 * cr + 32768) >> 16)))
        y0 = _clip(255 - (y + ((116130 * cb + 32768) >> 16)))
        cmyk0 = [c0, m0, y0, s[3]]
    else:
        cmyk0 = s
    c, m, y, k = (255 - p for p in cmyk0)
    nk = 255 - k

    def ch(x):
        t = x * nk + 128
        return _clip(nk - (((t >> 8) + t) >> 8))
    return np.stack([c, m, y, k], -1).astype(np.uint8), np.stack([ch(c), ch(m), ch(y)], -1).astype(np.uint8)


def statement(dec, img, planes, d=1, islow=True):
    """steps 1-2 on the host stage's four planes -> (CMYK;I bytes, RGB bytes) of the W' x H' image"""
    comps = [dec.component(z) for z in range(4)]
    hmax, vmax = max(c.h_samp for c in comps), max(c.v_samp for c in comps)
    s0 = 8 // d
    W, H = -(-img.width // d), -(-img.height // d)
    up = []
    for c, plane in zip(comps, planes):
        h, v, ss = c.h_samp, c.v_samp, s0
        while ss < 8 and (hmax * s0) % (2 * h * ss) == 0 and (vmax * s0) % (2 * v * ss) == 0:
            ss *= 2
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
        rh, rv = hmax * s0 // (h * ss), vmax * s0 // (v * ss)
        fancy = s0 > 1
        if (rh, rv) == (2, 1):
            a = _upsample(a, 2, 1) if fancy and dw > 2 else np.repeat(a, 2, 1)
        elif (rh, rv) == (1, 2):
            a = _upsample(a, 1, 2) if fancy else np.repeat(a, 2, 0)
        elif (rh, rv) == (2, 2):
            a = _upsample(a, 2, 2) if fancy and dw > 2 else np.repeat(np.repeat(a, 2, 0), 2, 1)
        up.append(a[:H, :W])
    return cmyk_to_pillow(up, dec.jpeg_colorspace() == ColorSpace.YCCK)


def to_output(cmyk, rgb, cs):
    if cs == ColorSpace.CMYK:
        return cmyk
    if cs == ColorSpace.GRAYSCALE:
        r, g, b = (rgb[..., k].astype(np.int64) for k in range(3))
        return ((19595 * r + 38470 * g + 7471 * b + 32768) >> 16).astype(np.uint8)[..., None]
    if cs in (ColorSpace.RGBA, ColorSpace.RGBX):
        return np.concatenate([rgb, np.full(rgb.shape[:2] + (1,), 255, np.uint8)], -1)
    return rgb


def pillow(data, cs, d=1):
    """Pillow's pixels; d > 1: after its draft to 1/d, or None where Pillow does not draft that far.  (GRAYSCALE of a YCbCr file:
    libjpeg's grayscale output, the luma plane, through draft("L"), which is what libjpeg output gives for it.)"""
    im = Image.open(io.BytesIO(data))
    luma = cs == ColorSpace.GRAYSCALE and im.mode != "CMYK"
    if d > 1 or luma:
        w, h = im.size
        im.draft("L" if luma else im.mode, (max(w // d, 1), max(h // d, 1)))
        if im.size != _ffi.scaled_size(w, h, d):
            return None
    if cs == ColorSpace.CMYK:
        return np.asarray(im)
    a = np.asarray(im.convert({ColorSpace.GRAYSCALE: "L", ColorSpace.RGBA: "RGBA", ColorSpace.RGBX: "RGBA"}.get(cs, "RGB")))
    return a[..., None] if a.ndim == 2 else a


def options(cs=ColorSpace.RGB, mode="libjpeg", d=1, orient=False):
    o = ZuneJpegOptions().set_out_colorspace(cs).set_num_threads(4)
    o = o.set_spec_output(True) if mode == "spec" else o.set_libjpeg_output(True)
    if d > 1:
        o = o.set_scale_denom(d)
    return o.set_exif_orientation(True) if orient else o


# ------------------------------------------------------------------------------------------------ CPU: headers and host stage
FILES = {
    "444": lambda: cmyk_jpeg(1, 61, 45),
    "420c": lambda: cmyk_jpeg(2, 70, 37, sub=2),
    "prog": lambda: cmyk_jpeg(3, 53, 66, progressive=True),
    "prog420c": lambda: cmyk_jpeg(4, 40, 41, sub=2, progressive=True),
    "dri": lambda: cmyk_jpeg(5, 90, 50, restart=1),
    "dri420c": lambda: cmyk_jpeg(6, 45, 80, sub=2, restart=2),
    "ycck": lambda: set_transform(cmyk_jpeg(7, 77, 39), 2),
    "ycck420c_prog": lambda: set_transform(cmyk_jpeg(8, 33, 70, sub=2, progressive=True), 2),
    "ycck_assumed": lambda: set_transform(cmyk_jpeg(9, 50, 50), 7),
    "no_adobe": lambda: drop_app14(cmyk_jpeg(10, 31, 29)),
    "ids1234": lambda: rewrite_ids(cmyk_jpeg(11, 47, 21, sub=2), [1, 2, 3, 4]),
    "ids_prog": lambda: rewrite_ids(cmyk_jpeg(12, 20, 30, progressive=True), [200, 0, 17, 3]),
    "tiny1x1": lambda: cmyk_jpeg(13, 1, 1),
    "tiny2x3_420c": lambda: cmyk_jpeg(14, 2, 3, sub=2),
    "odd17x9_ycck": lambda: set_transform(cmyk_jpeg(15, 17, 9, sub=2), 2),
}


def _cmyk_files():
    return {k: f() for k, f in FILES.items()}


@pytest.mark.parametrize("name", sorted(FILES))
@pytest.mark.parametrize("mode,d", [("spec", 1), ("libjpeg", 1), ("libjpeg", 2), ("libjpeg", 4), ("libjpeg", 8)])
def test_statement_on_host_planes_equals_pillow(name, mode, d):
    data = FILES[name]()
    dec = Decoder.new_with_options(options(ColorSpace.RGB, mode, d))
    img, planes = dec.decode_coefficients(data)
    assert img.n_comp == 4 and len(planes) == 4
    if mode == "spec":
        # spec output differs from Pillow only in its IDCT (the GPU tests check it against the statement): its host stage is
        # libjpeg output's
        _, lplanes = Decoder.new_with_options(options(ColorSpace.RGB, "libjpeg")).decode_coefficients(data)
        assert all(np.array_equal(a, b) for a, b in zip(planes, lplanes))
        assert img.flags & _ffi.FLAG_ISLOW == 0
        return
    cmyk, rgb = statement(dec, img, planes, d)
    for cs in (ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.GRAYSCALE, ColorSpace.CMYK):
        want = pillow(data, cs, d)
        if want is None:
            continue
        got = to_output(cmyk, rgb, cs)
        assert got.shape == want.shape, (cs, got.shape, want.shape)
        assert np.array_equal(got, want), (cs, int(np.abs(got.astype(int) - want.astype(int)).max()))


def test_ycck_layout_2211_equals_pillow():
    for restart in (0, 3):
        for w, h in ((40, 24), (33, 17), (3, 5)):
            data = ycck_2211_jpeg(w * h + restart, w, h, restart=restart)
            for d in (1, 2, 4, 8):
                dec = Decoder.new_with_options(options(ColorSpace.RGB, "libjpeg", d))
                img, planes = dec.decode_coefficients(data)
                assert dec.jpeg_colorspace() == ColorSpace.YCCK
                assert [dec.component(z).h_samp for z in range(4)] == [2, 1, 1, 2]
                cmyk, rgb = statement(dec, img, planes, d)
                if pillow(data, ColorSpace.RGB, d) is None:
                    continue
                assert np.array_equal(rgb, pillow(data, ColorSpace.RGB, d)), (w, h, d, restart)
                assert np.array_equal(cmyk, pillow(data, ColorSpace.CMYK, d)), (w, h, d, restart)


def test_rgb_equals_torchvision():
    torch = pytest.importorskip("torch")
    tv_io = pytest.importorskip("torchvision.io")
    for name in ("444", "420c", "prog", "ycck", "dri"):
        data = FILES[name]()
        dec = Decoder.new_with_options(options())
        img, planes = dec.decode_coefficients(data)
        _, rgb = statement(dec, img, planes)
        tv = tv_io.decode_jpeg(torch.frombuffer(bytearray(data), dtype=torch.uint8), mode=tv_io.ImageReadMode.RGB)
        assert np.array_equal(rgb, tv.permute(1, 2, 0).numpy()), name


def _pillow_transform(data):
    im = Image.open(io.BytesIO(data))
    return im.info.get("adobe_transform")


@pytest.mark.parametrize("case", ["pillow", "t2", "t1", "t255", "none", "short", "truncated_marker", "repeated", "repeated_last_0"])
def test_colour_model(case):
    base = cmyk_jpeg(20, 16, 16)
    data = {
        "pillow": base,
        "t2": set_transform(base, 2),
        "t1": set_transform(base, 1),
        "t255": set_transform(base, 255),
        "none": drop_app14(base),
        "short": insert_app14(drop_app14(base), adobe(2)[:11]),                  # 11 bytes: not an Adobe marker
        "truncated_marker": insert_app14(drop_app14(base), b"Adob"),
        "repeated": insert_app14(set_transform(base, 0), adobe(2)),             # the later one (transform 0) wins
        "repeated_last_0": insert_app14(set_transform(base, 2), adobe(0)),      # the later one (transform 2) wins
    }[case]
    dec = Decoder.new_with_options(options())
    dec.read_headers(data)
    segs = [data[p + 4:p + 2 + n] for p, m, n in _header_segments(data) if m == 0xEE]
    t = next((s[11] for s in reversed(segs) if len(s) >= 12 and s[:5] == b"Adobe"), None)
    want = ColorSpace.CMYK if t in (None, 0) else ColorSpace.YCCK
    assert dec.jpeg_colorspace() == want
    if case in ("pillow", "t2", "t1", "t255", "none"):
        assert _pillow_transform(data) == t
    # and the decode follows it: the host planes give Pillow's pixels
    img, planes = dec.decode_coefficients(data)
    _, rgb = statement(dec, img, planes)
    assert np.array_equal(rgb, pillow(data, ColorSpace.RGB))
    assert dec.info().components == 4


def test_three_component_colour_model_unchanged():
    b = io.BytesIO()
    Image.fromarray(np.zeros((8, 8, 3), np.uint8)).save(b, "JPEG")
    dec = Decoder.new_with_options(options())
    dec.read_headers(b.getvalue())
    assert dec.jpeg_colorspace() == ColorSpace.YCbCr


@pytest.mark.parametrize("unsafe", [0, 1])
def test_as_written_options_still_reject(unsafe):
    for data, want in ((FILES["444"](), 67), (FILES["ids1234"](), 4)):
        dec = Decoder.new_with_options(ZuneJpegOptions().set_use_unsafe(bool(unsafe)))
        with pytest.raises(DecodeErrors) as e:
            dec.decode_coefficients(data)
        assert e.value.kind == 1
        assert e.value.display == f"Unknown component id found,{want}, expected value between 1 and 3\nNote I and Q components are not supported yet"


def test_bad_four_component_frames():
    base = cmyk_jpeg(21, 16, 16)
    dup = rewrite_ids(base, [1, 2, 1, 4])
    with pytest.raises(DecodeErrors):
        Decoder.new_with_options(options()).decode_coefficients(dup)
    # YCBCR and YCCK output have no statement for four components
    for cs in (ColorSpace.YCbCr, ColorSpace.YCCK):
        dec = Decoder.new_with_options(options(cs))
        img, planes = dec.decode_coefficients(base)
        assert img.n_comp == 4 and img.out_cs == cs


def test_abi():
    lib = _ffi.load()
    assert C.sizeof(_ffi.ZjImage) == 6 * 4 + 3 * C.sizeof(_ffi.ZjComponent)
    dec = Decoder.new_with_options(options())
    img, planes = dec.decode_coefficients(FILES["420c"]())
    k = dec.component(3)
    assert k.n_i16 == planes[3].size and k.h_samp == 1 and k.width_stride % 8 == 0
    with pytest.raises(IndexError):
        dec.component(4)
    # the planes-in entry points refuse n_comp = 4
    assert lib.zj_validate_image(C.byref(img)) == _ffi.ERR_INVALID_ARG
    assert lib.zj_output_size(C.byref(img)) == 0


# ------------------------------------------------------------------------------------------------ GPU
def _want(data, cs, d=1, orient=False):
    """Pillow's pixels (after draft for d > 1), with exif_transpose applied when orient"""
    w = pillow(data, cs, d)
    if orient and w is not None:
        im = Image.open(io.BytesIO(data))
        o = im.getexif().get(0x0112, 1)
        ops = {2: Image.Transpose.FLIP_LEFT_RIGHT, 3: Image.Transpose.ROTATE_180, 4: Image.Transpose.FLIP_TOP_BOTTOM,
               5: Image.Transpose.TRANSPOSE, 6: Image.Transpose.ROTATE_270, 7: Image.Transpose.TRANSVERSE, 8: Image.Transpose.ROTATE_90}
        if o in ops:   # (exif_transpose's transform, applied to each channel plane)
            w = np.stack([np.asarray(Image.fromarray(np.ascontiguousarray(w[..., k])).transpose(ops[o])) for k in range(w.shape[-1])], -1)
    return w


def _oriented(seed, w, h, o, **kw):
    ex = Image.Exif()
    ex[0x0112] = o
    return cmyk_jpeg(seed, w, h, exif=ex.tobytes(), **kw)


CS_ALL = [ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.RGBX, ColorSpace.GRAYSCALE, ColorSpace.CMYK]


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 2, 4, 8])
def test_decode_buffer_and_into_equal_pillow(d):
    from zune_jpeg_b200.gpu import PinnedBuffer
    files = _cmyk_files()
    files["2211"] = ycck_2211_jpeg(3, 70, 45)
    files["2211_dri"] = ycck_2211_jpeg(4, 35, 50, restart=2)
    for name, data in files.items():
        dec = Decoder.new_with_options(options(ColorSpace.RGB, "libjpeg", d))
        img, planes = dec.decode_coefficients(data)
        cmyk, rgb = statement(dec, img, planes, d)
        for cs in CS_ALL:
            want = _want(data, cs, d)
            if want is None:   # (Pillow does not draft that far: the statement, checked against Pillow where it does)
                want = to_output(cmyk, rgb, cs)
            got = Decoder.new_with_options(options(cs, "libjpeg", d)).decode_buffer(data)
            assert np.array_equal(np.frombuffer(got, np.uint8), want.reshape(-1)), (name, cs, d)
            pb = PinnedBuffer(want.size + 13)
            n = Decoder.new_with_options(options(cs, "libjpeg", d)).decode_into(data, pb.array[5:])
            assert n == want.size and np.array_equal(pb.array[5:5 + n], want.reshape(-1)), (name, cs, d, "into")


@pytest.mark.gpu
def test_spec_output_equals_statement():
    for name, data in _cmyk_files().items():
        dec = Decoder.new_with_options(options(ColorSpace.RGB, "spec"))
        img, planes = dec.decode_coefficients(data)
        cmyk, rgb = statement(dec, img, planes, islow=False)
        for cs in CS_ALL:
            got = Decoder.new_with_options(options(cs, "spec")).decode_buffer(data)
            assert np.array_equal(np.frombuffer(got, np.uint8), to_output(cmyk, rgb, cs).reshape(-1)), (name, cs)


def _mixed_inputs():
    """CMYK / YCCK files of every layout with YCbCr, gray, scaled and oriented neighbours: (data, options, want)"""
    out = []
    for i, (name, data) in enumerate(sorted(_cmyk_files().items())):
        out.append((data, 1, False))
        if i % 3 == 0:
            b = io.BytesIO()
            _content(i, 37, 23).convert("RGB").save(b, "JPEG", quality=85)
            out.append((b.getvalue(), 1, False))
        if i % 3 == 1:
            b = io.BytesIO()
            _content(i, 29, 31).convert("L").save(b, "JPEG", quality=85)
            out.append((b.getvalue(), 1, False))
    for o in (3, 6, 8):
        out.append((_oriented(30 + o, 45, 27, o, sub=2), 1, True))
    return out


@pytest.mark.gpu
@pytest.mark.parametrize("d", [1, 4])
@pytest.mark.parametrize("cs", [ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.GRAYSCALE])
def test_decode_batch_mixed(d, cs):
    inputs = _mixed_inputs()
    orient = any(o for _, _, o in inputs)
    opts = options(cs, "libjpeg", d, orient=True)
    res = decode_batch([x[0] for x in inputs], opts, threads=3)
    for (data, _, o), r in zip(inputs, res):
        assert not isinstance(r, Exception), r
        want = _want(data, cs, d, orient=o)
        if want is None:   # (Pillow does not draft that far)
            continue
        assert np.array_equal(np.frombuffer(r, np.uint8), want.reshape(-1))
    assert orient


@pytest.mark.gpu
def test_decode_batch_device_out_and_multi():
    torch = pytest.importorskip("torch")
    inputs = _mixed_inputs()
    datas = [x[0] for x in inputs]
    opts = options(ColorSpace.RGB, "libjpeg", 1, orient=True)
    wants = [_want(data, ColorSpace.RGB, 1, orient=o) for data, _, o in inputs]
    bufs = [torch.empty(w.size, dtype=torch.uint8, device="cuda:0") for w in wants]
    res = decode_batch(datas, opts, device_out=[(b.data_ptr(), b.numel()) for b in bufs])
    for r, b, w in zip(res, bufs, wants):
        assert not isinstance(r, Exception), r
        assert np.array_equal(b.cpu().numpy(), w.reshape(-1))
    n_dev = torch.cuda.device_count()
    for devs in ([0], [0, 1]) if n_dev > 1 else ([0],):
        res = decode_batch(datas, opts, devices=devs)
        for r, w in zip(res, wants):
            assert np.array_equal(np.frombuffer(r, np.uint8), w.reshape(-1))
        res = decode_batch(datas[:1], opts, devices=devs)
        assert np.array_equal(np.frombuffer(res[0], np.uint8), wants[0].reshape(-1))


@pytest.mark.gpu
def test_device_out_f16_chw():
    torch = pytest.importorskip("torch")
    from zune_jpeg_b200 import gpu
    datas = [FILES[n]() for n in ("444", "ycck", "prog420c")]
    mean, std = [120.0, 110.0, 100.0], [60.0, 61.0, 62.0]
    desc = gpu.OutputDesc(layout="CHW", dtype="f16", mean=mean, inv_std=[1.0 / v for v in std])
    wants = [_want(d, ColorSpace.RGB) for d in datas]
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
    datas = [cmyk_jpeg(40, 300, 200), set_transform(cmyk_jpeg(41, 260, 330, sub=2), 2), ycck_2211_jpeg(42, 280, 250),
             _oriented(43, 310, 240, 6)]
    S, out = 256, 224
    tf = T.Compose([T.Resize(S, interpolation=T.InterpolationMode.BICUBIC), T.CenterCrop(out)])
    opts = options(ColorSpace.RGB, "libjpeg", 1, orient=True)
    arr, errs = decode_batch_resized(datas, gpu.Resize((out, out), filter="pil_bicubic", short_side=S), options=opts)
    assert errs == [None] * len(datas)
    t = arr.to_torch().cpu().numpy()
    for i, data in enumerate(datas):
        im = ImageOps.exif_transpose(Image.open(io.BytesIO(data)).convert("RGB")) if i == 3 else Image.open(io.BytesIO(data)).convert("RGB")
        want = np.asarray(tf(im))
        got = t[i]
        if got.shape[0] == 3:
            got = got.transpose(1, 2, 0)
        assert np.array_equal(got, want), i
