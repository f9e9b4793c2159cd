"""EXIF orientation of spec and libjpeg output (include/zune_jpeg_b200.h next to ZJ_FLAG_ORIENT_SHIFT, DESIGN.md section 4.6.3):
the parser against Pillow's decision, the numpy statement (the scaled / libjpeg statement, then Pillow's Transpose) against
ImageOps.exif_transpose and torchvision's decode_jpeg, the ABI, and on the GPU every route bit for bit against the statement."""
from __future__ import annotations

import ctypes as C
import io
import struct
import warnings

import numpy as np
import pytest
from PIL import Image, ImageOps

import jpeg_util
import oracle
import util
from test_scaled_output import MODES, QTS, _flags, scaled_expected
from test_spec_output import _device_run, spec_expected, spec_planes
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch

SPEC, ISLOW = _ffi.VARIANT_SPEC, _ffi.FLAG_ISLOW
XMP_HDR = b"http://ns.adobe.com/xap/1.0/\0"


# ------------------------------------------------------------------------------------------------ statement
def orient_pixels(px: np.ndarray, o: int) -> np.ndarray:
    """Pillow's Transpose for orientation o of an H x W x nc image (exif_transpose's table)"""
    return {1: lambda a: a, 2: lambda a: a[:, ::-1], 3: lambda a: a[::-1, ::-1], 4: lambda a: a[::-1],
            5: lambda a: a.transpose(1, 0, 2), 6: lambda a: np.rot90(a, -1), 7: lambda a: a[::-1, ::-1].transpose(1, 0, 2),
            8: lambda a: np.rot90(a, 1)}[o](px)


def orient_flags(o: int) -> int:
    return (o - 1) << _ffi.FLAG_ORIENT_SHIFT


def oriented_expected(img, planes) -> np.ndarray:
    """The statement: the image's scaled / libjpeg / spec statement, then the transform of its orientation bits"""
    o = ((img.flags & _ffi.FLAG_ORIENT_MASK) >> _ffi.FLAG_ORIENT_SHIFT) + 1
    flags = img.flags
    img.flags &= ~_ffi.FLAG_ORIENT_MASK
    try:
        flat = scaled_expected(img, planes) if img.flags & ISLOW else spec_expected(img, planes)
        w, h = _ffi.image_size(img)
    finally:
        img.flags = flags
    px = flat.reshape(h, w, -1)
    return np.ascontiguousarray(orient_pixels(px, o)).reshape(-1)


# ------------------------------------------------------------------------------------------------ crafted metadata
def with_app1(data: bytes, payloads) -> bytes:
    """`data` with APP1 segments holding `payloads` spliced in after SOI"""
    return data[:2] + b"".join(b"\xff\xe1" + struct.pack(">H", len(p) + 2) + p for p in payloads) + data[2:]


def tiff(entries, bo="<", ifd=8, extra=b"") -> bytes:
    """A TIFF header and IFD0 of `entries` = (tag, type, count, 4-byte value field)"""
    head = (b"II*\0" if bo == "<" else b"MM\0*") + struct.pack(bo + "I", ifd)
    body = struct.pack(bo + "H", len(entries)) + b"".join(struct.pack(bo + "HHI", t, ty, c) + v for t, ty, c, v in entries)
    return head + body + struct.pack(bo + "I", 0) + extra


def short(v, bo="<"):
    return struct.pack(bo + "HH", v, 0)


def exif(o, bo="<", typ=3):
    return b"Exif\0\0" + tiff([(0x0100, 4, 1, struct.pack(bo + "I", 64)), (0x0112, typ, 1, short(o, bo) if typ == 3 else struct.pack(bo + "I", o))], bo)


def pillow_orientation(data: bytes) -> int:
    """exif_transpose's decision: the orientation Pillow's getexif() gives if it is 2-8, else 1 (also where Pillow raises)"""
    with warnings.catch_warnings():
        warnings.simplefilter("ignore")
        try:
            o = Image.open(io.BytesIO(data)).getexif().get(0x0112, 1)
        except Exception:
            return 1
    return o if o in range(2, 9) else 1


BASE = jpeg_util.synth_jpeg(21, 37, 29, "420", 90)
EXIF_CASES = {
    **{f"ii_short_{o}": [exif(o)] for o in range(1, 9)},
    **{f"mm_short_{o}": [exif(o, ">")] for o in (3, 6)},
    **{f"ii_long_{o}": [exif(o, typ=4)] for o in (5, 8)},
    "mm_long_7": [exif(7, ">", 4)],
    "count_2": [b"Exif\0\0" + tiff([(0x0112, 3, 2, struct.pack("<HH", 6, 3))])],
    "count_3_at_offset": [b"Exif\0\0" + tiff([(0x0112, 3, 3, struct.pack("<I", 26))], extra=struct.pack("<HHH", 8, 3, 3))],
    "value_0": [exif(0)],
    "value_9": [exif(9)],
    "no_tag": [b"Exif\0\0" + tiff([(0x0100, 4, 1, struct.pack("<I", 64))])],
    "ifd0_past_the_data": [b"Exif\0\0" + tiff([(0x0112, 3, 1, short(6))], ifd=4000)],
    "truncated_header": [b"Exif\0\0II*\0\x08"],
    "bad_header": [b"Exif\0\0XX*\0" + b"\0" * 24],
    "bad_data_offset_before_the_tag": [b"Exif\0\0" + tiff([(0x0100, 4, 4, struct.pack("<I", 5000)), (0x0112, 3, 1, short(6))])],
    "truncated_after_the_tag": [(b"Exif\0\0" + tiff([(0x0112, 3, 1, short(6)), (0x0100, 3, 1, short(6))]))[:6 + 8 + 2 + 12 + 5]],
    "byte_type": [b"Exif\0\0" + tiff([(0x0112, 1, 1, b"\x06\0\0\0")])],
    "repeated_tag": [b"Exif\0\0" + tiff([(0x0112, 3, 1, short(6)), (0x0112, 3, 1, short(8))])],
    "two_exif_segments": [(b"Exif\0\0" + tiff([(0x0112, 3, 1, short(6))]))[:18], b"Exif\0\0" + (b"Exif\0\0" + tiff([(0x0112, 3, 1, short(6))]))[18:]],
    "xmp_attribute_6": [XMP_HDR + b'<x:xmpmeta><rdf:Description tiff:Orientation="6"/></x:xmpmeta>'],
    "xmp_element_8": [XMP_HDR + b"<tiff:Orientation>8</tiff:Orientation>"],
    "xmp_last_segment_wins": [XMP_HDR + b'tiff:Orientation="3"', XMP_HDR + b'tiff:Orientation="5"'],
    "xmp_first_match": [XMP_HDR + b'tiff:Orientation="x" tiff:Orientation>7 tiff:Orientation="2"'],
    "exif_1_with_xmp_6": [exif(1), XMP_HDR + b'tiff:Orientation="6"'],
    "no_tag_with_xmp_6": [b"Exif\0\0" + tiff([(0x0100, 4, 1, struct.pack("<I", 64))]), XMP_HDR + b'tiff:Orientation="6"'],
    "ifd0_past_the_data_with_xmp_7": [b"Exif\0\0" + tiff([(0x0112, 3, 1, short(6))], ifd=4000), XMP_HDR + b'tiff:Orientation="7"'],
    "empty_exif_with_xmp_4": [b"Exif\0\0", XMP_HDR + b'tiff:Orientation="4"'],
    "bad_header_with_xmp_6": [b"Exif\0\0XX", XMP_HDR + b'tiff:Orientation="6"'],
    "other_app1": [b"Other\0" + tiff([(0x0112, 3, 1, short(6))])],
    # the tag in the 11th of 13 Exif segments (3 TIFF bytes each): every segment's bytes are appended, however many there are
    "thirteen_exif_segments": [b"Exif\0\0" + _t[k:k + 3] for _t in [tiff([(0x0100, 4, 1, struct.pack("<I", 64)), (0x0112, 3, 1, short(7))])]
                               for k in range(0, len(_t), 3)],
}


def exif_decoder(scale=1, cs=ColorSpace.RGB, orient=True, threads=4):
    opts = ZuneJpegOptions().set_out_colorspace(cs).set_num_threads(threads)
    opts = opts.set_libjpeg_output(True).set_scale_denom(scale) if scale else opts.set_spec_output(True)
    return Decoder.new_with_options(opts.set_exif_orientation(orient))


@pytest.mark.parametrize("name", list(EXIF_CASES))
def test_parser_matches_pillow_decision(name):
    data = with_app1(BASE, EXIF_CASES[name])
    want = pillow_orientation(data)
    for dec in (exif_decoder(), Decoder.new_with_options(ZuneJpegOptions())):   # read whatever the options
        dec.read_headers(data)
        assert dec.exif_orientation() == want, (name, want)
    img, _ = exif_decoder().decode_coefficients(data)
    assert (img.flags & _ffi.FLAG_ORIENT_MASK) >> _ffi.FLAG_ORIENT_SHIFT == want - 1


def test_pillow_saved_exif_and_markers_after_the_first_sos():
    """Files Pillow writes with save(exif=...); an APP1 after the first SOS (between progressive scans) is not read"""
    for o in range(1, 9):
        e = Image.Exif()
        e[0x0112] = o
        bio = io.BytesIO()
        jpeg_util.smooth_image(3, 40, 24, False).save(bio, "JPEG", exif=e.tobytes())
        dec = exif_decoder()
        dec.read_headers(bio.getvalue())
        assert dec.exif_orientation() == pillow_orientation(bio.getvalue()) == o
    prog = jpeg_util.synth_jpeg(4, 64, 48, "420", 90, progressive=True)
    sos = prog.index(b"\xff\xda")
    nxt = prog.index(b"\xff\xc4", sos)   # the DHT of the second scan
    late = prog[:nxt] + b"\xff\xe1" + struct.pack(">H", len(exif(6)) + 2) + exif(6) + prog[nxt:]
    dec = exif_decoder()
    img, _ = dec.decode_coefficients(late)
    assert dec.exif_orientation() == 1 and img.flags & _ffi.FLAG_ORIENT_MASK == 0
    assert Decoder.new_with_options(ZuneJpegOptions()).exif_orientation() == 1   # before any headers


SYNTH = [  # (seed, width, height, subsampling, progressive, gray): every sampling, sizes not multiples of 8
    (31, 157, 93, "420", False, False), (32, 130, 77, "422", False, False), (33, 101, 67, "444", False, False),
    (34, 99, 45, "444", False, True), (35, 123, 71, "420", True, False), (36, 21, 13, "420", False, False),
]


def _synth(case, o):
    seed, w, h, sub, prog, gray = case
    return with_app1(jpeg_util.synth_jpeg(seed, w, h, sub, 90, prog, gray), [exif(o)]), gray


def _pillow_oriented(data, d, gray):
    """Pillow: draft to 1/d (when Pillow drafts that far), then exif_transpose; None otherwise"""
    im = Image.open(io.BytesIO(data))
    mode = "L" if gray else "RGB"
    w, h = im.size
    if d > 1:
        im.draft(mode, (max(w // d, 1), max(h // d, 1)))
        if im.size != _ffi.scaled_size(w, h, d):
            return None
    return np.asarray(ImageOps.exif_transpose(im.convert(mode)))


@pytest.mark.parametrize("case", SYNTH, ids=lambda c: "%dx%d_%s%s%s" % (c[1], c[2], c[3], "_prog" if c[4] else "", "_gray" if c[5] else ""))
def test_statement_equals_pillow_exif_transpose(case):
    n = 0
    for d in (1, 2, 4, 8):
        data, gray = _synth(case, 1)
        cs = ColorSpace.GRAYSCALE if gray else ColorSpace.RGB
        img, planes = exif_decoder(scale=d, cs=cs, orient=False).decode_coefficients(data)
        for o in range(1, 9):
            data, _ = _synth(case, o)
            want = _pillow_oriented(data, d, gray)
            if want is None:
                continue
            oimg, oplanes = exif_decoder(scale=d, cs=cs).decode_coefficients(data)
            assert oimg.flags == img.flags | orient_flags(o)
            assert all(np.array_equal(a, b) for a, b in zip(planes, oplanes))
            got = oriented_expected(oimg, oplanes)
            assert _ffi.image_size(oimg) == (want.shape[1], want.shape[0])
            assert int(np.abs(got.astype(int) - want.reshape(-1).astype(int)).max()) == 0, (case, d, o)
            n += 1
    assert n >= 8


@pytest.mark.parametrize("case", SYNTH[:3], ids=["420", "422", "444"])
def test_statement_equals_torchvision_decode_jpeg(case):
    tv = pytest.importorskip("torchvision.io")
    import torch
    for o in range(1, 9):
        data, _ = _synth(case, o)
        img, planes = exif_decoder(scale=1).decode_coefficients(data)
        w, h = _ffi.image_size(img)
        t = tv.decode_jpeg(torch.frombuffer(bytearray(data), dtype=torch.uint8), mode=tv.ImageReadMode.RGB, apply_exif_orientation=True)
        assert np.array_equal(oriented_expected(img, planes), t.permute(1, 2, 0).contiguous().numpy().reshape(-1)), (case, o)


def test_abi_flags_sizes_and_use_unsafe():
    lib = _ffi.load()
    rng = np.random.default_rng(3)
    planes = spec_planes(rng, 41, 23, 3, 2, 2)
    img = util.make_image(41, 23, planes, QTS, 2, 2, _ffi.CS_RGBA, SPEC)
    desc = _ffi.ZjOutputDesc()
    lib.zj_output_desc_default(C.byref(desc))
    ow, oh, oc = C.c_uint32(), C.c_uint32(), C.c_uint32()
    for base in (0, ISLOW, _flags(4)):
        sw, sh = _ffi.scaled_size(41, 23, 4 if base & _ffi.FLAG_SCALE_MASK else 1)
        for o in range(1, 9):
            img.flags = base | orient_flags(o)
            assert lib.zj_validate_image(C.byref(img)) == 0
            assert lib.zj_output_size(C.byref(img)) == sw * sh * 4
            assert lib.zj_consumer_output_shape(C.byref(img), C.byref(desc), C.byref(ow), C.byref(oh), C.byref(oc)) == 0
            assert (ow.value, oh.value) == ((sh, sw) if o >= 5 else (sw, sh)) == _ffi.image_size(img)
    # the bits are valid on spec images only; strip cuts stay refused
    for variant in (_ffi.VARIANT_X86, _ffi.VARIANT_SCALAR):
        img.variant, img.flags = variant, orient_flags(6)
        assert lib.zj_validate_image(C.byref(img)) == _ffi.ERR_INVALID_ARG and lib.zj_output_size(C.byref(img)) == 0
    img.variant = SPEC
    sub, off, nb = _ffi.ZjImage(), C.c_size_t(), C.c_size_t()
    assert lib.zj_image_strip_range(C.byref(img), 0, 1, C.byref(sub), C.byref(off), C.byref(nb), None) == _ffi.ERR_UNSUPPORTED
    # use_unsafe: ZJ_USE_EXIF_ORIENTATION ORed into 2, 3 and 3 | k << 4 orients; every other value keeps its meaning
    data = with_app1(jpeg_util.synth_jpeg(5, 61, 35, "422", 90), [exif(6)])
    for v, variant, flags in ((0x102, SPEC, orient_flags(6)), (0x103, SPEC, ISLOW | orient_flags(6)),
                              (0x123, SPEC, ISLOW | _flags(4) | orient_flags(6)), (0x100, _ffi.VARIANT_X86, 0), (0x101, _ffi.VARIANT_X86, 0),
                              (0x112, _ffi.VARIANT_X86, 0), (0x143, _ffi.VARIANT_X86, 0), (0x02, SPEC, 0), (0x13, SPEC, ISLOW | _flags(2))):
        o = _ffi.ZjOptions()
        lib.zj_options_default(C.byref(o))
        o.use_unsafe = v
        dec = Decoder.new_with_options(ZuneJpegOptions())
        lib.zj_decoder_free(dec._h)
        dec._h = lib.zj_decoder_new(C.byref(o))
        got, _ = dec.decode_coefficients(data)
        assert (got.variant, got.flags & ~_ffi.FLAG_PROGRESSIVE) == (variant, flags), hex(v)
        assert dec.exif_orientation() == 6
    assert C.sizeof(_ffi.ZjOptions) == 32


def test_options_builder():
    o = ZuneJpegOptions()
    assert o.get_exif_orientation() is False
    e = o.set_exif_orientation(True)
    assert e.get_exif_orientation() and not o.get_exif_orientation()
    assert e.set_spec_output(True)._raw().use_unsafe == 0x102
    assert e.set_libjpeg_output(True)._raw().use_unsafe == 0x103
    assert e.set_libjpeg_output(True).set_scale_denom(8)._raw().use_unsafe == 0x133
    with pytest.raises(ValueError):
        e._raw()
    with pytest.raises(ValueError):
        Decoder.new_with_options(e.set_use_unsafe(False))
    assert _ffi.oriented_size(5, 3, 6) == (3, 5) and _ffi.oriented_size(5, 3, 4) == (5, 3)


# ------------------------------------------------------------------------------------------------ GPU
def _planes_image(rng, w, h, mode, cs, kind, o=1, n_comp=3):
    """kind: 0 X86, 1 spec, 2 libjpeg, 3-5 libjpeg at 1/2, 1/4, 1/8; o: orientation (spec kinds)"""
    hs, vs = MODES[mode]
    planes = spec_planes(rng, w, h, n_comp, hs, vs)
    img = util.make_image(w, h, planes, QTS[:n_comp], hs, vs, cs, SPEC if kind else _ffi.VARIANT_X86)
    img.flags = (0 if kind < 2 else (ISLOW if kind == 2 else _flags(1 << (kind - 2)))) | (orient_flags(o) if kind else 0)
    want = oracle.reconstruct(img) if kind == 0 else oriented_expected(img, planes)
    return img, planes, want


@pytest.mark.gpu
def test_planes_routes_mixed_call():
    """One call mixing X86, spec, libjpeg and scaled images, oriented ones at every o: host, device (offset 0 and 1) and zj_batch"""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(4000)
    shapes = [(640, 362, "hv", 0), (333, 250, "h", 0), (255, 33, "v", 2), (100, 17, "none", 5), (17, 9, "hv", 1), (637, 480, "hv", 0),
              (99, 45, "none", 1), (321, 40, "h", 6), (1023, 77, "hv", 5), (64, 64, "v", 0), (1, 7, "hv", 0), (3, 2, "h", 5)]
    imgs, keep, wants = [], [], []
    for k in range(48):
        w, h, mode, cs = shapes[k % len(shapes)]
        img, planes, want = _planes_image(rng, w, h, mode, cs, k % 6, 1 + (k * 5) % 8)
        imgs.append(img); keep.append(planes); wants.append(want)
    assert {((im.flags >> 4) & 7) for im in imgs if im.variant == SPEC} == set(range(8))
    for use_batch in (False, True):
        for off in (0, 1):
            for g, want, img in zip(_device_run(imgs, keep, use_batch, off), wants, imgs):
                assert np.array_equal(g, want), (img.width, img.height, img.flags, use_batch, off)
    for g, want in zip(gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want)
    devs = [0, 1] if gpu.device_count() >= 2 else [0, 0]
    for g, want in zip(gpu.reconstruct_multi(imgs[1:2], devs) + gpu.reconstruct_multi(imgs, devs), wants[1:2] + wants):
        assert np.array_equal(g, want)


@pytest.mark.gpu
def test_narrow_images_and_unaligned_edges():
    """widths of 1, 3 and 5 pixels (and their transposes), RGB and RGBA, every orientation, outputs at offsets 0-3"""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(4100)
    imgs, keep, wants = [], [], []
    for w, h in ((1, 1), (1, 70), (3, 67), (5, 131), (70, 3), (131, 5), (67, 1), (5, 5)):
        for cs in (_ffi.CS_RGB, _ffi.CS_RGBA):
            for o in range(1, 9):
                img, planes, want = _planes_image(rng, w, h, "hv", cs, 2 if o % 2 else 1, o)
                imgs.append(img); keep.append(planes); wants.append(want)
    for off in (0, 1, 2, 3):
        for g, want, img in zip(_device_run(imgs, keep, True, off), wants, imgs):
            assert np.array_equal(g, want), (img.width, img.height, img.out_cs, img.flags, off)
    for g, want in zip(gpu.reconstruct(imgs), wants):
        assert np.array_equal(g, want)


def _pillow_files():
    return [with_app1(jpeg_util.synth_jpeg(40 + o, 157 + 7 * o, 93 + 3 * o, ("420", "422", "444")[o % 3], 90, o == 4), [exif(o)])
            for o in range(1, 9)] + [with_app1(jpeg_util.synth_jpeg(49, 130, 77, "420", 90), [XMP_HDR + b'tiff:Orientation="6"'])]


@pytest.mark.gpu
def test_jpeg_bytes_equal_pillow_exif_transpose():
    """decode_buffer, decode_into (also >= 4 MP into pinned memory), decode_batch (one and two device slots) and device_out"""
    from zune_jpeg_b200 import gpu
    datas = _pillow_files()
    for opts in (ZuneJpegOptions().set_libjpeg_output(True), ZuneJpegOptions().set_libjpeg_output(True).set_scale_denom(2)):
        opts = opts.set_exif_orientation(True)
        d = opts.get_scale_denom()
        wants = [_pillow_oriented(data, d, False) for data in datas]
        for data, want in zip(datas, wants):
            assert Decoder.new_with_options(opts).decode_buffer(data) == want.tobytes()
            buf = np.full(want.size + 7, 0xAB, np.uint8)
            assert Decoder.new_with_options(opts).decode_into(data, buf) == want.size and buf[:want.size].tobytes() == want.tobytes()
            assert (buf[want.size:] == 0xAB).all()
        for devices in (None, [0, 1] if gpu.device_count() >= 2 else [0, 0]):
            got = decode_batch(datas, opts, threads=4, devices=devices)
            assert [g == w.tobytes() for g, w in zip(got, wants)] == [True] * len(datas), devices
        outs = [gpu.DeviceBuffer(w.size) for w in wants]
        got = decode_batch(datas, opts, threads=4, device_out=[(b.ptr, w.size) for b, w in zip(outs, wants)])
        assert got == [w.size for w in wants]
        for b, w in zip(outs, wants):
            assert b.download(w.size).tobytes() == w.tobytes()
        desc = gpu.OutputDesc("CHW", "f16", False, 0, (120.0, 110.0, 100.0, 0.0), (1 / 60, 1 / 57, 1 / 58, 1.0))
        outs = [gpu.DeviceBuffer(w.size * 2) for w in wants]
        got = decode_batch(datas, opts, threads=4, device_out=[(b.ptr, w.size * 2) for b, w in zip(outs, wants)], desc=desc)
        assert got == [w.size * 2 for w in wants]
        for b, w in zip(outs, wants):
            assert b.download(w.size * 2).tobytes() == desc.expected(w.reshape(-1), w.shape[1], w.shape[0], 3).tobytes()
    # a >= 4 MP image (the strip-pipeline size) into pinned memory
    big = with_app1(jpeg_util.synth_jpeg(50, 2600, 1700, "420", 90), [exif(8)])
    want = _pillow_oriented(big, 1, False)
    pin = gpu.PinnedBuffer(want.size)
    opts = ZuneJpegOptions().set_libjpeg_output(True).set_exif_orientation(True)
    assert Decoder.new_with_options(opts).decode_into(big, pin.array) == want.size
    assert pin.array[:want.size].tobytes() == want.tobytes()


@pytest.mark.gpu
def test_batch_resized_displayed_rois_equal_pillow():
    """decode_batch_resized with rois drawn on the displayed image: Pillow's exif_transpose -> crop -> resize, byte for byte; and
    the planes route (gpu.reconstruct_device_resized), which orients only the rectangle it reads"""
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import decode_batch_resized
    datas = _pillow_files()
    opts = ZuneJpegOptions().set_libjpeg_output(True).set_exif_orientation(True)
    ims = [ImageOps.exif_transpose(Image.open(io.BytesIO(d)).convert("RGB")) for d in datas]
    rois = [(3 + k, 5 + 2 * k, ims[k].size[0] - 9 - k, ims[k].size[1] // 2 + k) for k in range(len(datas))]
    rois[1] = None
    size, S = (40, 48), 48   # (short_side covers both output sides: Resize(S) + CenterCrop never pads)
    for rz in (gpu.Resize(size, "pil_bicubic", short_side=S), gpu.Resize(size, "pil_bilinear"), gpu.Resize(size, "bilinear")):
        out, errs = decode_batch_resized(datas, rz, gpu.OutputDesc(), rois, opts, threads=4)
        assert errs == [None] * len(datas)
        got = out.download()
        for k, im in enumerate(ims):
            px = np.asarray(im)
            want = rz.expected(px.reshape(-1), px.shape[1], px.shape[0], 3, gpu.OutputDesc(), rois[k])
            assert got[k].tobytes() == want.tobytes(), (rz, k)
            if rz.c.filter == _ffi.FILTER_PIL_BICUBIC:
                c = im.crop((rois[k][0], rois[k][1], rois[k][0] + rois[k][2], rois[k][1] + rois[k][3])) if rois[k] else im
                rw, rh, left, top = gpu.pil_geometry(c.size[0], c.size[1], size[1], size[0], S)
                pil = np.asarray(c.resize((rw, rh), Image.BICUBIC).crop((left, top, left + size[1], top + size[0])))
                assert got[k].tobytes() == pil.tobytes(), k
        # the planes route on the host stage's planes, uploaded
        keep, dimgs = [], []
        for data in datas:
            img, planes = Decoder.new_with_options(opts).decode_coefficients(data)
            bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
            for b, p in zip(bufs, planes):
                b.upload(p)
            di = _ffi.ZjImage()
            C.memmove(C.byref(di), C.byref(img), C.sizeof(di))
            for z, b in enumerate(bufs):
                di.comp[z].coeff = b.ptr
            keep.append(bufs); dimgs.append(di)
        gpu.synchronize()
        planes_out = gpu.reconstruct_device_resized(dimgs, rz, gpu.OutputDesc(), rois)
        gpu.synchronize()
        assert planes_out.download().tobytes() == got.tobytes(), rz


@pytest.mark.gpu
def test_resized_sub_batches_count_the_orientation_scratch():
    """An oriented image of the resized planes route is charged its whole stored size (the scratch its batch reconstructs into), not
    only the small rectangle it orients: with a 1 MB sub-batch budget, 0.9 MB images with 24 x 20 rois take one sub-batch each
    (reconstruction, orientation and resize: three launches per image)."""
    import os
    import subprocess
    import sys
    if os.environ.get("ZJ_CONSUMER_CHUNK_MB") != "1":      # the budget is read once per process: run this test in a child
        env = dict(os.environ, ZJ_CONSUMER_CHUNK_MB="1")
        r = subprocess.run([sys.executable, "-m", "pytest", "-x", "-q", "-m", "gpu", __file__ + "::test_resized_sub_batches_count_the_orientation_scratch"],
                           env=env, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout[-2000:] + r.stderr[-2000:]
        return
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(4200)
    n = 6
    keep, dimgs, wants = [], [], []
    for k in range(n):
        img, planes, want = _planes_image(rng, 640, 480, "hv", _ffi.CS_RGB, 2, 5 + k % 4)
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b, p in zip(bufs, planes):
            b.upload(p)
        for z, b in enumerate(bufs):
            img.comp[z].coeff = b.ptr
        keep.append((planes, bufs)); dimgs.append(img); wants.append(want)
    gpu.synchronize()
    rois = [(7 * k, 100 + 11 * k, 24, 20) for k in range(n)]
    rz = gpu.Resize((8, 12), "bilinear")
    before = gpu.launch_count()
    out = gpu.reconstruct_device_resized(dimgs, rz, gpu.OutputDesc(), rois)
    gpu.synchronize()
    assert gpu.launch_count() - before == 3 * n
    got = out.download()
    for k in range(n):
        assert got[k].tobytes() == rz.expected(wants[k], 480, 640, 3, gpu.OutputDesc(), rois[k]).tobytes(), k
