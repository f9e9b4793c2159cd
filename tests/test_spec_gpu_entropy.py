"""GPU entropy decoding of spec and libjpeg output (ZJ_USE_GPU_ENTROPY): the interval kernel's spec form for scans with
restart markers and the self-synchronising decode for scans without them.  Every result must equal the host route's."""
import ctypes as C
import io
import os
import subprocess
import sys

import numpy as np
import pytest
from PIL import Image, ImageOps

import jpeg_util
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, Decoder, DecodeErrors, ZuneJpegOptions, decode_batch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _enc(seed, w, h, sub="420", q=90, gray=False, optimize=False, noise=4, **kw):
    im = jpeg_util.smooth_image(seed, w, h, gray, noise)
    bio = io.BytesIO()
    args = dict(quality=q, optimize=optimize, **kw)
    if not gray:
        args["subsampling"] = jpeg_util.SUBSAMPLING[sub]
    im.save(bio, "JPEG", **args)
    return bio.getvalue()


def _libjpeg(bit=False, cs=ColorSpace.RGB):
    o = ZuneJpegOptions().set_out_colorspace(cs).set_libjpeg_output(True)
    return o.set_gpu_entropy(True) if bit else o


# ---------------------------------------------------------------------------------------------------- ABI (CPU)
def test_abi_value_and_options_size():
    assert _ffi.USE_GPU_ENTROPY == 0x200
    assert C.sizeof(_ffi.ZjOptions) == 32
    header = open(os.path.join(ROOT, "include", "zune_jpeg_b200.h")).read()
    assert "ZJ_USE_GPU_ENTROPY = 0x200" in header


def test_options_builder_needs_spec_or_libjpeg_output():
    with pytest.raises(ValueError):
        ZuneJpegOptions().set_gpu_entropy(True)._raw()
    assert ZuneJpegOptions().set_spec_output(True).set_gpu_entropy(True)._raw().use_unsafe == _ffi.USE_SPEC_OUTPUT | 0x200
    o = ZuneJpegOptions().set_libjpeg_output(True).set_scale_denom(4).set_exif_orientation(True).set_gpu_entropy(True)
    assert o.get_gpu_entropy() and o._raw().use_unsafe == _ffi.USE_LIBJPEG_OUTPUT | 2 << _ffi.USE_SCALE_SHIFT | 0x100 | 0x200
    assert ZuneJpegOptions().set_libjpeg_output(True)._raw().use_unsafe == _ffi.USE_LIBJPEG_OUTPUT


def _opts(spec):
    return ZuneJpegOptions().set_spec_output(True) if spec else ZuneJpegOptions().set_libjpeg_output(True)


@pytest.mark.parametrize("spec", [False, True])
def test_coefficients_ignore_the_bit(spec):
    data = _enc(3, 61, 45, "420", 85)
    ia, pa = Decoder.new_with_options(_opts(spec)).decode_coefficients(data)
    ib, pb = Decoder.new_with_options(_opts(spec).set_gpu_entropy(True)).decode_coefficients(data)
    assert (ia.width, ia.height, ia.flags) == (ib.width, ib.height, ib.flags)
    assert len(pa) == len(pb) and all(np.array_equal(x, y) for x, y in zip(pa, pb))


@pytest.mark.gpu
@pytest.mark.parametrize("spec", [False, True])
def test_decode_buffer_ignores_the_bit(spec):
    data = _enc(3, 61, 45, "420", 85)
    assert Decoder.new_with_options(_opts(spec)).decode_buffer(data) == Decoder.new_with_options(_opts(spec).set_gpu_entropy(True)).decode_buffer(data)


# ---------------------------------------------------------------------------------------------------- GPU corpus
def _corpus():
    files = []
    k = 0
    for sub in ("420", "422", "444", "gray"):
        for q in (50, 75, 90, 100):
            for opt in (False, True):
                for (w, h) in ((1, 1), (17, 9), (99, 70), (333, 250)):
                    if (w, h) == (333, 250) and q != 90:
                        continue
                    k += 1
                    files.append(_enc(k, w, h, sub if sub != "gray" else "444", q, gray=sub == "gray", optimize=opt))
    return files


DRI_CASES = [("420", dict(restart_marker_rows=1)), ("420", dict(restart_marker_rows=2)), ("422", dict(restart_marker_rows=1)),
             ("444", dict(restart_marker_blocks=1)), ("420", dict(restart_marker_blocks=1)), ("420", dict(restart_marker_blocks=2)),
             ("444", dict(restart_marker_blocks=2)), ("422", dict(restart_marker_blocks=1))]


def _dri_corpus():
    # (scans of more than 64 KB: the host stage's interval-parallel form, which applies the GPU kernel's acceptance rule, runs)
    return [_enc(100 + k, 701, 487, sub, 95, noise=16, **kw) for k, (sub, kw) in enumerate(DRI_CASES)]


def _interval_form_accepts(data):
    """the host stage's interval-parallel form took every interval (the rule the spec interval kernel applies)"""
    d = Decoder.new_with_options(_libjpeg().set_num_threads(4))
    d.decode_coefficients(data)
    return d.entropy_segments() > 0


def test_dri_corpus_is_taken_by_the_interval_rule():
    # with Q8 the countdown ticks once per component, yet for these files every interval ends where the next one starts
    assert [_interval_form_accepts(d) for d in _dri_corpus()] == [True] * len(DRI_CASES)


def _pillow(data, gray=False):
    im = Image.open(io.BytesIO(data))
    return np.asarray(im.convert("L" if gray else "RGB"))


def _both(files, opts_bit, opts_plain, **kw):
    s1, s0 = {}, {}
    got = decode_batch(files, opts_bit, threads=4, gpu_entropy=True, stats=s1, **kw)
    want = decode_batch(files, opts_plain, threads=4, gpu_entropy=True, stats=s0, **kw)
    return got, want, s1["gpu_entropy"], s0["gpu_entropy"]


@pytest.mark.gpu
def test_no_dri_files_equal_the_host_route_and_pillow():
    files = _corpus()
    got, want, n1, n0 = _both(files, _libjpeg(True), _libjpeg(False))
    assert n0 == 0 and n1 == len(files)
    assert [g == w for g, w in zip(got, want)] == [True] * len(files)
    assert [g == _pillow(d).tobytes() for g, d in zip(got, files)] == [True] * len(files)
    # spec output too
    spec = ZuneJpegOptions().set_spec_output(True)
    got, want, n1, n0 = _both(files, spec.set_gpu_entropy(True), spec)
    assert n1 == len(files) and got == want


@pytest.mark.gpu
def test_dri_files_take_the_spec_interval_kernel():
    files = _dri_corpus()
    got, want, n1, n0 = _both(files, _libjpeg(True), _libjpeg(False))
    assert n0 == 0 and n1 == sum(_interval_form_accepts(d) for d in files) == len(files)
    assert [g == w for g, w in zip(got, want)] == [True] * len(files)
    # whole MCU rows per interval: Pillow's pixels (with DRI = 1 or 2 MCUs the host stage's Q8 bookkeeping decides what the
    # countdown does, and the GPU form gives the host stage's pixels)
    assert [g == _pillow(d).tobytes() for g, d in zip(got[:3], files[:3])] == [True] * 3


@pytest.mark.gpu
def test_large_image_scaled_and_oriented():
    big = _enc(7, 8192, 8192, "420", 90)
    files = [big, _enc(8, 1000, 700, "420", 90)]
    got, want, n1, _ = _both(files, _libjpeg(True), _libjpeg(False))
    assert n1 == 2 and got == want
    o = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB).set_libjpeg_output(True).set_scale_denom(4)
    got, want, n1, _ = _both(files[1:], o.set_gpu_entropy(True), o)
    assert n1 == 1 and got == want
    im = jpeg_util.smooth_image(9, 203, 101)
    ex = im.getexif()
    ex[0x0112] = 6
    bio = io.BytesIO()
    im.save(bio, "JPEG", quality=90, exif=ex.tobytes())
    data = bio.getvalue()
    o = _libjpeg().set_exif_orientation(True)
    got, want, n1, _ = _both([data], o.set_gpu_entropy(True), o)
    assert n1 == 1 and got == want
    assert got[0] == np.asarray(ImageOps.exif_transpose(Image.open(io.BytesIO(data))).convert("RGB")).tobytes()


def _damaged():
    base = _enc(20, 200, 150, "420", 90)
    sos = base.index(b"\xff\xda")
    body = sos + 2 + int.from_bytes(base[sos + 2:sos + 4], "big")
    out = []
    out.append(base[:len(base) - 2000])                                       # truncated, no EOI
    flipped = bytearray(base)
    flipped[body + 300:body + 308] = b"\xff\x00" * 4
    out.append(bytes(flipped))                                                # 32 one bits: a code no table holds
    stray = bytearray(base)
    stray[body + 500:body + 502] = b"\xff\xc4"
    out.append(bytes(stray))                                                  # stray marker in the scan
    rst = bytearray(base)
    rst[body + 700:body + 702] = b"\xff\xd3"
    out.append(bytes(rst))                                                    # RSTn without DRI
    out.append(base[:len(base) - 600] + b"\xff\xd9")                          # data ends mid-scan
    dri = _enc(21, 200, 150, "420", 90, restart_marker_rows=1)
    d = dri.index(b"\xff\xdd")
    out.append(dri[:d + 4] + (3).to_bytes(2, "big") + dri[d + 6:])          # mis-declared DRI
    prog = _enc(22, 200, 150, "420", 90, progressive=True)
    s2 = prog.index(b"\xff\xda", prog.index(b"\xff\xda") + 2)
    out.append(base[:-2] + prog[s2:])                                         # a trailing second scan
    return out


@pytest.mark.gpu
def test_mixed_and_damaged_files_give_the_host_results():
    good = [_enc(30, 120, 90, "420", 90), _enc(31, 120, 90, "420", 90, restart_marker_rows=1)]
    other = [_enc(32, 120, 90, "420", 90, progressive=True), _enc(33, 97, 61, "444", 80)]
    cmyk = Image.fromarray(np.random.default_rng(1).integers(0, 255, (40, 48, 4), np.uint8), "CMYK")
    bio = io.BytesIO()
    cmyk.save(bio, "JPEG", quality=90)
    other.append(bio.getvalue())
    other.append(b"\xff\xd8\xff\xc0\x00\x05")                                # header error
    damaged = _damaged()
    files = good + other + damaged
    got, want, n1, n0 = _both(files, _libjpeg(True), _libjpeg(False))
    # the two good files and the 4:4:4 one; no progressive, CMYK, header-error or damaged file
    assert n0 == 0 and n1 == 3
    for d in damaged:
        s = {}
        decode_batch([d], _libjpeg(True), threads=4, gpu_entropy=True, stats=s)
        assert s["gpu_entropy"] == 0
    for g, w in zip(got, want):
        if isinstance(w, DecodeErrors):
            assert isinstance(g, DecodeErrors) and str(g) == str(w) and g.args == w.args
        else:
            assert g == w


@pytest.mark.gpu
def test_device_out_and_resized_equal_the_host_route():
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import decode_batch_resized
    files = [_enc(40, 640, 362, "420", 90), _enc(41, 333, 250, "422", 95, optimize=True), _enc(42, 500, 301, "444", 85),
             _enc(43, 401, 299, "420", 90, restart_marker_rows=1)]
    pil = [_pillow(d) for d in files]
    for desc in (None, gpu.OutputDesc("CHW", "f16", False, 0, (0.0,) * 4, (1.0,) * 4)):
        res = []
        for bit in (True, False):
            es = 1 if desc is None else 2
            outs = [gpu.DeviceBuffer(p.size * es) for p in pil]
            stats = {}
            r = decode_batch(files, _libjpeg(bit), threads=4, device_out=[(o.ptr, o.nbytes) for o in outs], desc=desc, stats=stats)
            assert r == [o.nbytes for o in outs]
            assert stats["gpu_entropy"] == (len(files) if bit else 0)
            res.append([o.download().tobytes() for o in outs])
        assert res[0] == res[1]
        if desc is None:
            assert res[0] == [p.tobytes() for p in pil]
    rz = gpu.Resize((224, 224), "pil_bicubic", short_side=256)
    for desc in (None, gpu.OutputDesc("CHW", "f16", False, 0, (0.0,) * 4, (1.0,) * 4)):
        outs = []
        for bit in (True, False):
            stats = {}
            out, errs = decode_batch_resized(files, rz, desc, None, _libjpeg(bit), threads=4, stats=stats)
            assert errs == [None] * len(files) and stats["gpu_entropy"] == (len(files) if bit else 0)
            outs.append(out.download())
        assert outs[0].tobytes() == outs[1].tobytes()
        if desc is None:   # u8 HWC: Pillow's decode, torchvision's Resize(256) + CenterCrop(224) on it
            from torchvision.transforms import InterpolationMode, v2
            tv = v2.Compose([v2.Resize(256, interpolation=InterpolationMode.BICUBIC), v2.CenterCrop(224)])
            for k, p in enumerate(pil):
                assert outs[0][k].tobytes() == np.asarray(tv(Image.fromarray(p))).tobytes(), k


@pytest.mark.gpu
def test_small_budget_covers_several_sub_batches():
    code = ("import sys; sys.path[:0] = [%r, %r]\n"
            "from test_spec_gpu_entropy import _corpus, _libjpeg\n"
            "from zune_jpeg_b200.decoder import decode_batch\n"
            "from test_spec_gpu_entropy import _enc\n"
            "files = [_enc(60 + k, 1200, 900, '420', 90) for k in range(24)] + _corpus()[:16]\n"
            "s = {}\n"
            "a = decode_batch(files, _libjpeg(True), threads=4, gpu_entropy=True, stats=s)\n"
            "b = decode_batch(files, _libjpeg(False), threads=4)\n"
            "assert a == b and s['gpu_entropy'] == len(files), s\n"
            "print('ok')\n") % (ROOT, os.path.join(ROOT, "tests"))
    env = dict(os.environ, ZJ_GPU_ENTROPY_BUDGET_MB="64")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-2000:]
