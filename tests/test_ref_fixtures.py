"""The reference's own JPEG files through the PRODUCT path on the GPU (BASELINE configs[0] and the inputs of the
reference's integration tests, tests/{large,medium,random}_images.rs, which only eyeball their outputs).

Every file under tests/golden/ref/ (verbatim copies of files of the reference's test-images/ and tests/inputs/, see
tests/ref_files.py) is decoded by Decoder.decode_buffer, decode_batch and decode_batch(gpu_entropy=True) and must
equal, byte for byte, the oracle fed with the planes of the SEQUENTIAL host stage."""
import glob
import hashlib
import os

import numpy as np
import pytest

import oracle
import ref_files
from zune_jpeg_b200.decoder import ColorSpace, DecodeErrors, Decoder, ZuneJpegOptions, decode_batch


def _want(data: bytes, out_cs: ColorSpace):
    """oracle pixels from the planes of the sequential host stage (1 thread = the reference's loop), or the DecodeErrors"""
    opts = ZuneJpegOptions().set_out_colorspace(out_cs).set_num_threads(1)
    try:
        img, planes = Decoder.new_with_options(opts).decode_coefficients(data)
    except DecodeErrors as e:
        return e
    for z in range(img.n_comp):
        img.comp[z].coeff = planes[z].ctypes.data if planes[z].size else None
    return oracle.reconstruct(img, threads=os.cpu_count() or 1)


def test_fixture_copies_are_the_reference_files():
    """tests/golden/ref/ holds the files of its manifest and nothing else, and each, as ref_files.read() returns it, has
    the recorded length and SHA-256."""
    stored = sorted(os.path.basename(p) for p in glob.glob(os.path.join(ref_files.DIR, "*.jp*g")))
    assert len(stored) >= 7 and stored == ref_files.NAMES
    for name in ref_files.NAMES:
        data = ref_files.read(name)
        assert len(data) == ref_files.MANIFEST[name]["bytes"], name
        assert hashlib.sha256(data).hexdigest() == ref_files.MANIFEST[name]["sha256"], name


@pytest.mark.gpu
@pytest.mark.parametrize("name", ref_files.NAMES)
def test_reference_file_through_the_product(name):
    data = ref_files.read(name)
    for out_cs in (ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.GRAYSCALE, ColorSpace.YCbCr):
        want = _want(data, out_cs)
        opts = ZuneJpegOptions().set_out_colorspace(out_cs)
        if isinstance(want, DecodeErrors):      # test-arithmetic-coding.jpg: same variant and message from every front door
            with pytest.raises(DecodeErrors) as e:
                Decoder.new_with_options(opts).decode_buffer(data)
            assert (e.value.variant, e.value.message) == (want.variant, want.message)
            assert isinstance(decode_batch([data], opts, threads=2)[0], DecodeErrors)
            continue
        d = Decoder.new_with_options(opts)      # default 4 threads: restart-interval-parallel host stage when DRI is present
        got = np.frombuffer(d.decode_buffer(data), np.uint8)
        assert got.size == d.width() * d.height() * d.get_output_colorspace().num_components()
        assert np.array_equal(got, want), (name, out_cs, "decode_buffer")
        if out_cs in (ColorSpace.RGB, ColorSpace.GRAYSCALE):
            a, b = decode_batch([data, data], opts, threads=2)
            assert a == want.tobytes() and b == a, (name, out_cs, "decode_batch")
            stats = {}
            g = decode_batch([data], opts, threads=2, gpu_entropy=True, stats=stats)[0]
            assert g == want.tobytes(), (name, out_cs, "decode_batch gpu_entropy", stats)


@pytest.mark.gpu
def test_single_qt_restart_fixture_takes_the_gpu_entropy_route():
    """single_qt.jpeg (DRI = 1005 MCUs: not row-aligned, 4:2:2) is the reference's one real restart-marker file."""
    data = ref_files.read("single_qt.jpeg")
    stats = {}
    got = decode_batch([data], threads=2, gpu_entropy=True, stats=stats)[0]
    assert got == _want(data, ColorSpace.RGB).tobytes()
    d = Decoder.new()
    d.decode_coefficients(data)
    assert d.entropy_segments() > 0            # host form: intervals side by side
    assert stats["gpu_entropy"] == 1           # GPU form accepted every interval
