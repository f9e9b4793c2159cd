"""Isolation of the host-stage quirks Q9 / Q10 / Q11 (DESIGN.md section 2) on the reference's OWN fixtures.

The product reproduces three bugs of the reference's entropy stage on purpose, so its pixels deliberately disagree with
libjpeg on some files.  This test shows that each disagreement comes from exactly the cited reference lines: the host stage
has one test-only switch per quirk (zj_host_set_quirks); its coefficient planes are rebuilt by a spec-correct numpy pipeline
(tests/sane_ref.py: none of the pixel-path quirks) and compared with libjpeg-turbo (Pillow):

    quirks as written -> the deviation listed below;   the ONE named quirk off -> within +-5 of libjpeg everywhere.

Files: tests/golden/ref/ = copies of the reference's {test-images,tests/inputs} (reference-held vectors, tests/ref_files.py)."""
import io

import numpy as np
import pytest
from PIL import Image

import ref_files
from sane_ref import sane_pixels
from zune_jpeg_b200 import _ffi
from zune_jpeg_b200.decoder import ColorSpace, DecodeErrors, Decoder, ZuneJpegOptions

Q9, Q10, Q11, ALL = _ffi.QUIRK_Q9, _ffi.QUIRK_Q10, _ffi.QUIRK_Q11, _ffi.QUIRK_ALL


@pytest.fixture(autouse=True)
def _restore_quirks():
    yield
    _ffi.load().zj_host_set_quirks(ALL)


def _deviation(data: bytes, mask: int):
    """(max |delta|, share of pixels with |delta| > 8) of host-stage planes -> spec-correct pixels against libjpeg"""
    _ffi.load().zj_host_set_quirks(mask)
    ref = np.asarray(Image.open(io.BytesIO(data)).convert("RGB")).astype(np.int16)
    h, w, _ = ref.shape
    img, planes = Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB)).decode_coefficients(data)
    px, rows = sane_pixels(img, planes, w, h)
    d = np.abs(px - ref[:rows]).max(axis=2)
    return int(d.max()), float((d > 8).mean())


# file, the quirk that explains its deviation (None: the host stage already agrees with libjpeg), (min max-delta, min share > 8)
# with the quirks as written.  Measured values: test-progressive 255 / 1.45 %, huffman_third_index 238 / 7.53 %, medium_* 21-22.
CASES = [
    ("test-baseline.jpg", None, None),              # BASELINE configs[0]: 4:4:4 baseline, standard-sized codes
    ("single_qt.jpeg", None, None),                 # 4:2:2, DRI = 1005 (the one restart fixture): Q8 stays benign, planes end at row 1072 (Q1)
    ("test-progressive.jpg", Q9, (200, 0.010)),     # optimised Huffman tables: short codes for |k| >= 32 (209 -> -49 ...)
    ("huffman_third_index.jpg", Q9, (200, 0.050)),
    ("medium_no_samp_2500x1786.jpg", Q11, (15, 0.0)),    # last MCU: Cb / Cr (and trailing Y blocks) stay zero
    ("medium_horiz_samp_2500x1786.jpg", Q11, (15, 0.0)),
    ("medium_vertical_samp_2500x1786.jpg", Q11, (15, 0.0)),
]


@pytest.mark.parametrize("name,quirk,as_written", CASES)
def test_fixture_deviation_is_the_cited_quirk(name, quirk, as_written):
    data = ref_files.read(name)
    mx, share = _deviation(data, ALL)
    if quirk is None:
        assert mx <= 5, (name, mx)
        return
    assert mx >= as_written[0] and share >= as_written[1], (name, mx, share)      # the deviation is there ...
    mx_off, share_off = _deviation(data, ALL & ~quirk)
    assert mx_off <= 5 and share_off == 0.0, (name, mx_off, share_off)            # ... and gone with that ONE switch off
    for other in (Q9, Q10, Q11):
        if other != quirk:
            mx_o, _ = _deviation(data, ALL & ~other)
            assert mx_o == mx, (name, other, mx_o)                                # the other two switches do not touch it


def test_q10_dc_refill_underrun():
    """Q10 (bitstream.rs:278-281): no reference fixture has DC differences large enough (category >= 10 needs > 16 bits), so
    the input is synthetic: random black / white 8x8 blocks at quality 100, 4:2:0.  As written the reader under-runs and the
    stream mis-syncs until a code is invalid -- the reference REJECTS a valid JPEG; with the refill fixed it decodes to +-5."""
    rng = np.random.default_rng(5)
    w, h = 640, 480
    rng.integers(0, 2, size=(h // 8, w // 8, 3)); rng.integers(-20, 21, size=(h, w, 3))     # (the stream of the first draw is skipped)
    blocks = rng.integers(0, 2, size=(h // 8, w // 8, 3)).astype(np.uint8) * 255
    a = np.kron(blocks, np.ones((8, 8, 1), np.uint8)).astype(np.int16) + rng.integers(-20, 21, size=(h, w, 3))
    bio = io.BytesIO()
    Image.fromarray(np.clip(a, 0, 255).astype(np.uint8), "RGB").save(bio, "JPEG", quality=100, subsampling=2)
    data = bio.getvalue()
    for mask in (ALL, ALL & ~Q9, ALL & ~Q11):
        try:
            mx, share = _deviation(data, mask)
        except DecodeErrors as e:
            assert e.variant == "HuffmanDecode"
        else:
            assert mx > 8 and share > 0.01, (mask, mx, share)
    mx, share = _deviation(data, ALL & ~Q10)
    assert mx <= 5 and share == 0.0


def test_switches_default_on_and_gate_gpu_entropy():
    lib = _ffi.load()
    assert lib.zj_host_get_quirks() == ALL
    lib.zj_host_set_quirks(0xFFFFFFFF)
    assert lib.zj_host_get_quirks() == ALL
