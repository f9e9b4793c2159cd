"""GPU parity: the fused CUDA path (through the C ABI) must equal the oracle byte-for-byte."""
import numpy as np
import pytest

import oracle
import util

pytestmark = pytest.mark.gpu

QTS = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]
MODES = {"444": (1, 1), "422": (2, 1), "440": (1, 2), "420": (2, 2)}


def _run_case(rng, w, h, mode, out_cs, variant, n_comp=3, progressive=False, **kw):
    from zune_jpeg_b200 import gpu
    hs, vs = MODES[mode]
    planes = util.random_planes(rng, w, h, n_comp, hs, vs, **kw)
    img = util.make_image(w, h, planes, QTS[:n_comp], hs, vs, out_cs, variant, progressive)
    try:
        want = oracle.reconstruct(img)
    except RuntimeError as e:
        assert "rc=-5" in str(e), e
        assert gpu.validate(img) == -5, "GPU path must refuse what the reference panics on"
        return "panic"
    got = gpu.reconstruct([img])[0]
    if not np.array_equal(got, want):
        bad = np.nonzero(got != want)[0]
        nc = len(want) // (w * h)
        first = bad[:6]
        where = [(int(b // (w * nc)), int((b % (w * nc)))) for b in first]
        raise AssertionError(f"{w}x{h} {mode} out={out_cs} var={variant}: {bad.size} bytes differ, first (row,byte)={where} got={got[first]} want={want[first]}")
    return "ok"


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("mode", list(MODES))
@pytest.mark.parametrize("out_cs", [0, 5, 2, 1])
def test_random_sizes(mode, out_cs, variant):
    rng = np.random.default_rng(hash((mode, out_cs, variant)) & 0xFFFF)
    sizes = [(64, 64), (100, 70), (1000, 96), (333, 130), (16, 16), (17, 40), (640, 33), (2500, 48), (1288, 64)]
    for (w, h) in sizes:
        _run_case(rng, w, h, mode, out_cs, variant)


@pytest.mark.parametrize("variant", [0, 1])
@pytest.mark.parametrize("mode", list(MODES))
def test_small_widths(mode, variant):
    rng = np.random.default_rng(5)
    for w in range(1, 40):
        for out_cs in (0, 5):
            _run_case(rng, w, 37, mode, out_cs, variant)


@pytest.mark.parametrize("variant", [0, 1])
def test_extreme_coefficients(variant):
    rng = np.random.default_rng(11)
    for mode in MODES:
        _run_case(rng, 264, 72, mode, 0, variant, extreme=True)


@pytest.mark.parametrize("variant", [0, 1])
def test_grayscale_input(variant):
    rng = np.random.default_rng(3)
    for (w, h) in [(64, 64), (1001, 77), (4096, 64), (57, 9), (200, 8)]:
        _run_case(rng, w, h, "444", 1, variant, n_comp=1)
        _run_case(rng, w, h, "444", 0, variant, n_comp=1)  # GRAY -> RGB: the reference writes nothing


def test_unwritten_pairs_are_zero():
    rng = np.random.default_rng(4)
    _run_case(rng, 128, 64, "420", 3, 0)  # YCbCr -> CMYK: zeros
    _run_case(rng, 128, 64, "444", 4, 1)  # YCbCr -> YCCK: zeros


def test_batch_mixed():
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(9)
    imgs, keep, wants = [], [], []
    for (w, h, mode, out_cs, variant) in [(640, 480, "420", 0, 0), (320, 200, "444", 0, 0), (500, 100, "422", 5, 1),
                                          (1920, 64, "420", 0, 0), (256, 256, "440", 2, 0), (300, 300, "420", 1, 0),
                                          (777, 123, "420", 0, 1), (4000, 40, "420", 5, 0)]:
        hs, vs = MODES[mode]
        planes = util.random_planes(rng, w, h, 3, hs, vs)
        keep.append(planes)
        img = util.make_image(w, h, planes, QTS, hs, vs, out_cs, variant)
        imgs.append(img)
        wants.append(oracle.reconstruct(img))
    gots = gpu.reconstruct(imgs)
    for i, (g, wv) in enumerate(zip(gots, wants)):
        assert np.array_equal(g, wv), f"image {i} differs"


def test_4k_420_full_size():
    """BASELINE config 2 geometry (3840x2160 4:2:0 -> RGB), one image, against the oracle."""
    rng = np.random.default_rng(21)
    assert _run_case(rng, 3840, 2160, "420", 0, 0) == "ok"


def test_device_resident_batch_plan():
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(13)
    w, h = 1280, 720
    planes = util.random_planes(rng, w, h, 3, 2, 2)
    host_img = util.make_image(w, h, planes, QTS, 2, 2, 0, 0)
    want = oracle.reconstruct(host_img)
    bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
    for b, p in zip(bufs, planes):
        b.upload(p)
    out = gpu.DeviceBuffer(len(want))
    out.memset(0xAB)  # the kernel must define every byte itself
    img = util.make_image(w, h, planes, QTS, 2, 2, 0, 0, ptrs=[b.ptr for b in bufs])
    batch = gpu.Batch([img], [out.ptr], [len(want)])
    before = gpu.launch_count()
    batch.run()
    batch.run()
    assert gpu.launch_count() - before == 2 * batch.launches
    got = out.download()
    assert np.array_equal(got, want)
    # algorithmic bytes = coefficient bytes of the strips the reference processes + output bytes (DESIGN.md 4.1): 4:2:0 strips
    # are two MCU rows (mcu.rs:155-159; 720 rows = 45 MCU rows -> 22 strips, the odd MCU row is dropped, Q1)
    mcu_x, mcu_y = util.geometry(w, h, 2, 2)
    n_strips = mcu_y // 2
    assert n_strips == 22
    assert batch.algorithmic_bytes == n_strips * (4 * 2 * mcu_x + 2 * 2 * mcu_x) * 64 * 2 + len(want)


# ------------------------------------------------------------------ the producer / consumer kernel's own corners
def _device_case(rng, w, h, mode, out_cs, out_offset=0, coeff_offset=0):
    """Device-resident planes / output at chosen byte offsets; returns (got, want) or the error status."""
    from zune_jpeg_b200 import gpu
    hs, vs = MODES[mode]
    planes = util.random_planes(rng, w, h, 3, hs, vs)
    host_img = util.make_image(w, h, planes, QTS, hs, vs, out_cs, 0)
    want = oracle.reconstruct(host_img)
    bufs = [gpu.DeviceBuffer(p.nbytes + 64) for p in planes]
    for b, p in zip(bufs, planes):
        b.upload(p, offset=coeff_offset)
    out = gpu.DeviceBuffer(len(want) + 64)
    out.memset(0xCD)
    img = util.make_image(w, h, planes, QTS, hs, vs, out_cs, 0, ptrs=[b.ptr + coeff_offset for b in bufs])
    try:
        batch = gpu.Batch([img], [out.ptr + out_offset], [len(want)])
    except gpu.ZjError as e:
        return e.status, None
    batch.run()
    got = out.download()
    assert np.all(got[:out_offset] == 0xCD) and np.all(got[out_offset + len(want):] == 0xCD), "wrote outside the output"
    return got[out_offset:out_offset + len(want)], want


@pytest.mark.parametrize("mode", list(MODES))
def test_output_alignment_classes(mode):
    """16-byte aligned rows take 128-bit stores, 4-byte aligned ones word stores, anything else the generic kernel."""
    rng = np.random.default_rng(31)
    for (w, h, out_cs) in [(640, 96, 0), (644, 64, 0), (1000, 70, 5), (333, 40, 0)]:
        for off in (0, 4, 16, 1, 2):
            got, want = _device_case(rng, w, h, mode, out_cs, out_offset=off)
            assert np.array_equal(got, want), f"{w}x{h} {mode} out={out_cs} offset {off}"


def test_misaligned_device_planes_are_refused():
    rng = np.random.default_rng(32)
    status, _ = _device_case(rng, 320, 64, "420", 0, coeff_offset=2)
    assert status == -1  # ZJ_ERR_INVALID_ARG: device planes are read with 128-bit accesses


def test_wide_and_partial_tiles():
    """Many tiles per strip, a partial last tile, widths with W % 16 == 8, the "RGBA" zero columns spread over all tiles."""
    rng = np.random.default_rng(33)
    for (w, h, mode, out_cs) in [(8192, 64, "420", 5), (4100, 48, "420", 0), (4120, 40, "422", 0), (4104, 24, "444", 0),
                                 (4104, 40, "440", 5), (2056, 70, "420", 2), (1032, 130, "420", 0), (264, 600, "420", 0)]:
        assert _run_case(rng, w, h, mode, out_cs, 0) == "ok"


@pytest.mark.parametrize("spc", [1, 2, 3, 5])
def test_strips_per_cta(spc):
    """ZJ_SPC (strips per CTA of the fast kernel) is read once per process: run the cases in a fresh interpreter."""
    import os
    import subprocess
    import sys
    code = (
        "import sys, numpy as np\n"
        "sys.path[:0] = [%r, %r]\n"
        "import oracle, util\n"
        "from zune_jpeg_b200 import gpu\n"
        "rng = np.random.default_rng(41)\n"
        "qts = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]\n"
        "for (w, h, hs, vs, cs) in [(640, 480, 2, 2, 0), (320, 200, 1, 1, 0), (500, 330, 2, 1, 5), (256, 256, 1, 2, 2), (1000, 96, 2, 2, 0)]:\n"
        "    planes = util.random_planes(rng, w, h, 3, hs, vs)\n"
        "    img = util.make_image(w, h, planes, qts, hs, vs, cs, 0)\n"
        "    assert np.array_equal(gpu.reconstruct([img])[0], oracle.reconstruct(img)), (w, h, hs, vs, cs)\n"
        "print('ok')\n"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, ZJ_SPC=str(spc))
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_generic_kernel_still_matches():
    """ZJ_NO_FAST routes everything through zj::reconstruct_kernel (the path SCALAR / unaligned images take)."""
    import os
    import subprocess
    import sys
    code = (
        "import sys, numpy as np\n"
        "sys.path[:0] = [%r, %r]\n"
        "import oracle, util\n"
        "from zune_jpeg_b200 import gpu\n"
        "rng = np.random.default_rng(42)\n"
        "qts = [util.std_qt(False), util.std_qt(True), util.std_qt(True)]\n"
        "for (w, h, hs, vs, cs) in [(640, 480, 2, 2, 0), (333, 130, 1, 1, 0), (500, 330, 2, 1, 5), (256, 256, 1, 2, 2)]:\n"
        "    planes = util.random_planes(rng, w, h, 3, hs, vs)\n"
        "    img = util.make_image(w, h, planes, qts, hs, vs, cs, 0)\n"
        "    assert np.array_equal(gpu.reconstruct([img])[0], oracle.reconstruct(img)), (w, h, hs, vs, cs)\n"
        "print('ok')\n"
    ) % (os.path.dirname(os.path.dirname(os.path.abspath(__file__))), os.path.dirname(os.path.abspath(__file__)))
    env = dict(os.environ, ZJ_NO_FAST="1")
    r = subprocess.run([sys.executable, "-c", code], env=env, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "ok" in r.stdout, r.stdout + r.stderr


def test_sparse_and_dense_blocks_mix():
    """The rolled IDCT picks its short forms per warp: DC-only blocks, 4x4 blocks and dense blocks side by side."""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(43)
    w, h = 1024, 128
    for mode in MODES:
        hs, vs = MODES[mode]
        planes = util.random_planes(rng, w, h, 3, hs, vs)
        for p in planes:
            blk = p.reshape(-1, 64)
            kind = rng.integers(0, 4, size=blk.shape[0])
            blk[kind == 0, 1:] = 0                                   # DC only
            m4 = np.ones(64, bool).reshape(8, 8); m4[:4, :4] = False
            blk[np.ix_(kind == 1, m4.ravel())] = 0                   # top-left 4x4
            m6 = np.ones(64, bool).reshape(8, 8); m6[:6, :] = False
            blk[np.ix_(kind == 2, m6.ravel())] = 0                   # rows 6, 7 empty
        img = util.make_image(w, h, planes, QTS, hs, vs, 0, 0)
        want = oracle.reconstruct(img)
        got = gpu.reconstruct([img])[0]
        assert np.array_equal(got, want), mode


@pytest.mark.parametrize("mode", list(MODES))
def test_warp_uniform_sparsity_classes_at_the_limits(mode):
    """Every short form of the rolled IDCT taken by WHOLE warps (the class is the same in every block of a plane), with
    coefficients over the full i16 range and quantisers up to 255: the regrouped butterflies (idct8 / idct8_lo4 / idct8_lo6 --
    multiply-adds re-associated in Z/2^32) and the 4- / 6- / 8-input column passes must wrap exactly like the
    oracle's literal form.  Classes = (rows kept, columns kept)."""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(4242)
    hs, vs = MODES[mode]
    w, h = 528, 96
    qts = [rng.integers(1, 256, size=64).astype(np.int32) for _ in range(3)]
    qts[1][:] = 255
    for (rk, ck) in [(8, 8), (6, 8), (6, 4), (4, 8), (4, 4), (8, 4), (7, 8), (5, 6), (2, 2), (1, 8), (8, 1), (6, 2)]:
        for out_cs in (0, 2):
            planes = util.random_planes(rng, w, h, 3, hs, vs, extreme=True, dc_only_frac=0.05)
            for p in planes:
                blk = p.reshape(-1, 8, 8)
                blk[:, rk:, :] = 0
                blk[:, :, ck:] = 0
            img = util.make_image(w, h, planes, qts, hs, vs, out_cs, 0)
            want = oracle.reconstruct(img)
            got = gpu.reconstruct([img])[0]
            assert np.array_equal(got, want), (mode, rk, ck, out_cs, int((got != want).sum()))


def test_gray_fast_kernel_corners():
    """Luma-only output through gray_fast_kernel: odd block-row counts, ragged widths, colour inputs of every sub-sampling,
    unaligned output pointers."""
    rng = np.random.default_rng(51)
    for (w, h) in [(520, 24), (1001, 77), (33, 9), (2056, 40), (512, 16), (528, 8), (5000, 72)]:
        assert _run_case(rng, w, h, "444", 1, 0, n_comp=1) in ("ok", "panic")
        for mode in MODES:
            assert _run_case(rng, w, h, mode, 1, 0) in ("ok", "panic")
    for off in (0, 1, 4, 16):
        got, want = _device_case(rng, 640, 56, "420", 1, out_offset=off)
        assert np.array_equal(got, want), off


def test_decode_batch_matches_single_image_decodes():
    """zj_decode_batch (host threads entropy-decode different images while the GPU reconstructs finished ones) returns exactly
    what one Decoder per image returns, in input order, with per-image errors."""
    import json
    import os
    import jpeg_util
    from zune_jpeg_b200.decoder import ColorSpace, DecodeErrors, Decoder, ZuneJpegOptions, decode_batch
    golden = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    man = json.load(open(os.path.join(golden, "manifest.json")))
    rgb = [c for c in man["cases"] if c["out"] == "RGB" and c["variant"] == "X86"]
    jpegs = [open(os.path.join(golden, c["jpeg"]), "rb").read() for c in rgb]
    wants = [np.fromfile(os.path.join(golden, c["pixels"]), np.uint8).tobytes() for c in rgb]
    for i in range(6):   # a few bigger ones: 4:2:0, 4:4:4, 4:2:2 progressive, grayscale
        sub, prog, gray = [("420", False, False), ("444", False, False), ("422", True, False), ("444", False, True)][i % 4]
        jpegs.append(jpeg_util.synth_jpeg(100 + i, 640 + 16 * i, 360 + 8 * i, sub, 90, prog, gray))
        wants.append(Decoder.new().decode_buffer(jpegs[-1]))
    bad = bytes([0xff, 0xd8, 0xa4])
    batch = jpegs[:3] + [bad] + jpegs[3:] + jpegs   # every image twice, one broken stream in between
    res = decode_batch(batch, threads=5)
    expect = wants[:3] + [None] + wants[3:] + wants
    assert len(res) == len(expect)
    for r, w in zip(res, expect):
        if w is None:
            assert isinstance(r, DecodeErrors) and r.status == -9
        else:
            assert r == w
    # caller-provided (pinned) output buffers, non-default options
    from zune_jpeg_b200 import gpu
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGBA)
    sizes = [len(Decoder.new_with_options(opts).decode_buffer(j)) for j in jpegs]
    pinned = gpu.PinnedBuffer(sum(sizes))
    offs = np.concatenate([[0], np.cumsum(sizes)])
    outs = [pinned.array[offs[i]:offs[i + 1]] for i in range(len(jpegs))]
    res = decode_batch(jpegs, opts, threads=0, out=outs)
    assert res == sizes
    for j, o in zip(jpegs, outs):
        assert o.tobytes() == Decoder.new_with_options(opts).decode_buffer(j)
    # the workers' pooled decoders can be dropped between calls
    from zune_jpeg_b200 import _ffi
    _ffi.load().zj_release_host_caches()
    assert decode_batch(jpegs[:3], threads=2) == wants[:3]


@pytest.mark.parametrize("w,h,mode", [(2500, 1786, "444"), (2500, 1786, "422"), (2500, 1786, "440"), (3024, 4032, "420"),
                                      (1920, 1080, "422"), (7680, 4320, "444"), (7680, 4320, "422"), (7680, 4320, "440")])
def test_reference_fixture_geometries(w, h, mode):
    """The shapes of the reference's own integration fixtures (tests/inputs/medium_*_2500x1786, google_pixel 3024x4032 2x2,
    single_qt 1920x1080 2x1, large_*_7680_4320; SURVEY section 4) with random coefficient planes: the reference only eyeballs
    these outputs, here they must equal the oracle byte for byte."""
    rng = np.random.default_rng(hash((w, h, mode)) & 0xFFFF)
    assert _run_case(rng, w, h, mode, 0, 0) == "ok"


@pytest.mark.parametrize("name,w,h,sub,prog,gray,out_cs,rst", [
    ("c3_444", 4096, 4096, "444", False, False, 0, 0),
    ("c3_gray", 4096, 4096, "444", False, True, 1, 0),
    ("c4", 1920, 1080, "422", True, False, 0, 0),
    ("c5", 8192, 8192, "420", False, False, 5, 1),
])
def test_baseline_configs_from_jpeg_bytes(name, w, h, sub, prog, gray, out_cs, rst):
    """BASELINE configs[2..4] at full size, from JPEG bytes: Decoder.decode_buffer (host stage on 4 threads -- for c5 that is
    the restart-interval-parallel entropy decode -- then the GPU) against the oracle fed with the planes of the sequential
    host stage."""
    import os
    import jpeg_util
    from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions
    data = jpeg_util.synth_jpeg(7, w, h, sub, 90, prog, gray, rst)
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace(out_cs))
    seq = Decoder.new_with_options(opts.set_num_threads(1))
    img, planes = seq.decode_coefficients(data)
    for z in range(img.n_comp):
        img.comp[z].coeff = planes[z].ctypes.data if planes[z].size else None
    want = oracle.reconstruct(img, threads=os.cpu_count() or 1)
    d = Decoder.new_with_options(opts.set_num_threads(4))
    got = np.frombuffer(d.decode_buffer(data), np.uint8)
    assert got.size == w * h * ColorSpace(out_cs).num_components()
    assert np.array_equal(got, want)
    assert (d.entropy_segments() > 0) == bool(rst)


def test_c2_from_jpeg_bytes_all_bench_images():
    """BASELINE configs[1] from JPEG bytes: the eight distinct 3840x2160 4:2:0 images bench.py cycles through its batch of 256
    (same seeds, quality 90), decoded by decode_batch (host stage + GPU) and checked against the oracle -- all eight, not
    only the first one the bench itself checks."""
    import os
    import jpeg_util
    from zune_jpeg_b200.decoder import ColorSpace, Decoder, ZuneJpegOptions, decode_batch
    opts = ZuneJpegOptions().set_out_colorspace(ColorSpace.RGB)
    datas = [jpeg_util.synth_jpeg(i, 3840, 2160, "420", 90) for i in range(8)]      # bench.make_pool: seed = 1000 * rank + i
    got = decode_batch(datas, opts, threads=8)
    for data, g in zip(datas, got):
        seq = Decoder.new_with_options(opts.set_num_threads(1))
        img, planes = seq.decode_coefficients(data)
        for z in range(img.n_comp):                      # (the descriptor points into the decoder: re-point it at the copies)
            img.comp[z].coeff = planes[z].ctypes.data if planes[z].size else None
        want = oracle.reconstruct(img, threads=os.cpu_count() or 1)
        assert isinstance(g, bytes) and len(g) == 3840 * 2160 * 3
        assert np.array_equal(np.frombuffer(g, np.uint8), want)


def test_mixed_geometry_batch_launch_groups():
    """A heterogeneous device-resident batch: images are grouped by kernel (luma-only / fast / mode / variant), one launch per
    group, and a group's grid is sized by its LARGEST member -- a 4000-wide and an 80-wide image in one group (very different tile
    counts), several modes, both variants, a luma-only output.  zj_batch_launches must equal the number of groups."""
    from zune_jpeg_b200 import gpu
    rng = np.random.default_rng(77)
    cases = [(4000, 64, "420", 0, 0), (80, 400, "420", 0, 0), (640, 480, "420", 0, 0),       # one group: HV fast, 1 .. 16 tiles, 2 .. 15 strips
             (333, 100, "444", 0, 0), (1000, 96, "422", 5, 0),                                 # NONE fast, H fast
             (200, 64, "420", 0, 1), (264, 100, "440", 2, 1),                                   # SCALAR variant: generic kernels (HV, V)
             (520, 90, "420", 1, 0), (72, 40, "444", 1, 0)]                                     # luma-only output: gray fast kernel, two modes
    imgs, wants, outs, keep = [], [], [], []
    for (w, h, mode, out_cs, variant) in cases:
        hs, vs = MODES[mode]
        planes = util.random_planes(rng, w, h, 3, hs, vs)
        wants.append(oracle.reconstruct(util.make_image(w, h, planes, QTS, hs, vs, out_cs, variant)))
        bufs = [gpu.DeviceBuffer(p.nbytes) for p in planes]
        for b, p in zip(bufs, planes):
            b.upload(p)
        o = gpu.DeviceBuffer(len(wants[-1]))
        o.memset(0x5A)
        keep.append((planes, bufs))
        outs.append(o)
        imgs.append(util.make_image(w, h, planes, QTS, hs, vs, out_cs, variant, ptrs=[b.ptr for b in bufs]))
    batch = gpu.Batch(imgs, [o.ptr for o in outs], [len(w_) for w_ in wants])
    assert batch.launches == 7          # HV fast | NONE fast | H fast | HV generic SCALAR | V generic SCALAR | gray HV | gray NONE
    before = gpu.launch_count()
    batch.run()
    assert gpu.launch_count() - before == 7
    for (case, o, want) in zip(cases, outs, wants):
        assert np.array_equal(o.download(), want), case


def test_gpu_entropy_decode_matches_host_stage():
    """zj_decode_batch_gpu: restart intervals entropy-decoded one per GPU thread (zj_entropy.cu) give the pixels of the host
    stage (the reference's sequential loop); images without restart markers, progressive ones, streams whose declared DRI does
    not match their markers and damaged streams silently take the host route and still give identical results / errors."""
    import jpeg_util
    from zune_jpeg_b200.decoder import ColorSpace, DecodeErrors, decode_batch, ZuneJpegOptions
    cases = []   # (jpeg, expected to run on the GPU)
    for i, (w, h, sub, gray, rows, q) in enumerate([(1024, 768, "420", False, 1, 90), (1000, 1016, "420", False, 2, 75), (1280, 720, "422", False, 1, 85),
                                                     (800, 600, "444", False, 3, 95), (2048, 1024, "444", True, 1, 90), (3840, 2160, "420", False, 1, 98),
                                                     (640, 480, "440", False, 1, 60)]):
        if sub == "440":
            continue
        cases.append((jpeg_util.synth_jpeg(30 + i, w, h, sub, q, False, gray, rows), True))
    cases.append((jpeg_util.synth_jpeg(40, 800, 608, "420", 90), False))                       # no DRI
    cases.append((jpeg_util.synth_jpeg(41, 800, 608, "422", 90, True), False))                 # progressive
    base = jpeg_util.synth_jpeg(42, 1024, 512, "420", 80, restart_rows=1)
    i = base.index(b"\xff\xdd")
    cases.append((base[:i + 4] + bytes([0, 7]) + base[i + 6:], False))                         # DRI does not match the markers (Q8 territory)
    cut = bytearray(base); del cut[len(cut) // 2:]
    cases.append((bytes(cut), False))                                                          # truncated
    flip = bytearray(base); flip[len(flip) // 2] ^= 0x10
    cases.append((bytes(flip), None))                                                          # damaged entropy data: either route
    cases.append((bytes([0xff, 0xd8, 0xa4]), False))                                           # header error
    fill = bytearray(base)                                                                     # 0xFF fill bytes in front of every RSTn (legal)
    sos = base.index(b"\xff\xda")
    for k, p_ in enumerate(reversed([i for i in range(sos, len(base) - 1) if base[i] == 0xFF and 0xD0 <= base[i + 1] <= 0xD7])):
        fill[p_:p_] = b"\xff" * (1 + k % 3)
    cases.append((bytes(fill), True))
    jpegs = [c[0] for c in cases]
    for out_cs in (ColorSpace.RGB, ColorSpace.RGBA, ColorSpace.GRAYSCALE):
        opts = ZuneJpegOptions().set_out_colorspace(out_cs)
        want = decode_batch(jpegs, opts, threads=4)
        stats = {}
        got = decode_batch(jpegs, opts, threads=4, gpu_entropy=True, stats=stats)
        for k, (g, w_) in enumerate(zip(got, want)):
            if isinstance(w_, DecodeErrors):
                assert isinstance(g, DecodeErrors) and g.status == w_.status, k
            else:
                assert g == w_, f"image {k} out_cs={out_cs}"
        sure = sum(1 for c in cases if c[1] is True)
        maybe = sum(1 for c in cases if c[1] is None)
        assert sure <= stats["gpu_entropy"] <= sure + maybe, stats


def test_gpu_entropy_decode_device_outputs():
    """zj_decode_batch_gpu_device: pixels stay in device memory; GPU-entropy images and host-route images (no DRI) both land
    there with the bytes Decoder.decode_buffer returns; a too small device buffer is a per-image error."""
    import jpeg_util
    from zune_jpeg_b200 import gpu
    from zune_jpeg_b200.decoder import DecodeErrors, Decoder, decode_batch
    jpegs = [jpeg_util.synth_jpeg(50, 1024, 768, "420", 90, restart_rows=1), jpeg_util.synth_jpeg(51, 800, 608, "420", 90),
             jpeg_util.synth_jpeg(52, 1280, 720, "422", 85, restart_rows=2), jpeg_util.synth_jpeg(53, 640, 480, "444", 90, gray=True, restart_rows=1)]
    wants = [Decoder.new().decode_buffer(j) for j in jpegs]
    pinned_in = gpu.PinnedBuffer(sum(len(j) for j in jpegs))
    ins, off = [], 0
    for j in jpegs:
        pinned_in.array[off:off + len(j)] = np.frombuffer(j, np.uint8)
        ins.append(pinned_in.array[off:off + len(j)])
        off += len(j)
    bufs = [gpu.DeviceBuffer(len(w_) + 64) for w_ in wants]
    stats = {}
    res = decode_batch(ins, threads=4, device_out=[(b.ptr, b.nbytes) for b in bufs], stats=stats)
    assert stats["gpu_entropy"] == 3
    for r, w_, b in zip(res, wants, bufs):
        assert r == len(w_)
        assert b.download(len(w_)).tobytes() == w_
    res = decode_batch(ins, threads=4, device_out=[(b.ptr, 1000) for b in bufs])
    assert all(isinstance(r, DecodeErrors) for r in res)


def test_gpu_entropy_decode_fuzz():
    """Damaged restart-marker streams, many at once: whatever route an image ends up on (GPU intervals accepted, or the host
    stage after a rejected interval), pixels and per-image errors equal those of the host stage alone."""
    import jpeg_util
    from zune_jpeg_b200.decoder import DecodeErrors, decode_batch
    rng = np.random.default_rng(77)
    bases = [jpeg_util.synth_jpeg(60, 640, 480, "420", 85, restart_rows=1), jpeg_util.synth_jpeg(61, 512, 384, "444", 92, restart_rows=2),
             jpeg_util.synth_jpeg(62, 768, 256, "422", 70, restart_rows=1), jpeg_util.synth_jpeg(63, 512, 512, "444", 90, gray=True, restart_rows=1)]
    jpegs = []
    for k in range(64):
        d = bytearray(bases[k % len(bases)])
        sos = bytes(d).index(b"\xff\xda")
        kind = k % 6
        if kind == 0:      # bit flips in the entropy-coded data
            for p in rng.integers(sos + 14, len(d) - 2, size=int(rng.integers(1, 5))):
                d[p] ^= 1 << int(rng.integers(0, 8))
        elif kind == 1:    # truncation
            del d[int(rng.integers(sos + 14, len(d) - 2)):]
        elif kind == 2:    # a restart marker removed / duplicated
            marks = [i for i in range(sos, len(d) - 1) if d[i] == 0xFF and 0xD0 <= d[i + 1] <= 0xD7]
            p = marks[int(rng.integers(0, len(marks)))]
            if k % 12 < 6:
                del d[p:p + 2]
            else:
                d[p:p] = d[p:p + 2]
        elif kind == 3:    # a foreign marker / stuffed 0xFF bytes inside the scan
            p = int(rng.integers(sos + 14, len(d) - 2))
            d[p:p] = [b"\xff\xd9", b"\xff\xc4", b"\xff\xff\xff\x00", b"\xff\x01"][k // 6 % 4]
        elif kind == 4:    # DRI changed
            i = bytes(d).index(b"\xff\xdd")
            v = int(rng.integers(1, 400))
            d[i + 4:i + 6] = bytes([v >> 8, v & 255])
        # kind 5: untouched
        jpegs.append(bytes(d))
    want = decode_batch(jpegs, threads=4)
    stats = {}
    got = decode_batch(jpegs, threads=4, gpu_entropy=True, stats=stats)
    assert stats["gpu_entropy"] >= 64 // 6
    for k, (g, w_) in enumerate(zip(got, want)):
        if isinstance(w_, DecodeErrors):
            assert isinstance(g, DecodeErrors) and g.status == w_.status, k
        else:
            assert g == w_, f"image {k} (kind {k % 6})"
