"""Host-side mirror of the reference's public API (reference src/lib.rs:89-91, src/decoder.rs, src/options.rs,
src/misc.rs, src/errors.rs) on top of the C ABI.

    from zune_jpeg_b200 import Decoder, ZuneJpegOptions, ColorSpace
    pixels = Decoder.new_with_options(ZuneJpegOptions().set_out_colorspace(ColorSpace.RGBA)).decode_buffer(data)

Same names, argument meaning and error behaviour as the Rust crate: `Result<_, DecodeErrors>` becomes a raised
`DecodeErrors` whose `.variant` / `.message` carry the enum variant and its payload.  Headers and Huffman
decoding run in the C++ host front-end, everything after that on the GPU; there is no CPU pixel path.
"""
from __future__ import annotations

import ctypes as C
import enum

import numpy as np

from . import _ffi
from ._ffi import ZjImage, ZjImageInfo, ZjOptions


class ColorSpace(enum.IntEnum):
    """src/misc.rs:88-106"""
    RGB = 0
    GRAYSCALE = 1
    YCbCr = 2
    CMYK = 3
    YCCK = 4
    RGBA = 5
    RGBX = 6

    def num_components(self) -> int:
        return {0: 3, 2: 3, 1: 1}.get(int(self), 4)


class DecodeErrors(Exception):
    """src/errors.rs:16-43; `variant` is the enum variant name, `message` its payload."""
    VARIANTS = {1: "Format", 2: "FormatStatic", 3: "IllegalMagicBytes", 4: "HuffmanDecode", 5: "ZeroError",
                6: "DqtError", 7: "SosError", 8: "SofError", 9: "Unsupported", 10: "MCUError",
                11: "ExhaustedData", 12: "LargeDimensions", 13: "Gpu"}

    def __init__(self, kind: int, display: str, status: int = _ffi.ERR_DECODE):
        super().__init__(display)
        self.kind = kind
        self.variant = self.VARIANTS.get(kind, "Format")
        self.display = display
        self.status = status

    @property
    def message(self) -> str:
        """The variant's payload (what the reference's tests compare with `x == "..."`)."""
        prefixes = {"HuffmanDecode": "Error decoding huffman tables.Reason:", "DqtError": "Error parsing DQT segment. Reason:",
                    "SosError": "Error parsing SOS Segment. Reason:", "SofError": "Error parsing SOF segment. Reason:",
                    "MCUError": "Error in decoding MCU. Reason ", "IllegalMagicBytes": "Error parsing image. Illegal start bytes:"}
        d = self.display
        if self.variant == "FormatStatic" and len(d) >= 2 and d[0] == '"' and d[-1] == '"':
            return d[1:-1]
        p = prefixes.get(self.variant)
        return d[len(p):] if p and d.startswith(p) else d


class ImageInfo:
    """src/decoder.rs:652-668"""

    def __init__(self, raw: ZjImageInfo):
        self.width, self.height = raw.width, raw.height
        self.pixel_density = raw.pixel_density
        self.sof = raw.sof
        self.x_density, self.y_density = raw.x_density, raw.y_density
        self.components = raw.components

    def __repr__(self):
        return f"ImageInfo(width={self.width}, height={self.height}, components={self.components}, sof={self.sof})"


class ZuneJpegOptions:
    """src/options.rs:6-160 -- a by-value builder: every setter returns a new options object."""

    def __init__(self):
        self._use_unsafe = True
        self._out_colorspace = ColorSpace.RGB
        self._num_threads = 4
        self._max_width = 1 << 14
        self._max_height = 1 << 14
        self._max_scans = 64
        self._strict_mode = False
        self._device = 0
        self._spec_output = False
        self._libjpeg_output = False
        self._scale_denom = 1
        self._exif_orientation = False

    @staticmethod
    def new() -> "ZuneJpegOptions":
        return ZuneJpegOptions()

    def _with(self, **kw) -> "ZuneJpegOptions":
        o = ZuneJpegOptions()
        o.__dict__.update(self.__dict__)
        o.__dict__.update(kw)
        return o

    def get_out_colorspace(self): return self._out_colorspace
    def set_out_colorspace(self, colorspace): return self._with(_out_colorspace=ColorSpace(colorspace))
    def get_use_unsafe(self): return self._use_unsafe
    def set_use_unsafe(self, choice: bool): return self._with(_use_unsafe=bool(choice))
    def get_threads(self): return self._num_threads

    def set_num_threads(self, count: int):
        if count <= 0:
            raise ValueError("NonZeroU32")
        return self._with(_num_threads=int(count))

    def get_max_width(self): return self._max_width
    def set_max_width(self, w: int): return self._with(_max_width=int(w) & 0xFFFF)
    def get_max_height(self): return self._max_height
    def set_max_height(self, h: int): return self._with(_max_height=int(h) & 0xFFFF)
    def get_max_scans(self): return self._max_scans
    def set_max_scans(self, scans: int): return self._with(_max_scans=int(scans))
    def get_strict_mode(self): return self._strict_mode
    def set_strict_mode(self, choice: bool): return self._with(_strict_mode=bool(choice))
    # not in the reference: which GPU runs the pixel path
    def get_device(self): return self._device
    def set_device(self, device: int): return self._with(_device=int(device))
    # not in the reference: spec-correct output (every row decoded, libjpeg-style chroma up-sampling, JFIF colour, opaque
    # alpha; the statement is in include/zune_jpeg_b200.h, ZJ_VARIANT_SPEC)
    def get_spec_output(self): return self._spec_output
    def set_spec_output(self, choice: bool): return self._with(_spec_output=bool(choice))
    # not in the reference: libjpeg-turbo-exact output (spec output with libjpeg-turbo's islow IDCT: byte for byte what Pillow
    # and other libjpeg-turbo decodes with default settings give; ZJ_FLAG_ISLOW).  Takes precedence over spec output.
    def get_libjpeg_output(self): return self._libjpeg_output
    def set_libjpeg_output(self, choice: bool): return self._with(_libjpeg_output=bool(choice))
    # not in the reference: libjpeg-turbo's DCT-scaled decode of libjpeg output to ceil(width / d) x ceil(height / d), d = 1, 2, 4
    # or 8 -- what Pillow's Image.draft gives (ZJ_FLAG_SCALE_*; draft_scale picks d as Pillow does).  d > 1 needs libjpeg output.
    def get_scale_denom(self): return self._scale_denom

    def set_scale_denom(self, d: int):
        if d not in (1, 2, 4, 8):
            raise ValueError(f"scale denominator must be 1, 2, 4 or 8, not {d!r}")
        return self._with(_scale_denom=int(d))

    # not in the reference: the EXIF orientation applied to spec or libjpeg output, as Pillow's ImageOps.exif_transpose does
    # (ZJ_FLAG_ORIENT_*; sizes and rois are then those of the displayed image, oriented_size).  Needs spec or libjpeg output.
    def get_exif_orientation(self): return self._exif_orientation
    def set_exif_orientation(self, choice: bool): return self._with(_exif_orientation=bool(choice))

    def _raw(self) -> ZjOptions:
        o = ZjOptions()
        if self._scale_denom > 1 and not self._libjpeg_output:
            raise ValueError("a scale denominator above 1 needs libjpeg output (set_libjpeg_output(True))")
        if self._exif_orientation and not (self._libjpeg_output or self._spec_output):
            raise ValueError("EXIF orientation needs spec or libjpeg output (set_spec_output(True) or set_libjpeg_output(True))")
        if self._libjpeg_output:
            o.use_unsafe = _ffi.USE_LIBJPEG_OUTPUT | (self._scale_denom.bit_length() - 1) << _ffi.USE_SCALE_SHIFT
        else:
            o.use_unsafe = _ffi.USE_SPEC_OUTPUT if self._spec_output else int(self._use_unsafe)
        if self._exif_orientation:
            o.use_unsafe |= _ffi.USE_EXIF_ORIENTATION
        o.out_colorspace = int(self._out_colorspace)
        o.num_threads = self._num_threads
        o.max_width, o.max_height = self._max_width, self._max_height
        o.max_scans = self._max_scans
        o.strict_mode = int(self._strict_mode)
        o.device = self._device
        return o


class Decoder:
    """src/decoder.rs:60-647"""

    def __init__(self, options: ZuneJpegOptions | None = None):
        self._lib = _ffi.load()
        self.options = options if options is not None else ZuneJpegOptions()
        self._h = None
        self._rebuild()

    # constructors with the reference's names
    @staticmethod
    def new() -> "Decoder":
        return Decoder()

    @staticmethod
    def new_with_options(options: ZuneJpegOptions) -> "Decoder":
        return Decoder(options)

    def _rebuild(self):
        if self._h:
            self._lib.zj_decoder_free(self._h)
        raw = self.options._raw()
        self._h = self._lib.zj_decoder_new(C.byref(raw))
        if not self._h:
            raise MemoryError("zj_decoder_new")

    def __del__(self):
        try:
            if self._h:
                self._lib.zj_decoder_free(self._h)
                self._h = None
        except Exception:
            pass

    def _raise(self, status: int):
        kind = self._lib.zj_decoder_error_kind(self._h)
        text = self._lib.zj_decoder_error(self._h).decode("utf-8", "replace")
        if kind == 0:
            kind, text = 13, self._lib.zj_gpu_strerror(status).decode()
        raise DecodeErrors(kind, text, status)

    # ---- decoding
    def decode_buffer(self, buf: bytes) -> bytes:
        """Decoder::decode_buffer (decoder.rs:178): JPEG bytes -> width*height*components pixel bytes (with a scale denominator
        d: ceil(width / d) * ceil(height / d) * components)."""
        buf = bytes(buf)
        out = C.POINTER(C.c_uint8)()
        n = C.c_size_t()
        rc = self._lib.zj_decoder_decode_buffer(self._h, buf, len(buf), C.byref(out), C.byref(n))
        if rc != 0:
            self._raise(rc)
        try:
            return C.string_at(out, n.value)
        finally:
            self._lib.zj_buffer_free(out)

    decode = decode_buffer  # name used by later zune-jpeg releases

    def decode_into(self, buf, out) -> int:
        """JpegDecoder::decode_into of later zune-jpeg releases: the pixels go into `out` (a writable uint8 buffer, e.g. a
        PinnedBuffer.array slice); returns the number of bytes written (the scaled size's with a scale denominator).  Baseline
        images of >= 4 MP run as a strip pipeline (zj_decoder_decode_into): finished strip ranges are on their way through the GPU
        while the host still entropy-decodes."""
        import numpy as np
        data = buf if isinstance(buf, np.ndarray) else bytes(buf)
        p = data.ctypes.data if isinstance(data, np.ndarray) else C.cast(C.c_char_p(data), C.c_void_p).value
        n_in = data.nbytes if isinstance(data, np.ndarray) else len(data)
        view = out if isinstance(out, np.ndarray) else np.frombuffer(out, dtype=np.uint8)
        n = C.c_size_t()
        rc = self._lib.zj_decoder_decode_into(self._h, p, n_in, view.ctypes.data, view.nbytes, C.byref(n))
        if rc != 0:
            self._raise(rc)
        return int(n.value)

    def decode_file(self, path) -> bytes:
        """Decoder::decode_file (decoder.rs:193)"""
        try:
            with open(path, "rb") as f:
                data = f.read()
        except OSError as e:
            raise DecodeErrors(1, f"Error decoding an image:\n {e}")
        return self.decode_buffer(data)

    def read_headers(self, buf: bytes) -> None:
        """Decoder::read_headers (decoder.rs:452)"""
        buf = bytes(buf)
        rc = self._lib.zj_decoder_read_headers(self._h, buf, len(buf))
        if rc != 0:
            self._raise(rc)

    def decode_coefficients(self, buf: bytes):
        """Host stage only (headers + entropy decode): returns (zj_image descriptor, [int16 plane copies]); the descriptor's
        plane pointers refer to those copies."""
        buf = bytes(buf)
        img = ZjImage()
        rc = self._lib.zj_decoder_decode_coefficients(self._h, buf, len(buf), C.byref(img))
        if rc != 0:
            self._raise(rc)
        planes = []
        for z in range(img.n_comp):
            c = img.comp[z]
            if c.coeff and c.n_i16:
                a = np.ctypeslib.as_array((C.c_int16 * c.n_i16).from_address(c.coeff)).copy()
            else:
                a = np.zeros(0, np.int16)
            planes.append(a)
            # the descriptor is handed out pointing at the COPIES (kept alive by the descriptor object), not into the decoder's own
            # planes, which the next decode overwrites and the decoder's destruction frees
            c.coeff = a.ctypes.data if a.size else None
        img._planes = planes
        return img, planes

    def entropy_segments(self) -> int:
        """Restart intervals the last decode entropy-decoded side by side on `num_threads` host threads (0 = the
        reference's sequential loop, mcu.rs:253-351, ran instead)."""
        return int(self._lib.zj_decoder_entropy_segments(self._h))

    # ---- queries
    def info(self):
        """Decoder::info (decoder.rs:210): None until headers were parsed."""
        raw = ZjImageInfo()
        self._lib.zj_decoder_info(self._h, C.byref(raw))
        return ImageInfo(raw) if raw.valid else None

    def width(self) -> int:
        raw = ZjImageInfo()
        self._lib.zj_decoder_info(self._h, C.byref(raw))
        return raw.width

    def height(self) -> int:
        raw = ZjImageInfo()
        self._lib.zj_decoder_info(self._h, C.byref(raw))
        return raw.height

    def get_output_colorspace(self) -> ColorSpace:
        return ColorSpace(self._lib.zj_decoder_out_colorspace(self._h))

    def exif_orientation(self) -> int:
        """The EXIF orientation (1-8) of the file whose headers were read last, whatever the options: 1 before headers or when
        the file has none.  Pillow's rule (getexif + exif_transpose; the header states it next to ZJ_FLAG_ORIENT_SHIFT)."""
        return int(self._lib.zj_decoder_orientation(self._h))

    # ---- deprecated setters kept by the reference (decoder.rs:531-603)
    def rgba(self):
        self.set_output_colorspace(ColorSpace.RGBA)

    def set_limits(self, width: int, height: int):
        self.options = self.options.set_max_width(width).set_max_height(height)
        self._rebuild()

    def set_output_colorspace(self, colorspace):
        self.options = self.options.set_out_colorspace(colorspace)
        self._rebuild()

    def set_num_threads(self, threads: int):
        if threads == 0:
            raise DecodeErrors(2, '"Cannot set zero threads to decode image"')
        self.options = self.options.set_num_threads(threads)
        self._rebuild()


# names later zune-jpeg releases use for the same objects
JpegDecoder = Decoder
DecoderOptions = ZuneJpegOptions
UnsupportedSchemes = enum.Enum("UnsupportedSchemes", "ExtendedSequentialHuffman LosslessHuffman ExtendedSequentialDctArithmetic ProgressiveDctArithmetic LosslessArithmetic")


# names of later zune-jpeg releases (BASELINE north_star: `JpegDecoder::new(..).decode()/decode_into()` + `DecoderOptions`)
JpegDecoder = Decoder
DecoderOptions = ZuneJpegOptions


def draft_scale(width: int, height: int, size):
    """Pillow's Image.draft rule for a width x height JPEG drafted to size = (w, h): d = the largest of 8, 4, 2, 1 with
    min(width // w, height // h) >= d.  Returns (d, (ceil(width / d), ceil(height / d))), the denominator for
    ZuneJpegOptions.set_scale_denom and the size the decode then has."""
    scale = min(width // size[0], height // size[1])
    d = next(a for a in (8, 4, 2, 1) if scale >= a or a == 1)
    return d, _ffi.scaled_size(width, height, d)


def _input_arrays(buffers):
    """(keep, bufs, lens): the inputs as bytes or uint8 arrays (the caller keeps them alive during the call) and the pointer and
    length arrays the batch calls take"""
    n = len(buffers)
    keep = [b if isinstance(b, np.ndarray) else bytes(b) for b in buffers]
    bufs = (C.c_void_p * n)(*[b.ctypes.data if isinstance(b, np.ndarray) else C.cast(C.c_char_p(b), C.c_void_p).value for b in keep])
    lens = (C.c_size_t * n)(*[b.nbytes if isinstance(b, np.ndarray) else len(b) for b in keep])
    return keep, bufs, lens


def _image_error(lib, i: int, status: int, batch_errors: bool = True) -> DecodeErrors:
    """image i's failure in a batch call: the variant and text Decoder.decode_buffer raises for the same input
    (zj_batch_error_kind / zj_batch_error, which the call records when `batch_errors`)"""
    kind = lib.zj_batch_error_kind(i) if batch_errors else 0
    text = lib.zj_batch_error(i).decode(errors="replace") if kind else lib.zj_gpu_strerror(status).decode()
    return DecodeErrors(kind or (13 if status != _ffi.ERR_DECODE else 1), text, status)


def decode_batch(buffers, options: ZuneJpegOptions | None = None, threads: int = 0, out=None, gpu_entropy: bool = False, stats: dict | None = None,
                 device_out=None, desc=None, devices=None):
    """zj_decode_batch: JPEG byte strings in, pixel bytes out, `threads` host threads (0 = one per hardware thread)
    running the host stage of different images side by side while the GPU reconstructs the finished ones.
    `gpu_entropy=True` (zj_decode_batch_gpu): baseline JPEGs with restart markers are entropy-decoded on the GPU as well, one
    restart interval per thread; same results, `stats["gpu_entropy"]` = how many images took that route.
    `device_out=[(device_ptr, nbytes), ...]` (zj_decode_batch_gpu_device): the pixels stay in device memory; with
    `desc=gpu.OutputDesc(...)` (zj_decode_batch_gpu_device_ex) in the layout / type / scale a GPU consumer wants.
    `devices=[0, 1, ...]` (zj_decode_batch_multi): the batch is cut into contiguous image ranges, one per device of the box
    (strip ranges when there are fewer images than devices).

    Returns a list with one entry per input: `bytes` (or, with `out` / `device_out`, the number of bytes written) for a decoded
    image, a `DecodeErrors` instance for a failed one.  `out`: optional list of writable buffers (e.g. PinnedBuffer.array
    slices), one per image, large enough for width*height*components (ceil(width / d) * ceil(height / d) * components with the
    options' scale denominator d).  Inputs may be `bytes` or uint8 numpy arrays (e.g. views of pinned memory, which upload at the
    full PCIe rate)."""
    lib = _ffi.load()
    options = options if options is not None else ZuneJpegOptions()
    raw = options._raw()
    raw.num_threads = int(threads)
    n = len(buffers)
    keep, bufs, lens = _input_arrays(buffers)
    outs = (C.c_void_p * n)()
    out_len = (C.c_size_t * n)()
    status = (C.c_int * n)()
    if device_out is not None:
        for i, (ptr, nbytes) in enumerate(device_out):
            outs[i] = ptr
            out_len[i] = nbytes
    elif out is not None:
        views = [np.frombuffer(o, dtype=np.uint8) if not isinstance(o, np.ndarray) else o for o in out]
        for i, v in enumerate(views):
            outs[i] = v.ctypes.data
            out_len[i] = v.nbytes
    if devices is not None:
        devs = (C.c_int * len(devices))(*devices)
        rc = lib.zj_decode_batch_multi(C.byref(raw), devs, len(devices), bufs, lens, n, outs, out_len, status)
    elif gpu_entropy or device_out is not None:
        n_gpu = C.c_size_t(0)
        if device_out is not None and desc is not None:
            rc = lib.zj_decode_batch_gpu_device_ex(C.byref(raw), bufs, lens, n, C.byref(desc.c), outs, out_len, status, C.byref(n_gpu))
        else:
            fn = lib.zj_decode_batch_gpu_device if device_out is not None else lib.zj_decode_batch_gpu
            rc = fn(C.byref(raw), bufs, lens, n, outs, out_len, status, C.byref(n_gpu))
        if stats is not None:
            stats["gpu_entropy"] = int(n_gpu.value)
    else:
        rc = lib.zj_decode_batch(C.byref(raw), bufs, lens, n, outs, out_len, status)
    if rc < 0:
        raise DecodeErrors(13, lib.zj_gpu_strerror(rc).decode(), rc)
    res = []
    for i in range(n):
        if status[i] != 0:
            res.append(_image_error(lib, i, status[i], batch_errors=devices is None))
        elif out is not None or device_out is not None:
            res.append(int(out_len[i]))
        else:
            try:
                res.append(C.string_at(outs[i], out_len[i]))
            finally:
                lib.zj_buffer_free(outs[i])
    return res


def decode_batch_resized(buffers, resize, desc=None, rois=None, options: ZuneJpegOptions | None = None, threads: int = 0):
    """zj_decode_batch_gpu_device_resized: JPEG byte strings in, one batch tensor in device memory out -- every image decoded
    whole, its crop resized to `resize` (a gpu.Resize) in the layout / type / normalisation of `desc` (a gpu.OutputDesc, scale
    must be full size; default HWC u8).  rois: None, or one (x, y, w, h) or None (= the whole image) per image, in the
    coordinates of the decoded image (ceil(width / d) x ceil(height / d) with the options' scale denominator d; with EXIF
    orientation, of the displayed image: oriented_size).

    Returns (gpu.DeviceArray of shape (N, C, OH, OW) or (N, OH, OW, C), [None | DecodeErrors per image]).  The errors are the
    ones decode_batch reports for the same inputs; a crop that does not fit its image, or an image whose channel count is not
    the one the options' colourspace gives, fails with status ZJ_ERR_INVALID_ARG.  The slot of a failed image is not written."""
    from . import gpu
    lib = _ffi.load()
    options = options if options is not None else ZuneJpegOptions()
    desc = desc if desc is not None else gpu.OutputDesc()
    raw = options._raw()
    raw.num_threads = int(threads)
    n = len(buffers)
    keep, bufs, lens = _input_arrays(buffers)
    sizes = [(0, 0)] * n
    if rois is not None and any(r is None for r in rois) and not all(r is None for r in rois):
        # whole-image entries next to crops: the sizes come from the headers (a file whose headers fail reports that error)
        for i, r in enumerate(rois):
            if r is None:
                d = Decoder(options)
                try:
                    d.read_headers(keep[i])
                    sizes[i] = _ffi.scaled_size(d.width(), d.height(), options.get_scale_denom())
                    if options.get_exif_orientation():
                        sizes[i] = _ffi.oriented_size(*sizes[i], d.exif_orientation())
                except DecodeErrors:
                    sizes[i] = (1, 1)
    nc = ColorSpace(options.get_out_colorspace()).num_components()
    slot = resize.slot_size(desc, nc)
    out = gpu.DeviceBuffer(max(slot * n, 1), options.get_device())
    status = (C.c_int * n)()
    n_gpu = C.c_size_t(0)
    rc = lib.zj_decode_batch_gpu_device_resized(C.byref(raw), bufs, lens, n, gpu._roi_array(rois, sizes), C.byref(desc.c), C.byref(resize.c),
                                                out.ptr, slot * n, status, C.byref(n_gpu))
    if rc < 0:
        raise DecodeErrors(13, lib.zj_gpu_strerror(rc).decode(), rc)
    errs = [_image_error(lib, i, status[i]) if status[i] != 0 else None for i in range(n)]
    return gpu.DeviceArray(out, (n, *resize.slot_shape(desc, nc)), desc.c.dtype), errs
