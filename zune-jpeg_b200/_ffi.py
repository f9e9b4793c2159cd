"""ctypes view of include/zune_jpeg_b200.h and the loader for the C-ABI shared library.

There is no fallback: if ``libzune_jpeg_b200.so`` has not been built (``python -c 'import __graft_entry__ as
g; g.build()'``) importing the product path raises.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("ZJ_LIB_PATH") or os.path.join(_HERE, "csrc", "libzune_jpeg_b200.so")  # env override: tuning builds only

# zj_colorspace / zj_variant / zj_status -------------------------------------------------------
CS_RGB, CS_GRAYSCALE, CS_YCBCR, CS_CMYK, CS_YCCK, CS_RGBA, CS_RGBX = range(7)
VARIANT_X86, VARIANT_SCALAR, VARIANT_SPEC = 0, 1, 2
USE_SPEC_OUTPUT = 2   # zj_options.use_unsafe value that selects VARIANT_SPEC
USE_LIBJPEG_OUTPUT = 3   # zj_options.use_unsafe value that selects VARIANT_SPEC with FLAG_ISLOW
FLAG_PROGRESSIVE, FLAG_ISLOW = 1, 2
FLAG_SCALE_SHIFT, FLAG_SCALE_MASK = 2, 3 << 2   # zj_image.flags bits 2-3: k of a DCT-scaled (1/2^k) image
USE_SCALE_SHIFT = 4   # zj_options.use_unsafe = USE_LIBJPEG_OUTPUT | k << USE_SCALE_SHIFT, k = 1..3: libjpeg output at 1/2^k


def scaled_size(width: int, height: int, denom: int):
    """The output size of a DCT-scaled decode to 1/denom: (ceil(width / denom), ceil(height / denom))"""
    return -(-width // denom), -(-height // denom)


FLAG_ORIENT_SHIFT, FLAG_ORIENT_MASK = 4, 7 << 4   # zj_image.flags bits 4-6: EXIF orientation o - 1 (spec images only)
USE_EXIF_ORIENTATION = 0x100   # ORed into a spec / libjpeg / scaled zj_options.use_unsafe value: the output is oriented
USE_GPU_ENTROPY = 0x200        # ORed into a spec / libjpeg / scaled value: zj_decode_batch_gpu* may entropy-decode on the GPU
USE_GPU_PROGRESSIVE = 0x400    # ... next to USE_GPU_ENTROPY: progressive images too


def oriented_size(width: int, height: int, orientation: int):
    """The size of a width x height image after EXIF orientation `orientation` (1-8): 5-8 swap the two"""
    return (height, width) if orientation >= 5 else (width, height)


def image_size(img) -> tuple:
    """(width, height) of a zj_image's output: its size, or the scaled size of a DCT-scaled image (ZJ_FLAG_SCALE_*), oriented
    (ZJ_FLAG_ORIENT_*)"""
    w, h = scaled_size(img.width, img.height, 1 << ((img.flags & FLAG_SCALE_MASK) >> FLAG_SCALE_SHIFT))
    return oriented_size(w, h, ((img.flags & FLAG_ORIENT_MASK) >> FLAG_ORIENT_SHIFT) + 1)
QUIRK_Q9, QUIRK_Q10, QUIRK_Q11, QUIRK_ALL = 1, 2, 4, 7   # zj_host_set_quirks (tests only)
OK = 0
ERR_INVALID_ARG, ERR_UNSUPPORTED, ERR_SHORT_PLANE, ERR_SHORT_OUTPUT = -1, -2, -3, -4
ERR_REF_PANIC, ERR_NO_DEVICE, ERR_CUDA, ERR_OOM, ERR_DECODE = -5, -6, -7, -8, -9


class ZjComponent(C.Structure):
    _fields_ = [
        ("coeff", C.c_void_p),
        ("n_i16", C.c_uint64),
        ("qt", C.c_int32 * 64),
        ("h_samp", C.c_uint32),
        ("v_samp", C.c_uint32),
        ("width_stride", C.c_uint32),
        ("reserved", C.c_uint32),
    ]


class ZjImage(C.Structure):
    _fields_ = [
        ("width", C.c_uint32),
        ("height", C.c_uint32),
        ("n_comp", C.c_uint32),
        ("out_cs", C.c_uint32),
        ("variant", C.c_uint32),
        ("flags", C.c_uint32),
        ("comp", ZjComponent * 3),
    ]


LAYOUT_HWC, LAYOUT_CHW = 0, 1
DTYPE_U8, DTYPE_F16, DTYPE_F32 = 0, 1, 2


class ZjOutputDesc(C.Structure):
    _fields_ = [
        ("layout", C.c_uint32),
        ("dtype", C.c_uint32),
        ("scale_log2", C.c_uint32),
        ("channels", C.c_uint32),
        ("mean", C.c_float * 4),
        ("inv_std", C.c_float * 4),
    ]


FILTER_AREA, FILTER_BILINEAR, FILTER_PIL_BILINEAR, FILTER_PIL_BICUBIC = 0, 1, 18, 19


class ZjRoi(C.Structure):
    _fields_ = [("x", C.c_uint32), ("y", C.c_uint32), ("w", C.c_uint32), ("h", C.c_uint32)]


class _ZjResizeLast(C.Union):
    _fields_ = [("reserved", C.c_uint32), ("short_side", C.c_uint32)]


class ZjResize(C.Structure):
    _anonymous_ = ("_u",)
    _fields_ = [("out_w", C.c_uint32), ("out_h", C.c_uint32), ("filter", C.c_uint32), ("_u", _ZjResizeLast)]


class ZjOptions(C.Structure):
    _fields_ = [
        ("use_unsafe", C.c_uint32),
        ("out_colorspace", C.c_uint32),
        ("num_threads", C.c_uint32),
        ("max_width", C.c_uint32),
        ("max_height", C.c_uint32),
        ("max_scans", C.c_uint32),
        ("strict_mode", C.c_uint32),
        ("device", C.c_int32),
    ]


class ZjImageInfo(C.Structure):
    _fields_ = [
        ("width", C.c_uint16),
        ("height", C.c_uint16),
        ("pixel_density", C.c_uint8),
        ("sof", C.c_uint8),
        ("x_density", C.c_uint16),
        ("y_density", C.c_uint16),
        ("components", C.c_uint8),
        ("valid", C.c_uint8),
    ]


# every symbol include/zune_jpeg_b200.h declares: name -> (restype, argtypes)
_P = C.c_void_p
_PP = C.POINTER(C.c_void_p)
SYMBOLS = {
    "zj_gpu_device_count": (C.c_int, []),
    "zj_output_size": (C.c_size_t, [C.POINTER(ZjImage)]),
    "zj_validate_image": (C.c_int, [C.POINTER(ZjImage)]),
    "zj_gpu_reconstruct": (C.c_int, [C.c_int, _P, C.POINTER(ZjImage), C.c_size_t, _PP, C.POINTER(C.c_size_t)]),
    "zj_gpu_reconstruct_submit": (C.c_int, [C.c_int, _P, C.POINTER(ZjImage), C.c_size_t, _PP, C.POINTER(C.c_size_t), _PP]),
    "zj_gpu_reconstruct_finish": (C.c_int, [_P]),
    "zj_gpu_reconstruct_multi": (C.c_int, [C.POINTER(C.c_int), C.c_size_t, C.POINTER(ZjImage), C.c_size_t, _PP, C.POINTER(C.c_size_t)]),
    "zj_partition": (None, [C.c_size_t, C.c_size_t, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]),
    "zj_image_strip_range": (C.c_int, [C.POINTER(ZjImage), C.c_uint32, C.c_uint32, C.POINTER(ZjImage), C.POINTER(C.c_size_t), C.POINTER(C.c_size_t), C.POINTER(C.c_uint32)]),
    "zj_decode_batch_multi": (C.c_int, [C.POINTER(ZjOptions), C.POINTER(C.c_int), C.c_size_t, C.POINTER(_P), C.POINTER(C.c_size_t), C.c_size_t,
                                        C.POINTER(_P), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]),
    "zj_gpu_reconstruct_device": (C.c_int, [C.c_int, _P, C.POINTER(ZjImage), C.c_size_t, _PP, C.POINTER(C.c_size_t)]),
    "zj_batch_create": (C.c_int, [C.c_int, C.POINTER(ZjImage), C.c_size_t, _PP, C.POINTER(C.c_size_t), _PP]),
    "zj_batch_run": (C.c_int, [_P, _P]),
    "zj_batch_launches": (C.c_int, [_P]),
    "zj_batch_algorithmic_bytes": (C.c_uint64, [_P]),
    "zj_batch_destroy": (None, [_P]),
    "zj_output_desc_default": (None, [C.POINTER(ZjOutputDesc)]),
    "zj_output_desc_is_default": (C.c_int, [C.POINTER(ZjOutputDesc)]),
    "zj_consumer_output_size": (C.c_size_t, [C.POINTER(ZjImage), C.POINTER(ZjOutputDesc)]),
    "zj_consumer_output_shape": (C.c_int, [C.POINTER(ZjImage), C.POINTER(ZjOutputDesc), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32)]),
    "zj_gpu_convert_device": (C.c_int, [C.c_int, _P, _P, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(ZjOutputDesc), _P, C.c_size_t]),
    "zj_gpu_reconstruct_device_ex": (C.c_int, [C.c_int, _P, C.POINTER(ZjImage), C.c_size_t, C.POINTER(ZjOutputDesc), _PP, C.POINTER(C.c_size_t)]),
    "zj_decode_batch_gpu_device_ex": (C.c_int, [C.POINTER(ZjOptions), C.POINTER(_P), C.POINTER(C.c_size_t), C.c_size_t, C.POINTER(ZjOutputDesc),
                                                C.POINTER(_P), C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "zj_resize_slot_size": (C.c_size_t, [C.POINTER(ZjOutputDesc), C.POINTER(ZjResize), C.c_uint32]),
    "zj_image_rows": (C.c_int, [C.POINTER(ZjImage), C.c_uint32, C.c_uint32, C.POINTER(ZjImage), C.POINTER(C.c_uint32)]),
    "zj_gpu_resize_device": (C.c_int, [C.c_int, _P, _P, C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(ZjRoi), C.POINTER(ZjOutputDesc),
                                       C.POINTER(ZjResize), _P, C.c_size_t]),
    "zj_gpu_reconstruct_device_resized": (C.c_int, [C.c_int, _P, C.POINTER(ZjImage), C.c_size_t, C.POINTER(ZjRoi), C.POINTER(ZjOutputDesc),
                                                    C.POINTER(ZjResize), _P, C.c_size_t]),
    "zj_decode_batch_gpu_device_resized": (C.c_int, [C.POINTER(ZjOptions), C.POINTER(_P), C.POINTER(C.c_size_t), C.c_size_t, C.POINTER(ZjRoi),
                                                     C.POINTER(ZjOutputDesc), C.POINTER(ZjResize), _P, C.c_size_t, C.POINTER(C.c_int),
                                                     C.POINTER(C.c_size_t)]),
    "zj_gpu_pinned_alloc": (C.c_int, [C.c_size_t, _PP]),
    "zj_gpu_pinned_free": (C.c_int, [_P]),
    "zj_gpu_device_alloc": (C.c_int, [C.c_int, C.c_size_t, _PP]),
    "zj_gpu_device_free": (C.c_int, [C.c_int, _P]),
    "zj_gpu_memcpy_h2d": (C.c_int, [C.c_int, _P, _P, _P, C.c_size_t]),
    "zj_gpu_memcpy_d2h": (C.c_int, [C.c_int, _P, _P, _P, C.c_size_t]),
    "zj_gpu_memset": (C.c_int, [C.c_int, _P, _P, C.c_int, C.c_size_t]),
    "zj_gpu_stream_create": (C.c_int, [C.c_int, _PP]),
    "zj_gpu_stream_destroy": (C.c_int, [C.c_int, _P]),
    "zj_gpu_stream_synchronize": (C.c_int, [C.c_int, _P]),
    "zj_gpu_event_create": (C.c_int, [C.c_int, _PP]),
    "zj_gpu_event_record": (C.c_int, [C.c_int, _P, _P]),
    "zj_gpu_event_elapsed_ms": (C.c_int, [C.c_int, _P, _P, C.POINTER(C.c_float)]),
    "zj_gpu_event_destroy": (C.c_int, [C.c_int, _P]),
    "zj_gpu_strerror": (C.c_char_p, [C.c_int]),
    "zj_gpu_last_cuda_error": (C.c_char_p, []),
    "zj_gpu_launch_count": (C.c_uint64, []),
    "zj_options_default": (None, [C.POINTER(ZjOptions)]),
    "zj_decoder_new": (_P, [C.POINTER(ZjOptions)]),
    "zj_decoder_free": (None, [_P]),
    "zj_decoder_read_headers": (C.c_int, [_P, _P, C.c_size_t]),
    "zj_decoder_info": (C.c_int, [_P, C.POINTER(ZjImageInfo)]),
    "zj_decoder_out_colorspace": (C.c_uint32, [_P]),
    "zj_decoder_orientation": (C.c_uint32, [_P]),
    "zj_decoder_jpeg_colorspace": (C.c_uint32, [_P]),
    "zj_decoder_component": (C.c_int, [_P, C.c_uint32, C.POINTER(ZjComponent)]),
    "zj_decoder_decode_coefficients": (C.c_int, [_P, _P, C.c_size_t, C.POINTER(ZjImage)]),
    "zj_decoder_decode_buffer": (C.c_int, [_P, _P, C.c_size_t, C.POINTER(C.POINTER(C.c_uint8)), C.POINTER(C.c_size_t)]),
    "zj_buffer_free": (None, [_P]),
    "zj_decoder_decode_into": (C.c_int, [_P, _P, C.c_size_t, _P, C.c_size_t, C.POINTER(C.c_size_t)]),
    "zj_decode_batch": (C.c_int, [C.POINTER(ZjOptions), C.POINTER(_P), C.POINTER(C.c_size_t), C.c_size_t,
                                  C.POINTER(_P), C.POINTER(C.c_size_t), C.POINTER(C.c_int)]),
    "zj_decode_batch_gpu": (C.c_int, [C.POINTER(ZjOptions), C.POINTER(_P), C.POINTER(C.c_size_t), C.c_size_t,
                                      C.POINTER(_P), C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "zj_decode_batch_gpu_device": (C.c_int, [C.POINTER(ZjOptions), C.POINTER(_P), C.POINTER(C.c_size_t), C.c_size_t,
                                             C.POINTER(_P), C.POINTER(C.c_size_t), C.POINTER(C.c_int), C.POINTER(C.c_size_t)]),
    "zj_batch_error_kind": (C.c_int, [C.c_size_t]),
    "zj_batch_error": (C.c_char_p, [C.c_size_t]),
    "zj_release_host_caches": (None, []),
    "zj_release_device_caches": (None, []),
    "zj_host_set_quirks": (None, [C.c_uint32]),
    "zj_host_get_quirks": (C.c_uint32, []),
    "zj_decoder_entropy_segments": (C.c_size_t, [_P]),
    "zj_decoder_error_kind": (C.c_int, [_P]),
    "zj_decoder_error": (C.c_char_p, [_P]),
}

_lib = None


def load() -> C.CDLL:
    """Load libzune_jpeg_b200.so and type every exported symbol.  Raises if it is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            f"{LIB_PATH} not built -- run `python -c 'import __graft_entry__ as g; g.build()'`; "
            "zune_jpeg_b200 has no CPU fallback"
        )
    lib = C.CDLL(LIB_PATH)
    for name, (res, args) in SYMBOLS.items():
        fn = getattr(lib, name)  # AttributeError if the library does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib
