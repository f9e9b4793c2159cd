"""zune_jpeg_b200 -- B200-native pixel-reconstruction path of etemesi254/zune-jpeg behind the reference's
`Decoder` / `ZuneJpegOptions` API (reference src/lib.rs:89-91)."""
from ._ffi import (  # noqa: F401
    CS_CMYK, CS_GRAYSCALE, CS_RGB, CS_RGBA, CS_RGBX, CS_YCBCR, CS_YCCK, FLAG_PROGRESSIVE,
    VARIANT_SCALAR, VARIANT_X86, ZjComponent, ZjImage, ZjImageInfo, ZjOptions,
)

__all__ = ["Decoder", "ZuneJpegOptions", "JpegDecoder", "DecoderOptions", "ColorSpace", "DecodeErrors", "ImageInfo", "reconstruct", "decode_batch",
           "decode_batch_resized", "Resize", "draft_scale"]


def __getattr__(name):  # lazy: importing the package must not require the built library
    if name in ("Decoder", "ZuneJpegOptions", "ColorSpace", "DecodeErrors", "ImageInfo", "UnsupportedSchemes", "decode_batch",
                "decode_batch_resized", "JpegDecoder", "DecoderOptions", "draft_scale"):
        from . import decoder as _d
        return getattr(_d, name)
    if name in ("reconstruct", "Batch", "DeviceBuffer", "PinnedBuffer", "make_image", "Resize"):
        from . import gpu as _g
        return getattr(_g, name)
    raise AttributeError(name)
