"""Thin Python view of the GPU half of the C ABI (include/zune_jpeg_b200.h).  Every call goes through
libzune_jpeg_b200.so; nothing here computes pixels and there is no CPU fallback."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _ffi
from ._ffi import ZjImage


class ZjError(RuntimeError):
    def __init__(self, status: int, where: str = ""):
        lib = _ffi.load()
        msg = lib.zj_gpu_strerror(status).decode()
        if status == _ffi.ERR_CUDA or status == _ffi.ERR_OOM:
            msg += " -- " + lib.zj_gpu_last_cuda_error().decode()
        super().__init__(f"{where}: [{status}] {msg}" if where else f"[{status}] {msg}")
        self.status = status


def _check(status: int, where: str = "") -> None:
    if status != 0:
        raise ZjError(status, where)


def device_count() -> int:
    return _ffi.load().zj_gpu_device_count()


def launch_count() -> int:
    return int(_ffi.load().zj_gpu_launch_count())


def output_size(img: ZjImage) -> int:
    """zj_output_size: bytes of the image's output (width x height, or the scaled size of a DCT-scaled image, x components)"""
    return int(_ffi.load().zj_output_size(C.byref(img)))


def validate(img: ZjImage) -> int:
    return int(_ffi.load().zj_validate_image(C.byref(img)))


def _img_array(images):
    arr = (ZjImage * len(images))()
    for i, im in enumerate(images):
        C.memmove(C.byref(arr[i]), C.byref(im), C.sizeof(ZjImage))
    return arr


def reconstruct(images, device: int = 0, stream=None):
    """zj_gpu_reconstruct: host coefficient planes in, host pixels out (numpy uint8 arrays)."""
    lib = _ffi.load()
    n = len(images)
    arr = _img_array(images)
    outs = []
    ptrs = (C.c_void_p * n)()
    lens = (C.c_size_t * n)()
    for i, im in enumerate(images):
        sz = output_size(im)
        if sz == 0:
            _check(validate(im) or _ffi.ERR_INVALID_ARG, "zj_validate_image")
        o = np.empty(sz, np.uint8)
        outs.append(o)
        ptrs[i] = o.ctypes.data
        lens[i] = sz
    _check(lib.zj_gpu_reconstruct(device, stream, arr, n, ptrs, lens), "zj_gpu_reconstruct")
    return outs


def reconstruct_multi(images, devices):
    """zj_gpu_reconstruct_multi: one batch over several devices of one box (image ranges, or strip ranges when there are fewer
    images than devices); host planes in, host pixels out."""
    lib = _ffi.load()
    n = len(images)
    arr = _img_array(images)
    outs, ptrs, lens = [], (C.c_void_p * n)(), (C.c_size_t * n)()
    for i, im in enumerate(images):
        sz = output_size(im)
        if sz == 0:
            _check(validate(im) or _ffi.ERR_INVALID_ARG, "zj_validate_image")
        o = np.empty(sz, np.uint8)
        outs.append(o)
        ptrs[i], lens[i] = o.ctypes.data, sz
    devs = (C.c_int * len(devices))(*devices)
    _check(lib.zj_gpu_reconstruct_multi(devs, len(devices), arr, n, ptrs, lens), "zj_gpu_reconstruct_multi")
    return outs


class DeviceBuffer:
    """cudaMalloc'd bytes owned through the C ABI."""

    def __init__(self, nbytes: int, device: int = 0):
        self.device, self.nbytes = device, int(nbytes)
        p = C.c_void_p()
        _check(_ffi.load().zj_gpu_device_alloc(device, self.nbytes, C.byref(p)), "zj_gpu_device_alloc")
        self.ptr = p.value

    def upload(self, host: np.ndarray, stream=None, offset: int = 0):
        host = np.ascontiguousarray(host)
        _check(_ffi.load().zj_gpu_memcpy_h2d(self.device, stream, self.ptr + offset, host.ctypes.data, host.nbytes), "h2d")

    def download(self, nbytes: int | None = None, stream=None, offset: int = 0) -> np.ndarray:
        nbytes = self.nbytes - offset if nbytes is None else nbytes
        out = np.empty(nbytes, np.uint8)
        lib = _ffi.load()
        _check(lib.zj_gpu_memcpy_d2h(self.device, stream, out.ctypes.data, self.ptr + offset, nbytes), "d2h")
        _check(lib.zj_gpu_stream_synchronize(self.device, stream), "sync")
        return out

    def memset(self, value: int, stream=None):
        _check(_ffi.load().zj_gpu_memset(self.device, stream, self.ptr, value, self.nbytes), "memset")

    def free(self):
        if self.ptr:
            _ffi.load().zj_gpu_device_free(self.device, self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class PinnedBuffer:
    """cudaHostAlloc'd bytes exposed as a numpy array."""

    def __init__(self, nbytes: int):
        self.nbytes = int(nbytes)
        p = C.c_void_p()
        _check(_ffi.load().zj_gpu_pinned_alloc(self.nbytes, C.byref(p)), "zj_gpu_pinned_alloc")
        self.ptr = p.value
        self.array = np.ctypeslib.as_array((C.c_uint8 * self.nbytes).from_address(self.ptr))

    def free(self):
        if self.ptr:
            self.array = None
            _ffi.load().zj_gpu_pinned_free(self.ptr)
            self.ptr = None

    def __del__(self):
        try:
            self.free()
        except Exception:
            pass


class Batch:
    """zj_batch_*: a reusable launch plan over device-resident planes and outputs."""

    def __init__(self, images, out_ptrs, out_lens, device: int = 0):
        lib = _ffi.load()
        n = len(images)
        self.device = device
        arr = _img_array(images)
        ptrs = (C.c_void_p * n)(*out_ptrs)
        lens = (C.c_size_t * n)(*out_lens)
        h = C.c_void_p()
        _check(lib.zj_batch_create(device, arr, n, ptrs, lens, C.byref(h)), "zj_batch_create")
        self.handle = h

    def run(self, stream=None):
        _check(_ffi.load().zj_batch_run(self.handle, stream), "zj_batch_run")

    @property
    def launches(self) -> int:
        return _ffi.load().zj_batch_launches(self.handle)

    @property
    def algorithmic_bytes(self) -> int:
        return int(_ffi.load().zj_batch_algorithmic_bytes(self.handle))

    def destroy(self):
        if self.handle:
            _ffi.load().zj_batch_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.destroy()
        except Exception:
            pass


def synchronize(device: int = 0, stream=None):
    _check(_ffi.load().zj_gpu_stream_synchronize(device, stream), "sync")


class Stream:
    def __init__(self, device: int = 0):
        self.device = device
        p = C.c_void_p()
        _check(_ffi.load().zj_gpu_stream_create(device, C.byref(p)), "stream_create")
        self.ptr = p.value

    def synchronize(self):
        synchronize(self.device, self.ptr)

    def destroy(self):
        if self.ptr:
            _ffi.load().zj_gpu_stream_destroy(self.device, self.ptr)
            self.ptr = None


class Event:
    def __init__(self, device: int = 0):
        self.device = device
        p = C.c_void_p()
        _check(_ffi.load().zj_gpu_event_create(device, C.byref(p)), "event_create")
        self.ptr = p.value

    def record(self, stream=None):
        _check(_ffi.load().zj_gpu_event_record(self.device, self.ptr, stream), "event_record")

    def elapsed_ms(self, stop: "Event") -> float:
        ms = C.c_float()
        _check(_ffi.load().zj_gpu_event_elapsed_ms(self.device, self.ptr, stop.ptr, C.byref(ms)), "event_elapsed")
        return float(ms.value)


# ------------------------------------------------------------------ device-side consumers (SURVEY.md 8(f).4)
_NP_DTYPES = {_ffi.DTYPE_U8: np.uint8, _ffi.DTYPE_F16: np.float16, _ffi.DTYPE_F32: np.float32}
_TYPESTR = {_ffi.DTYPE_U8: "|u1", _ffi.DTYPE_F16: "<f2", _ffi.DTYPE_F32: "<f4"}


class OutputDesc:
    """zj_output_desc: layout 'HWC' | 'CHW', dtype 'u8' | 'f16' | 'f32', half = 2x2 box down-scale, channels 0 (all) | 3,
    per-channel mean / inv_std in u8 units.  Float values are (float(u8) - mean) * inv_std of the reference's exact bytes."""

    def __init__(self, layout: str = "HWC", dtype: str = "u8", half: bool = False, channels: int = 0,
                 mean=(0.0, 0.0, 0.0, 0.0), inv_std=(1.0, 1.0, 1.0, 1.0)):
        d = _ffi.ZjOutputDesc()
        d.layout = {"HWC": _ffi.LAYOUT_HWC, "CHW": _ffi.LAYOUT_CHW}[layout]
        d.dtype = {"u8": _ffi.DTYPE_U8, "f16": _ffi.DTYPE_F16, "f32": _ffi.DTYPE_F32}[dtype]
        d.scale_log2 = 1 if half else 0
        d.channels = channels
        mean, inv_std = list(mean) + [0.0] * 4, list(inv_std) + [1.0] * 4
        for c in range(4):
            d.mean[c], d.inv_std[c] = float(mean[c]), float(inv_std[c])
        self.c = d

    @property
    def chw(self) -> bool:
        return self.c.layout == _ffi.LAYOUT_CHW

    @property
    def np_dtype(self):
        return _NP_DTYPES[self.c.dtype]

    def out_channels(self, nc: int) -> int:
        """channels written per pixel of nc source bytes (channels=3 drops the fourth byte)"""
        return 3 if (self.c.channels == 3 and nc == 4) else nc

    def shape_of(self, img: ZjImage):
        w, h, ch = C.c_uint32(), C.c_uint32(), C.c_uint32()
        _check(_ffi.load().zj_consumer_output_shape(C.byref(img), C.byref(self.c), C.byref(w), C.byref(h), C.byref(ch)), "zj_consumer_output_shape")
        return (ch.value, h.value, w.value) if self.chw else (h.value, w.value, ch.value)

    def expected(self, u8: np.ndarray, width: int, height: int, nc: int) -> np.ndarray:
        """The specification, applied to the reference's bytes with numpy (tests: `u8` comes from the oracle)."""
        a = np.asarray(u8, np.uint8).reshape(height, width, nc)
        oc = 3 if (self.c.channels == 3 and nc == 4) else nc
        a = a[:, :, :oc]
        mean = np.array(list(self.c.mean)[:oc], np.float32)
        inv = np.array(list(self.c.inv_std)[:oc], np.float32)
        if self.c.scale_log2:
            h2, w2 = height // 2, width // 2
            s = a[: 2 * h2, : 2 * w2].astype(np.uint32).reshape(h2, 2, w2, 2, oc).sum(axis=(1, 3))
            r = ((s + 2) >> 2).astype(np.uint8) if self.c.dtype == _ffi.DTYPE_U8 else ((s.astype(np.float32) * np.float32(0.25) - mean) * inv)
        else:
            r = a if self.c.dtype == _ffi.DTYPE_U8 else ((a.astype(np.float32) - mean) * inv)
        r = r.astype(self.np_dtype)
        return np.ascontiguousarray(r.transpose(2, 0, 1)) if self.chw else np.ascontiguousarray(r)


class DeviceArray:
    """A typed view of device memory produced by the consumer kernels.  Exposes ``__cuda_array_interface__`` (version 3), so
    ``torch.as_tensor(a, device='cuda')``, ``cupy.asarray(a)`` and numba read it in place; ``__dlpack__`` goes through torch."""

    def __init__(self, buf: DeviceBuffer, shape, dtype_code: int):
        self.buf, self.shape, self.dtype_code = buf, tuple(int(x) for x in shape), dtype_code

    @property
    def __cuda_array_interface__(self):
        return {"shape": self.shape, "typestr": _TYPESTR[self.dtype_code], "data": (int(self.buf.ptr or 0), False), "version": 3, "strides": None}

    def to_torch(self):
        import torch
        return torch.as_tensor(self, device=f"cuda:{self.buf.device}")

    def __dlpack__(self, stream=None):
        return self.to_torch().__dlpack__(stream=stream)

    def __dlpack_device__(self):
        return (2, self.buf.device)   # kDLCUDA

    def download(self) -> np.ndarray:
        n = int(np.prod(self.shape)) * np.dtype(_NP_DTYPES[self.dtype_code]).itemsize
        return self.buf.download(n).view(_NP_DTYPES[self.dtype_code]).reshape(self.shape)


def reconstruct_device_ex(images, desc: OutputDesc, device: int = 0, stream=None):
    """zj_gpu_reconstruct_device_ex: `images` carry DEVICE coefficient planes; returns one DeviceArray per image."""
    lib = _ffi.load()
    n = len(images)
    arr = _img_array(images)
    outs, ptrs, lens = [], (C.c_void_p * n)(), (C.c_size_t * n)()
    for i, im in enumerate(images):
        sz = int(lib.zj_consumer_output_size(C.byref(im), C.byref(desc.c)))
        if sz == 0 and output_size(im) == 0:
            _check(validate(im) or _ffi.ERR_INVALID_ARG, "zj_validate_image")
        b = DeviceBuffer(max(sz, 1), device)
        outs.append(DeviceArray(b, desc.shape_of(im), desc.c.dtype))
        ptrs[i], lens[i] = b.ptr, sz
    _check(lib.zj_gpu_reconstruct_device_ex(device, stream, arr, n, C.byref(desc.c), ptrs, lens), "zj_gpu_reconstruct_device_ex")
    return outs


def convert_device(src: DeviceBuffer, width: int, height: int, nc: int, desc: OutputDesc, device: int = 0, stream=None) -> DeviceArray:
    """zj_gpu_convert_device: the consumer alone over interleaved u8 pixels already in device memory."""
    lib = _ffi.load()
    ow, oh = width >> desc.c.scale_log2, height >> desc.c.scale_log2
    oc = desc.out_channels(nc)
    sz = ow * oh * oc * np.dtype(desc.np_dtype).itemsize
    b = DeviceBuffer(max(sz, 1), device)
    _check(lib.zj_gpu_convert_device(device, stream, src.ptr, width, height, nc, C.byref(desc.c), b.ptr, sz), "zj_gpu_convert_device")
    synchronize(device, stream)
    return DeviceArray(b, (oc, oh, ow) if desc.chw else (oh, ow, oc), desc.c.dtype)


# ------------------------------------------------------------------ cropped, resized batch tensors (DESIGN.md section 4.5.1)
_FILTERS = {"area": _ffi.FILTER_AREA, "bilinear": _ffi.FILTER_BILINEAR, "pil_bilinear": _ffi.FILTER_PIL_BILINEAR,
            "pil_bicubic": _ffi.FILTER_PIL_BICUBIC}


def _pil_filter(x: float, bicubic: bool) -> float:
    x = -x if x < 0.0 else x
    if not bicubic:
        return 1.0 - x if x < 1.0 else 0.0
    a = -0.5
    if x < 1.0:
        return ((a + 2.0) * x - (a + 3.0)) * x * x + 1
    if x < 2.0:
        return (((x - 5) * x + 8) * x - 4) * a
    return 0.0


def pil_coefficients(n_in: int, n_out: int, bicubic: bool, first: int = 0, count: int | None = None):
    """Rule 2 of the PIL filters for indices [first, first + count) of an axis resized from n_in to n_out: per index (xmin,
    int64 weights).  Python floats are IEEE doubles and Python evaluates in the order written, without FMA."""
    scale = n_in / n_out
    fs = max(scale, 1.0)
    support = (2.0 if bicubic else 1.0) * fs
    ss = 1.0 / fs
    out = []
    for i in range(first, first + (n_out - first if count is None else count)):
        center = (i + 0.5) * scale
        xmin = max(int(center - support + 0.5), 0)
        xmax = min(int(center + support + 0.5), n_in) - xmin
        k = [_pil_filter((x + xmin - center + 0.5) * ss, bicubic) for x in range(xmax)]
        ww = 0.0
        for w in k:
            ww += w
        if ww != 0.0:
            k = [w / ww for w in k]
        out.append((xmin, np.array([int(-0.5 + w * (1 << 22)) if w < 0 else int(0.5 + w * (1 << 22)) for w in k], np.int64)))
    return out


def pil_geometry(w: int, h: int, out_w: int, out_h: int, short_side: int = 0):
    """Rule 1 of the PIL filters: (RW, RH, left, top) for a w x h crop, or None where the call is ZJ_ERR_INVALID_ARG"""
    if not short_side:
        return out_w, out_h, 0, 0
    short, long = (w, h) if w <= h else (h, w)
    new_long = int(short_side * long / short)
    rw, rh = (short_side, new_long) if w <= h else (new_long, short_side)
    if rw < out_w or rh < out_h or rw > 65535 or rh > 65535:
        return None
    return rw, rh, int(round((rw - out_w) / 2.0)), int(round((rh - out_h) / 2.0))      # (round: half to even)


def _nc_of(img: ZjImage) -> int:
    return {0: 3, 1: 1, 2: 3}.get(int(img.out_cs), 4)


def _roi_array(rois, sizes):
    """zj_roi[n] for a list of (x, y, w, h) or None (= the whole image, sizes[i] = (width, height)) entries; None -> NULL"""
    if rois is None or all(r is None for r in rois):
        return None
    arr = (_ffi.ZjRoi * len(rois))()
    for i, r in enumerate(rois):
        arr[i].x, arr[i].y, arr[i].w, arr[i].h = r if r is not None else (0, 0, *sizes[i])
    return arr


class Resize:
    """zj_resize: each image's crop resized to size = (OH, OW) with filter "area" (adaptive average pooling: the anti-aliased
    choice for down-scales), "bilinear" (torch interpolate, align_corners=False, antialias=False), or Pillow's Image.resize
    with "pil_bilinear" / "pil_bicubic" (torchvision's resized_crop on a PIL image).  With a PIL filter, short_side = S is
    torchvision's Resize(S) of the crop followed by CenterCrop(size).  Every value is the function of the crop's u8 bytes that
    expected() states."""

    def __init__(self, size, filter: str = "area", short_side: int | None = None):
        oh, ow = size
        r = _ffi.ZjResize()
        r.out_w, r.out_h, r.filter = int(ow), int(oh), _FILTERS[filter]
        if short_side is not None:
            if filter not in ("pil_bilinear", "pil_bicubic"):
                raise ValueError("short_side needs a PIL filter")
            r.short_side = int(short_side)
        self.c = r

    @property
    def size(self):
        return (self.c.out_h, self.c.out_w)

    def slot_shape(self, desc: OutputDesc, nc: int):
        oc = desc.out_channels(nc)
        return (oc, self.c.out_h, self.c.out_w) if desc.chw else (self.c.out_h, self.c.out_w, oc)

    def slot_size(self, desc: OutputDesc, nc: int) -> int:
        return int(_ffi.load().zj_resize_slot_size(C.byref(desc.c), C.byref(self.c), nc))

    def expected(self, u8: np.ndarray, width: int, height: int, nc: int, desc: OutputDesc | None = None, roi=None) -> np.ndarray:
        """The specification, applied to the reference's bytes with numpy (tests: `u8` comes from the oracle).  Every float32
        operation is one numpy float32 operation, in the order the header states."""
        desc = desc if desc is not None else OutputDesc()
        f32 = np.float32
        x, y, w, h = roi if roi is not None else (0, 0, width, height)
        oc = 3 if (desc.c.channels == 3 and nc == 4) else nc
        p = np.asarray(u8, np.uint8).reshape(height, width, nc)[y:y + h, x:x + w, :oc]
        OH, OW = self.c.out_h, self.c.out_w
        u8_out = desc.c.dtype == _ffi.DTYPE_U8
        if self.c.filter in (_ffi.FILTER_PIL_BILINEAR, _ffi.FILTER_PIL_BICUBIC):
            g = pil_geometry(w, h, OW, OH, self.c.short_side)
            if g is None:
                raise ValueError(f"a {w}x{h} crop resized to short side {self.c.short_side} does not cover {OW}x{OH}")
            rw, rh, left, top = g
            bicubic = self.c.filter == _ffi.FILTER_PIL_BICUBIC
            cx = pil_coefficients(w, rw, bicubic, left, OW)
            cy = pil_coefficients(h, rh, bicubic, top, OH)
            y0, y1 = cy[0][0], cy[-1][0] + len(cy[-1][1])

            def clip8(s):
                return np.clip(s >> 22, 0, 255)
            q = p[y0:y1].astype(np.int64)
            tmp = np.empty((y1 - y0, OW, oc), np.int64)                 # the horizontal pass's u8 intermediate
            for j, (xm, k) in enumerate(cx):
                tmp[:, j] = clip8((1 << 21) + np.einsum("ywc,w->yc", q[:, xm:xm + len(k)], k))
            v = np.empty((OH, OW, oc), np.int64)
            for i, (ym, k) in enumerate(cy):
                v[i] = clip8((1 << 21) + np.einsum("ywc,y->wc", tmp[ym - y0:ym - y0 + len(k)], k))
            v = v.astype(np.uint8)
            if not u8_out:
                v = v.astype(f32)
        elif self.c.filter == _ffi.FILTER_AREA:
            def windows(n_out, n_in):
                i = np.arange(n_out, dtype=np.int64)
                return (i * n_in) // n_out, ((i + 1) * n_in + n_out - 1) // n_out
            r0, r1 = windows(OH, h)
            c0, c1 = windows(OW, w)
            sat = np.zeros((h + 1, w + 1, oc), np.uint64)           # summed-area table: exact window sums
            sat[1:, 1:] = p.astype(np.uint64).cumsum(axis=0).cumsum(axis=1)
            s = sat[r1][:, c1] - sat[r0][:, c1] - sat[r1][:, c0] + sat[r0][:, c0]
            n = ((r1 - r0)[:, None] * (c1 - c0)[None, :]).astype(np.uint64)[:, :, None]
            v = ((s + n // np.uint64(2)) // n).astype(np.uint8) if u8_out else s.astype(f32) / n.astype(f32)
        else:
            def coords(n_out, n_in):
                sc = f32(n_in) / f32(n_out)
                f = (np.arange(n_out, dtype=f32) + f32(0.5)) * sc - f32(0.5)
                f = np.maximum(f, f32(0))
                i0 = np.minimum(f.astype(np.int64), n_in - 1)
                i1 = np.minimum(i0 + 1, n_in - 1)
                a = f - i0.astype(f32)
                return i0, i1, a, f32(1) - a
            r0, r1, ay, by = coords(OH, h)
            c0, c1, ax, bx = coords(OW, w)
            q = p.astype(f32)
            ax, bx, ay, by = ax[None, :, None], bx[None, :, None], ay[:, None, None], by[:, None, None]
            top = bx * q[r0][:, c0] + ax * q[r0][:, c1]
            bot = bx * q[r1][:, c0] + ax * q[r1][:, c1]
            v = by * top + ay * bot
            if u8_out:
                v = np.clip(np.rint(v), 0, 255).astype(np.uint8)    # (rint: round half to even)
        if not u8_out:
            mean = np.array(list(desc.c.mean)[:oc], f32)
            inv = np.array(list(desc.c.inv_std)[:oc], f32)
            v = (v - mean) * inv
        v = v.astype(desc.np_dtype)
        return np.ascontiguousarray(v.transpose(2, 0, 1)) if desc.chw else np.ascontiguousarray(v)


def resize_device(src: DeviceBuffer, width: int, height: int, nc: int, resize: Resize, desc: OutputDesc | None = None, roi=None,
                  device: int = 0, stream=None) -> DeviceArray:
    """zj_gpu_resize_device: the resize alone over interleaved u8 pixels already in device memory; roi = (x, y, w, h) or None."""
    lib = _ffi.load()
    desc = desc if desc is not None else OutputDesc()
    sz = resize.slot_size(desc, nc)
    b = DeviceBuffer(max(sz, 1), device)
    r = _roi_array([roi], [(width, height)])
    _check(lib.zj_gpu_resize_device(device, stream, src.ptr, width, height, nc, r, C.byref(desc.c), C.byref(resize.c), b.ptr, sz),
           "zj_gpu_resize_device")
    synchronize(device, stream)
    return DeviceArray(b, resize.slot_shape(desc, nc), desc.c.dtype)


def reconstruct_device_resized(images, resize: Resize, desc: OutputDesc | None = None, rois=None, device: int = 0, stream=None) -> DeviceArray:
    """zj_gpu_reconstruct_device_resized: `images` carry DEVICE coefficient planes; returns one (N, C, OH, OW) or (N, OH, OW, C)
    DeviceArray.  rois: None, or one (x, y, w, h) or None (= the whole image) per image, in the coordinates of the image's output
    (the scaled size of a DCT-scaled image); only the strips that hold a crop's rows are reconstructed."""
    lib = _ffi.load()
    desc = desc if desc is not None else OutputDesc()
    n = len(images)
    nc = _nc_of(images[0]) if n else 3
    slot = resize.slot_size(desc, nc)
    b = DeviceBuffer(max(slot * n, 1), device)
    arr = _img_array(images)
    r = _roi_array(rois, [_ffi.image_size(im) for im in images])
    _check(lib.zj_gpu_reconstruct_device_resized(device, stream, arr, n, r, C.byref(desc.c), C.byref(resize.c), b.ptr, slot * n),
           "zj_gpu_reconstruct_device_resized")
    return DeviceArray(b, (n, *resize.slot_shape(desc, nc)), desc.c.dtype)
