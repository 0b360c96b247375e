"""ctypes binding of the C ABI (include/aa_resize.h) -- the same calls a cgo/JNI/FFI host makes.

The parity tests (`-m gpu`) go through this module so that they exercise the C-ABI entry points
directly; torch is used only to allocate device memory and hand over raw pointers.
There is no fallback: a missing library raises at import of the symbol table.
"""
import ctypes
import os

from ._build_ext import LIB

BOX, TRIANGLE, CUBIC = 0, 1, 2
U8, F32, F64, F16, BF16 = 0, 1, 2, 3, 4
FLAG_AUTO, FLAG_FORCE_GENERAL, FLAG_FORCE_STREAM, FLAG_STREAM_TMA, FLAG_STREAM_LDG, FLAG_ROUND_NEAREST = 0, 1, 2, 4, 8, 32
FLAG_VMMA = 64
FLAG_STRICT_NONFINITE = 128
FLAG_ASSUME_FINITE = 256  # skip the drain launch behind the fast float kernels (csrc/aa_redo.cu)
FILL_NONE, FILL_INPUT, FILL_OUTPUT = 0, 1, 2  # aa_fill modes of aa_resize_crops_pad
FILTERS = {"nearest": BOX, "box": BOX, "bilinear": TRIANGLE, "linear": TRIANGLE, "bicubic": CUBIC, "cubic": CUBIC}

EXPORTS = [
    "aa_abi_version", "aa_last_error", "aa_interp_size", "aa_host_tables", "aa_build_tables", "aa_build_tables_sf", "aa_warm_tables",
    "aa_clear_table_cache", "aa_check_device", "aa_debug_counters", "aa_resize_forward", "aa_resize_forward_sf", "aa_resize_backward_sf", "aa_resize_forward_ex", "aa_resize_forward_ragged", "aa_resize_crops", "aa_resize_crops_ex", "aa_resize_crops_pad", "aa_resize_backward",
    "aa_resize_backward_nonaa_bilinear", "aa_resize_forward_host", "aa_resize_forward_host_multi", "aa_launch_count",
]


class TensorDesc(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("dtype", ctypes.c_int32), ("device", ctypes.c_int32),
                ("n", ctypes.c_int64), ("c", ctypes.c_int64), ("h", ctypes.c_int64), ("w", ctypes.c_int64),
                ("stride_n", ctypes.c_int64), ("stride_c", ctypes.c_int64), ("stride_h", ctypes.c_int64),
                ("stride_w", ctypes.c_int64)]


class TablesDesc(ctypes.Structure):
    _fields_ = [("xmin", ctypes.c_void_p), ("xsize", ctypes.c_void_p), ("weights", ctypes.c_void_p),
                ("interp_size", ctypes.c_int32)]


class Epilogue(ctypes.Structure):
    _fields_ = [("normalize", ctypes.c_int32), ("scale", ctypes.c_float * 4), ("bias", ctypes.c_float * 4)]


class ImageDesc(ctypes.Structure):
    _fields_ = [("data", ctypes.c_void_p), ("h", ctypes.c_int64), ("w", ctypes.c_int64), ("stride_h", ctypes.c_int64),
                ("stride_c", ctypes.c_int64)]


class Crop(ctypes.Structure):
    """aa_crop: a box (top, left, height, width) in pixels of its image and an optional horizontal flip."""
    _fields_ = [("top", ctypes.c_int64), ("left", ctypes.c_int64), ("height", ctypes.c_int64), ("width", ctypes.c_int64),
                ("hflip", ctypes.c_int32)]


class CropEx(ctypes.Structure):
    """aa_crop_ex: a box of its image, the size it is resized to, the origin of the stored window in the resized image and
    the flip bits (0: horizontal, 1: vertical)."""
    _fields_ = [("top", ctypes.c_int64), ("left", ctypes.c_int64), ("height", ctypes.c_int64), ("width", ctypes.c_int64),
                ("resized_h", ctypes.c_int64), ("resized_w", ctypes.c_int64), ("crop_top", ctypes.c_int64),
                ("crop_left", ctypes.c_int64), ("flip", ctypes.c_int32)]


class Fill(ctypes.Structure):
    """aa_fill: how aa_resize_crops_pad fills outputs outside the resized image (FILL_NONE, FILL_INPUT: a pixel value of the
    input that goes through the epilogue, FILL_OUTPUT: a value stored as it is) and the value per channel."""
    _fields_ = [("mode", ctypes.c_int32), ("value", ctypes.c_float * 4)]


def crop_ex_dtype():
    """numpy structured dtype laid out as aa_crop_ex (72 bytes): an array of it is passed to the C ABI as it stands, so a
    batch of thousands of crops needs no ctypes object per crop."""
    import numpy as np
    return np.dtype(CropEx)


def image_desc_dtype():
    """numpy structured dtype laid out as aa_image_desc (40 bytes)."""
    import numpy as np
    return np.dtype(ImageDesc)


class Scales(ctypes.Structure):
    _fields_ = [("scale_h", ctypes.c_double), ("scale_w", ctypes.c_double)]


class AAError(RuntimeError):
    pass


_lib = None


def lib():
    """Loads libaa_resize_b200.so (RTLD_GLOBAL so the torch extension resolves against it)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB):
            raise AAError(f"{LIB} is missing: run `python -c 'import __graft_entry__ as g; g.build()'` "
                          "(there is no CPU or PyTorch fallback)")
        L = ctypes.CDLL(LIB, mode=ctypes.RTLD_GLOBAL)
        i32, i64, u32, vp = ctypes.c_int32, ctypes.c_int64, ctypes.c_uint32, ctypes.c_void_p
        P = ctypes.POINTER
        L.aa_abi_version.restype = i32
        L.aa_last_error.restype = ctypes.c_char_p
        L.aa_interp_size.argtypes = [i64, i64, i32, i32, i32, P(i32)]
        L.aa_build_tables.argtypes = [i64, i64, i32, i32, i32, i32, P(TablesDesc), vp]
        L.aa_build_tables_sf.argtypes = [i64, i64, i32, i32, i32, ctypes.c_double, i32, P(TablesDesc), vp]
        L.aa_host_tables.argtypes = [i64, i64, i32, i32, i32, ctypes.c_double, vp, vp]
        L.aa_warm_tables.argtypes = [i64, i64, i64, i64, i32, i32, i32, i32, vp]
        L.aa_resize_forward.argtypes = [P(TensorDesc), P(TensorDesc), i32, i32, u32, vp]
        L.aa_resize_forward_sf.argtypes = [P(TensorDesc), P(TensorDesc), i32, i32, P(Scales), u32, vp]
        L.aa_resize_backward_sf.argtypes = [P(TensorDesc), P(TensorDesc), i32, i32, P(Scales), u32, vp]
        L.aa_resize_forward_ex.argtypes = [P(TensorDesc), P(TensorDesc), i32, i32, u32, P(Epilogue), vp]
        L.aa_resize_forward_ragged.argtypes = [vp, i32, i32, i64, i32, P(TensorDesc), i32, i32, u32, P(Epilogue), vp, P(i32)]
        L.aa_resize_crops.argtypes = [vp, vp, i32, i32, i64, i32, P(TensorDesc), i32, i32, u32, P(Epilogue), vp, P(i32)]
        L.aa_resize_crops_ex.argtypes = [vp, vp, i32, i32, i64, i32, P(TensorDesc), i32, i32, u32, P(Epilogue), vp, P(i32)]
        L.aa_resize_crops_pad.argtypes = [vp, vp, i32, i32, i64, i32, P(TensorDesc), i32, i32, u32, P(Epilogue), P(Fill), vp,
                                          P(i32)]
        L.aa_resize_backward.argtypes = [P(TensorDesc), P(TensorDesc), i32, i32, u32, vp]
        L.aa_resize_backward_nonaa_bilinear.argtypes = [P(TensorDesc), P(TensorDesc), i32, vp]
        L.aa_resize_forward_host.argtypes = [P(TensorDesc), P(TensorDesc), i32, i32, u32]
        L.aa_resize_forward_host_multi.argtypes = [P(TensorDesc), P(TensorDesc), i32, i32, u32, P(i32), i32]
        L.aa_check_device.argtypes = [i32]
        L.aa_debug_counters.argtypes = [i32, vp, i32]
        L.aa_launch_count.argtypes = [i32]
        L.aa_launch_count.restype = i64
        _lib = L
    return _lib


def check(rc):
    if rc != 0:
        raise AAError(f"aa_resize error {rc}: {lib().aa_last_error().decode()}")


def _dtype_code(t):
    import torch
    return {torch.uint8: U8, torch.float32: F32, torch.float64: F64, torch.float16: F16, torch.bfloat16: BF16}[t.dtype]


def desc(t, device=None):
    """TensorDesc for a 4-D torch tensor (CUDA, or host when `device` is given)."""
    assert t.dim() == 4
    dev = t.device.index if t.is_cuda else device
    return TensorDesc(t.data_ptr() if t.numel() else None, _dtype_code(t), dev, *t.shape, *t.stride())


def _stream(t):
    import torch
    return ctypes.c_void_p(torch.cuda.current_stream(t.device).cuda_stream)


def _filter(f):
    return FILTERS[f] if isinstance(f, str) else int(f)


def interp_size(in_size, out_size, filter, align_corners=False, dtype=F32):
    k = ctypes.c_int32(0)
    check(lib().aa_interp_size(in_size, out_size, _filter(filter), int(align_corners), dtype, ctypes.byref(k)))
    return k.value


def host_tables(in_size, out_size, filter, align_corners=False, dtype=F32, scale=None):
    """-> (xmin, xsize) int64 numpy arrays computed on the host (no device): the launch planners' view of the tables."""
    import numpy as np
    xmin = np.empty(out_size, np.int64)
    xsize = np.empty(out_size, np.int64)
    check(lib().aa_host_tables(in_size, out_size, _filter(filter), int(align_corners), dtype, float(scale or 0.0),
                               xmin.ctypes.data, xsize.ctypes.data))
    return xmin, xsize


def build_tables(in_size, out_size, filter, align_corners=False, dtype=None, device=0, scale=None):
    """-> (xmin int64[out], xsize int64[out], weights [out, K]) as CUDA tensors, built by the table kernel."""
    import torch
    dtype = dtype or torch.float32
    code = F64 if dtype == torch.float64 else F32
    if scale and not align_corners:
        import numpy as np  # K = ceil(support)*2+1 with support from the caller's scale (aa_interpolation_impl.h:208-210)
        sc = np.float32(1.0 / scale) if code == F32 else np.float64(1.0 / scale)
        base = {BOX: 0.5, TRIANGLE: 1.0, CUBIC: 2.0}[_filter(filter)]
        sup = (np.float32(base * np.float64(sc)) if code == F32 else base * sc) if sc >= 1.0 else base
        K = int(np.ceil(np.float32(sup))) * 2 + 1
    else:
        K = interp_size(in_size, out_size, filter, align_corners, code)
    dev = torch.device("cuda", device)
    xmin = torch.empty(out_size, dtype=torch.int64, device=dev)
    xsize = torch.empty(out_size, dtype=torch.int64, device=dev)
    w = torch.empty((out_size, K), dtype=dtype, device=dev)
    td = TablesDesc(xmin.data_ptr(), xsize.data_ptr(), w.data_ptr(), 0)
    with torch.cuda.device(dev):
        check(lib().aa_build_tables_sf(in_size, out_size, _filter(filter), int(align_corners), code, float(scale or 0.0),
                                       device, ctypes.byref(td), _stream(xmin)))
    assert td.interp_size == K
    return xmin, xsize, w


def resize_forward(x, output_size, filter, align_corners=False, flags=FLAG_AUTO, out=None, out_u8=False, scales=None):
    """C-ABI forward on a CUDA tensor already contiguous in channels_first or channels_last.
    out_u8=True allocates a uint8 output: the clamp + truncate/round epilogue is fused (FLAG_ROUND_NEAREST).
    scales=(sh, sw): the reference's `scale_factors` (aa_resize_forward_sf)."""
    import torch
    N, C, H, W = x.shape
    oH, oW = int(output_size[0]), int(output_size[1])
    if out is None:
        cl = x.is_contiguous(memory_format=torch.channels_last) and not x.is_contiguous()
        out = torch.empty((N, C, oH, oW), dtype=torch.uint8 if out_u8 else (torch.float64 if x.dtype == torch.float64 else torch.float32),
                          device=x.device, memory_format=torch.channels_last if cl else torch.contiguous_format)
    di, do = desc(x), desc(out)
    if scales is not None:
        sc = Scales(float(scales[0] or 0.0), float(scales[1] or 0.0))
        check(lib().aa_resize_forward_sf(ctypes.byref(di), ctypes.byref(do), _filter(filter), int(align_corners),
                                         ctypes.byref(sc), flags, _stream(x)))
    else:
        check(lib().aa_resize_forward(ctypes.byref(di), ctypes.byref(do), _filter(filter), int(align_corners), flags, _stream(x)))
    return out


def resize_forward_ex(x, output_size, filter, out, scale=None, bias=None, align_corners=False, flags=FLAG_AUTO):
    """C-ABI forward with the decode-adjacent epilogue: `out` may be f16/bf16/f32/u8 and channels_first for a
    channels_last `x`; scale/bias (per channel, <= 4) apply v*scale[c] + bias[c] at the store."""
    e = _epilogue(scale, bias)
    di, do = desc(x), desc(out)
    check(lib().aa_resize_forward_ex(ctypes.byref(di), ctypes.byref(do), _filter(filter), int(align_corners), flags,
                                     ctypes.byref(e), _stream(x)))
    return out


def _is_hwc(t):
    """A 3-D image is taken as [H, W, C] (what a decoder emits) when its last axis is a dense interleave of at most 4 channels,
    else as planar [C, H, W]."""
    return t.dim() == 3 and t.stride(-1) == 1 and t.shape[-1] <= 4 and t.stride(1) == t.shape[-1]


def _epilogue(scale, bias):
    e = Epilogue()
    e.normalize = 1 if scale is not None else 0
    for i in range(4):
        e.scale[i] = float(scale[i]) if scale is not None and i < len(scale) else 1.0
        e.bias[i] = float(bias[i]) if bias is not None and i < len(bias) else 0.0
    return e


def resize_forward_ragged(images, output_size, filter, out=None, align_corners=False, flags=FLAG_AUTO, scale=None, bias=None):
    """Variable-size images -> one fixed-size batch (aa_resize_forward_ragged).  `images`: list of CUDA tensors, all [C,H_i,W_i]
    (planar) or all [H_i,W_i,C] (HWC, as a decoder emits), same dtype.  Returns (out [N,C,oH,oW], launches)."""
    import torch
    hwc = _is_hwc(images[0])
    C = images[0].shape[-1] if hwc else images[0].shape[0]
    oH, oW = int(output_size[0]), int(output_size[1])
    if out is None:
        out = torch.empty((len(images), C, oH, oW), dtype=torch.float32, device=images[0].device,
                          memory_format=torch.channels_last if hwc else torch.contiguous_format)
    rows = image_descs(images, hwc)
    # an (empty) epilogue is what lets the call store f16/bf16, or planar output from HWC input
    e = None
    if scale is not None or out.dtype in (torch.float16, torch.bfloat16) or (hwc and out.is_contiguous() and C > 1):
        e = _epilogue(scale, bias)
    n = ctypes.c_int32(0)
    do = desc(out)
    check(lib().aa_resize_forward_ragged(rows.ctypes.data, len(images), _dtype_code(images[0]), C, int(hwc), ctypes.byref(do),
                                         _filter(filter), int(align_corners), flags, ctypes.byref(e) if e is not None else None,
                                         _stream(out), ctypes.byref(n)))
    return out, n.value


def _crops_batch(name, images, n_rows, out, output_size):
    """-> (hwc, channels, input dtype code, out) of a crops call: `out` defaults to a contiguous float32 [N,C,oH,oW]."""
    import torch
    n = len(images)
    if n_rows != n:
        raise ValueError(f"{name}: images and crops must have the same length")
    hwc = bool(n) and _is_hwc(images[0])
    if n:
        C = images[0].shape[-1] if hwc else images[0].shape[0]
    elif out is not None:
        C = out.shape[1]
    else:
        raise ValueError(f"{name}: an empty batch needs `out`")
    if out is None:
        out = torch.empty((n, C, int(output_size[0]), int(output_size[1])), dtype=torch.float32, device=images[0].device)
    return hwc, C, _dtype_code(images[0]) if n else F32, out


def resize_crops(images, boxes, output_size, filter, out=None, hflip=None, scale=None, bias=None, align_corners=False, flags=FLAG_AUTO):
    """Batched resized crops (aa_resize_crops): out[i] = resize(images[i][top:top+height, left:left+width]) to output_size,
    flipped horizontally where hflip[i].  `images`: list of CUDA tensors, all [H_i,W_i,C] (HWC) or all [C,H_i,W_i] (planar), same
    dtype (uint8 or float32); an image may repeat.  `boxes`: (top, left, height, width) per image.  `out` defaults to a
    contiguous float32 [N,C,oH,oW]; scale/bias (per channel, <= 4) apply v*scale[c] + bias[c] at the store.
    Returns (out, launches)."""
    import numpy as np
    n = len(images)
    if len(boxes) != n or (hflip is not None and len(hflip) != n):
        raise ValueError("resize_crops: images, boxes and hflip must have the same length")
    hwc, C, dtype, out = _crops_batch("resize_crops", images, n, out, output_size)
    crops = np.zeros(n, np.dtype(Crop))
    if n:
        crops["top"], crops["left"], crops["height"], crops["width"] = np.array(boxes, np.int64).reshape(n, 4).T
        if hflip is not None:
            crops["hflip"] = [bool(f) for f in hflip]
    rows = image_descs(images, hwc)  # held until the call returns: only its address is passed
    e = _epilogue(scale, bias)
    k = ctypes.c_int32(0)
    do = desc(out)
    check(lib().aa_resize_crops(rows.ctypes.data, crops.ctypes.data, n, dtype, C, int(hwc), ctypes.byref(do), _filter(filter),
                                int(align_corners), flags, ctypes.byref(e), _stream(out), ctypes.byref(k)))
    return out, k.value


def image_descs(images, hwc):
    """aa_image_desc rows (an image_desc_dtype array) of a list of [H,W,C] (hwc) or [C,H,W] CUDA tensors."""
    import numpy as np
    if hwc:
        rows = [(t.data_ptr(), t.shape[0], t.shape[1], t.stride(0), 1) for t in images]
    else:
        rows = [(t.data_ptr(), t.shape[1], t.shape[2], t.stride(1), t.stride(0)) for t in images]
    return np.array(rows, dtype=image_desc_dtype())


def crop_ex_array(crops):
    """aa_crop_ex rows (a crop_ex_dtype array) from (top, left, height, width, resized_h, resized_w, crop_top, crop_left, flip)
    tuples, an [N, 9] integer array or a crop_ex_dtype array."""
    import numpy as np
    if isinstance(crops, np.ndarray) and crops.dtype == crop_ex_dtype():
        return np.ascontiguousarray(crops.reshape(-1))
    rows = np.asarray(crops, dtype=np.int64).reshape(-1, 9)
    arr = np.zeros(rows.shape[0], crop_ex_dtype())
    for k, f in enumerate(arr.dtype.names):
        arr[f] = rows[:, k]
    if not np.array_equal(arr["flip"], rows[:, 8]):
        raise ValueError("crop_ex_array: flip does not fit in 32 bits")
    return arr


def fill_struct(mode, value):
    """Fill of `mode` with `value`: a number for every channel or one number per channel (at most 4)."""
    f = Fill()
    f.mode = int(mode)
    v = [float(value)] * 4 if isinstance(value, (int, float)) else [float(t) for t in value]
    if not 1 <= len(v) <= 4:
        raise ValueError(f"fill value: one number or one per channel (at most 4), got {value}")
    v = v * 4 if len(v) == 1 else v + [0.0] * (4 - len(v))
    for i in range(4):
        f.value[i] = v[i]
    return f


def launch_crops(image_rows, crop_rows, dtype, channels, hwc, out, filter, scale=None, bias=None, align_corners=False,
                 flags=FLAG_AUTO, fill=None):
    """The crops kernel on descriptor arrays (image_descs / crop_ex_array, one row per crop) into `out`; -> launches.
    Without `fill` it calls aa_resize_crops_ex; with one, a (mode, value) pair or a Fill, aa_resize_crops_pad."""
    assert len(image_rows) == len(crop_rows) and image_rows.dtype == image_desc_dtype() and crop_rows.dtype == crop_ex_dtype()
    assert image_rows.flags.c_contiguous and crop_rows.flags.c_contiguous
    args = [image_rows.ctypes.data, crop_rows.ctypes.data, len(crop_rows), dtype, channels, int(hwc), ctypes.byref(desc(out)),
            _filter(filter), int(align_corners), flags, ctypes.byref(_epilogue(scale, bias))]
    if fill is None:
        call = lib().aa_resize_crops_ex
    else:
        call = lib().aa_resize_crops_pad
        args.append(ctypes.byref(fill if isinstance(fill, Fill) else fill_struct(*fill)))
    k = ctypes.c_int32(0)
    check(call(*args, _stream(out), ctypes.byref(k)))
    return k.value


def _resize_crops(name, images, crops, output_size, filter, out, scale, bias, align_corners, flags, fill):
    rows = crop_ex_array(crops)
    hwc, C, dtype, out = _crops_batch(name, images, len(rows), out, output_size)
    return out, launch_crops(image_descs(images, hwc), rows, dtype, C, hwc, out, filter, scale, bias, align_corners, flags, fill)


def resize_crops_ex(images, crops, output_size, filter, out=None, scale=None, bias=None, align_corners=False, flags=FLAG_AUTO):
    """Batched resize-then-crop (aa_resize_crops_ex): out[i] = the output_size window at (crop_top, crop_left) of
    resize(images[i][top:top+height, left:left+width]) to (resized_h, resized_w), flipped horizontally where bit 0 of flip is
    set and vertically where bit 1 is.  `images` as in resize_crops; `crops`: one aa_crop_ex row per image, tuples
    (top, left, height, width, resized_h, resized_w, crop_top, crop_left, flip), an [N, 9] integer array or a crop_ex_dtype
    array.  `out` defaults to a contiguous float32 [N,C,oH,oW]; scale/bias as in resize_crops.  Returns (out, launches)."""
    return _resize_crops("resize_crops_ex", images, crops, output_size, filter, out, scale, bias, align_corners, flags, None)


def resize_crops_pad(images, crops, output_size, filter, fill=0.0, fill_mode=FILL_INPUT, out=None, scale=None, bias=None,
                     align_corners=False, flags=FLAG_AUTO):
    """Padded resize-then-crop (aa_resize_crops_pad): resize_crops_ex whose windows may reach past the resized image (a
    negative crop_top / crop_left, or past its end); outputs there store `fill` (one number, or one per channel), as a
    pixel value of the input (FILL_INPUT) or as it is (FILL_OUTPUT).  Arguments as in resize_crops_ex.
    Returns (out, launches)."""
    return _resize_crops("resize_crops_pad", images, crops, output_size, filter, out, scale, bias, align_corners, flags,
                         (fill_mode, fill))


def resize_backward(grad_out, input_size, filter, align_corners=False, nonaa=False, flags=FLAG_AUTO, scales=None, out=None):
    import torch
    cl = grad_out.is_contiguous(memory_format=torch.channels_last) and not grad_out.is_contiguous()
    gin = out if out is not None else torch.empty(tuple(input_size), dtype=grad_out.dtype, device=grad_out.device,
                                                  memory_format=torch.channels_last if cl else torch.contiguous_format)
    dg, di = desc(grad_out), desc(gin)
    if scales is not None:
        sc = Scales(float(scales[0] or 0.0), float(scales[1] or 0.0))
        check(lib().aa_resize_backward_sf(ctypes.byref(dg), ctypes.byref(di), _filter(filter), int(align_corners),
                                          ctypes.byref(sc), flags, _stream(grad_out)))
    elif nonaa:
        check(lib().aa_resize_backward_nonaa_bilinear(ctypes.byref(dg), ctypes.byref(di), int(align_corners), _stream(grad_out)))
    else:
        check(lib().aa_resize_backward(ctypes.byref(dg), ctypes.byref(di), _filter(filter), int(align_corners), flags, _stream(grad_out)))
    return gin


def resize_forward_host(x_host, out_host, filter, align_corners=False, flags=FLAG_AUTO, device=0):
    """Host-buffer entry point (H2D, resize, D2H inside the call); tensors are CPU tensors, ideally pinned."""
    di, do = desc(x_host, device), desc(out_host, device)
    check(lib().aa_resize_forward_host(ctypes.byref(di), ctypes.byref(do), _filter(filter), int(align_corners), flags))
    return out_host


def resize_forward_host_multi(x_host, out_host, filter, align_corners=False, flags=FLAG_AUTO, devices=None):
    """One process, several GPUs: shards the host batch by image over `devices` (None: all visible) and returns when done."""
    di, do = desc(x_host, 0), desc(out_host, 0)
    if devices is None:
        arr, n = None, 0
    else:
        n = len(devices)
        arr = (ctypes.c_int32 * n)(*devices)
    check(lib().aa_resize_forward_host_multi(ctypes.byref(di), ctypes.byref(do), _filter(filter), int(align_corners), flags, arr, n))
    return out_host


def check_device(device=0):
    """Raises if a kernel watchdog fired on `device` since the last call (call after torch.cuda.synchronize())."""
    check(lib().aa_check_device(device))


def debug_counters(device=0, reset=True):
    """AA_VMMA_PROF=1 wait-time counters of the tensor-core kernel (include/aa_resize.h: aa_debug_counters)."""
    buf = (ctypes.c_uint64 * 16)()
    check(lib().aa_debug_counters(device, ctypes.cast(buf, ctypes.c_void_p), int(reset)))
    return list(buf)


def launch_count(reset=False):
    return lib().aa_launch_count(int(reset))
