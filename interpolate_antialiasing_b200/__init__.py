"""interpolate_antialiasing_b200 -- B200-native (sm_100a) anti-aliased bilinear/bicubic resize.

Drop-in for ONE hot path of vfdev-5/interpolate-antialiasing: the functions below have the names,
positional signatures and semantics of the reference's pybind module
(/root/reference/step_two_dot_two/extension_interpolate.cpp:46-51) and are backed by the torch C++
extension in csrc/torch_binding.cpp, which calls the C ABI in include/aa_resize.h, which launches
hand-written CUDA kernels.  There is no CPU path and no PyTorch fallback: importing works anywhere,
calling needs the built extension and a CUDA device and fails loudly otherwise.

    import interpolate_antialiasing_b200 as aa
    y = aa.linear_forward(x_cuda, (oH, oW), False)
    aa_interp = aa.load()          # the pybind module itself, e.g. to pass to the reference's test.py helpers
"""
import importlib.util
import numbers
import os

from . import capi
from ._build_ext import EXT, EXT_NAME, LIB

__all__ = ["load", "linear_forward", "cubic_forward", "nearest_forward", "linear_backward", "cubic_backward",
           "nearest_backward", "linear_backward_nonaa", "forward_with_flags", "resize_to_uint8", "decode_resize_normalize", "resized_crops", "resized_output_size",
           "resize_center_crop", "five_crop", "ten_crop", "resize_pad_batch", "AAResize", "aa_resize", "capi"]

_ext = None


def load():
    """Returns the compiled pybind module (same exported names as the reference's `aa_interp`)."""
    global _ext
    if _ext is None:
        if not os.path.exists(EXT) or not os.path.exists(LIB):
            raise capi.AAError(
                f"native extension not built ({EXT}); run `python -c 'import __graft_entry__ as g; g.build()'`. "
                "There is no CPU or PyTorch fallback for this op.")
        import torch  # noqa: F401
        capi.lib()  # load libaa_resize_b200.so first (RTLD_GLOBAL) so the extension binds to it
        spec = importlib.util.spec_from_file_location(EXT_NAME, EXT)
        mod = importlib.util.module_from_spec(spec)
        spec.loader.exec_module(mod)
        _ext = mod
    return _ext


def _sz(v):
    return None if v is None else [int(t) for t in v]


def _sf(v):
    return None if v is None else [float(t) for t in v]


# `scale_factors` is the optional argument of the reference's ti_upsample_*2d_cpu (aa_interpolation_impl.h:735) that its
# shim always leaves empty; with it output_size may be None (floor(in * scale)) and the table scale is 1/scale_factor.
def linear_forward(input, output_size, align_corners=False, scale_factors=None):
    return load().linear_forward(input, _sz(output_size), align_corners, _sf(scale_factors))


def cubic_forward(input, output_size, align_corners=False, scale_factors=None):
    return load().cubic_forward(input, _sz(output_size), align_corners, _sf(scale_factors))


def nearest_forward(input, output_size, align_corners=False, scale_factors=None):
    return load().nearest_forward(input, _sz(output_size), align_corners, _sf(scale_factors))


def linear_backward(grad_output, output_size, input_size, align_corners=False, scale_factors=None):
    return load().linear_backward(grad_output, _sz(output_size), list(input_size), align_corners, _sf(scale_factors))


def cubic_backward(grad_output, output_size, input_size, align_corners=False, scale_factors=None):
    return load().cubic_backward(grad_output, _sz(output_size), list(input_size), align_corners, _sf(scale_factors))


def nearest_backward(grad_output, output_size, input_size, align_corners=False, scale_factors=None):
    return load().nearest_backward(grad_output, _sz(output_size), list(input_size), align_corners, _sf(scale_factors))


def linear_backward_nonaa(grad_output, output_size, input_size, align_corners=False):
    return load().linear_backward_nonaa(grad_output, list(output_size), list(input_size), align_corners)


def forward_with_flags(input, output_size, align_corners, filter, flags):
    return load().forward_with_flags(input, list(output_size), align_corners, capi.FILTERS.get(filter, filter), flags)


def resize_to_uint8(input, output_size, mode="bilinear", align_corners=False, round_nearest=True):
    """uint8/float32 in -> uint8 out with the clamp + round epilogue fused into the kernel's store
    (round_nearest=False reproduces the reference harness' clamp + `.byte()` truncation, test.py:71-75)."""
    return load().forward_u8(input, list(output_size), align_corners, capi.FILTERS[mode], round_nearest)


def decode_resize_normalize(x_hwc_u8, output_size, mean, std, mode="bilinear", out_dtype=None, align_corners=False):
    """Decode-adjacent fused op (SURVEY 8(f) row 4): [N,H,W,C] uint8 (as a JPEG decoder emits) -> anti-aliased
    resize -> (x/255 - mean)/std -> [N,C,oH,oW] contiguous float16/bfloat16/float32, all in ONE kernel."""
    import torch
    assert x_hwc_u8.dim() == 4 and x_hwc_u8.is_cuda
    N, H, W, C = x_hwc_u8.shape
    x = x_hwc_u8.permute(0, 3, 1, 2)  # a channels_last NCHW view of the same memory, no copy
    out = torch.empty((N, C, int(output_size[0]), int(output_size[1])), dtype=out_dtype or torch.float16, device=x.device)
    scale = [1.0 / (255.0 * s) for s in std]
    bias = [-m / s for m, s in zip(mean, std)]
    return capi.resize_forward_ex(x, output_size, mode, out, scale, bias, align_corners)


def _image_batch(images):
    """The `images` argument of resized_crops and the eval-crop helpers -> (list of 3-D CUDA tensors, hwc, channels,
    [(h, w)] per image)."""
    import torch
    if torch.is_tensor(images):
        assert images.dim() == 4 and images.is_cuda
        cl = images.is_contiguous(memory_format=torch.channels_last) and not images.is_contiguous()
        images = [t.permute(1, 2, 0) if cl else t for t in images.unbind(0)]
    hwc = capi._is_hwc(images[0])
    C = images[0].shape[-1] if hwc else images[0].shape[0]
    hw = [(t.shape[0], t.shape[1]) if hwc else (t.shape[1], t.shape[2]) for t in images]
    return images, hwc, C, hw


def _normalize_args(mean, std, out_dtype):
    """-> (scale, bias, out dtype, flags) of the (x/255 - mean)/std epilogue, or none of it."""
    import torch
    scale = bias = None
    if mean is not None or std is not None:
        scale = [1.0 / (255.0 * s) for s in std]
        bias = [-m / s for m, s in zip(mean, std)]
        out_dtype = out_dtype or torch.float16
    out_dtype = out_dtype or torch.float32
    return scale, bias, out_dtype, capi.FLAG_ROUND_NEAREST if out_dtype == torch.uint8 else capi.FLAG_AUTO


def resized_crops(images, boxes, size, mode="bilinear", hflip=None, mean=None, std=None, out_dtype=None, align_corners=False):
    """RandomResizedCrop + RandomHorizontalFlip of a batch in one kernel launch: torchvision's
    `resized_crop(img, top, left, height, width, size, antialias=True)` per image, with its own box, optionally flipped.

    images: a list of CUDA tensors, all [H,W,C] (HWC uint8 as a decoder emits; C <= 4) or all [C,H,W], uint8 or float32,
            or one 4-D [N,C,H,W] tensor (contiguous or channels_last).  An image may repeat (several boxes of one image).
    boxes:  (top, left, height, width) per image, e.g. from torchvision.transforms.RandomResizedCrop.get_params; each box
            must lie inside its image.
    hflip:  optional booleans per image.
    mean/std: the affine map of decode_resize_normalize, (x/255 - mean)/std, fused into the store; the output is float16
            unless out_dtype says otherwise.  Without them the output is float32, or uint8 rounded to nearest with
            out_dtype=torch.uint8.
    Returns a contiguous [N,C,oH,oW] tensor."""
    import torch
    images, _, C, _ = _image_batch(images)
    if isinstance(boxes, torch.Tensor):
        boxes = boxes.tolist()
    if hflip is not None and isinstance(hflip, torch.Tensor):
        hflip = hflip.tolist()
    oH, oW = (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[1]))
    scale, bias, out_dtype, flags = _normalize_args(mean, std, out_dtype)
    out = torch.empty((len(images), C, oH, oW), dtype=out_dtype, device=images[0].device)
    return capi.resize_crops(images, boxes, (oH, oW), mode, out=out, hflip=hflip, scale=scale, bias=bias,
                             align_corners=align_corners, flags=flags)[0]


def resized_output_size(h, w, size, max_size=None):
    """The (height, width) torchvision.transforms.v2.functional.resize(img, size, max_size=max_size) gives an h x w image,
    host-only.  size: an int or [int] for the shorter edge (the longer one becomes int(size * long / short), the aspect ratio
    kept), (h, w) for both, or None with max_size (the longer edge becomes max_size).  max_size caps the longer edge of the
    int / [int] form and must then exceed the requested shorter edge; it cannot be combined with (h, w)."""
    if isinstance(size, numbers.Integral):
        size = [int(size)]
    elif size is not None:
        size = [int(v) for v in size]
        if len(size) not in (1, 2):
            raise ValueError(f"size must be an int or a sequence of one or two ints, got {size}")
        if max_size is not None and len(size) != 1:
            raise ValueError("max_size should only be passed if size is None or specifies the length of the smaller edge, "
                             "i.e. size should be an int or a sequence of length 1")
    short, long = (w, h) if w <= h else (h, w)
    if size is None:
        if not isinstance(max_size, numbers.Integral):
            raise ValueError(f"max_size must be an integer when size is None, but got {max_size} instead.")
        new_short, new_long = int(max_size * short / long), int(max_size)
    elif len(size) == 1:
        new_short, new_long = size[0], int(size[0] * long / short)
        if max_size is not None:
            if max_size <= size[0]:
                raise ValueError(f"max_size = {max_size} must be strictly greater than the requested size for the smaller "
                                 f"edge size = {size}")
            if new_long > max_size:
                new_short, new_long = int(max_size * new_short / new_long), int(max_size)
    else:
        return size[0], size[1]
    return (new_long, new_short) if w <= h else (new_short, new_long)


def _crop_hw(crop_size):
    """torchvision's CenterCrop / FiveCrop size argument: an int, [int] or (h, w)."""
    if isinstance(crop_size, numbers.Integral):
        return int(crop_size), int(crop_size)
    crop_size = [int(v) for v in crop_size]
    if len(crop_size) == 1:
        return crop_size[0], crop_size[0]
    if len(crop_size) != 2:
        raise ValueError(f"crop size must be an int or (h, w), got {crop_size}")
    return crop_size[0], crop_size[1]


def _eval_crops(hw, size, crop_size, kind, vertical_flip=False, max_size=None, pad=False):
    """Host-only: the aa_crop_ex rows ([N, kinds] of capi.crop_ex_dtype) of Resize(size, max_size) followed by
    CenterCrop ("center"), FiveCrop ("five") or TenCrop ("ten") of crop_size, for images of sizes hw ([N, 2]: h, w).
    pad (CenterCrop only): a crop larger than the resized image gets the window torchvision's zero padding gives."""
    import numpy as np
    ch, cw = _crop_hw(crop_size)
    hw = np.asarray(hw, np.int64).reshape(-1, 2)
    R = np.array([resized_output_size(int(h), int(w), size, max_size) for h, w in hw], np.int64).reshape(-1, 2)
    small = np.nonzero((R[:, 0] < ch) | (R[:, 1] < cw))[0]
    if len(small) and not (pad and kind == "center"):
        i = int(small[0])
        raise ValueError(f"crop size {(ch, cw)} is larger than the resized image {tuple(int(v) for v in R[i])} of image {i}: "
                         "zero padding is not supported")
    dy, dx = R[:, 0] - ch, R[:, 1] - cw
    # torchvision's anchor int(round(d / 2.0)): Python's round, half to even, which np.round also does
    cy, cx = np.round(dy / 2.0).astype(np.int64), np.round(dx / 2.0).astype(np.int64)
    # v2 center_crop pads a too small axis by (c - R) // 2 before and (c - R + 1) // 2 after, then crops at 0 on it
    cy, cx = np.where(dy < 0, -((-dy) // 2), cy), np.where(dx < 0, -((-dx) // 2), cx)
    z = np.zeros_like(dy)
    five = [(z, z, 0), (z, dx, 0), (dy, z, 0), (dy, dx, 0), (cy, cx, 0)]  # torchvision's order: tl, tr, bl, br, center
    if kind == "center":
        windows = five[4:]
    elif kind == "five":
        windows = five
    elif kind == "ten":
        # a crop of the flipped resized image is the flip of the mirrored window of the unflipped one
        windows = five + [(dy - t, l, 2) if vertical_flip else (t, dx - l, 1) for t, l, _ in five]
    else:
        raise ValueError(f"unknown crop kind {kind!r}")
    crops = np.zeros((len(hw), len(windows)), capi.crop_ex_dtype())
    crops["height"], crops["width"] = hw[:, :1], hw[:, 1:]
    crops["resized_h"], crops["resized_w"] = R[:, :1], R[:, 1:]
    for j, (top, left, flip) in enumerate(windows):
        crops["crop_top"][:, j], crops["crop_left"][:, j], crops["flip"][:, j] = top, left, flip
    return crops


def _resize_then_crop(images, size, crop_size, kind, vertical_flip, mode, max_size, mean, std, out_dtype, pad=False):
    """_eval_crops of every image in one aa_resize_crops_ex call, or one aa_resize_crops_pad call with a zero input fill when
    pad (ceil(crops / 512) launches) -> [N * kinds, C, ch, cw]."""
    import numpy as np
    import torch
    images, hwc, C, hw = _image_batch(images)
    crops = _eval_crops(hw, size, crop_size, kind, vertical_flip, max_size, pad)
    scale, bias, out_dtype, flags = _normalize_args(mean, std, out_dtype)
    ch, cw = _crop_hw(crop_size)
    out = torch.empty((crops.size, C, ch, cw), dtype=out_dtype, device=images[0].device)
    rows = np.repeat(capi.image_descs(images, hwc), crops.shape[1])
    capi.launch_crops(rows, crops.reshape(-1), capi._dtype_code(images[0]), C, hwc, out, mode, scale, bias, flags=flags,
                      fill=(capi.FILL_INPUT, 0.0) if pad else None)
    return out


def resize_center_crop(images, size, crop_size, mode="bilinear", max_size=None, mean=None, std=None, out_dtype=None,
                       pad=False):
    """The evaluation transform CenterCrop(crop_size)(Resize(size, antialias=True, max_size=max_size)(img)) of a batch in
    one kernel launch: every image resized with its own aspect ratio (resized_output_size), then the centre window at
    torchvision's anchor int(round((R - c) / 2.0)) stored; only the window's outputs are computed.  images, mode, mean/std
    and out_dtype as in resized_crops.  A crop larger than a resized image raises ValueError unless pad=True, which
    zero-pads it as torchvision v2 center_crop does: (c - R) // 2 zeros before and (c - R + 1) // 2 after on each axis that
    is too small, zeros of the input (they go through mean/std like pixels), still in one launch.
    Returns a contiguous [N,C,ch,cw] tensor."""
    return _resize_then_crop(images, size, crop_size, "center", False, mode, max_size, mean, std, out_dtype, pad)


def five_crop(images, size, crop_size, mode="bilinear", max_size=None, mean=None, std=None, out_dtype=None):
    """FiveCrop(crop_size) after Resize(size, antialias=True, max_size=max_size), one kernel launch per 512 crops.
    Returns a contiguous [N,5,C,ch,cw] tensor in torchvision's order: top-left, top-right, bottom-left, bottom-right,
    centre.  Other arguments as in resize_center_crop."""
    y = _resize_then_crop(images, size, crop_size, "five", False, mode, max_size, mean, std, out_dtype)
    return y.view(-1, 5, *y.shape[1:])


def ten_crop(images, size, crop_size, vertical_flip=False, mode="bilinear", max_size=None, mean=None, std=None,
             out_dtype=None):
    """TenCrop(crop_size, vertical_flip) after Resize(size, antialias=True, max_size=max_size), one kernel launch per 512
    crops.  Returns a contiguous [N,10,C,ch,cw] tensor in torchvision's order: the five crops of five_crop, then the five
    crops of the flipped resized image.  Each of those is computed as the flip of the mirrored window of the unflipped
    image: the flipped top-left is the flipped window at left = W - cw, the flipped centre the one at
    left = W - cw - round((W - cw) / 2), one column right of the unflipped centre when W - cw is odd (rows and the
    vertical flip likewise).  Other arguments as in resize_center_crop."""
    y = _resize_then_crop(images, size, crop_size, "ten", vertical_flip, mode, max_size, mean, std, out_dtype)
    return y.view(-1, 10, *y.shape[1:])


def _pad_layout(hw, size, max_size=None, size_divisible=32, canvas=None, align="top_left"):
    """Host-only: (resized sizes [N, 2], canvas (Hc, Wc), placements [N, 4] as (top, left, h, w)) of resize_pad_batch."""
    import numpy as np
    hw = np.asarray(hw, np.int64).reshape(-1, 2)
    per_image = size is not None and not isinstance(size, numbers.Integral) and len(size) > 0 and \
        not isinstance(size[0], numbers.Integral)
    if per_image:
        R = np.asarray([[int(v) for v in s] for s in size], np.int64).reshape(-1, 2)
        if len(R) != len(hw):
            raise ValueError(f"resize_pad_batch: {len(R)} sizes for {len(hw)} images")
        if (R < 1).any():
            raise ValueError("resize_pad_batch: every resized size must be at least 1x1")
    else:
        R = np.array([resized_output_size(int(h), int(w), size, max_size) for h, w in hw], np.int64).reshape(-1, 2)
    if canvas is None:
        d = int(size_divisible or 1)
        Hc, Wc = (int(-(-int(R[:, k].max()) // d) * d) for k in (0, 1))
    else:
        Hc, Wc = _crop_hw(canvas)
        big = np.nonzero((R[:, 0] > Hc) | (R[:, 1] > Wc))[0]
        if len(big):
            i = int(big[0])
            raise ValueError(f"resized image {tuple(int(v) for v in R[i])} of image {i} is larger than the canvas {(Hc, Wc)}")
    if align == "top_left":
        top, left = np.zeros(len(R), np.int64), np.zeros(len(R), np.int64)
    elif align == "center":
        top, left = (Hc - R[:, 0]) // 2, (Wc - R[:, 1]) // 2
    else:
        raise ValueError(f"align must be 'top_left' or 'center', got {align!r}")
    return R, (Hc, Wc), np.stack([top, left, R[:, 0], R[:, 1]], axis=1)


def resize_pad_batch(images, size, max_size=None, size_divisible=32, canvas=None, align="top_left", fill=None, pad_value=None,
                     mode="bilinear", mean=None, std=None, out_dtype=None):
    """Variable-size images -> one padded batch in one kernel launch per 512 images: each image resized with torchvision v2
    `resize(img, size, max_size=max_size, antialias=True)` (not the non-antialiased resize of torchvision's detection
    transform) and placed on a common canvas whose other outputs hold a constant.  Letterboxing is
    canvas=(640, 640), align="center", fill=114; pad-to-batch (torchvision detection's batch_images, DETR's nested tensors)
    is the default: the canvas is the largest resized size rounded up to size_divisible, images at the top left, zeros
    after normalisation.

    images: as in resized_crops.
    size:   what resized_output_size takes, or one (h, w) per image for a caller with its own size rule.
    canvas: None (see above) or a fixed (H, W); an image resized larger than it raises ValueError.
    align:  "top_left", or "center" with offsets ((Hc - h) // 2, (Wc - w) // 2).
    fill / pad_value: the constant, one number or one per channel; at most one of them may be given.  fill is a pixel value
            of the input and goes through mean/std like a pixel; pad_value is stored as it is.  The default is pad_value=0.
    mean/std/out_dtype: as in resized_crops.
    Returns (batch [N, C, Hc, Wc] contiguous, placements): placements is an int64 CPU tensor [N, 4] with (top, left, h, w)
    of each resized image in the canvas, what a caller needs to map boxes and to build masks."""
    import numpy as np
    import torch
    if fill is not None and pad_value is not None:
        raise ValueError("resize_pad_batch: give fill or pad_value, not both")
    fill_mode, value = (capi.FILL_INPUT, fill) if fill is not None else (capi.FILL_OUTPUT, 0.0 if pad_value is None else pad_value)
    images, hwc, C, hw = _image_batch(images)
    R, (Hc, Wc), place = _pad_layout(hw, size, max_size, size_divisible, canvas, align)
    crops = np.zeros(len(R), capi.crop_ex_dtype())
    crops["height"], crops["width"] = [h for h, _ in hw], [w for _, w in hw]
    crops["resized_h"], crops["resized_w"] = R[:, 0], R[:, 1]
    crops["crop_top"], crops["crop_left"] = -place[:, 0], -place[:, 1]
    scale, bias, out_dtype, flags = _normalize_args(mean, std, out_dtype)
    out = torch.empty((len(R), C, Hc, Wc), dtype=out_dtype, device=images[0].device)
    capi.launch_crops(capi.image_descs(images, hwc), crops, capi._dtype_code(images[0]), C, hwc, out, mode, scale, bias,
                      flags=flags, fill=(fill_mode, value))
    return out, torch.from_numpy(place)


from .functional import AAResize, aa_resize  # noqa: E402
