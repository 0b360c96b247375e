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
import os

from . import capi
from ._build_ext import EXT, EXT_NAME, LIB

__all__ = ["load", "linear_forward", "cubic_forward", "nearest_forward", "linear_backward", "cubic_backward",
           "nearest_backward", "linear_backward_nonaa", "forward_with_flags", "resize_to_uint8", "decode_resize_normalize", "resized_crops", "AAResize", "aa_resize", "capi"]

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
    if torch.is_tensor(images):
        assert images.dim() == 4 and images.is_cuda
        cl = images.is_contiguous(memory_format=torch.channels_last) and not images.is_contiguous()
        images = [t.permute(1, 2, 0) if cl else t for t in images.unbind(0)]
    if isinstance(boxes, torch.Tensor):
        boxes = boxes.tolist()
    if hflip is not None and isinstance(hflip, torch.Tensor):
        hflip = hflip.tolist()
    oH, oW = (int(size), int(size)) if isinstance(size, int) else (int(size[0]), int(size[1]))
    hwc = capi._is_hwc(images[0])
    C = images[0].shape[-1] if hwc else images[0].shape[0]
    scale = bias = None
    if mean is not None or std is not None:
        scale = [1.0 / (255.0 * s) for s in std]
        bias = [-m / s for m, s in zip(mean, std)]
        out_dtype = out_dtype or torch.float16
    out = torch.empty((len(images), C, oH, oW), dtype=out_dtype or torch.float32, device=images[0].device)
    flags = capi.FLAG_ROUND_NEAREST if out.dtype == torch.uint8 else capi.FLAG_AUTO
    return capi.resize_crops(images, boxes, (oH, oW), mode, out=out, hflip=hflip, scale=scale, bias=bias,
                             align_corners=align_corners, flags=flags)[0]


from .functional import AAResize, aa_resize  # noqa: E402
