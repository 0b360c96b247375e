"""Helpers shared by the tests of the three batched-crop entry points (aa_resize_crops, aa_resize_crops_ex,
aa_resize_crops_pad): case lists, bitwise comparison, and the one reference all three are held to.

The reference never goes through the crops kernel: each crop is aa_resize_forward_ex of the box's view to the resized size
with FLAG_FORCE_GENERAL, sliced to the window and flipped with torch.flip.  With a fill, the window starts as the 1x1
resize of the fill and only its part inside the resized image is taken from the resize.  An aa_resize_crops crop
(top, left, h, w) with hflip is the aa_crop_ex (top, left, h, w, oH, oW, 0, 0, hflip)."""
import numpy as np

FILL_NAN = float("nan")

# aa_crop_ex rows every entry point accepts (the output is 32x48)
OK = [(0, 0, 300, 400, 32, 48, 0, 0, 0), (10, 20, 100, 100, 200, 150, 168, 102, 3)]

# (image index, box): 4x upsampling, about 1x, 0.75x from the top-left corner, a full 1080p frame to 224^2, 1-pixel-high and
# 1-pixel-wide boxes (the latter on the right edge), the bottom-right corner of both images, the same image several times
BOXES = [(0, (100, 120, 56, 56)), (0, (10, 20, 224, 230)), (0, (0, 0, 299, 299)), (1, (0, 0, 1080, 1920)),
         (0, (150, 30, 1, 200)), (0, (40, 399, 150, 1)), (0, (180, 200, 120, 200)), (0, (5, 5, 290, 390)),
         (1, (500, 900, 580, 1020))]

# output size -> [(image index, aa_crop_ex without flip)]; the flips cycle through 0..3
WINDOWS = {
    (48, 64): [
        (0, (0, 0, 300, 400, 48, 64, 0, 0)),            # the whole resized image
        (0, (0, 0, 300, 400, 120, 160, 30, 41)),        # interior windows
        (0, (0, 0, 300, 400, 333, 181, 200, 97)),
        (0, (0, 0, 300, 400, 100, 90, 0, 13)),          # touching the top edge
        (0, (0, 0, 300, 400, 100, 90, 52, 26)),         # the bottom and the right edge
        (0, (0, 0, 300, 400, 100, 90, 20, 0)),          # the left edge
        (0, (0, 0, 300, 400, 48, 200, 0, 70)),          # the full height of the resized image
        (0, (100, 120, 20, 25, 80, 100, 17, 19)),       # a window of a 4x upscale
        (1, (0, 0, 1080, 1920, 72, 128, 12, 40)),       # 15x downscale: bicubic windows of 61-63 taps
        (1, (500, 900, 580, 1020, 150, 200, 77, 101)),  # a box smaller than the image, combined with a window
        (0, (5, 7, 290, 380, 60, 80, 12, 16)),          # ... at the bottom-right corner of its resized image
        (0, (299, 0, 1, 400, 48, 300, 0, 236)),         # a 1-pixel-high box, upscaled
    ],
    (1, 37): [(0, (0, 0, 300, 400, 90, 120, 0, 0)), (0, (0, 0, 300, 400, 90, 120, 89, 83)),
              (1, (10, 20, 700, 900, 256, 329, 128, 150))],  # 1-pixel-high windows
    (29, 1): [(0, (0, 0, 300, 400, 90, 120, 61, 119)), (0, (0, 399, 300, 1, 29, 1, 0, 0)),
              (0, (0, 399, 300, 1, 64, 5, 35, 4))],  # 1-pixel-wide windows
}

OUTS = {  # name: (torch dtype name, flags, affine)
    "f32": ("float32", 0, False),
    "u8": ("uint8", 0, False),
    "u8_round": ("uint8", "FLAG_ROUND_NEAREST", False),
    "f16_affine": ("float16", 0, True),
    "bf16_affine": ("bfloat16", 0, True),
}
SCALE, BIAS = [0.0174, -0.031, 2.5, 1.0 / 255], [-2.1, 0.75, -300.0, 0.5]


def _host_args(capi, crops, img_hw=(300, 400), C=3, oHW=(32, 48), out_dtype=None, cl=1):
    """Descriptor arrays for `crops` (aa_crop_ex tuples) on fake device pointers: enough for every check that runs before
    the device is touched.  Returns (image rows, crop rows, out desc); pass rows.ctypes.data."""
    out_dtype = capi.F32 if out_dtype is None else out_dtype
    n = len(crops)
    H, W = img_hw
    imgs = np.zeros(n, capi.image_desc_dtype())
    for i in range(n):
        imgs[i] = (0x10000, H, W, W * C if cl else W, 1 if cl else H * W)
    rows = capi.crop_ex_array(crops)
    oH, oW = oHW
    out = capi.TensorDesc(0x20000 if n else None, out_dtype, 0, n, C, oH, oW, C * oH * oW, oH * oW, oW, 1)
    return imgs, rows, out


def _view(img, hwc, box):
    top, left, h, w = box
    if hwc:
        return img[top:top + h, left:left + w, :].permute(2, 0, 1).unsqueeze(0)
    return img[:, top:top + h, left:left + w].unsqueeze(0)


def _bits(t):
    import torch
    return t.view({4: torch.int32, 2: torch.int16, 1: torch.uint8}[t.element_size()])


def _assert_same_bits(got, want, what):
    import torch
    g, w = _bits(got.contiguous()), _bits(want.contiguous())
    if not torch.equal(g, w):
        bad = (g != w).nonzero()
        raise AssertionError(f"{what}: {bad.shape[0]} of {g.numel()} outputs differ, first at {bad[0].tolist()}: "
                             f"{got[tuple(bad[0])].item()} vs {want[tuple(bad[0])].item()}")


def _images(kind, C, dev, seed):
    """Two images per kind: 300x400 and a 1080p frame, as HWC or planar tensors."""
    import torch
    g = torch.Generator(device=dev).manual_seed(seed)
    hwc = kind.endswith("hwc")
    imgs = []
    for H, W in ((300, 400), (1080, 1920)):
        shape = (H, W, C) if hwc else (C, H, W)
        if kind.startswith("u8"):
            imgs.append(torch.randint(0, 256, shape, generator=g, device=dev, dtype=torch.uint8))
        else:
            imgs.append(torch.rand(shape, generator=g, device=dev) * 255)
    return imgs


def _fill_value(capi, C, fill, mode, out_dtype, scale, bias, flags, dev):
    """[C] tensor: the 1x1 resize of a [1, C, 1, 1] float32 tensor holding the fill."""
    import torch
    x = torch.tensor(fill[:C] if len(fill) >= C else fill * C, dtype=torch.float32, device=dev).view(1, C, 1, 1)
    o = torch.empty((1, C, 1, 1), dtype=out_dtype, device=dev)
    if mode == capi.FILL_OUTPUT:
        scale = bias = None
    capi.resize_forward_ex(x, (1, 1), "bilinear", o, scale, bias, False, flags | capi.FLAG_FORCE_GENERAL)
    return o.view(C)


def _reference(capi, images, crops, osize, filt, align, out_dtype, scale=None, bias=None, flags=0, fill=None,
               fill_mode=None):
    """The expected [N, C, oH, oW] output of aa_crop_ex rows `crops`.  Without `fill` every window must lie inside its
    resized image; with one (values per channel and a FILL_* mode) the outputs outside it hold the fill."""
    import torch
    hwc = capi._is_hwc(images[0])
    C = images[0].shape[-1] if hwc else images[0].shape[0]
    oH, oW = osize
    if fill is not None:
        fv = _fill_value(capi, C, fill, fill_mode, out_dtype, scale, bias, flags, images[0].device)
    outs = []
    for img, c in zip(images, crops):
        top, left, h, w, rh, rw, ct, cl, flip = (int(v) for v in c)
        y0, y1, x0, x1 = max(ct, 0), min(ct + oH, rh), max(cl, 0), min(cl + oW, rw)
        if fill is None:
            assert (y0, y1, x0, x1) == (ct, ct + oH, cl, cl + oW), ("window outside the resized image", c)
            win = torch.empty((1, C, oH, oW), dtype=out_dtype, device=img.device)
        else:
            win = fv.view(1, C, 1, 1).expand(1, C, oH, oW).clone()
        if y0 < y1 and x0 < x1:
            r = torch.empty((1, C, rh, rw), dtype=out_dtype, device=img.device)
            capi.resize_forward_ex(_view(img, hwc, (top, left, h, w)), (rh, rw), filt, r, scale, bias, align,
                                   flags | capi.FLAG_FORCE_GENERAL)
            win[:, :, y0 - ct:y1 - ct, x0 - cl:x1 - cl] = r[:, :, y0:y1, x0:x1]
        dims = ([-1] if flip & 1 else []) + ([-2] if flip & 2 else [])
        outs.append(win.flip(dims) if dims else win)
    return torch.cat(outs)
