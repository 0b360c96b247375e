"""Padded resize-then-crop (aa_resize_crops_pad; aa.resize_center_crop(pad=True), aa.resize_pad_batch): the windows of
aa_resize_crops_ex may reach past the resized image, and their outputs there hold a constant fill.

Outputs inside the resized image must be bit-identical to aa_resize_forward_ex of the box's view with FLAG_FORCE_GENERAL;
outputs outside must be bit-identical to aa_resize_forward_ex of a [1, C, 1, 1] float32 tensor holding the fill, resized to
1x1 with the same out dtype and flags, and with the same epilogue (FILL_INPUT) or none (FILL_OUTPUT).  Argument errors, the
fill struct layout and the geometry of the helpers are checked without a device (the non-GPU tests at the top)."""
import ctypes
import random

import pytest

from crops_common import BIAS, OK, OUTS, SCALE, WINDOWS, _assert_same_bits, _host_args, _images, _reference, _view


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _call(capi, images, crops, count, dtype, channels, channels_last, out, fill=None, filt=1, flags=0):
    n = ctypes.c_int32(-1)
    rc = capi.lib().aa_resize_crops_pad(images, crops, count, dtype, channels, channels_last,
                                        ctypes.byref(out) if out is not None else None, filt, 0, flags, None,
                                        ctypes.byref(fill) if fill is not None else None, None, ctypes.byref(n))
    return rc, capi.lib().aa_last_error().decode(), n.value


# windows that aa_resize_crops_ex refuses as outside the resized image (test_crops_ex_refusals_without_device), and more:
# wholly outside, negative origins, larger than the resized image
OUTSIDE = [(0, 0, 300, 400, 40, 60, -1, 0, 0), (0, 0, 300, 400, 40, 60, 0, -1, 0), (0, 0, 300, 400, 40, 60, 9, 0, 0),
           (0, 0, 300, 400, 40, 60, 0, 13, 0), (0, 0, 300, 400, 31, 48, 0, 0, 0), (0, 0, 300, 400, 32, 47, 0, 0, 0)]
PADDED_ONLY = [(0, 0, 300, 400, 40, 60, -5000, 7, 1), (0, 0, 300, 400, 40, 60, 3, 900, 2), (0, 0, 3, 4, 1, 1, -16, -24, 3),
               (0, 0, 300, 400, 20, 24, -21, -30, 0), ((0, 0, 300, 400, 100, 90, -(1 << 31), -(1 << 31), 0))]


def test_crops_pad_refusals_without_device():
    from interpolate_antialiasing_b200 import capi
    # no fill, or AA_FILL_NONE: every window aa_resize_crops_ex refuses, with the new name
    for fill in (None, capi.fill_struct(capi.FILL_NONE, 5.0)):
        for c in OUTSIDE + PADDED_ONLY:
            imgs, rows, out = _host_args(capi, OK + [c])
            rc, msg, n = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out, fill)
            assert rc == -1 and "crop 2" in msg and msg.startswith("aa_resize_crops_pad") and n == 0, (c, rc, msg, n)
    imgs, rows, out = _host_args(capi, OK + [PADDED_ONLY[0]])
    # an unknown mode
    for mode in (3, -1, 1 << 20):
        rc, msg, _ = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out, capi.fill_struct(mode, 0))
        assert rc == -1 and "fill mode" in msg, (mode, rc, msg)
    # more than 4 channels with a fill (planar)
    imgs5, rows5, out5 = _host_args(capi, OK + [PADDED_ONLY[0]], C=5, cl=0)
    for mode in (capi.FILL_INPUT, capi.FILL_OUTPUT):
        rc, msg, _ = _call(capi, imgs5.ctypes.data, rows5.ctypes.data, 3, capi.F32, 5, 0, out5, capi.fill_struct(mode, 0))
        assert rc == -2 and "4 channels" in msg, (rc, msg)
    # an edge of the window outside int32 (the output is 32x48)
    for ct, cl in ((-(1 << 31) - 1, 0), (0, -(1 << 31) - 1), ((1 << 31) - 32, 0), (0, (1 << 31) - 48), (1 << 40, 0),
                   (0, -(1 << 62))):
        imgs, rows, out = _host_args(capi, OK + [(0, 0, 300, 400, 40, 60, ct, cl, 0)])
        for mode in (capi.FILL_INPUT, capi.FILL_OUTPUT):
            rc, msg, n = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out, capi.fill_struct(mode, 1))
            assert rc == -2 and "crop 2" in msg and "int32" in msg and n == 0, (ct, cl, rc, msg)
    # the other refusals of aa_resize_crops_ex still apply with a fill: a box outside its image, an empty resized size
    for c in ((-1, 0, 10, 10, 32, 48, -3, 0, 0), (0, 0, 300, 400, 0, 48, -3, 0, 0), (0, 0, 300, 400, 32, 48, 0, 0, 4)):
        imgs, rows, out = _host_args(capi, OK + [c])
        rc, msg, _ = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out, capi.fill_struct(capi.FILL_INPUT, 0))
        assert rc == -1 and "crop 2" in msg, (c, rc, msg)


def test_crops_pad_valid_arguments_need_a_device():
    import torch
    from interpolate_antialiasing_b200 import capi
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    for c in OUTSIDE + PADDED_ONLY:
        imgs, rows, out = _host_args(capi, OK + [c])
        for mode in (capi.FILL_INPUT, capi.FILL_OUTPUT):
            rc, msg, _ = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out, capi.fill_struct(mode, 114))
            assert rc == -3 and "CUDA error" in msg, (c, rc, msg)
    # four channels with a fill are fine
    imgs, rows, out = _host_args(capi, OK + [PADDED_ONLY[1]], C=4)
    rc, msg, _ = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 4, 1, out,
                       capi.fill_struct(capi.FILL_INPUT, [1, 2, 3, 4]))
    assert rc == -3, (rc, msg)


def test_fill_struct_layout():
    from interpolate_antialiasing_b200 import capi
    assert ctypes.sizeof(capi.Fill) == 20  # static_assert in aa_api.cu
    assert (capi.Fill.mode.offset, capi.Fill.value.offset) == (0, 4)
    f = capi.fill_struct(capi.FILL_OUTPUT, 2.5)
    assert f.mode == 2 and list(f.value) == [2.5] * 4
    assert list(capi.fill_struct(1, [1, 2, 3]).value) == [1, 2, 3, 0]
    assert list(capi.fill_struct(1, [7]).value) == [7] * 4
    with pytest.raises(ValueError):
        capi.fill_struct(1, [1, 2, 3, 4, 5])


def test_padded_center_crop_origins_against_torchvision():
    pytest.importorskip("torchvision")
    from torchvision.transforms.v2.functional._geometry import (_center_crop_compute_crop_anchor,
                                                                 _center_crop_compute_padding)
    import interpolate_antialiasing_b200 as aa
    checked = padded = 0
    # resized sizes (Resize with (h, w): no aspect rule) against crops with odd and even differences, one axis or both too
    # small, and none
    for rh, rw in ((256, 256), (200, 341), (341, 200), (1, 1), (223, 224), (7, 300)):
        for ch, cw in ((224, 224), (256, 256), (257, 258), (300, 100), (100, 345), (1, 1), (225, 224), (8, 301)):
            rows = aa._eval_crops([(rh, rw)], (rh, rw), (ch, cw), "center", pad=True)[0]
            assert len(rows) == 1
            left, top, right, bottom = _center_crop_compute_padding(ch, cw, rh, rw)
            at, al = _center_crop_compute_crop_anchor(ch, cw, rh + top + bottom, rw + left + right)
            got = (int(rows[0]["crop_top"]), int(rows[0]["crop_left"]))
            assert got == (at - top, al - left), ((rh, rw), (ch, cw), got, (at - top, al - left))
            assert int(rows[0]["flip"]) == 0 and (int(rows[0]["resized_h"]), int(rows[0]["resized_w"])) == (rh, rw)
            checked += 1
            padded += bool(top or left)
    assert checked == 48 and padded >= 25, (checked, padded)
    # without pad the same crops are refused; five / ten crops refuse even with pad
    with pytest.raises(ValueError, match="zero padding"):
        aa._eval_crops([(200, 341)], (200, 341), 224, "center")
    with pytest.raises(ValueError, match="zero padding"):
        aa._eval_crops([(200, 341)], (200, 341), 224, "five", pad=True)


def test_resize_pad_batch_layout():
    import interpolate_antialiasing_b200 as aa
    hw = [(480, 640), (1080, 1920), (640, 480), (333, 500)]
    # pad-to-batch: Resize(800, max_size=1333), canvas = largest size rounded up to 32, images at the top left
    R, canvas, place = aa._pad_layout(hw, 800, 1333)
    want_R = [aa.resized_output_size(h, w, 800, 1333) for h, w in hw]
    assert [tuple(r) for r in R.tolist()] == want_R
    Hm, Wm = max(r[0] for r in want_R), max(r[1] for r in want_R)
    assert canvas == (-(-Hm // 32) * 32, -(-Wm // 32) * 32)
    assert place.tolist() == [[0, 0, h, w] for h, w in want_R]
    assert aa._pad_layout(hw, 800, 1333, size_divisible=1)[1] == (Hm, Wm)
    assert aa._pad_layout(hw, 800, 1333, size_divisible=None)[1] == (Hm, Wm)
    assert aa._pad_layout([(100, 101)], (100, 101), size_divisible=64)[1] == (128, 128)
    # letterbox: a fixed canvas, centred with (Hc - h) // 2, (Wc - w) // 2
    sizes = [(480, 640), (640, 427), (640, 640), (359, 640)]
    R, canvas, place = aa._pad_layout(hw, sizes, canvas=(640, 640), align="center")
    assert canvas == (640, 640) and R.tolist() == [list(s) for s in sizes]
    assert place.tolist() == [[(640 - h) // 2, (640 - w) // 2, h, w] for h, w in sizes]
    assert place[3].tolist() == [140, 0, 359, 640]
    assert aa._pad_layout(hw[:1], [(3, 5)], canvas=8, align="center")[2].tolist() == [[2, 1, 3, 5]]
    # per-image sizes with the automatic canvas
    R, canvas, place = aa._pad_layout(hw[:2], [(10, 20), (33, 7)], size_divisible=16)
    assert canvas == (48, 32) and place.tolist() == [[0, 0, 10, 20], [0, 0, 33, 7]]
    # errors: an image larger than a fixed canvas, a wrong number of sizes, an unknown alignment
    with pytest.raises(ValueError, match="larger than the canvas"):
        aa._pad_layout(hw, 640, canvas=(640, 640))
    with pytest.raises(ValueError):
        aa._pad_layout(hw, [(10, 10)] * 3)
    with pytest.raises(ValueError):
        aa._pad_layout(hw, 256, align="bottom")
    with pytest.raises(ValueError):
        aa.resize_pad_batch([], 256, fill=1, pad_value=0)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: reference = aa_resize_forward_ex of the box's view (FLAG_FORCE_GENERAL) written into a window pre-filled with the
# 1x1 resize of the fill, then flipped
# ---------------------------------------------------------------------------------------------------------------------
FILL = [114.6, -0.0, 300.5, 7.3]  # a u8 clamp and rounding, a negative zero, a value no half-precision type holds


# output size -> [(image index, aa_crop_ex without flip)]; image 0 is 300x400, image 1 1080x1920
PAD_WINDOWS = {
    (48, 64): [
        (0, (0, 0, 300, 400, 120, 160, 30, 41)),        # inside
        (0, (0, 0, 300, 400, 100, 90, -1, 13)),         # 1 px over each edge
        (0, (0, 0, 300, 400, 100, 90, 53, 13)),
        (0, (0, 0, 300, 400, 100, 90, 20, -1)),
        (0, (0, 0, 300, 400, 100, 90, 20, 27)),
        (0, (0, 0, 300, 400, 100, 90, -1, -1)),         # 1 px over each corner
        (0, (0, 0, 300, 400, 100, 90, -1, 27)),
        (0, (0, 0, 300, 400, 100, 90, 53, -1)),
        (0, (0, 0, 300, 400, 100, 90, 53, 27)),
        (0, (0, 0, 300, 400, 20, 30, -10, -17)),        # larger than the resized image on both axes
        (0, (0, 0, 300, 400, 100, 90, -5000, 3)),       # wholly outside
        (0, (0, 0, 300, 400, 100, 90, 10, 91)),
        (0, (10, 10, 2, 3, 1, 1, -20, -30)),            # a 1-pixel resized image
        (0, (100, 120, 20, 25, 80, 100, -5, 50)),       # a 4x upscale
        (1, (0, 0, 1080, 1920, 72, 128, -10, -20)),     # 15x downscale: bicubic windows of 61-63 taps
        (0, (299, 0, 1, 400, 48, 300, 7, 250)),         # a 1-pixel-high box
    ],
    (80, 150): [
        (0, (0, 0, 300, 400, 100, 200, -40, -70)),      # over the top-left by more than a tile (32 rows, 64 columns)
        (0, (0, 0, 300, 400, 100, 200, 60, 120)),       # ... and the bottom-right
        (0, (0, 0, 300, 400, 32, 64, 0, 0)),            # resized edges on the tile boundaries (planar: 64 columns)
        (0, (0, 0, 300, 400, 64, 128, -32, -64)),       # origin on a tile boundary
        (1, (500, 900, 580, 1020, 150, 200, -33, -65)),
        (0, (0, 0, 300, 400, 40, 50, -20, -50)),        # larger than the resized image
        (0, (0, 0, 300, 400, 100, 200, -300, 0)),       # wholly outside
        (0, (0, 0, 300, 400, 100, 200, 0, 250)),
        (0, (10, 10, 2, 3, 1, 1, -40, -75)),            # a 1-pixel resized image
    ],
    (29, 1): [(0, (0, 0, 300, 400, 90, 120, 70, -1)), (0, (0, 399, 300, 1, 29, 1, -3, 0))],
}


@pytest.mark.gpu
@pytest.mark.parametrize("fill_mode", ["input", "output"])
@pytest.mark.parametrize("out_kind", list(OUTS))
@pytest.mark.parametrize("kind", ["u8_hwc", "u8_planar", "f32_planar", "f32_hwc"])
@pytest.mark.parametrize("filt,align", [("box", 0), ("box", 1), ("bilinear", 0), ("bilinear", 1), ("bicubic", 0), ("bicubic", 1)])
def test_crops_pad_parity_matrix(cuda, filt, align, kind, out_kind, fill_mode):
    import torch
    from interpolate_antialiasing_b200 import capi
    dt_name, flag_name, affine = OUTS[out_kind]
    out_dtype = getattr(torch, dt_name)
    flags = getattr(capi, flag_name) if flag_name else 0
    mode = capi.FILL_INPUT if fill_mode == "input" else capi.FILL_OUTPUT
    for C in (1, 3, 4):
        imgs = _images(kind, C, cuda, seed=C)
        scale, bias = (SCALE[:C], BIAS[:C]) if affine else (None, None)
        for osize, windows in PAD_WINDOWS.items():
            images = [imgs[i] for i, _ in windows]
            crops = [c + ((j + C) % 4,) for j, (_, c) in enumerate(windows)]
            out = torch.empty((len(crops), C) + osize, dtype=out_dtype, device=cuda)
            got, launches = capi.resize_crops_pad(images, crops, osize, filt, FILL[:C], mode, out=out, scale=scale, bias=bias,
                                                  align_corners=bool(align), flags=flags)
            want = _reference(capi, images, crops, osize, filt, bool(align), out_dtype, scale, bias, flags, fill=FILL[:C],
                              fill_mode=mode)
            assert launches == 1
            _assert_same_bits(got, want, f"{kind} C={C} {filt} align={align} {out_kind} {fill_mode} {osize}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["u8_hwc", "f32_planar"])
def test_crops_pad_without_fill_is_crops_ex(cuda, kind):
    import torch
    from interpolate_antialiasing_b200 import capi
    imgs = _images(kind, 3, cuda, seed=5)
    for osize, windows in WINDOWS.items():
        images = [imgs[i] for i, _ in windows]
        crops = [c + (j % 4,) for j, (_, c) in enumerate(windows)]
        want, n_ex = capi.resize_crops_ex(images, crops, osize, "bicubic", scale=SCALE[:3], bias=BIAS[:3],
                                          out=torch.empty((len(crops), 3) + osize, dtype=torch.float16, device=cuda))
        rows, descs = capi.crop_ex_array(crops), capi.image_descs(images, capi._is_hwc(images[0]))
        for fill in (None, capi.fill_struct(capi.FILL_NONE, 9.0), capi.fill_struct(capi.FILL_INPUT, 9.0)):
            got = torch.empty_like(want)
            n = ctypes.c_int32(0)
            e = capi._epilogue(SCALE[:3], BIAS[:3])
            do = capi.desc(got)
            capi.check(capi.lib().aa_resize_crops_pad(descs.ctypes.data, rows.ctypes.data, len(rows), capi._dtype_code(images[0]),
                                                      3, int(capi._is_hwc(images[0])), ctypes.byref(do), capi.CUBIC, 0, 0,
                                                      ctypes.byref(e), ctypes.byref(fill) if fill is not None else None,
                                                      capi._stream(got), ctypes.byref(n)))
            assert n.value == n_ex == 1
            _assert_same_bits(got, want, f"no fill {kind} {osize} {fill and fill.mode}")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["u8", "f32"])
def test_random_crop_with_padding_against_torchvision(cuda, kind):
    """RandomCrop(size, padding=p, fill=v) + RandomHorizontalFlip: the box filter at scale 1 is one tap of weight 1, so a
    window of the image itself at an origin in [-p, p] is pad + crop + hflip, bit for bit."""
    import torch
    tv = pytest.importorskip("torchvision.transforms.v2.functional")
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(41)
    g = torch.Generator(device=cuda).manual_seed(41)
    H, W, C, p = 32, 40, 3, 4
    if kind == "u8":
        imgs = [torch.randint(0, 256, (C, H, W), generator=g, device=cuda, dtype=torch.uint8) for _ in range(64)]
        fill = 114
    else:
        imgs = [torch.rand((C, H, W), generator=g, device=cuda) * 255 + 0.25 for _ in range(64)]  # finite, no -0.0
        fill = 0.5
    crops, want = [], []
    for k, im in enumerate(imgs):
        i, j, flip = rnd.randint(-p, p), rnd.randint(-p, p), k % 2
        if k < 4:
            i, j = (-p, p, -p, p)[k], (-p, -p, p, p)[k]
        crops.append((0, 0, H, W, H, W, i, j, flip))
        r = tv.pad(im, [p], fill=fill)[:, i + p:i + p + H, j + p:j + p + W]
        want.append(tv.horizontal_flip(r) if flip else r)
    out = torch.empty((64, C, H, W), dtype=imgs[0].dtype, device=cuda)
    got, n = capi.resize_crops_pad(imgs, crops, (H, W), "box", fill, capi.FILL_INPUT, out=out)
    assert n == 1
    _assert_same_bits(got, torch.stack(want), f"RandomCrop padding {kind}")


def _tv_normalize(x, mean, std):
    import torch
    m = torch.tensor(mean, dtype=torch.float64).view(-1, 1, 1) * 255
    s = torch.tensor(std, dtype=torch.float64).view(-1, 1, 1) * 255
    return (x.double() - m) / s


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["bilinear", "bicubic"])
def test_padded_helpers_against_torchvision(cuda, mode):
    import torch
    tv = pytest.importorskip("torchvision.transforms.v2.functional")
    from torchvision.transforms import InterpolationMode
    import interpolate_antialiasing_b200 as aa
    im = InterpolationMode.BILINEAR if mode == "bilinear" else InterpolationMode.BICUBIC
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    g = torch.Generator().manual_seed(43)
    imgs = [torch.rand((3, H, W), generator=g) * 255 for H, W in ((480, 640), (300, 250), (200, 700), (641, 479))]

    def close(a, b, what):
        a, b = a.cpu().double(), b.double()
        err = (a - b).abs()
        assert a.shape == b.shape and bool((err <= 1e-3 + 1e-5 * b.abs()).all()), (what, float(err.max()))

    # Resize(256) + CenterCrop larger than some resized images, zero padding, normalised
    for crop in (300, (256, 400), (200, 224)):
        got = aa.resize_center_crop([x.to(cuda) for x in imgs], 256, crop, mode=mode, mean=mean, std=std,
                                    out_dtype=torch.float32, pad=True)
        for k, x in enumerate(imgs):
            r = tv.center_crop(tv.resize(x, 256, interpolation=im, antialias=True), crop)
            close(got[k], _tv_normalize(r, mean, std), f"center crop {crop} image {k}")
    # letterbox: 512x512 canvas, centred, fill 114 in the input's domain, normalised
    batch, place = aa.resize_pad_batch([x.to(cuda) for x in imgs], None, max_size=512, canvas=(512, 512), align="center",
                                       fill=114, mode=mode, mean=mean, std=std, out_dtype=torch.float32)
    assert batch.shape == (4, 3, 512, 512) and place.dtype == torch.int64 and place.device.type == "cpu"
    for k, x in enumerate(imgs):
        r = tv.resize(x, None, max_size=512, interpolation=im, antialias=True)
        t, l, h, w = place[k].tolist()
        assert (h, w) == tuple(r.shape[-2:])
        p = tv.pad(r, [l, t, 512 - w - l, 512 - h - t], fill=114)
        close(batch[k], _tv_normalize(p, mean, std), f"letterbox image {k}")
    # pad-to-batch: Resize(256, max_size=400), top left, zeros after normalisation, canvas rounded up to 32
    batch, place = aa.resize_pad_batch([x.to(cuda) for x in imgs], 256, max_size=400, mode=mode, mean=mean, std=std,
                                       out_dtype=torch.float32)
    rs = [tv.resize(x, 256, max_size=400, interpolation=im, antialias=True) for x in imgs]
    Hc, Wc = (-(-max(r.shape[d] for r in rs) // 32) * 32 for d in (1, 2))
    assert batch.shape == (4, 3, Hc, Wc)
    for k, r in enumerate(rs):
        want = torch.zeros((3, Hc, Wc), dtype=torch.float64)
        want[:, :r.shape[1], :r.shape[2]] = _tv_normalize(r, mean, std)
        assert place[k].tolist() == [0, 0, r.shape[1], r.shape[2]]
        close(batch[k], want, f"pad-to-batch image {k}")


@pytest.mark.gpu
def test_padded_helpers_bitwise(cuda):
    """The helpers' outputs are the aa_resize_crops_pad reference, bit for bit: HWC uint8 in, normalised fp16 out."""
    import torch
    import interpolate_antialiasing_b200 as aa
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(47)
    g = torch.Generator(device=cuda).manual_seed(47)
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    scale, bias = [1.0 / (255.0 * s) for s in std], [-m / s for m, s in zip(mean, std)]
    imgs = [torch.randint(0, 256, (rnd.randint(150, 400), rnd.randint(150, 400), 3), generator=g, device=cuda,
                          dtype=torch.uint8) for _ in range(9)]
    y = aa.resize_center_crop(imgs, 200, 256, mean=mean, std=std, pad=True)
    rows = aa._eval_crops([t.shape[:2] for t in imgs], 200, 256, "center", pad=True).reshape(-1)
    want = _reference(capi, imgs, [tuple(int(v) for v in r) for r in rows], (256, 256), "bilinear", False, torch.float16,
                      scale, bias, fill=[0.0], fill_mode=capi.FILL_INPUT)
    _assert_same_bits(y, want, "resize_center_crop(pad=True)")
    # nothing to pad: the same bits as pad=False
    _assert_same_bits(aa.resize_center_crop(imgs, 256, 150, mean=mean, std=std, pad=True),
                      aa.resize_center_crop(imgs, 256, 150, mean=mean, std=std), "pad=True without padding")
    for kw, mode in ((dict(fill=(114, 20, 3)), capi.FILL_INPUT), (dict(pad_value=-1.5), capi.FILL_OUTPUT), ({}, capi.FILL_OUTPUT)):
        for align in ("top_left", "center"):
            batch, place = aa.resize_pad_batch(imgs, 224, max_size=300, align=align, mean=mean, std=std, **kw)
            crops = [(0, 0, t.shape[0], t.shape[1], h, w, -top, -left, 0) for t, (top, left, h, w) in zip(imgs, place.tolist())]
            value = list(kw.get("fill", (kw.get("pad_value", 0.0),)))
            want = _reference(capi, imgs, crops, tuple(batch.shape[-2:]), "bilinear", False, torch.float16, scale, bias,
                              fill=value * 3 if len(value) == 1 else value, fill_mode=mode)
            _assert_same_bits(batch, want, f"resize_pad_batch {kw} {align}")


@pytest.mark.gpu
@pytest.mark.parametrize("hwc", [True, False])
def test_crops_pad_read_inside_boxes_store_inside_output(cuda, hwc):
    import torch
    from interpolate_antialiasing_b200 import capi
    crops = [(0, 0, 80, 90, 100, 120, -30, 40, 0), (37, 11, 5, 140, 70, 300, -40, 250, 1), (100, 150, 50, 50, 64, 72, 0, 0, 2),
             (0, 199, 150, 1, 200, 72, 170, -10, 3), (149, 0, 1, 200, 64, 90, -900, 9, 1), (20, 30, 100, 120, 30, 40, -11, -14, 2)]
    C = 3
    g = torch.Generator(device=cuda).manual_seed(11)

    def image(fill, dtype, c):
        shape = (150, 200, C) if hwc else (C, 150, 200)
        t = torch.full(shape, fill, dtype=dtype, device=cuda)
        v = _view(t, hwc, c[:4])[0]
        if dtype == torch.uint8:
            v.copy_(torch.randint(0, 256, v.shape, generator=g, device=cuda, dtype=torch.uint8))
        else:
            v.copy_(torch.rand(v.shape, generator=g, device=cuda) * 255)
        return t

    for mode in ("box", "bilinear", "bicubic"):
        # float: every pixel outside the box is NaN, no output may be
        imgs = [image(float("nan"), torch.float32, c) for c in crops]
        got, _ = capi.resize_crops_pad(imgs, crops, (64, 72), mode, [1.0, 2.0, 3.0], capi.FILL_INPUT)
        assert bool(torch.isfinite(got).all()), mode
        _assert_same_bits(got, _reference(capi, imgs, crops, (64, 72), mode, False, torch.float32, fill=[1.0, 2.0, 3.0],
                                          fill_mode=capi.FILL_INPUT), f"NaN parents {mode}")
        # uint8: canary 0 and 255 outside the boxes give the same bits
        g.manual_seed(12)
        a = [image(0, torch.uint8, c) for c in crops]
        g.manual_seed(12)
        z = [image(255, torch.uint8, c) for c in crops]
        ya, _ = capi.resize_crops_pad(a, crops, (64, 72), mode, 9.0, capi.FILL_INPUT)
        yz, _ = capi.resize_crops_pad(z, crops, (64, 72), mode, 9.0, capi.FILL_INPUT)
        _assert_same_bits(ya, yz, f"uint8 canaries {mode}")
    # output through a padded, unaligned view: every cell outside it keeps its canary
    imgs = [image(float("nan"), torch.float32, c) for c in crops]
    for dt, canary in ((torch.float32, float("nan")), (torch.float16, float("nan")), (torch.uint8, 77)):
        parent = torch.full((len(crops) + 1, C + 1, 64 + 3, 72 + 9), canary, dtype=dt, device=cuda)
        out = parent[1:, 1:, 2:66, 1:73]
        scale = [1.0] * C if dt == torch.float16 else None
        for mode in (capi.FILL_INPUT, capi.FILL_OUTPUT):
            capi.resize_crops_pad(imgs, crops, (64, 72), "bicubic", 5.0, mode, out=out, scale=scale)
            _assert_same_bits(out, _reference(capi, imgs, crops, (64, 72), "bicubic", False, dt, scale, fill=[5.0] * 3,
                                              fill_mode=mode), f"padded view {dt}")
            mask = torch.ones(parent.shape, dtype=torch.bool, device=cuda)
            mask[1:, 1:, 2:66, 1:73] = False
            outside = parent[mask]
            if dt == torch.uint8:
                assert bool((outside == canary).all()), dt
            else:
                assert bool(torch.isnan(outside).all()), dt


@pytest.mark.gpu
@pytest.mark.parametrize("hwc", [True, False])
def test_crops_pad_nonfinite_placement(cuda, hwc):
    import torch
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator(device=cuda).manual_seed(13)
    img = torch.rand((200, 260, 3) if hwc else (3, 200, 260), generator=g, device=cuda) * 255
    for (y, x, c), v in (((0, 0, 0), float("nan")), ((120, 30, 1), float("inf")), ((199, 259, 2), float("-inf")),
                         ((10, 200, 1), float("nan"))):
        if hwc:
            img[y, x, c] = v
        else:
            img[c, y, x] = v
    for mode in ("box", "bilinear", "bicubic"):
        for osize in ((64, 80), (17, 23)):
            oH, oW = osize
            crops = []
            for j, (rh, rw) in enumerate(((200, 260), (70, 91), (256, 341), (30, 40))):
                for k, (ct, cl) in enumerate(((-7, -9), (rh - oH + 5, rw - oW + 6), (-oH // 2, rw - oW // 2),
                                              (rh * 50 // 200 - 3, rw * 60 // 260 - 2))):
                    crops.append((0, 0, 200, 260, rh, rw, ct, cl, (j + k) % 4))
            for fill in (0.0, float("nan")):
                got, n = capi.resize_crops_pad([img] * len(crops), crops, osize, mode, fill, capi.FILL_INPUT)
                want = _reference(capi, [img] * len(crops), crops, osize, mode, False, torch.float32, fill=[fill] * 3,
                                  fill_mode=capi.FILL_INPUT)
                assert n == 1
                assert torch.equal(torch.isnan(got), torch.isnan(want)), (mode, osize, fill)
                assert fill != 0.0 or not bool(torch.isfinite(got).all()), (mode, osize)
                fin = ~torch.isnan(want)
                _assert_same_bits(got[fin], want[fin], f"non-finite {mode} {osize} {fill}")


@pytest.mark.gpu
def test_crops_pad_launches_and_graph_capture(cuda):
    import torch
    import interpolate_antialiasing_b200 as aa
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(3)
    g = torch.Generator(device=cuda).manual_seed(3)
    # 1100 images into one padded batch: ceil(1100 / 512) = 3 launches
    imgs = [torch.randint(0, 256, (rnd.randint(20, 60), rnd.randint(20, 60), 3), generator=g, device=cuda, dtype=torch.uint8)
            for _ in range(1100)]
    torch.cuda.synchronize()
    capi.launch_count(reset=True)
    batch, place = aa.resize_pad_batch(imgs, 32, max_size=48, canvas=(48, 48), align="center", fill=114, mode="bicubic")
    assert capi.launch_count(reset=True) == 3
    assert batch.shape == (1100, 3, 48, 48) and batch.dtype == torch.float32 and batch.is_contiguous()
    crops = [(0, 0, t.shape[0], t.shape[1], h, w, -top, -left, 0) for t, (top, left, h, w) in zip(imgs, place.tolist())]
    _assert_same_bits(batch, _reference(capi, imgs, crops, (48, 48), "bicubic", False, torch.float32, fill=[114.0] * 3,
                                        fill_mode=capi.FILL_INPUT), "1100 crops")
    # float input: one launch (no drain); capture once, replay on new pixel data
    imgs = [torch.rand((rnd.randint(64, 200), rnd.randint(64, 200), 3), generator=g, device=cuda) * 255 for _ in range(512)]
    crops = []
    for im in imgs:
        H, W = im.shape[:2]
        h, w = rnd.randint(1, H), rnd.randint(1, W)
        rh, rw = rnd.randint(20, 140), rnd.randint(20, 140)
        crops.append((rnd.randint(0, H - h), rnd.randint(0, W - w), h, w, rh, rw, rnd.randint(-60, rh), rnd.randint(-60, rw),
                      rnd.randint(0, 3)))
    out = torch.empty((512, 3, 56, 56), dtype=torch.float16, device=cuda)
    kw = dict(scale=[0.5, 1, 2], bias=[0, 1, 2])
    torch.cuda.synchronize()
    capi.launch_count(reset=True)
    _, n = capi.resize_crops_pad(imgs, crops, (56, 56), "bilinear", [3, 4, 5], capi.FILL_OUTPUT, out=out, **kw)
    assert n == 1 and capi.launch_count(reset=True) == 1
    _assert_same_bits(out, _reference(capi, imgs, crops, (56, 56), "bilinear", False, torch.float16, fill=[3, 4, 5],
                                      fill_mode=capi.FILL_OUTPUT, **kw), "512 crops")
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            capi.resize_crops_pad(imgs, crops, (56, 56), "bilinear", [3, 4, 5], capi.FILL_OUTPUT, out=out, **kw)
    torch.cuda.current_stream().wait_stream(s)
    for step in range(2):
        for im in imgs:
            im.copy_(torch.rand(im.shape, generator=g, device=cuda) * 255)
        graph.replay()
        torch.cuda.synchronize()
        want, _ = capi.resize_crops_pad(imgs, crops, (56, 56), "bilinear", [3, 4, 5], capi.FILL_OUTPUT,
                                        out=torch.empty_like(out), **kw)
        _assert_same_bits(out, want, f"graph replay {step}")


@pytest.mark.gpu
def test_crops_pad_64bit_offsets(cuda):
    """One HWC uint8 image of 2.25e9 elements; the boxes start past element 2^31 and the windows overhang."""
    import torch
    from interpolate_antialiasing_b200 import capi
    H, W, C = 50000, 15000, 3
    nbytes = H * W * C
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + (4 << 30):
        pytest.skip(f"needs {nbytes / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    img = torch.empty((H, W, C), dtype=torch.uint8, device=cuda)
    crops = [(48000, 14000, 1500, 1000, 300, 200, -20, 100, 3), (49900, 0, 100, 3000, 150, 400, 50, -30, 1),
             (0, 0, 300, 300, 400, 400, 300, -60, 2), (47000, 0, 3000, 15000, 200, 1000, -40, 900, 0)]
    assert crops[0][0] * W * C > 2 ** 31
    g = torch.Generator(device=cuda).manual_seed(19)
    for c in crops:
        v = img[c[0]:c[0] + c[2], c[1]:c[1] + c[3]]
        v.copy_(torch.randint(0, 256, v.shape, generator=g, device=cuda, dtype=torch.uint8))
    got, _ = capi.resize_crops_pad([img] * len(crops), crops, (150, 120), "bicubic", 50.0, capi.FILL_INPUT)
    want = _reference(capi, [img] * len(crops), crops, (150, 120), "bicubic", False, torch.float32, fill=[50.0] * 3,
                      fill_mode=capi.FILL_INPUT)
    _assert_same_bits(got, want, "64-bit offsets")
    del img
    torch.cuda.empty_cache()
