"""Batched resize-then-crop (aa_resize_crops_ex; aa.resize_center_crop / five_crop / ten_crop / resized_output_size): a box
per crop resized to its own size, one (oH, oW) window of the resized image stored per crop, flipped horizontally and/or
vertically.

Every crop must be bit-identical to aa_resize_forward_ex of the box's view to the resized size with FLAG_FORCE_GENERAL,
sliced to the window and flipped with torch.flip.  The size and anchor arithmetic of the evaluation helpers must equal
torchvision's.  Argument errors, the output-size rules, the crop anchors and the descriptor layout are checked without a
device (the non-GPU tests at the top)."""
import ctypes
import random

import pytest

from crops_common import (BIAS, BOXES, FILL_NAN, OK, OUTS, SCALE, WINDOWS, _assert_same_bits, _host_args, _images, _reference,
                          _view)


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _call(capi, images, crops, count, dtype, channels, channels_last, out, filt=1, align=0, flags=0, epi=None):
    n = ctypes.c_int32(-1)
    rc = capi.lib().aa_resize_crops_ex(images, crops, count, dtype, channels, channels_last,
                                       ctypes.byref(out) if out is not None else None, filt, align, flags,
                                       ctypes.byref(epi) if epi is not None else None, None, ctypes.byref(n))
    return rc, capi.lib().aa_last_error().decode(), n.value


def test_crops_ex_refusals_without_device():
    from interpolate_antialiasing_b200 import capi
    invalid = [
        # everything aa_resize_crops refuses in a box
        (-1, 0, 10, 10, 32, 48, 0, 0, 0), (0, -1, 10, 10, 32, 48, 0, 0, 0), (0, 0, 0, 10, 32, 48, 0, 0, 0),
        (0, 0, 10, 0, 32, 48, 0, 0, 0), (291, 0, 10, 10, 32, 48, 0, 0, 0), (0, 391, 10, 10, 32, 48, 0, 0, 0),
        (0, 0, 301, 10, 32, 48, 0, 0, 0), (0, 0, 10, 401, 32, 48, 0, 0, 0),
        # an empty resized size
        (0, 0, 300, 400, 0, 48, 0, 0, 0), (0, 0, 300, 400, 32, 0, 0, 0, 0), (0, 0, 300, 400, -5, 48, 0, 0, 0),
        # a window outside the resized image (no zero padding)
        (0, 0, 300, 400, 40, 60, -1, 0, 0), (0, 0, 300, 400, 40, 60, 0, -1, 0), (0, 0, 300, 400, 40, 60, 9, 0, 0),
        (0, 0, 300, 400, 40, 60, 0, 13, 0), (0, 0, 300, 400, 31, 48, 0, 0, 0), (0, 0, 300, 400, 32, 47, 0, 0, 0),
        # flip bits other than 0 and 1
        (0, 0, 300, 400, 32, 48, 0, 0, 4), (0, 0, 300, 400, 32, 48, 0, 0, 8), (0, 0, 300, 400, 32, 48, 0, 0, -1),
    ]
    for c in invalid:
        imgs, rows, out = _host_args(capi, OK + [c])
        rc, msg, n = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out)
        assert rc == -1 and "crop 2" in msg and n == 0, (c, rc, msg, n)
    # an image with no data, and one whose rows overlap
    for bad in ((0, 300, 400, 1200, 1), (0x10000, 300, 400, 1199, 1)):
        imgs, rows, out = _host_args(capi, OK + [OK[0]])
        imgs[2] = bad
        rc, msg, n = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out)
        assert rc == -1 and "crop 2" in msg and n == 0, (bad, rc, msg)
    imgs, rows, out = _host_args(capi, OK)
    # out not [count, channels, oH, oW]; null pointers; a negative count
    for n_, c_ in ((3, 3), (2, 4)):
        o = capi.TensorDesc(0x20000, capi.F32, 0, n_, c_, 32, 48, 3 * 32 * 48, 32 * 48, 48, 1)
        assert _call(capi, imgs.ctypes.data, rows.ctypes.data, 2, capi.U8, 3, 1, o)[::2] == (-1, 0)
    assert _call(capi, None, rows.ctypes.data, 2, capi.U8, 3, 1, out)[::2] == (-1, 0)
    assert _call(capi, imgs.ctypes.data, None, 2, capi.U8, 3, 1, out)[::2] == (-1, 0)
    assert _call(capi, imgs.ctypes.data, rows.ctypes.data, 2, capi.U8, 3, 1, None)[::2] == (-1, 0)
    assert _call(capi, imgs.ctypes.data, rows.ctypes.data, -1, capi.U8, 3, 1, out)[::2] == (-1, 0)
    # f64 input and the path-forcing flags: unsupported
    assert _call(capi, imgs.ctypes.data, rows.ctypes.data, 2, capi.F64, 3, 1, out)[::2] == (-2, 0)
    for f in (capi.FLAG_FORCE_STREAM, capi.FLAG_STREAM_TMA, capi.FLAG_STREAM_LDG, capi.FLAG_VMMA, capi.FLAG_FORCE_GENERAL):
        assert _call(capi, imgs.ctypes.data, rows.ctypes.data, 2, capi.U8, 3, 1, out, flags=f)[::2] == (-2, 0), f
    unsupported = [
        # a window longer than 65 taps for box -> resized (not box -> output): bicubic 1080 -> 60 rows and 1920 -> 100
        # columns are 18x and 19.2x downscales (> 16x)
        ((0, 0, 1080, 1920, 60, 1920, 0, 0, 0), (1080, 1920), capi.CUBIC),
        ((0, 0, 1080, 1920, 224, 100, 5, 7, 1), (1080, 1920), capi.CUBIC),
        # resized sizes past 2^31 - 1
        ((0, 0, 300, 400, 1 << 31, 48, 0, 0, 0), (300, 400), capi.TRIANGLE),
        ((0, 0, 300, 400, 32, 1 << 31, 0, 0, 0), (300, 400), capi.TRIANGLE),
        # a box past 2^31 - 1 rows
        ((0, 0, 1 << 31, 400, 32, 48, 0, 0, 0), (1 << 32, 400), capi.TRIANGLE),
    ]
    for c, hw, filt in unsupported:
        imgs, rows, out = _host_args(capi, [OK[0], OK[0], c], img_hw=hw)
        rc, msg, n = _call(capi, imgs.ctypes.data, rows.ctypes.data, 3, capi.U8, 3, 1, out, filt=filt)
        assert rc == -2 and "crop 2" in msg and n == 0, (c, rc, msg)
    # count == 0: a no-op
    imgs, rows, out = _host_args(capi, [])
    assert _call(capi, imgs.ctypes.data, rows.ctypes.data, 0, capi.U8, 3, 1, out)[::2] == (0, 0)
    assert _call(capi, None, None, 0, capi.U8, 3, 1, out)[::2] == (0, 0)


def test_crops_ex_valid_arguments_need_a_device():
    import torch
    from interpolate_antialiasing_b200 import capi
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    crops = OK + [(0, 0, 1080, 1920, 256, 455, 16, 115, 2), (0, 0, 1080, 1920, 68, 120, 0, 0, 1)]  # the last: 65 taps
    imgs, rows, out = _host_args(capi, crops, img_hw=(1080, 1920))
    for flags in (0, capi.FLAG_ASSUME_FINITE, capi.FLAG_STRICT_NONFINITE, capi.FLAG_ROUND_NEAREST):
        rc, msg, _ = _call(capi, imgs.ctypes.data, rows.ctypes.data, 4, capi.U8, 3, 1, out, filt=capi.CUBIC, flags=flags)
        assert rc == -3 and "CUDA error" in msg, (rc, msg)


def test_descriptor_dtypes_match_the_structs():
    from interpolate_antialiasing_b200 import capi
    for dt, st in ((capi.crop_ex_dtype(), capi.CropEx), (capi.image_desc_dtype(), capi.ImageDesc)):
        assert dt.itemsize == ctypes.sizeof(st)
        assert list(dt.names) == [f for f, _ in st._fields_]
        for f, ct in st._fields_:
            assert dt.fields[f][1] == getattr(st, f).offset, f
            assert dt.fields[f][0].itemsize == ctypes.sizeof(ct), f
    assert ctypes.sizeof(capi.CropEx) == 72  # eight int64, an int32, padding to 8 bytes
    # the same bytes as a ctypes array built field by field
    rows = capi.crop_ex_array([(1, 2, 3, 4, 5, 6, 7, 8, 3), (-1, 1 << 40, 9, 10, 11, 12, 13, 14, 0)])
    ref = (capi.CropEx * 2)(capi.CropEx(1, 2, 3, 4, 5, 6, 7, 8, 3), capi.CropEx(-1, 1 << 40, 9, 10, 11, 12, 13, 14, 0))
    assert rows.tobytes() == bytes(ref)
    with pytest.raises(ValueError):
        capi.crop_ex_array([(0, 0, 1, 1, 1, 1, 0, 0, 1 << 32)])


H_W = [(256, 341), (341, 256), (480, 640), (640, 480), (300, 300), (224, 224), (375, 500), (1080, 1920), (33, 2000),
       (2000, 33), (257, 256)]
SIZES = [(256, None), ([256], None), (224, None), ((224, 300), None), ([300, 200], None), (256, 300), ([256], 400),
         (256, 257), (256, 256), (256, 100), ((224, 224), 300), (None, 320), (None, 1000), (None, None)]


def test_resized_output_size_against_torchvision():
    import torch
    tv = pytest.importorskip("torchvision.transforms.v2.functional")
    import interpolate_antialiasing_b200 as aa
    checked = errors = 0
    for h, w in H_W:
        x = torch.zeros((1, h, w))
        for size, max_size in SIZES:
            try:
                want = tuple(tv.resize(x, size, max_size=max_size, antialias=True).shape[-2:])
            except ValueError:
                with pytest.raises(ValueError):
                    aa.resized_output_size(h, w, size, max_size)
                errors += 1
                continue
            assert aa.resized_output_size(h, w, size, max_size) == want, (h, w, size, max_size)
            checked += 1
    assert checked >= 100 and errors >= 30, (checked, errors)


def _coordinates(H, W):
    """A 2-channel image whose values are the row and the column index."""
    import torch
    return torch.stack([torch.arange(H).view(H, 1).expand(H, W), torch.arange(W).view(1, W).expand(H, W)]).float()


def _origin_and_flip(crop):
    """(top, left, flip bits, the flip bits that are visible) of a crop of a _coordinates image, from its corner values: the
    flip of a 1-pixel-wide (-high) crop along that axis does not show."""
    t0, l0, t1, l1 = int(crop[0, 0, 0]), int(crop[1, 0, 0]), int(crop[0, -1, -1]), int(crop[1, -1, -1])
    visible = (1 if crop.shape[-1] > 1 else 0) | (2 if crop.shape[-2] > 1 else 0)
    return min(t0, t1), min(l0, l1), (1 if l1 < l0 else 0) | (2 if t1 < t0 else 0), visible


@pytest.mark.parametrize("kind", ["center", "five", "ten", "ten_vflip"])
def test_crop_anchors_against_torchvision(kind):
    tv = pytest.importorskip("torchvision.transforms.v2.functional")
    import interpolate_antialiasing_b200 as aa
    # (image h, w), Resize size, crop size: odd R - c on one axis (256x341 - 224), on both (256x256 - 223, 341x256 - 223),
    # a crop the size of the resized image, non-square crops
    cases = [((480, 640), 256, 224), ((640, 480), 256, 224), ((300, 300), 256, 223), ((500, 375), 256, [223]),
             ((256, 341), 256, (224, 200)), ((600, 400), (300, 201), (101, 200)), ((224, 224), 224, 224),
             ((1080, 1920), [256], (255, 1)), ((331, 517), 256, (1, 99))]
    hw = [c[0] for c in cases]
    for (h, w), size, crop in cases:
        rows = aa._eval_crops([(h, w)], size, crop, "ten" if kind.startswith("ten") else kind, kind == "ten_vflip")
        assert rows.shape[0] == 1
        rows = rows[0]
        R = aa.resized_output_size(h, w, size)
        img = _coordinates(*R)
        if kind == "center":
            want = [tv.center_crop(img, crop)]
        elif kind == "five":
            want = tv.five_crop(img, crop)
        else:
            want = tv.ten_crop(img, crop, vertical_flip=kind == "ten_vflip")
        assert len(rows) == len(want)
        for r, c in zip(rows, want):
            assert (int(r["top"]), int(r["left"]), int(r["height"]), int(r["width"])) == (0, 0, h, w)
            assert (int(r["resized_h"]), int(r["resized_w"])) == tuple(R)
            top, left, flip, visible = _origin_and_flip(c)
            got = (int(r["crop_top"]), int(r["crop_left"]), int(r["flip"]) & visible)
            assert got == (top, left, flip), ((h, w), size, crop, got, (top, left, flip))
    # the issue's example: on a 256x341 resized image the flipped centre covers columns 59..282, the unflipped one 58..281
    rows = aa._eval_crops([(256, 341)], 256, 224, "ten")[0]
    assert (int(rows[4]["crop_left"]), int(rows[9]["crop_left"])) == (58, 59)
    # one call for a batch gives the rows of each image
    batch = aa._eval_crops(hw[:4], 256, 200, "five")
    for i, (h, w) in enumerate(hw[:4]):
        assert batch[i].tobytes() == aa._eval_crops([(h, w)], 256, 200, "five")[0].tobytes()


def test_crop_larger_than_the_resized_image_is_refused():
    import interpolate_antialiasing_b200 as aa
    for crop in (257, (224, 342), (257, 1)):
        for kind in ("center", "five", "ten"):
            with pytest.raises(ValueError, match="zero padding"):
                aa._eval_crops([(256, 300), (480, 640)], 256, crop, kind)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: reference = aa_resize_forward_ex of the box's view to the resized size with FLAG_FORCE_GENERAL, sliced and flipped
# (crops_common._reference)
# ---------------------------------------------------------------------------------------------------------------------
def _rows(crops):
    """aa_crop_ex rows of a crop_ex_dtype array as plain tuples (for _reference)."""
    return [tuple(int(v) for v in r) for r in crops]


@pytest.mark.gpu
@pytest.mark.parametrize("out_kind", list(OUTS))
@pytest.mark.parametrize("kind", ["u8_hwc", "u8_planar", "f32_planar", "f32_hwc"])
@pytest.mark.parametrize("filt,align", [("box", 0), ("box", 1), ("bilinear", 0), ("bilinear", 1), ("bicubic", 0), ("bicubic", 1)])
def test_crops_ex_parity_matrix(cuda, filt, align, kind, out_kind):
    import torch
    from interpolate_antialiasing_b200 import capi
    dt_name, flag_name, affine = OUTS[out_kind]
    out_dtype = getattr(torch, dt_name)
    flags = getattr(capi, flag_name) if flag_name else 0
    for C in (1, 3, 4):
        imgs = _images(kind, C, cuda, seed=C)
        scale, bias = (SCALE[:C], BIAS[:C]) if affine else (None, None)
        for osize, windows in WINDOWS.items():
            images = [imgs[i] for i, _ in windows]
            crops = [c + (j % 4,) for j, (_, c) in enumerate(windows)]
            out = torch.empty((len(crops), C) + osize, dtype=out_dtype, device=cuda)
            got, launches = capi.resize_crops_ex(images, crops, osize, filt, out=out, scale=scale, bias=bias,
                                                 align_corners=bool(align), flags=flags)
            want = _reference(capi, images, crops, osize, filt, bool(align), out_dtype, scale, bias, flags)
            assert launches == 1
            _assert_same_bits(got, want, f"{kind} C={C} {filt} align={align} {out_kind} {osize}")


@pytest.mark.gpu
def test_crops_ex_hwc_into_channels_last_output(cuda):
    import torch
    from interpolate_antialiasing_b200 import capi
    imgs = _images("u8_hwc", 3, cuda, seed=7)
    windows = WINDOWS[(48, 64)]
    images = [imgs[i] for i, _ in windows]
    crops = [c + ((j + 1) % 4,) for j, (_, c) in enumerate(windows)]
    out = torch.empty((len(crops), 3, 48, 64), device=cuda, memory_format=torch.channels_last)
    got, _ = capi.resize_crops_ex(images, crops, (48, 64), "bicubic", out=out)
    want = _reference(capi, images, crops, (48, 64), "bicubic", False, torch.float32)
    _assert_same_bits(got, want, "HWC -> channels_last")


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["u8_hwc", "f32_planar"])
@pytest.mark.parametrize("filt,align", [("box", 0), ("bilinear", 1), ("bicubic", 0)])
def test_crops_and_crops_ex_agree(cuda, filt, align, kind):
    """aa_resize_crops is aa_resize_crops_ex with resized = out size, the window at the origin and flip = hflip."""
    import torch
    from interpolate_antialiasing_b200 import capi
    imgs = _images(kind, 3, cuda, seed=29)
    images = [imgs[i] for i, _ in BOXES]
    boxes = [b for _, b in BOXES]
    hflip = [i % 2 == 0 for i in range(len(boxes))]
    for osize, dt, scale in (((224, 224), torch.float16, SCALE[:3]), ((100, 130), torch.float32, None)):
        a, _ = capi.resize_crops(images, boxes, osize, filt, out=torch.empty((len(boxes), 3) + osize, dtype=dt, device=cuda),
                                 hflip=hflip, scale=scale, bias=BIAS[:3] if scale else None, align_corners=bool(align))
        crops = [b + osize + (0, 0, int(f)) for b, f in zip(boxes, hflip)]
        b, n = capi.resize_crops_ex(images, crops, osize, filt, out=torch.empty_like(a), scale=scale,
                                    bias=BIAS[:3] if scale else None, align_corners=bool(align))
        assert n == 1
        _assert_same_bits(b, a, f"crops vs crops_ex {kind} {filt} {osize}")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["bilinear", "bicubic"])
def test_eval_crops_against_torchvision(cuda, mode):
    import torch
    tv = pytest.importorskip("torchvision.transforms.v2.functional")
    from torchvision.transforms import InterpolationMode
    import interpolate_antialiasing_b200 as aa
    im = InterpolationMode.BILINEAR if mode == "bilinear" else InterpolationMode.BICUBIC
    g = torch.Generator().manual_seed(31)
    # 480x640 -> 256x341 (odd R - c across), 256x300 is not resized by torchvision (shorter side already 256),
    # 300x300 -> 256x256 with a 223 crop (odd R - c on both axes), 500x375 -> 341x256 (odd R - c down)
    for (H, W), crop in (((480, 640), 224), ((256, 300), 224), ((300, 300), 223), ((500, 375), (224, 200))):
        img = torch.rand((3, H, W), generator=g) * 255
        r = tv.resize(img, 256, interpolation=im, antialias=True)
        x = img.to(cuda)
        got = {"center": aa.resize_center_crop([x], 256, crop, mode=mode)[0],
               "five": aa.five_crop([x], 256, crop, mode=mode)[0],
               "ten": aa.ten_crop([x], 256, crop, mode=mode)[0],
               "ten_vflip": aa.ten_crop([x], 256, crop, vertical_flip=True, mode=mode)[0]}
        want = {"center": tv.center_crop(r, crop).unsqueeze(0), "five": torch.stack(tv.five_crop(r, crop)),
                "ten": torch.stack(tv.ten_crop(r, crop)), "ten_vflip": torch.stack(tv.ten_crop(r, crop, vertical_flip=True))}
        for k in got:
            a, b = got[k].cpu().double().reshape(want[k].shape), want[k].double()
            err = (a - b).abs()
            assert bool((err <= 1e-3 + 1e-5 * b.abs()).all()), ((H, W), crop, k, float(err.max()))


@pytest.mark.gpu
@pytest.mark.parametrize("hwc", [True, False])
def test_crops_ex_read_inside_boxes_store_inside_output(cuda, hwc):
    import torch
    from interpolate_antialiasing_b200 import capi
    crops = [(0, 0, 80, 90, 100, 120, 30, 40, 0), (37, 11, 5, 140, 70, 300, 0, 228, 1), (100, 150, 50, 50, 64, 72, 0, 0, 2),
             (0, 199, 150, 1, 200, 72, 136, 0, 3), (149, 0, 1, 200, 64, 90, 0, 9, 1), (20, 30, 100, 120, 90, 100, 11, 14, 2)]
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
        imgs = [image(FILL_NAN, torch.float32, c) for c in crops]
        got, _ = capi.resize_crops_ex(imgs, crops, (64, 72), mode)
        assert bool(torch.isfinite(got).all()), mode
        _assert_same_bits(got, _reference(capi, imgs, crops, (64, 72), mode, False, torch.float32), f"NaN parents {mode}")
        # uint8: canary 0 and 255 outside the boxes give the same bits
        g.manual_seed(12)
        a = [image(0, torch.uint8, c) for c in crops]
        g.manual_seed(12)
        z = [image(255, torch.uint8, c) for c in crops]
        ya, _ = capi.resize_crops_ex(a, crops, (64, 72), mode)
        yz, _ = capi.resize_crops_ex(z, crops, (64, 72), mode)
        _assert_same_bits(ya, yz, f"uint8 canaries {mode}")
    # output through a padded, unaligned view: every cell outside it keeps its fill
    imgs = [image(FILL_NAN, torch.float32, c) for c in crops]
    for dt, fill in ((torch.float32, FILL_NAN), (torch.float16, FILL_NAN), (torch.uint8, 77)):
        parent = torch.full((len(crops) + 1, C + 1, 64 + 3, 72 + 9), fill, dtype=dt, device=cuda)
        out = parent[1:, 1:, 2:66, 1:73]
        scale = [1.0] * C if dt == torch.float16 else None
        capi.resize_crops_ex(imgs, crops, (64, 72), "bicubic", out=out, scale=scale)
        _assert_same_bits(out, _reference(capi, imgs, crops, (64, 72), "bicubic", False, dt, scale), f"padded view {dt}")
        mask = torch.ones(parent.shape, dtype=torch.bool, device=cuda)
        mask[1:, 1:, 2:66, 1:73] = False
        outside = parent[mask]
        if dt == torch.uint8:
            assert bool((outside == fill).all()), dt
        else:
            assert bool(torch.isnan(outside).all()), dt


@pytest.mark.gpu
@pytest.mark.parametrize("hwc", [True, False])
def test_crops_ex_nonfinite_placement(cuda, hwc):
    import torch
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator(device=cuda).manual_seed(13)
    img = torch.rand((200, 260, 3) if hwc else (3, 200, 260), generator=g, device=cuda) * 255
    for (y, x, c), v in (((50, 60, 0), float("nan")), ((120, 30, 1), float("inf")), ((199, 259, 2), float("-inf")),
                         ((10, 200, 1), float("nan"))):
        if hwc:
            img[y, x, c] = v
        else:
            img[c, y, x] = v
    for mode in ("box", "bilinear", "bicubic"):
        for osize in ((64, 80), (17, 23)):
            oH, oW = osize
            # resized sizes from 0.35x to 2.2x; windows at the corners, the centre and next to the non-finite pixels
            crops = []
            for j, (rh, rw) in enumerate(((200, 260), (70, 91), (256, 341), (440, 572), (17 + 60, 23 + 90))):
                rh, rw = max(rh, oH), max(rw, oW)
                for k, (ct, cl) in enumerate(((0, 0), (rh - oH, rw - oW), ((rh - oH) // 2, (rw - oW) // 2),
                                              (min(rh * 50 // 200, rh - oH), min(rw * 60 // 260, rw - oW)))):
                    crops.append((0, 0, 200, 260, rh, rw, ct, cl, (j + k) % 4))
            crops.append((100, 0, 100, 100, 150, 150, 70, 3, 3))
            got, n = capi.resize_crops_ex([img] * len(crops), crops, osize, mode)
            want = _reference(capi, [img] * len(crops), crops, osize, mode, False, torch.float32)
            assert n == 1
            assert torch.equal(torch.isnan(got), torch.isnan(want)), (mode, osize)
            assert bool(torch.isnan(got).any() or torch.isinf(got).any()), (mode, osize)
            fin = ~torch.isnan(want)
            _assert_same_bits(got[fin], want[fin], f"non-finite {mode} {osize}")


@pytest.mark.gpu
def test_ten_crop_more_than_one_launch(cuda):
    """ten_crop of 110 images: 1100 crops, ceil(1100 / 512) = 3 launches, every crop in its own output slot."""
    import torch
    import interpolate_antialiasing_b200 as aa
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(3)
    g = torch.Generator(device=cuda).manual_seed(3)
    imgs = [torch.randint(0, 256, (rnd.randint(40, 90), rnd.randint(40, 90), 3), generator=g, device=cuda, dtype=torch.uint8)
            for _ in range(110)]
    torch.cuda.synchronize()
    capi.launch_count(reset=True)
    y = aa.ten_crop(imgs, 32, (24, 20), mode="bicubic")
    assert capi.launch_count(reset=True) == 3
    assert y.shape == (110, 10, 3, 24, 20) and y.dtype == torch.float32 and y.is_contiguous()
    crops = aa._eval_crops([im.shape[:2] for im in imgs], 32, (24, 20), "ten").reshape(-1)
    images = [im for im in imgs for _ in range(10)]
    out = torch.empty((1100, 3, 24, 20), device=cuda)
    _, launches = capi.resize_crops_ex(images, crops, (24, 20), "bicubic", out=out)
    assert launches == 3 and capi.launch_count(reset=True) == 3
    _assert_same_bits(out, y.view(1100, 3, 24, 20), "ten_crop vs resize_crops_ex")
    want = _reference(capi, images, _rows(crops), (24, 20), "bicubic", False, torch.float32)
    _assert_same_bits(out, want, "1100 crops")


@pytest.mark.gpu
def test_crops_ex_one_launch_and_graph_capture(cuda):
    import torch
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(17)
    g = torch.Generator(device=cuda).manual_seed(17)
    imgs = [torch.rand((rnd.randint(64, 200), rnd.randint(64, 200), 3), generator=g, device=cuda) * 255 for _ in range(512)]
    crops = []
    for im in imgs:
        H, W = im.shape[:2]
        h, w = rnd.randint(1, H), rnd.randint(1, W)
        rh, rw = rnd.randint(56, 140), rnd.randint(56, 140)
        crops.append((rnd.randint(0, H - h), rnd.randint(0, W - w), h, w, rh, rw, rnd.randint(0, rh - 56),
                      rnd.randint(0, rw - 56), rnd.randint(0, 3)))
    out = torch.empty((512, 3, 56, 56), dtype=torch.float16, device=cuda)
    kw = dict(scale=[0.5, 1, 2], bias=[0, 1, 2])
    torch.cuda.synchronize()
    capi.launch_count(reset=True)
    _, n = capi.resize_crops_ex(imgs, crops, (56, 56), "bilinear", out=out, **kw)
    assert n == 1 and capi.launch_count(reset=True) == 1  # float input: no drain launch behind it
    _assert_same_bits(out, _reference(capi, imgs, crops, (56, 56), "bilinear", False, torch.float16, **kw), "512 crops")
    # capture once, replay on new pixel data
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            capi.resize_crops_ex(imgs, crops, (56, 56), "bilinear", out=out, **kw)
    torch.cuda.current_stream().wait_stream(s)
    for step in range(2):
        for im in imgs:
            im.copy_(torch.rand(im.shape, generator=g, device=cuda) * 255)
        graph.replay()
        torch.cuda.synchronize()
        want, _ = capi.resize_crops_ex(imgs, crops, (56, 56), "bilinear", out=torch.empty_like(out), **kw)
        _assert_same_bits(out, want, f"graph replay {step}")


@pytest.mark.gpu
def test_crops_ex_64bit_offsets(cuda):
    """One HWC uint8 image of 2.25e9 elements; the boxes start past element 2^31."""
    import torch
    from interpolate_antialiasing_b200 import capi
    H, W, C = 50000, 15000, 3
    nbytes = H * W * C
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + (4 << 30):
        pytest.skip(f"needs {nbytes / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    img = torch.empty((H, W, C), dtype=torch.uint8, device=cuda)
    crops = [(48000, 14000, 1500, 1000, 300, 200, 100, 50, 3), (49900, 0, 100, 3000, 150, 400, 0, 280, 1),
             (0, 0, 300, 300, 400, 400, 250, 0, 2), (47000, 0, 3000, 15000, 200, 1000, 0, 630, 0)]
    assert crops[0][0] * W * C > 2 ** 31
    g = torch.Generator(device=cuda).manual_seed(19)
    for c in crops:
        v = img[c[0]:c[0] + c[2], c[1]:c[1] + c[3]]
        v.copy_(torch.randint(0, 256, v.shape, generator=g, device=cuda, dtype=torch.uint8))
    got, _ = capi.resize_crops_ex([img] * len(crops), crops, (150, 120), "bicubic")
    want = _reference(capi, [img] * len(crops), crops, (150, 120), "bicubic", False, torch.float32)
    _assert_same_bits(got, want, "64-bit offsets")
    del img
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_eval_crop_helpers_end_to_end(cuda):
    import torch
    import interpolate_antialiasing_b200 as aa
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(23)
    g = torch.Generator(device=cuda).manual_seed(23)
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    scale, bias = [1.0 / (255.0 * s) for s in std], [-m / s for m, s in zip(mean, std)]
    hwc_list = [torch.randint(0, 256, (rnd.randint(256, 600), rnd.randint(256, 600), 3), generator=g, device=cuda,
                              dtype=torch.uint8) for _ in range(12)]
    hwc_list.append(torch.randint(0, 256, (256, 341, 3), generator=g, device=cuda, dtype=torch.uint8))
    chw_list = [t.permute(2, 0, 1).contiguous() for t in hwc_list]
    calls = {"center": (lambda x, **k: aa.resize_center_crop(x, 256, 224, **k), 1),
             "five": (lambda x, **k: aa.five_crop(x, 256, 224, **k), 5),
             "ten": (lambda x, **k: aa.ten_crop(x, 256, 224, **k), 10),
             "ten_vflip": (lambda x, **k: aa.ten_crop(x, [256], (224, 200), vertical_flip=True, **k), 10)}
    for kind, (f, k) in calls.items():
        crop = (224, 200) if kind == "ten_vflip" else 224
        sizes = [t.shape[:2] for t in hwc_list]
        crops = aa._eval_crops(sizes, 256, crop, "ten" if kind.startswith("ten") else kind, kind == "ten_vflip")
        rows = _rows(crops.reshape(-1))
        images = [t for t in hwc_list for _ in range(k)]
        shape = (len(hwc_list), k, 3) + ((224, 200) if kind == "ten_vflip" else (224, 224))
        # HWC list, normalised fp16
        y = f(hwc_list, mean=mean, std=std)
        y = y.unsqueeze(1) if kind == "center" else y
        assert y.dtype == torch.float16 and tuple(y.shape) == shape and y.is_contiguous(), (kind, y.shape)
        want = _reference(capi, images, rows, shape[-2:], "bilinear", False, torch.float16, scale, bias)
        _assert_same_bits(y.reshape(want.shape), want, f"{kind} HWC fp16")
        # CHW list, uint8 rounded to nearest, bicubic
        y8 = f(chw_list, mode="bicubic", out_dtype=torch.uint8)
        assert y8.dtype == torch.uint8 and y8.numel() == want.numel()
        want8 = _reference(capi, [t for t in chw_list for _ in range(k)], rows, shape[-2:], "bicubic", False, torch.uint8,
                           flags=capi.FLAG_ROUND_NEAREST)
        _assert_same_bits(y8.reshape(want8.shape), want8, f"{kind} CHW uint8")
    # one 4-D tensor, contiguous and channels_last, float32 output
    x = torch.rand((4, 3, 300, 420), generator=g, device=cuda) * 255
    w = aa.ten_crop(list(x.unbind(0)), 256, 224)
    for xx in (x, x.contiguous(memory_format=torch.channels_last)):
        y = aa.ten_crop(xx, 256, 224)
        assert y.dtype == torch.float32 and y.shape == (4, 10, 3, 224, 224) and y.is_contiguous()
        _assert_same_bits(y, w, "4-D input")
    rows = _rows(aa._eval_crops([(300, 420)] * 4, 256, 224, "ten").reshape(-1))
    want = _reference(capi, [t for t in x.unbind(0) for _ in range(10)], rows, (224, 224), "bilinear", False, torch.float32)
    _assert_same_bits(w.view(40, 3, 224, 224), want, "4-D input vs general")
    with pytest.raises(ValueError, match="zero padding"):
        aa.resize_center_crop(x, 200, 224)
