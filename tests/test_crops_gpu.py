"""Batched resized crops (aa_resize_crops / aa.resized_crops): per-image boxes and horizontal flips resized into one batch.

Every crop must be bit-identical to aa_resize_forward_ex on its view with FLAG_FORCE_GENERAL (plus torch.flip where the crop
is flipped): the crops kernel computes its tables in-kernel with the K1 arithmetic and sums in the general kernel's order.
Argument errors come back as status codes without a device (the non-GPU tests at the top)."""
import ctypes
import random

import pytest

from crops_common import BIAS, BOXES, FILL_NAN, OUTS, SCALE, _assert_same_bits, _images, _reference, _view


# ---------------------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------------------
def _call(capi, images, crops, count, dtype, channels, channels_last, out, filt=1, align=0, flags=0, epi=None):
    n = ctypes.c_int32(-1)
    rc = capi.lib().aa_resize_crops(images, crops, count, dtype, channels, channels_last, ctypes.byref(out) if out is not None else None,
                                    filt, align, flags, ctypes.byref(epi) if epi is not None else None, None, ctypes.byref(n))
    return rc, capi.lib().aa_last_error().decode(), n.value


def _host_args(capi, boxes, img_hw=(300, 400), C=3, oHW=(32, 48), dtype=None, out_dtype=None, cl=1):
    """Descriptors for `boxes` on fake device pointers: enough for every check that runs before the device is touched."""
    dtype = capi.U8 if dtype is None else dtype
    out_dtype = capi.F32 if out_dtype is None else out_dtype
    n = len(boxes)
    H, W = img_hw
    imgs = (capi.ImageDesc * max(n, 1))()
    crops = (capi.Crop * max(n, 1))()
    for i, b in enumerate(boxes):
        imgs[i] = capi.ImageDesc(0x10000, H, W, W * C if cl else W, 1 if cl else H * W)
        crops[i] = capi.Crop(*b[:4], b[4] if len(b) > 4 else 0)
    oH, oW = oHW
    out = capi.TensorDesc(0x20000 if n else None, out_dtype, 0, n, C, oH, oW, C * oH * oW, oH * oW, oW, 1)
    return imgs, crops, out


def test_crops_refusals_without_device():
    from interpolate_antialiasing_b200 import capi
    ok = [(0, 0, 300, 400), (10, 20, 100, 100, 1)]
    bad_boxes = [(-1, 0, 10, 10), (0, -1, 10, 10), (0, 0, 0, 10), (0, 0, 10, 0), (291, 0, 10, 10), (0, 391, 10, 10),
                 (0, 0, 301, 10), (0, 0, 10, 401)]
    for b in bad_boxes:
        imgs, crops, out = _host_args(capi, ok + [b])
        rc, msg, n = _call(capi, imgs, crops, 3, capi.U8, 3, 1, out)
        assert rc == -1 and "crop 2" in msg and n == 0, (b, rc, msg)
    imgs, crops, out = _host_args(capi, ok)
    # out not [count, channels, oH, oW]
    for n_, c_ in ((3, 3), (2, 4)):
        o = capi.TensorDesc(0x20000, capi.F32, 0, n_, c_, 32, 48, 3 * 32 * 48, 32 * 48, 48, 1)
        assert _call(capi, imgs, crops, 2, capi.U8, 3, 1, o)[0] == -1
    # null pointers
    assert _call(capi, None, crops, 2, capi.U8, 3, 1, out)[0] == -1
    assert _call(capi, imgs, None, 2, capi.U8, 3, 1, out)[0] == -1
    assert _call(capi, imgs, crops, 2, capi.U8, 3, 1, None)[0] == -1
    imgs0, crops0, out0 = _host_args(capi, ok)
    imgs0[1] = capi.ImageDesc(None, 300, 400, 1200, 1)
    rc, msg, _ = _call(capi, imgs0, crops0, 2, capi.U8, 3, 1, out0)
    assert rc == -1 and "crop 1" in msg
    # f64 input and the path-forcing flags: unsupported
    assert _call(capi, imgs, crops, 2, capi.F64, 3, 1, out)[0] == -2
    for f in (capi.FLAG_FORCE_STREAM, capi.FLAG_STREAM_TMA, capi.FLAG_STREAM_LDG, capi.FLAG_VMMA, capi.FLAG_FORCE_GENERAL):
        assert _call(capi, imgs, crops, 2, capi.U8, 3, 1, out, flags=f)[0] == -2, f
    # a window longer than the kernel's shared weight rows: bicubic 1920 -> 100 is a 19.2x downscale (> 16x)
    imgs, crops, out = _host_args(capi, [(0, 0, 300, 400), (0, 0, 1080, 1920)], img_hw=(1080, 1920), oHW=(224, 100))
    rc, msg, _ = _call(capi, imgs, crops, 2, capi.U8, 3, 1, out, filt=capi.CUBIC)
    assert rc == -2 and "crop 1" in msg
    # count == 0: a no-op
    imgs, crops, out = _host_args(capi, [])
    assert _call(capi, imgs, crops, 0, capi.U8, 3, 1, out)[0] == 0


def test_crops_valid_arguments_need_a_device():
    import torch
    from interpolate_antialiasing_b200 import capi
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    boxes = [(0, 0, 300, 400, 0), (10, 20, 100, 100, 1), (0, 0, 1080, 1920, 0)]
    imgs, crops, out = _host_args(capi, boxes, img_hw=(1080, 1920), oHW=(224, 224))
    for flags in (0, capi.FLAG_ASSUME_FINITE, capi.FLAG_STRICT_NONFINITE, capi.FLAG_ROUND_NEAREST):
        rc, msg, _ = _call(capi, imgs, crops, 3, capi.U8, 3, 1, out, filt=capi.CUBIC, flags=flags)
        assert rc == -3 and "CUDA error" in msg, (rc, msg)


# ---------------------------------------------------------------------------------------------------------------------
# GPU: reference = aa_resize_forward_ex on the crop's view with FLAG_FORCE_GENERAL (crops_common._reference)
# ---------------------------------------------------------------------------------------------------------------------
def _as_ex(boxes, hflip, osize):
    """aa_resize_crops crops as aa_crop_ex rows for _reference: each box resized to the output size, the window at the
    origin, the horizontal flip bit from hflip."""
    return [tuple(b) + tuple(osize) + (0, 0, int(bool(f))) for b, f in zip(boxes, hflip)]


@pytest.mark.gpu
@pytest.mark.parametrize("out_kind", list(OUTS))
@pytest.mark.parametrize("kind", ["u8_hwc", "u8_planar", "f32_planar", "f32_hwc"])
@pytest.mark.parametrize("filt,align", [("box", 0), ("box", 1), ("bilinear", 0), ("bilinear", 1), ("bicubic", 0), ("bicubic", 1)])
def test_crops_parity_matrix(cuda, filt, align, kind, out_kind):
    import torch
    from interpolate_antialiasing_b200 import capi
    dt_name, flag_name, affine = OUTS[out_kind]
    out_dtype = getattr(torch, dt_name)
    flags = getattr(capi, flag_name) if flag_name else 0
    for C in (1, 3, 4):
        imgs = _images(kind, C, cuda, seed=C)
        images = [imgs[i] for i, _ in BOXES]
        boxes = [b for _, b in BOXES]
        hflip = [i % 2 == 1 for i in range(len(boxes))]
        scale, bias = (SCALE[:C], BIAS[:C]) if affine else (None, None)
        out = torch.empty((len(boxes), C, 224, 224), dtype=out_dtype, device=cuda)
        got, launches = capi.resize_crops(images, boxes, (224, 224), filt, out=out, hflip=hflip, scale=scale, bias=bias,
                                          align_corners=bool(align), flags=flags)
        want = _reference(capi, images, _as_ex(boxes, hflip, (224, 224)), (224, 224), filt, bool(align), out_dtype, scale,
                          bias, flags)
        assert launches == 1
        _assert_same_bits(got, want, f"{kind} C={C} {filt} align={align} {out_kind}")


@pytest.mark.gpu
def test_crops_hwc_into_channels_last_output(cuda):
    import torch
    from interpolate_antialiasing_b200 import capi
    imgs = _images("u8_hwc", 3, cuda, seed=7)
    images = [imgs[i] for i, _ in BOXES]
    boxes = [b for _, b in BOXES]
    hflip = [i % 3 == 0 for i in range(len(boxes))]
    out = torch.empty((len(boxes), 3, 100, 130), device=cuda, memory_format=torch.channels_last)
    got, _ = capi.resize_crops(images, boxes, (100, 130), "bicubic", out=out, hflip=hflip)
    want = _reference(capi, images, _as_ex(boxes, hflip, (100, 130)), (100, 130), "bicubic", False, torch.float32)
    _assert_same_bits(got, want, "HWC -> channels_last")


@pytest.mark.gpu
def test_crops_more_than_one_launch(cuda):
    """1100 crops: ceil(1100 / 512) = 3 launches, every crop in its own output slot."""
    import torch
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(3)
    g = torch.Generator(device=cuda).manual_seed(3)
    pool = [torch.randint(0, 256, (rnd.randint(40, 90), rnd.randint(40, 90), 3), generator=g, device=cuda, dtype=torch.uint8)
            for _ in range(16)]
    images, boxes, hflip = [], [], []
    for i in range(1100):
        img = pool[i % len(pool)]
        H, W = img.shape[:2]
        h, w = rnd.choice((8, 24, H)), rnd.choice((8, 30, W))
        h, w = min(h, H), min(w, W)
        images.append(img)
        boxes.append((rnd.randint(0, H - h), rnd.randint(0, W - w), h, w))
        hflip.append(rnd.random() < 0.5)
    capi.launch_count(reset=True)
    got, launches = capi.resize_crops(images, boxes, (20, 28), "bilinear", hflip=hflip)
    assert launches == 3 and capi.launch_count(reset=True) == 3
    want = _reference(capi, images, _as_ex(boxes, hflip, (20, 28)), (20, 28), "bilinear", False, torch.float32)
    _assert_same_bits(got, want, "1100 crops")


@pytest.mark.gpu
@pytest.mark.parametrize("mode", ["bilinear", "bicubic"])
def test_crops_against_torchvision(cuda, mode):
    import torch
    tv = pytest.importorskip("torchvision.transforms.v2.functional")
    from torchvision.transforms import InterpolationMode
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(5)
    img = torch.rand((3, 480, 640), generator=g) * 255
    boxes = [(0, 0, 480, 640), (100, 50, 60, 70), (13, 200, 301, 411), (479, 0, 1, 640), (0, 639, 480, 1)]
    hflip = [False, True, False, True, False]
    got, _ = capi.resize_crops([img.to(cuda)] * len(boxes), boxes, (224, 200), mode, hflip=hflip)
    got = got.cpu().double()
    im = InterpolationMode.BILINEAR if mode == "bilinear" else InterpolationMode.BICUBIC
    for i, (b, f) in enumerate(zip(boxes, hflip)):
        want = tv.resized_crop(img, *b, [224, 200], interpolation=im, antialias=True)
        want = (want.flip(-1) if f else want).double()
        err = (got[i] - want).abs()
        assert bool((err <= 1e-3 + 1e-5 * want.abs()).all()), (i, float(err.max()))


@pytest.mark.gpu
@pytest.mark.parametrize("hwc", [True, False])
def test_crops_read_only_inside_the_boxes(cuda, hwc):
    import torch
    from interpolate_antialiasing_b200 import capi
    boxes = [(0, 0, 80, 90), (37, 11, 5, 140), (100, 150, 50, 50), (0, 199, 150, 1), (149, 0, 1, 200), (20, 30, 100, 120)]
    hflip = [False, True, True, False, True, False]
    C = 3
    g = torch.Generator(device=cuda).manual_seed(11)

    def image(fill, dtype, box):
        shape = (150, 200, C) if hwc else (C, 150, 200)
        t = torch.full(shape, fill, dtype=dtype, device=cuda)
        v = _view(t, hwc, box)[0]
        if dtype == torch.uint8:
            v.copy_(torch.randint(0, 256, v.shape, generator=g, device=cuda, dtype=torch.uint8))
        else:
            v.copy_(torch.rand(v.shape, generator=g, device=cuda) * 255)
        return t

    # float: every pixel outside the box is NaN, no output may be
    for mode in ("box", "bilinear", "bicubic"):
        imgs = [image(FILL_NAN, torch.float32, b) for b in boxes]
        got, _ = capi.resize_crops(imgs, boxes, (64, 72), mode, hflip=hflip)
        assert bool(torch.isfinite(got).all()), mode
        # uint8: canary 0 and 255 outside the boxes give the same bits
        g.manual_seed(12)
        a = [image(0, torch.uint8, b) for b in boxes]
        g.manual_seed(12)
        z = [image(255, torch.uint8, b) for b in boxes]
        ya, _ = capi.resize_crops(a, boxes, (64, 72), mode, hflip=hflip)
        yz, _ = capi.resize_crops(z, boxes, (64, 72), mode, hflip=hflip)
        _assert_same_bits(ya, yz, f"uint8 canaries {mode}")
    # output through a padded, unaligned view: every cell outside it keeps its fill
    imgs = [image(FILL_NAN, torch.float32, b) for b in boxes]
    for dt, fill in ((torch.float32, FILL_NAN), (torch.float16, FILL_NAN), (torch.uint8, 77)):
        parent = torch.full((len(boxes) + 1, C + 1, 64 + 3, 72 + 9), fill, dtype=dt, device=cuda)
        out = parent[1:, 1:, 2:66, 1:73]
        got, _ = capi.resize_crops(imgs, boxes, (64, 72), "bicubic", out=out, hflip=hflip,
                                   scale=[1.0] * C if dt == torch.float16 else None)
        want = _reference(capi, imgs, _as_ex(boxes, hflip, (64, 72)), (64, 72), "bicubic", False, dt,
                          [1.0] * C if dt == torch.float16 else None)
        _assert_same_bits(out, want, f"padded view {dt}")
        mask = torch.ones(parent.shape, dtype=torch.bool, device=cuda)
        mask[1:, 1:, 2:66, 1:73] = False
        outside = parent[mask]
        if dt == torch.uint8:
            assert bool((outside == fill).all()), dt
        else:
            assert bool(torch.isnan(outside).all()), dt


@pytest.mark.gpu
@pytest.mark.parametrize("hwc", [True, False])
def test_crops_nonfinite_placement(cuda, hwc):
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
    boxes = [(0, 0, 200, 260), (40, 50, 30, 30), (100, 0, 100, 100), (150, 200, 50, 60), (5, 190, 20, 20), (0, 0, 40, 40)]
    hflip = [True, False, True, False, False, True]
    for mode in ("box", "bilinear", "bicubic"):
        for osize in ((224, 224), (17, 23)):
            got, n = capi.resize_crops([img] * len(boxes), boxes, osize, mode, hflip=hflip)
            want = _reference(capi, [img] * len(boxes), _as_ex(boxes, hflip, osize), osize, mode, False, torch.float32)
            assert n == 1
            assert torch.equal(torch.isnan(got), torch.isnan(want)), (mode, osize)
            assert bool(torch.isnan(got).any() or torch.isinf(got).any()), (mode, osize)
            fin = ~torch.isnan(want)
            _assert_same_bits(got[fin], want[fin], f"non-finite {mode} {osize}")


@pytest.mark.gpu
def test_crops_one_launch_and_graph_capture(cuda):
    import torch
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(17)
    g = torch.Generator(device=cuda).manual_seed(17)
    imgs = [torch.rand((rnd.randint(64, 200), rnd.randint(64, 200), 3), generator=g, device=cuda) * 255 for _ in range(512)]
    boxes = []
    for im in imgs:
        H, W = im.shape[:2]
        h, w = rnd.randint(1, H), rnd.randint(1, W)
        boxes.append((rnd.randint(0, H - h), rnd.randint(0, W - w), h, w))
    hflip = [rnd.random() < 0.5 for _ in imgs]
    out = torch.empty((512, 3, 56, 56), dtype=torch.float16, device=cuda)
    torch.cuda.synchronize()
    capi.launch_count(reset=True)
    _, n = capi.resize_crops(imgs, boxes, (56, 56), "bilinear", out=out, hflip=hflip, scale=[0.5, 1, 2], bias=[0, 1, 2])
    assert n == 1 and capi.launch_count(reset=True) == 1  # float input: no drain launch behind it
    # capture once, replay on new pixel data
    torch.cuda.synchronize()
    graph = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        with torch.cuda.graph(graph, stream=s):
            capi.resize_crops(imgs, boxes, (56, 56), "bilinear", out=out, hflip=hflip, scale=[0.5, 1, 2], bias=[0, 1, 2])
    torch.cuda.current_stream().wait_stream(s)
    for step in range(2):
        for im in imgs:
            im.copy_(torch.rand(im.shape, generator=g, device=cuda) * 255)
        graph.replay()
        torch.cuda.synchronize()
        want, _ = capi.resize_crops(imgs, boxes, (56, 56), "bilinear", out=torch.empty_like(out), hflip=hflip,
                                    scale=[0.5, 1, 2], bias=[0, 1, 2])
        _assert_same_bits(out, want, f"graph replay {step}")


@pytest.mark.gpu
def test_crops_64bit_offsets(cuda):
    """One HWC uint8 image of 2.25e9 elements; the box starts past element 2^31."""
    import torch
    from interpolate_antialiasing_b200 import capi
    H, W, C = 50000, 15000, 3
    nbytes = H * W * C
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes + (4 << 30):
        pytest.skip(f"needs {nbytes / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")
    img = torch.empty((H, W, C), dtype=torch.uint8, device=cuda)
    boxes = [(48000, 14000, 1500, 1000), (49900, 0, 100, 3000), (0, 0, 300, 300)]
    assert boxes[0][0] * W * C > 2 ** 31
    g = torch.Generator(device=cuda).manual_seed(19)
    for b in boxes:
        v = img[b[0]:b[0] + b[2], b[1]:b[1] + b[3]]
        v.copy_(torch.randint(0, 256, v.shape, generator=g, device=cuda, dtype=torch.uint8))
    got, _ = capi.resize_crops([img] * 3, boxes, (224, 224), "bicubic", hflip=[True, False, False])
    want = _reference(capi, [img] * 3, _as_ex(boxes, [True, False, False], (224, 224)), (224, 224), "bicubic", False,
                      torch.float32)
    _assert_same_bits(got, want, "64-bit offsets")
    del img
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_resized_crops_python_api(cuda):
    import torch
    T = pytest.importorskip("torchvision.transforms")
    import interpolate_antialiasing_b200 as aa
    from interpolate_antialiasing_b200 import capi
    torch.manual_seed(23)
    rnd = random.Random(23)
    g = torch.Generator(device=cuda).manual_seed(23)
    imgs = [torch.randint(0, 256, (rnd.randint(300, 600), rnd.randint(300, 600), 3), generator=g, device=cuda, dtype=torch.uint8)
            for _ in range(24)]
    boxes = [T.RandomResizedCrop.get_params(im.permute(2, 0, 1), scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3)) for im in imgs]
    hflip = [rnd.random() < 0.5 for _ in imgs]
    mean, std = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
    y = aa.resized_crops(imgs, boxes, 224, hflip=hflip, mean=mean, std=std)
    assert y.dtype == torch.float16 and y.shape == (24, 3, 224, 224) and y.is_contiguous()
    want, n = capi.resize_crops(imgs, boxes, (224, 224), "bilinear", out=torch.empty_like(y), hflip=hflip,
                                scale=[1.0 / (255.0 * s) for s in std], bias=[-m / s for m, s in zip(mean, std)])
    assert n == 1
    _assert_same_bits(y, want, "resized_crops fp16")
    ref = _reference(capi, imgs, _as_ex(boxes, hflip, (224, 224)), (224, 224), "bilinear", False, torch.float16,
                     [1.0 / (255.0 * s) for s in std], [-m / s for m, s in zip(mean, std)])
    _assert_same_bits(y, ref, "resized_crops vs general")
    y8 = aa.resized_crops(imgs, boxes, (200, 180), mode="bicubic", hflip=hflip, out_dtype=torch.uint8)
    want8 = _reference(capi, imgs, _as_ex(boxes, hflip, (200, 180)), (200, 180), "bicubic", False, torch.uint8,
                       flags=capi.FLAG_ROUND_NEAREST)
    _assert_same_bits(y8, want8, "resized_crops uint8")
    # one 4-D tensor, contiguous and channels_last, float32 output
    x = torch.rand((4, 3, 120, 160), generator=g, device=cuda) * 255
    b4 = [(0, 0, 120, 160), (10, 20, 50, 60), (60, 100, 60, 60), (0, 159, 120, 1)]
    for xx in (x, x.contiguous(memory_format=torch.channels_last)):
        y4 = aa.resized_crops(xx, b4, (64, 64), mode="bicubic", hflip=[False, True, False, True])
        assert y4.dtype == torch.float32 and y4.is_contiguous()
        w4 = _reference(capi, list(x.unbind(0)), _as_ex(b4, [False, True, False, True], (64, 64)), (64, 64), "bicubic", False,
                        torch.float32)
        _assert_same_bits(y4, w4, "4-D input")
