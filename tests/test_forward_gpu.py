"""K2 parity: forward through the C ABI against the oracle / golden fixtures.

Tolerances (BASELINE.json north_star): fp32 within 1e-5 relative / 1e-3 absolute on a [0,255]
scale (checked as |got-want| <= 1e-3 + 1e-5*|want|); uint8-rounded outputs within 1 LSB.
The general path (AA_FLAG_FORCE_GENERAL: H pass then V pass, no FMA) is held to BIT-EXACT."""
import numpy as np
import pytest
import torch

from oracle import aa_oracle as O

pytestmark = pytest.mark.gpu

ATOL, RTOL = 1e-3, 1e-5
MODES = ["linear", "cubic", "nearest"]
SIZES = [(320, 196), (460, 220), (120, 96), (1200, 196), (120, 1200)]  # PIL (w, h), reference test.py:15-21


def _close(got, want):
    got = got.astype(np.float64); want = want.astype(np.float64)
    err = np.abs(got - want)
    assert np.all(err <= ATOL + RTOL * np.abs(want)), f"max abs err {err.max():.3e}"
    return err.max()


def _run(capi, x, osize, mode, align, flags):
    y = capi.resize_forward(x, osize, mode, align, flags)
    torch.cuda.synchronize()
    return y


def test_small_cases_general_bit_exact(cuda, golden):
    from interpolate_antialiasing_b200 import capi
    for i in range(int(golden["n_cases"])):
        xn = golden[f"case{i}_x"]
        osize = tuple(int(v) for v in golden[f"case{i}_osize"])
        for cl in (False, True):
            x = torch.from_numpy(xn).to(cuda)
            if cl:
                x = x.contiguous(memory_format=torch.channels_last)
            for mode in MODES:
                for align in (0, 1):
                    y = _run(capi, x, osize, mode, bool(align), capi.FLAG_FORCE_GENERAL)
                    assert y.is_contiguous(memory_format=torch.channels_last if cl else torch.contiguous_format) or min(y.shape) == 1
                    assert np.array_equal(y.cpu().numpy(), golden[f"case{i}_{mode}_{align}"]), (i, cl, mode, align)


def test_small_cases_auto_within_tolerance(cuda, golden):
    from interpolate_antialiasing_b200 import capi
    for i in range(int(golden["n_cases"])):
        xn = golden[f"case{i}_x"]
        if xn.dtype != np.float32:
            continue
        osize = tuple(int(v) for v in golden[f"case{i}_osize"])
        for cl in (False, True):
            x = torch.from_numpy(xn).to(cuda)
            if cl:
                x = x.contiguous(memory_format=torch.channels_last)
            for mode in MODES:
                for align in (0, 1):
                    y = _run(capi, x, osize, mode, bool(align), capi.FLAG_AUTO)
                    _close(y.cpu().numpy(), golden[f"case{i}_{mode}_{align}"])


@pytest.mark.parametrize("flags_name", ["FLAG_FORCE_GENERAL", "FLAG_FORCE_STREAM", "FLAG_AUTO"])
def test_photo_all_sizes(cuda, photo, golden, flags_name):
    """cfg1 and the reference's 5 test sizes on its own fixture image, f32 and fused-uint8 input."""
    from interpolate_antialiasing_b200 import capi
    flags = getattr(capi, flags_name)
    xu8 = torch.from_numpy(photo.transpose(2, 0, 1)[None].copy()).to(cuda)
    xf = xu8.float()
    want_cache = {}
    for (w, h) in SIZES:
        for mode in MODES:
            want = O.forward(xf.cpu().numpy(), (h, w), mode)
            want_cache[(w, h, mode)] = want
            for x in (xf, xu8, xf.contiguous(memory_format=torch.channels_last), xu8.contiguous(memory_format=torch.channels_last)):
                try:
                    y = _run(capi, x, (h, w), mode, False, flags)
                except capi.AAError as e:
                    if flags == capi.FLAG_FORCE_STREAM and "-2" in str(e):
                        continue  # stream path legitimately ineligible (upsampling in H / alignment)
                    raise
                got = y.cpu().numpy()
                if flags == capi.FLAG_FORCE_GENERAL:
                    assert np.array_equal(got, want), (w, h, mode)
                else:
                    _close(got, want)
    # the reference's committed golden PNG: bilinear 320x196, .byte() truncation; general path is bit-exact
    y = _run(capi, xf, (196, 320), "linear", False, capi.FLAG_FORCE_GENERAL)
    assert np.array_equal(y[0].byte().permute(1, 2, 0).cpu().numpy(), golden["png_320x196"])
    # streaming path: within 1 LSB of it after the same truncation
    y = _run(capi, xf, (196, 320), "linear", False, capi.FLAG_AUTO)
    d = np.abs(y[0].byte().permute(1, 2, 0).cpu().numpy().astype(np.int32) - golden["png_320x196"].astype(np.int32))
    assert d.max() <= 1


def test_photo_vs_pil(cuda, photo):
    """Reference acceptance check test.py:360-379: bilinear MAE<1 & MaxAbsE<=1; bicubic MAE<1 & MaxAbsE<20."""
    from PIL import Image
    from interpolate_antialiasing_b200 import capi
    img = Image.fromarray(photo)
    xu8 = torch.from_numpy(photo.transpose(2, 0, 1)[None].copy()).to(cuda)
    for (w, h) in SIZES:
        for mode, resample, max_tol in (("linear", Image.BILINEAR, 1.0 + 1e-5), ("cubic", Image.BICUBIC, 20.0)):
            pil = np.asarray(img.resize((w, h), resample=resample)).transpose(2, 0, 1).astype(np.float32)
            y = _run(capi, xu8, (h, w), mode, False, capi.FLAG_AUTO)[0]
            if mode == "cubic":
                y = y.clamp(0, 255)
            y = y.byte().float().cpu().numpy()
            assert np.abs(y - pil).mean() < 1.0
            assert np.abs(y - pil).max() < max_tol


@pytest.mark.parametrize("C", [1, 3, 4])
@pytest.mark.parametrize("cl", [False, True])
def test_scale_sweep_medium(cuda, C, cl):
    """cfg5 at oracle-sized shapes: scale 0.125x..2x in both axes incl. mixed up/down, both filters."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(C * 2 + cl)
    H, W = 96, 128
    x = (torch.rand((2, C, H, W), generator=g) * 255)
    xc = x.to(cuda)
    if cl:
        xc = xc.contiguous(memory_format=torch.channels_last)
    for sh, sw in [(0.125, 0.125), (0.25, 0.5), (0.333, 0.333), (0.5, 0.25), (0.75, 0.75), (1, 1), (1.5, 1.5), (2, 2), (0.25, 2), (2, 0.25), (0.6, 1.3)]:
        osize = (max(1, round(H * sh)), max(1, round(W * sw)))
        for mode in ("linear", "cubic"):
            want = O.forward(x.numpy(), osize, mode, False)
            y = _run(capi, xc, osize, mode, False, capi.FLAG_AUTO)
            _close(y.cpu().numpy(), want)
            y = _run(capi, xc, osize, mode, False, capi.FLAG_FORCE_GENERAL)
            assert np.array_equal(y.cpu().numpy(), want), (sh, sw, mode)


def test_named_config_slices(cuda):
    """One-image slices of cfg2 (fp32 channels_last bilinear 1080x1920->224x224) and cfg3
    (uint8 channels_first bicubic 2160x3840->512x512) against the oracle."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(0)
    x = (torch.rand((2, 3, 1080, 1920), generator=g) * 255)
    want = O.forward(x.numpy(), (224, 224), "linear", False)
    y = _run(capi, x.to(cuda).contiguous(memory_format=torch.channels_last), (224, 224), "linear", False, capi.FLAG_AUTO)
    assert y.is_contiguous(memory_format=torch.channels_last)
    _close(y.cpu().numpy(), want)
    xu = torch.randint(0, 256, (1, 3, 2160, 3840), generator=g, dtype=torch.uint8)
    want = O.forward(xu.float().numpy(), (512, 512), "cubic", False)
    y = _run(capi, xu.to(cuda), (512, 512), "cubic", False, capi.FLAG_AUTO)
    e = _close(y.cpu().numpy(), want)
    # uint8-rounded (clamp + cast as the reference's caller does, test.py:71-75) within 1 LSB
    a = np.clip(y.cpu().numpy(), 0, 255).astype(np.uint8).astype(np.int32)
    b = np.clip(want, 0, 255).astype(np.uint8).astype(np.int32)
    assert np.abs(a - b).max() <= 1, e


def test_nonfinite_placement_tile_band_stream(cuda):
    """NaN/Inf pixels in every kernel regime (tile: upsampling; band: 0.75x; stream: downsampling; two launches: mixed),
    reference aa_interpolation_impl.h:73-85 (only taps j < xsize are touched, so an output is non-finite iff one of ITS
    taps is).  On EVERY path -- the fast kernels (AUTO: they check what they store and redo a region tap-exactly,
    aa_common.cuh aa_exact_region), AA_FLAG_STRICT_NONFINITE and AA_FLAG_FORCE_GENERAL -- the set of non-finite outputs
    equals the oracle's exactly; the finite ones are within tolerance on the fast path and bit-identical on the other two."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(17)
    for (H, W), osize, mode in [((40, 60), (80, 120), "cubic"), ((64, 96), (48, 72), "cubic"), ((64, 96), (48, 72), "linear"),
                                ((120, 160), (30, 40), "linear"), ((120, 160), (24, 50), "cubic"), ((50, 70), (50, 70), "linear"),
                                ((96, 64), (40, 150), "cubic"), ((64, 96), (100, 30), "linear"), ((300, 420), (37, 53), "cubic"),
                                ((24, 160), (72, 80), "cubic"), ((48, 200), (120, 60), "cubic")]:  # the last two: two launches
        x = torch.rand((2, 3, H, W), generator=g) * 255
        for (n, c, y, xx), val in [((0, 0, 5, 7), float("nan")), ((0, 2, H - 1, W - 1), float("inf")), ((1, 1, H // 2, W // 3), float("-inf")),
                                   ((1, 0, 0, 0), float("nan"))]:
            x[n, c, y, xx] = val
        for cl in (False, True):
            xc = x.to(cuda).contiguous(memory_format=torch.channels_last) if cl else x.to(cuda)
            want = O.forward(x.numpy(), osize, mode, False)
            wbad = ~np.isfinite(want)
            assert wbad.any() and not wbad.all()
            for flags in (capi.FLAG_STRICT_NONFINITE, capi.FLAG_FORCE_GENERAL):
                y = _run(capi, xc, osize, mode, False, flags).cpu().numpy()
                assert np.array_equal(~np.isfinite(y), wbad), (H, W, osize, mode, cl, flags)
                assert np.array_equal(y[~wbad], want[~wbad])
            for flags in (capi.FLAG_AUTO, capi.FLAG_FORCE_STREAM):
                if flags == capi.FLAG_FORCE_STREAM and osize[0] > H:
                    continue  # the streaming kernel does not upsample in H
                y = _run(capi, xc, osize, mode, False, flags).cpu().numpy()
                assert np.array_equal(~np.isfinite(y), wbad), (H, W, osize, mode, cl, flags)
                _close(y[~wbad], want[~wbad])
            # AA_FLAG_ASSUME_FINITE (no drain launch): nothing is lost, and what spreads stays within K-1 taps per axis
            y = _run(capi, xc, osize, mode, False, capi.FLAG_ASSUME_FINITE).cpu().numpy()
            ybad = ~np.isfinite(y)
            assert not np.any(wbad & ~ybad), "a non-finite output was lost"
            _close(y[~wbad & ~ybad], want[~wbad & ~ybad])
            Kh = int(np.ceil((capi.interp_size(H, osize[0], mode) - 1) * max(1.0, osize[0] / H))) + 1
            Kw = int(np.ceil((capi.interp_size(W, osize[1], mode) - 1) * max(1.0, osize[1] / W))) + 1
            for (n, c, oy, ox) in np.argwhere(ybad & ~wbad):
                assert wbad[n, c, max(0, oy - Kh):oy + Kh + 1, max(0, ox - Kw):ox + Kw + 1].any(), (H, W, osize, mode, cl, (n, c, oy, ox))
            # the adjoint kernels (backward): grad_in is non-finite iff a grad_out element whose window holds it is
            gy = torch.rand((2, 3) + tuple(osize), generator=g)
            gy[0, 1, osize[0] // 2, osize[1] // 2] = float("nan")
            gy[1, 2, 0, osize[1] - 1] = float("inf")
            gyc = gy.to(cuda).contiguous(memory_format=torch.channels_last) if cl else gy.to(cuda)
            gwant = O.backward_adjoint(gy.numpy(), (2, 3, H, W), mode, False)
            gbad = ~np.isfinite(gwant)
            gx = capi.resize_backward(gyc, (2, 3, H, W), mode, False).cpu().numpy()
            assert np.array_equal(~np.isfinite(gx), gbad), (H, W, osize, mode, cl, "backward")
            assert np.allclose(gx[~gbad], gwant[~gbad], rtol=1e-5, atol=4e-6)


def test_cfg3_eight_images_all_paths(cuda):
    """cfg3 at full per-image size on 8 images (24 planes): the tensor-core path (AUTO for uint8), the FP32-pipe streaming
    kernel and the bit-exact general path against the oracle, plane by plane (a work split that mixed planes up would
    show here, a single image would not)."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(3)
    xu = torch.randint(0, 256, (8, 3, 2160, 3840), generator=g, dtype=torch.uint8)
    xc = xu.to(cuda)
    ya = _run(capi, xc, (512, 512), "cubic", False, capi.FLAG_AUTO)
    ys = _run(capi, xc, (512, 512), "cubic", False, capi.FLAG_FORCE_STREAM)
    yg = _run(capi, xc, (512, 512), "cubic", False, capi.FLAG_FORCE_GENERAL)
    capi.check_device(0)
    for n in range(8):
        want = O.forward(xu[n:n + 1].float().numpy(), (512, 512), "cubic", False)
        _close(ya[n:n + 1].cpu().numpy(), want)
        _close(ys[n:n + 1].cpu().numpy(), want)
        assert np.array_equal(yg[n:n + 1].cpu().numpy(), want), n


def test_full_size_properties(cuda):
    """Size-independent properties at BASELINE sizes (a 16-image slab of cfg2; cfg3 full per-image size):
    constants are preserved (weights sum to 1), the op is linear, batch elements are independent,
    and channels_first / channels_last agree."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator(device="cuda").manual_seed(1)
    N = 16
    x = (torch.rand((N, 3, 1080, 1920), generator=g, device=cuda) * 255).contiguous(memory_format=torch.channels_last)
    y = _run(capi, x, (224, 224), "linear", False, capi.FLAG_AUTO)
    ones = torch.full_like(x, 37.0)
    yo = _run(capi, ones, (224, 224), "linear", False, capi.FLAG_AUTO)
    assert (yo - 37.0).abs().max().item() < 1e-3
    y2 = _run(capi, x * 0.5 + ones, (224, 224), "linear", False, capi.FLAG_AUTO)
    assert (y2 - (0.5 * y + yo)).abs().max().item() < 1e-3
    y3 = _run(capi, x[5:6], (224, 224), "linear", False, capi.FLAG_AUTO)
    assert torch.equal(y3, y[5:6])
    ycf = _run(capi, x.contiguous(), (224, 224), "linear", False, capi.FLAG_AUTO)
    assert (ycf - y).abs().max().item() < 1e-3
    # one image against the oracle
    _close(y[3:4].cpu().numpy(), O.forward(x[3:4].cpu().numpy(), (224, 224), "linear", False))


def test_edge_cases(cuda):
    from interpolate_antialiasing_b200 import capi
    # empty batch is allowed (aa_interpolation_impl.h:747-750)
    x = torch.empty((0, 3, 8, 8), device=cuda)
    y = capi.resize_forward(x, (4, 4), "linear")
    assert y.shape == (0, 3, 4, 4)
    # 1x1 in / 1x1 out / identity
    g = torch.Generator().manual_seed(4)
    for shp, osz in [((1, 2, 1, 1), (4, 5)), ((1, 3, 30, 50), (1, 1)), ((2, 2, 9, 9), (9, 9)), ((1, 1, 1, 37), (1, 5)), ((1, 1, 37, 1), (5, 1))]:
        x = torch.rand(shp, generator=g) * 255
        for mode in MODES:
            want = O.forward(x.numpy(), osz, mode, False)
            y = _run(capi, x.to(cuda), osz, mode, False, capi.FLAG_AUTO)
            _close(y.cpu().numpy(), want)
    # batch slice (stride_n != c*h*w) is read in place
    xb = (torch.rand((6, 3, 40, 48), generator=g) * 255).to(cuda)
    y = _run(capi, xb[1:5:2], (10, 12), "linear", False, capi.FLAG_AUTO)
    _close(y.cpu().numpy(), O.forward(xb[1:5:2].cpu().numpy(), (10, 12), "linear", False))
    # bad arguments surface as errors, not crashes
    with pytest.raises(capi.AAError):
        capi.resize_forward(torch.rand((1, 3, 8, 8), device=cuda), (4, 4), 7)
    with pytest.raises(capi.AAError):  # non-NCHW/NHWC strides
        capi.resize_forward(torch.rand((1, 3, 8, 16), device=cuda)[:, :, :, ::2], (4, 4), "linear")


def _guarded(shape, dtype, device, channels_last, fill, pad=4096, crop=None):
    """A tensor of `shape` carved out of a larger buffer filled with `fill` (the canary).  crop=(r0, c0, dh, dw): the
    tensor is the view [:, :, r0:r0+H, c0:c0+W] of a parent [N, C, H+dh, W+dw] (padded rows, a base pointer c0 elements
    past a row start, a batch stride larger than one image), the parent itself inside the guarded buffer."""
    N, C, H, W = shape
    r0, c0, dh, dw = crop or (0, 0, 0, 0)
    Hp, Wp = H + dh, W + dw
    n = N * C * Hp * Wp
    buf = torch.full((n + 2 * pad,), fill, dtype=dtype, device=device)
    core = buf[pad:pad + n]
    t = core.view(N, Hp, Wp, C).permute(0, 3, 1, 2) if channels_last else core.view(N, C, Hp, Wp)
    return buf, t[:, :, r0:r0 + H, c0:c0 + W]


def _untouched_outside(buf, view, fill):
    """Every element of `buf` outside `view` still holds `fill`."""
    b = buf.clone()
    b.as_strided(view.shape, view.stride(), view.storage_offset() - buf.storage_offset()).fill_(fill)
    return bool((b == fill).all())


# Input views of the canary test: dense, then crops whose base pointer is 1, 2, 4 and 16 elements past a row start
# (4/8/16-byte aligned fp32 rows: the streaming kernel's 1-, 2- and 4-wide vectors, TMA with padded rows; for uint8 the
# 16-byte aligned crop is the only one the tensor-core kernel takes).  Parent widths are multiples of 16 elements.
def _in_views(W):
    return [None] + [(3, c0, 5, (-W) % 16 + 32) for c0 in (1, 2, 4, 16)]


@pytest.mark.parametrize("flags_name", ["FLAG_AUTO", "FLAG_FORCE_STREAM", "FLAG_FORCE_GENERAL", "TMA"])
def test_no_out_of_bounds_access(cuda, flags_name):
    """Out-of-bounds traffic is caught with canaries: NaN margins around
    a float input poison the output if any kernel reads outside the tensor (even with a zero weight), and the output's
    margins must stay untouched.  A fast float kernel that stores a NaN/Inf gets the region recomputed tap-exactly by
    the drain kernel behind it (aa_redo.cu), which would repair exactly such a stray read; so every float case also runs
    with FLAG_ASSUME_FINITE (no drain): that output must be finite and match the oracle, and the default output must be
    bit-identical to it (finite data stores nothing non-finite, so the drain of a clean kernel has nothing to do).
    uint8 inputs run with canary 0 and canary 255: identical outputs mean no outside byte was read with any non-zero
    weight.  Inputs are dense tensors and cropped views of a larger image; outputs are written through `out=` into a
    dense tensor or into a view with padded rows and an unaligned base pointer."""
    from interpolate_antialiasing_b200 import capi
    flags = (capi.FLAG_FORCE_STREAM | capi.FLAG_STREAM_TMA) if flags_name == "TMA" else getattr(capi, flags_name)
    g = torch.Generator().manual_seed(5)
    cases = [((2, 3, 64, 96), (16, 24)), ((1, 4, 96, 128), (31, 45)), ((2, 1, 57, 64), (19, 20)), ((1, 3, 40, 48), (80, 96)),
             ((1, 3, 33, 64), (33, 64)), ((1, 2, 120, 36), (30, 72)), ((3, 3, 128, 128), (32, 32)),
             ((2, 3, 96, 128), (72, 96)),     # 0.75x: band kernel
             ((2, 1, 64, 64), (128, 112)),    # upsampling: tile kernel
             ((2, 3, 24, 160), (72, 80))]     # up in H, down in W: two launches
    ran = 0
    for shape, osize in cases:
        oshape = (shape[0], shape[1]) + osize
        for mode in ("linear", "cubic"):
            for dt in (torch.float32, torch.uint8):
                src = (torch.rand(shape, generator=g) * 255).to(dt)
                want = O.forward(src.float().numpy(), osize, mode, False)
                for cl in (False, True):
                    for crop in _in_views(shape[3]):
                        ocrop = None if crop is None else (1, 1, 2, 32 - osize[1] % 16)  # base pointer 1 pixel past a row start
                        runs = [(flags, float("nan")), (flags | capi.FLAG_ASSUME_FINITE, float("nan"))] if dt == torch.float32 else \
                               [(f, c) for f in ([flags, capi.FLAG_VMMA] if flags == capi.FLAG_AUTO else [flags]) for c in (0, 255)]
                        outs = {}
                        for fl, canary in runs:
                            _, x = _guarded(shape, dt, cuda, cl, canary, crop=crop)
                            x.copy_(src)
                            ob, out = _guarded(oshape, torch.float32, cuda, cl, -12345.0, crop=ocrop)
                            try:
                                capi.resize_forward(x, osize, mode, False, fl, out=out)
                            except capi.AAError as e:
                                if "-2" in str(e) and fl != capi.FLAG_AUTO:
                                    continue
                                raise
                            torch.cuda.synchronize()
                            assert _untouched_outside(ob, out, -12345.0), (shape, osize, cl, mode, dt, crop, fl, "wrote outside the output")
                            outs[(fl, str(canary))] = out.clone()
                        key = (shape, osize, cl, mode, dt, crop)
                        if dt == torch.float32:
                            if not outs:
                                continue
                            y = outs[(flags | capi.FLAG_ASSUME_FINITE, "nan")]
                            assert torch.isfinite(y).all(), key + ("read outside the input",)
                            _close(y.cpu().numpy(), want)
                            assert torch.equal(outs[(flags, "nan")], y), key + ("the drain repaired the output",)
                            ran += 1
                        else:
                            for fl in {f for f, _ in outs}:
                                assert torch.equal(outs[(fl, "0")], outs[(fl, "255")]), key + (fl, "read outside the input")
                                _close(outs[(fl, "0")].cpu().numpy(), want)
                                ran += 1
    assert ran > 0


def test_cuda_graph_capture_and_replay(cuda):
    """The C ABI is asynchronous and allocation-free once the table cache is warm (aa_warm_tables), so a
    forward + backward pair can be captured in a CUDA graph and replayed (SURVEY 7.3.7: cfg1/cfg4 are
    launch-latency-scale)."""
    import ctypes
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(8)
    x = (torch.rand((1, 3, 438, 906), generator=g) * 255).to(cuda)
    go = torch.rand((1, 3, 196, 320), generator=g).to(cuda)
    out = torch.empty((1, 3, 196, 320), device=cuda)
    gin = torch.empty_like(x)
    L = capi.lib()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        capi.check(L.aa_warm_tables(438, 906, 196, 320, capi.TRIANGLE, 0, capi.F32, 0, ctypes.c_void_p(s.cuda_stream)))
        capi.resize_forward(x, (196, 320), "linear", out=out)      # warm-up outside capture
    s.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        capi.resize_forward(x, (196, 320), "linear", out=out)
        dg, di = capi.desc(go), capi.desc(gin)
        capi.check(L.aa_resize_backward(ctypes.byref(dg), ctypes.byref(di), capi.TRIANGLE, 0, 0,
                                        ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
    out.zero_(); gin.zero_()
    x.mul_(0.5)                      # replay must see the new contents of the same buffers
    graph.replay()
    torch.cuda.synchronize()
    _close(out.cpu().numpy(), O.forward(x.cpu().numpy(), (196, 320), "linear", False))
    np.testing.assert_allclose(gin.cpu().numpy(), O.backward_adjoint(go.cpu().numpy(), x.shape, "linear", False), rtol=1e-5, atol=4e-6)


def test_fused_uint8_output(cuda, photo):
    """SURVEY 8(f) row 2: clamp + round + uint8 store fused into the kernels (all three forward kernels)."""
    from PIL import Image
    from interpolate_antialiasing_b200 import capi
    from test_epilogue_gpu import assert_rounded, fast_eps, got64, ref_forward
    img = Image.fromarray(photo)
    xu8 = torch.from_numpy(photo.transpose(2, 0, 1)[None].copy()).to(cuda)
    xs = {False: xu8, True: xu8.contiguous(memory_format=torch.channels_last)}
    for (w, h) in SIZES:
        for mode, resample, max_tol in (("linear", Image.BILINEAR, 1.0), ("cubic", Image.BICUBIC, 20.0)):
            pil = np.asarray(img.resize((w, h), resample=resample)).transpose(2, 0, 1).astype(np.int32)
            want_f = np.clip(O.forward(xu8.float().cpu().numpy(), (h, w), mode, False)[0], 0, 255)
            ref = ref_forward(xu8.cpu().numpy(), (h, w), mode)  # float64 sums: the rounding-window reference
            for cl in (False, True):
                for flags in (capi.FLAG_AUTO, capi.FLAG_FORCE_GENERAL):
                    # truncation = the reference caller's clamp + .byte() (test.py:71-75)
                    y = capi.resize_forward(xs[cl], (h, w), mode, False, flags, out_u8=True)
                    assert y.dtype == torch.uint8
                    assert_rounded(got64(y), ref, fast_eps(ref, ref), "u8", (w, h, mode, cl, flags))
                    if flags == capi.FLAG_FORCE_GENERAL:  # bit-exact float path -> identical bytes
                        assert np.array_equal(y[0].cpu().numpy(), want_f.astype(np.uint8))
                    # round to nearest = PIL's convention: closer to PIL than truncation
                    yr = capi.resize_forward(xs[cl], (h, w), mode, False, flags | capi.FLAG_ROUND_NEAREST, out_u8=True)
                    assert_rounded(got64(yr), ref, fast_eps(ref, ref), "u8r", (w, h, mode, cl, flags, "round"))
                    e = np.abs(yr[0].cpu().numpy().astype(np.int32) - pil)
                    assert e.max() <= max_tol and e.mean() < (0.25 if mode == "linear" else 0.6), (w, h, mode, e.max(), e.mean())
    # float32 input -> uint8 output through the torch extension
    import interpolate_antialiasing_b200 as aa
    y = aa.resize_to_uint8(xu8.float(), (196, 320), "bilinear", False, round_nearest=False)
    ref = ref_forward(xu8.cpu().numpy(), (196, 320), "linear")
    assert_rounded(got64(y), ref, fast_eps(ref, ref), "u8", "resize_to_uint8 fp32 input")


def test_extreme_shapes(cuda):
    """Very large scale factors in both directions, degenerate axes, odd widths that defeat every vector
    width, and windows longer than one strip: every case must land on SOME kernel and match the oracle."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(11)
    cases = [
        ((1, 1, 2048, 2048), (4, 4)),        # K = 1025 taps: a single window is wider than a strip
        ((1, 3, 1000, 37), (3, 50)),         # huge down in H, up in W
        ((1, 2, 8, 8), (128, 200)),          # 16x / 25x upsampling
        ((2, 3, 33, 907), (9, 111)),         # odd width: scalar loads
        ((1, 4, 300, 5), (7, 5)),            # identity in W, down in H
        ((1, 3, 5, 4097), (5, 13)),          # identity in H, 315x down in W
        ((1, 1, 1, 4096), (1, 64)), ((1, 1, 4096, 1), (64, 1)),
        ((1, 5, 64, 64), (17, 23)),          # C = 5 channels_last (odd interleave)
    ]
    for shape, osize in cases:
        for mode in ("linear", "cubic", "nearest"):
            x = torch.rand(shape, generator=g) * 255
            want = O.forward(x.numpy(), osize, mode, False)
            for cl in (False, True):
                for dt in (torch.float32, torch.uint8):
                    xs = x.to(dt)
                    wantd = want if dt == torch.float32 else O.forward(xs.float().numpy(), osize, mode, False)
                    xc = xs.to(cuda)
                    if cl:
                        xc = xc.contiguous(memory_format=torch.channels_last)
                    y = _run(capi, xc, osize, mode, False, capi.FLAG_AUTO)
                    _close(y.cpu().numpy(), wantd)


def test_band_walk_regime(cuda):
    """Scales 0.62x..1x with few taps (the band-walking kernel of aa_band.cu): tall images so one CTA walks
    several chunks and a band is cut into several segments, widths that defeat the 16-byte copies, output
    heights that are not a multiple of the chunk, uint8 input, both layouts, a view into a larger batch."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(23)
    cases = [
        ((1, 3, 400, 300), (300, 225)),      # 0.75x, W*C % 4 == 0 channels_first
        ((1, 3, 397, 301), (300, 226)),      # odd sizes: 4-byte copies
        ((2, 1, 333, 520), (333, 520)),      # identity (1 tap)
        ((1, 4, 512, 256), (330, 200)),      # 0.645x / 0.78x
        ((3, 2, 130, 1100), (100, 1000)),    # several column bands
        ((1, 3, 1000, 64), (777, 64)),       # many chunks per band, identity in W
    ]
    for shape, osize in cases:
        for mode in ("linear", "cubic"):
            x = torch.rand(shape, generator=g) * 255
            for dt in (torch.float32, torch.uint8):
                xs = x.to(dt)
                want = O.forward(xs.float().numpy(), osize, mode, False)
                for cl in (False, True):
                    xc = xs.to(cuda)
                    if cl:
                        xc = xc.contiguous(memory_format=torch.channels_last)
                    y = _run(capi, xc, osize, mode, False, capi.FLAG_AUTO)
                    _close(y.cpu().numpy(), want)
    # a batch slice of a larger tensor and the fused uint8 store
    big = (torch.rand((4, 3, 240, 320), generator=g) * 255).to(cuda)
    xs = big[1:3]
    want = O.forward(xs.cpu().numpy(), (180, 240), "linear", False)
    _close(_run(capi, xs, (180, 240), "linear", False, capi.FLAG_AUTO).cpu().numpy(), want)
    y8 = capi.resize_forward(xs, (180, 240), "linear", False, capi.FLAG_AUTO, out_u8=True)
    assert np.abs(y8.cpu().numpy().astype(np.int32) - np.clip(want, 0, 255).astype(np.uint8).astype(np.int32)).max() <= 1


def test_random_fuzz_all_paths(cuda):
    """20 s of scripts/fuzz_parity.py: random shapes / scales / layouts / dtypes through every forward path
    (general path bit-exact, fast paths within tolerance) and the backward, against the oracle."""
    import subprocess, sys, os
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    r = subprocess.run([sys.executable, os.path.join(root, "scripts", "fuzz_parity.py"), "20", "7"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout[-3000:] + r.stderr[-2000:]
    assert "0 failures" in r.stdout


def test_decode_adjacent_epilogue(cuda, photo):
    """SURVEY 8(f) row 4: HWC uint8 -> AA resize -> (x/255 - mean)/std -> CHW fp16/bf16/fp32 in one kernel
    (aa_resize_forward_ex: normalisation, half output and planar stores fused) on the reference photo, held to the
    rounding rule of tests/test_epilogue_gpu.py.  Its 906*3-byte rows are not 4-byte aligned, so the downsampling cases
    run on the general kernel; test_epilogue_gpu.py covers the other kernels."""
    import interpolate_antialiasing_b200 as aa
    from interpolate_antialiasing_b200 import capi
    from test_epilogue_gpu import affine_ref, assert_rounded, fast_eps, got64, ref_forward
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    scale, bias = [1 / (255 * s) for s in std], [-m / s for m, s in zip(mean, std)]   # what decode_resize_normalize passes
    hwc = torch.from_numpy(np.stack([photo, photo[::-1].copy()])).to(cuda)        # [2, 438, 906, 3] uint8
    xd = hwc.permute(0, 3, 1, 2).double().cpu().numpy()
    for osize, mode in (((224, 224), "bilinear"), ((196, 320), "bicubic"), ((600, 1200), "bilinear"), ((438, 906), "bicubic")):
        base = ref_forward(xd, osize, {"bilinear": "linear", "bicubic": "cubic"}[mode])
        want = affine_ref(base, scale, bias)
        eps = fast_eps(base, want, scale)
        for dt, kind in ((torch.float32, "f32"), (torch.float16, "f16"), (torch.bfloat16, "bf16")):
            y = aa.decode_resize_normalize(hwc, osize, mean, std, mode, dt)
            assert y.shape == (2, 3) + osize and y.dtype == dt and y.is_contiguous()
            assert_rounded(got64(y), want, eps, kind, (osize, mode, kind))
        # the same epilogue through the general (bit-exact accumulate) path
        out = torch.empty((2, 3) + osize, dtype=torch.float32, device=cuda)
        capi.resize_forward_ex(hwc.permute(0, 3, 1, 2), osize, mode, out, scale, bias, flags=capi.FLAG_FORCE_GENERAL)
        torch.cuda.synchronize()
        assert_rounded(got64(out), want, eps, "f32", (osize, mode, "general"))
    # planar output without normalisation, uint8 -> uint8 CHW
    out = torch.empty((2, 3, 196, 320), dtype=torch.uint8, device=cuda)
    capi.resize_forward_ex(hwc.permute(0, 3, 1, 2), (196, 320), "linear", out)
    base = ref_forward(xd, (196, 320), "linear")
    assert_rounded(got64(out), base, fast_eps(base, base), "u8", "planar uint8")
