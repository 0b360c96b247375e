"""K3 parity: gather-form adjoint through the C ABI / torch extension.
fp32 vs the adjoint oracle at north_star's tolerance carried to unit-scale gradients: 1e-5 relative + 1e-3/255 (4e-6)
absolute (grad_out is drawn on 0..1; the same bound as 1e-3 absolute on a 0..255 scale); fp64 gradcheck of the
forward/backward pair."""
import numpy as np
import pytest
import torch

from oracle import aa_oracle as O

pytestmark = pytest.mark.gpu
BWD_ATOL = 4e-6  # = 1e-3 / 255


def test_adjoint_vs_oracle(cuda):
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(2)
    shapes = [((2, 3, 37, 53), (11, 17)), ((2, 4, 16, 20), (33, 47)), ((1, 1, 40, 30), (13, 64)), ((3, 2, 9, 9), (9, 9)),
              ((1, 3, 30, 50), (1, 1)), ((1, 2, 1, 1), (4, 5)), ((2, 3, 128, 128), (32, 32))]
    for shp, osz in shapes:
        for mode in ("linear", "cubic", "nearest"):
            for align in (False, True):
                for tdt in (torch.float32, torch.float64):
                    for cl in (False, True):
                        go = torch.rand(shp[:2] + osz, generator=g, dtype=tdt)
                        want = O.backward_adjoint(go.numpy(), shp, mode, align)
                        gc = go.to(cuda)
                        if cl:
                            gc = gc.contiguous(memory_format=torch.channels_last)
                        got = capi.resize_backward(gc, shp, mode, align)
                        torch.cuda.synchronize()
                        tol = BWD_ATOL if tdt == torch.float32 else 1e-12
                        np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=tol)


def test_nonaa_backward_bit_exact_vs_reference_golden(cuda, golden):
    """The reference's exported linear_backward (non-AA) reproduced bit for bit (regression target)."""
    from interpolate_antialiasing_b200 import capi
    for i in range(int(golden["n_cases"])):
        x = golden[f"case{i}_x"]
        go = torch.from_numpy(golden[f"case{i}_gout"]).to(cuda)
        for align in (0, 1):
            got = capi.resize_backward(go, x.shape, "linear", bool(align), nonaa=True)
            torch.cuda.synchronize()
            assert np.array_equal(got.cpu().numpy(), golden[f"case{i}_linbwd_{align}"]), (i, align)


def test_gradcheck_fp64(cuda):
    """north_star: backward validated by gradcheck in fp64 (small shapes: down, up, mixed; both filters)."""
    import interpolate_antialiasing_b200 as aa
    torch.manual_seed(0)
    for shp, osz in [((1, 2, 12, 16), (5, 6)), ((1, 2, 6, 8), (12, 16)), ((2, 1, 10, 7), (4, 15))]:
        for mode in ("bilinear", "bicubic", "nearest"):
            for align in (False, True):
                x = torch.rand(shp, dtype=torch.float64, device=cuda, requires_grad=True)
                assert torch.autograd.gradcheck(lambda t: aa.aa_resize(t, osz, mode, align), (x,), eps=1e-6, atol=1e-6, rtol=1e-6,
                                                check_batched_grad=False, nondet_tol=0.0)


def test_cfg4_full_size_inner_product_and_torch(cuda):
    """cfg4: grad of bilinear AA [64,3,512,512] -> [128,128].  <A x, g> == <x, A^T g> ties the backward
    kernel to the forward kernel at full size; torch's own CUDA AA backward is a second opinion."""
    import interpolate_antialiasing_b200 as aa
    gen = torch.Generator(device="cuda").manual_seed(0)
    x = torch.rand((64, 3, 512, 512), generator=gen, device=cuda)
    go = torch.rand((64, 3, 128, 128), generator=gen, device=cuda)
    y = aa.linear_forward(x, (128, 128), False)
    gi = aa.linear_backward(go, (128, 128), x.shape, False)
    assert gi.shape == x.shape
    lhs = (y.double() * go.double()).sum().item()
    rhs = (x.double() * gi.double()).sum().item()
    assert abs(lhs - rhs) <= 1e-6 * abs(lhs)
    xt = x.clone().requires_grad_(True)
    yt = torch.nn.functional.interpolate(xt, size=(128, 128), mode="bilinear", antialias=True, align_corners=False)
    (gt,) = torch.autograd.grad(yt, xt, go)
    assert (gt - gi).abs().max().item() < 1e-5
    # one image against the adjoint oracle
    want = O.backward_adjoint(go[:1].cpu().numpy(), (1, 3, 512, 512), "linear", False)
    np.testing.assert_allclose(gi[:1].cpu().numpy(), want, rtol=1e-5, atol=1e-5)


def test_extension_matches_reference_api(cuda, golden):
    """The torch extension keeps the reference's names/positional signatures and error behaviour."""
    import interpolate_antialiasing_b200 as aa
    m = aa.load()
    for name in ("linear_forward", "cubic_forward", "nearest_forward", "linear_backward"):
        assert hasattr(m, name)
    x = torch.from_numpy(golden["case0_x"]).to(cuda)
    y = m.linear_forward(x, (11, 17), False)
    assert np.allclose(y.cpu().numpy(), golden["case0_linear_0"], rtol=1e-5, atol=1e-3)
    ycl = m.cubic_forward(x.contiguous(memory_format=torch.channels_last), (11, 17), False)
    assert ycl.is_contiguous(memory_format=torch.channels_last)
    with pytest.raises(RuntimeError):
        m.linear_forward(x[0], (11, 17), False)  # 3-D input
    with pytest.raises(RuntimeError):
        m.linear_forward(x.cpu(), (11, 17), False)  # no CPU fallback
    with pytest.raises(RuntimeError):
        m.linear_backward(y, (11, 18), list(x.shape), False)  # shape mismatch message path
    with pytest.raises(RuntimeError):
        m.linear_forward(x.half(), (11, 17), False)
    # uint8 in -> float32 out (fused cast)
    yu = m.linear_forward(x.byte(), (11, 17), False)
    assert yu.dtype == torch.float32


def test_backward_no_out_of_bounds_access(cuda):
    """NaN margins around grad_output, -12345 margins around grad_input.  The fast adjoint kernels are followed by the
    drain kernel, which would recompute a region that picked up a canary (aa_redo.cu); so each case runs with
    FLAG_ASSUME_FINITE (no drain), whose result must be finite and match the oracle, and with the default flags, whose
    result must be bit-identical to it.  The tile adjoint (backward of a downsampling) and the streaming adjoint
    (backward of an upsampling, forced) are both covered."""
    from interpolate_antialiasing_b200 import capi
    import ctypes
    g = torch.Generator().manual_seed(6)
    pad = 4096
    for shape, osize, flags in [((2, 3, 64, 96), (16, 24), capi.FLAG_AUTO), ((1, 4, 31, 45), (96, 128), capi.FLAG_AUTO),
                                ((2, 1, 57, 64), (19, 20), capi.FLAG_AUTO), ((3, 3, 128, 128), (32, 32), capi.FLAG_AUTO),
                                ((1, 3, 32, 48), (128, 192), capi.FLAG_FORCE_STREAM)]:
        for cl in (False, True):
            for mode in ("linear", "cubic"):
                gshape = (shape[0], shape[1]) + osize
                n_in = int(np.prod(gshape)); n_out = int(np.prod(shape))
                src = torch.rand(gshape, generator=g)
                res = []
                for fl in (flags | capi.FLAG_ASSUME_FINITE, flags):
                    gb = torch.full((n_in + 2 * pad,), float("nan"), device=cuda)
                    ob = torch.full((n_out + 2 * pad,), -12345.0, device=cuda)
                    if cl:
                        go = gb[pad:pad + n_in].view(gshape[0], gshape[2], gshape[3], gshape[1]).permute(0, 3, 1, 2)
                        gi = ob[pad:pad + n_out].view(shape[0], shape[2], shape[3], shape[1]).permute(0, 3, 1, 2)
                    else:
                        go = gb[pad:pad + n_in].view(gshape)
                        gi = ob[pad:pad + n_out].view(shape)
                    go.copy_(src)
                    dg, di = capi.desc(go), capi.desc(gi)
                    capi.check(capi.lib().aa_resize_backward(ctypes.byref(dg), ctypes.byref(di), capi.FILTERS[mode], 0, fl,
                                                              ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)))
                    torch.cuda.synchronize()
                    assert (ob[:pad] == -12345.0).all() and (ob[pad + n_out:] == -12345.0).all()
                    res.append(gi.clone())
                assert torch.isfinite(res[0]).all(), (shape, osize, cl, mode, "read outside grad_output")
                want = O.backward_adjoint(src.numpy(), shape, mode, False)
                np.testing.assert_allclose(res[0].cpu().numpy(), want, rtol=1e-5, atol=4e-6)
                assert torch.equal(res[1], res[0]), (shape, osize, cl, mode, "the drain repaired the result")


def test_custom_op_compile_and_autograd(cuda):
    """torch.ops.aa_b200.resize: fake kernel + autograd formula; traces under torch.compile without graph breaks."""
    import interpolate_antialiasing_b200 as aa  # noqa: F401  (registers the op)
    torch.manual_seed(0)
    x = torch.rand((2, 3, 64, 96), device=cuda, requires_grad=True)
    y = torch.ops.aa_b200.resize(x, [16, 24], "bilinear", False)
    y.square().sum().backward()
    xr = x.detach().clone().requires_grad_(True)
    yr = torch.nn.functional.interpolate(xr, size=(16, 24), mode="bilinear", antialias=True, align_corners=False)
    yr.square().sum().backward()
    assert torch.allclose(y, yr, rtol=1e-5, atol=1e-5) and torch.allclose(x.grad, xr.grad, rtol=1e-4, atol=1e-5)
    torch.library.opcheck(torch.ops.aa_b200.resize.default, (x.detach(), [16, 24], "bilinear", False),
                          test_utils=("test_schema", "test_faketensor"))

    def f(t):
        return torch.ops.aa_b200.resize(t * 2.0, [16, 24], "bicubic", False).sum()
    fc = torch.compile(f, fullgraph=True, backend="aot_eager")
    assert torch.allclose(fc(x.detach()), f(x.detach()))


def test_backward_of_upsampling_on_streaming_kernel(cuda):
    """When the forward was an upsampling, the backward is the many-taps, input-bound direction: it runs on
    the streaming kernel with the roles of the tables swapped (forced here; AUTO picks it when the tile kernel
    declines).  Also mixed directions and both layouts."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(21)
    cases = [((2, 3, 32, 48), (128, 192)), ((1, 4, 40, 64), (100, 200)), ((2, 1, 64, 64), (256, 96)),
             ((1, 3, 128, 128), (512, 512)), ((3, 3, 37, 53), (75, 211)), ((1, 3, 64, 64), (64, 64))]
    ran = 0
    for shp, osz in cases:
        for mode in ("linear", "cubic", "nearest"):
            for cl in (False, True):
                go = torch.rand(shp[:2] + osz, generator=g)
                want = O.backward_adjoint(go.numpy(), shp, mode, False)
                gc = go.to(cuda)
                if cl:
                    gc = gc.contiguous(memory_format=torch.channels_last)
                for flags in (capi.FLAG_AUTO, capi.FLAG_FORCE_STREAM):
                    try:
                        got = capi.resize_backward(gc, shp, mode, False, flags=flags)
                    except capi.AAError as e:
                        if "-2" in str(e) and flags == capi.FLAG_FORCE_STREAM:
                            continue
                        raise
                    torch.cuda.synchronize()
                    ran += flags == capi.FLAG_FORCE_STREAM
                    np.testing.assert_allclose(got.cpu().numpy(), want, rtol=1e-5, atol=4e-6)
    assert ran >= 12


def test_backward_with_uncovered_rows_and_columns(cuda):
    """align_corners with a 1-pixel output axis (scale 0: only input index 0 contributes) and the box filter leave
    grad_input rows / columns that NO grad_output element reaches: empty adjoint windows.  Their gathers must read
    initialised memory only (found by the fuzz: a zero weight times stale NaNs in shared memory).  Shared memory is
    pre-loaded with NaNs by resizing an all-NaN tensor through the same kernels right before every case, and the case
    runs once with FLAG_ASSUME_FINITE: without the drain kernel behind it, a stale NaN that was read stays visible."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(29)
    poison_f = torch.full((2, 5, 160, 64), float("nan"), device=cuda)
    poison_b = torch.full((2, 5, 40, 16), float("nan"), device=cuda)
    cases = [((2, 5, 145, 12), (145, 1)), ((2, 5, 12, 145), (1, 145)), ((1, 3, 33, 40), (1, 1)), ((1, 2, 300, 7), (5, 1)),
             ((2, 1, 64, 64), (1, 16)), ((1, 4, 9, 300), (1, 2))]
    for shp, osz in cases:
        for mode in ("linear", "cubic", "nearest"):
            for cl in (False, True):
                go = torch.rand(shp[:2] + osz, generator=g)
                want = O.backward_adjoint(go.numpy(), shp, mode, True)
                gc = go.to(cuda)
                if cl:
                    gc = gc.contiguous(memory_format=torch.channels_last)
                for flags in (capi.FLAG_ASSUME_FINITE, capi.FLAG_AUTO):
                    capi.resize_forward(poison_f, (120, 48), mode, False)          # band / tile kernels, NaN patches
                    capi.resize_backward(poison_b, (2, 5, 160, 64), mode, False)   # tile kernel (adjoint), NaN patches
                    got = capi.resize_backward(gc, shp, mode, True, flags=flags)
                    torch.cuda.synchronize()
                    a = got.cpu().numpy()
                    assert np.isfinite(a).all(), (shp, osz, mode, cl)
                    np.testing.assert_allclose(a, want, rtol=1e-5, atol=4e-6)


def test_scale_factors_and_uint8_box_through_the_binding(cuda):
    """(f3) `scale_factors` / `recompute_scale_factor` through the pybind module, the autograd wrapper and the custom op
    (reference: aa_interpolation_impl.h:735,740-742), against the oracle with the same factors; and the box filter's
    uint8 -> uint8 path (:566-570, :615-619) against the oracle's float result truncated."""
    import interpolate_antialiasing_b200 as aa
    g = torch.Generator().manual_seed(31)
    x = (torch.rand((2, 3, 57, 83), generator=g) * 255).to(cuda)
    for mode, fwd in (("linear", aa.linear_forward), ("cubic", aa.cubic_forward)):
        for sf in ((0.37, 0.37), (0.5, 0.81), (1.7, 0.4)):
            y = fwd(x, None, False, list(sf))
            osize = (int(57 * sf[0]), int(83 * sf[1]))
            assert tuple(y.shape[-2:]) == osize
            want = O.forward(x.cpu().numpy(), osize, mode, False, scale_factors=sf)
            assert np.abs(y.cpu().numpy() - want).max() <= 1e-3
            # F.interpolate-style front end: explicit factors vs recomputed ones
            y2 = aa.aa_resize(x, None, "bi" + mode, False, scale_factor=sf)
            assert torch.equal(y2, y)
            y3 = aa.aa_resize(x, None, "bi" + mode, False, scale_factor=sf, recompute_scale_factor=True)
            assert torch.equal(y3, fwd(x, osize, False))
            # backward with the same factors: adjoint of that forward
            go = torch.rand((2, 3) + osize, generator=g)
            gi = getattr(aa, mode + "_backward")(go.to(cuda), None, list(x.shape), False, list(sf))
            wantg = O.backward_adjoint(go.numpy(), x.shape, mode, False, scale_factors=sf)
            assert np.allclose(gi.cpu().numpy(), wantg, rtol=1e-5, atol=4e-6)
    # custom op + autograd with scale factors
    xr = x[:1].clone().requires_grad_(True)
    y = torch.ops.aa_b200.resize(xr, [28, 41], "bilinear", False, [0.5, 0.5])
    y.sum().backward()
    want = O.backward_adjoint(np.ones((1, 3, 28, 41), np.float32), xr.shape, "linear", False, scale_factors=(0.5, 0.5))
    assert np.allclose(xr.grad.cpu().numpy(), want, rtol=1e-5, atol=4e-6)
    with pytest.raises(RuntimeError, match="exactly one"):
        aa.linear_forward(x, (5, 5), False, [0.5, 0.5])
    # uint8 box filter keeps uint8
    xu = torch.randint(0, 256, (2, 3, 40, 64), dtype=torch.uint8, generator=g).to(cuda)
    for osize in ((10, 16), (13, 21), (80, 100)):
        for fmt in (torch.contiguous_format, torch.channels_last):
            yu = aa.nearest_forward(xu.contiguous(memory_format=fmt), osize, False)
            assert yu.dtype == torch.uint8 and yu.is_contiguous(memory_format=fmt)
            wantf = O.forward(xu.float().cpu().numpy(), osize, "nearest")
            d = np.abs(yu.cpu().numpy().astype(np.int32) - np.floor(np.clip(wantf, 0, 255)).astype(np.int32))
            assert d.max() <= 1 and (d != 0).mean() < 0.01
