"""K4 parity: the tensor-core vertical pass (tcgen05 kind::i8 + TMA, aa_vmma.cu) for uint8 inputs, through the C ABI,
against the oracle.  Tolerance as for every fast path: |got - want| <= 1e-3 + 1e-5*|want| on the 0..255 scale; the fused
uint8 output within 1 LSB.  Reference arithmetic: aa_interpolation_impl.h:60-87 (sums), :194-281 (tables)."""
import numpy as np
import pytest
import torch

from oracle import aa_oracle as O

pytestmark = pytest.mark.gpu
ATOL, RTOL = 1e-3, 1e-5


def _check(capi, x, osize, mode, align=False, flags=None):
    flags = capi.FLAG_VMMA if flags is None else flags
    y = capi.resize_forward(x, osize, mode, align, flags)
    torch.cuda.synchronize()
    capi.check_device(x.device.index)
    want = O.forward(x.float().cpu().numpy(), osize, mode, align)
    got = y.cpu().numpy().astype(np.float64)
    err = np.abs(got - want)
    assert np.all(err <= ATOL + RTOL * np.abs(want)), (tuple(x.shape), osize, mode, err.max())
    return y


@pytest.mark.parametrize("mode", ["linear", "cubic", "nearest"])
@pytest.mark.parametrize("cl", [False, True])
def test_vmma_shapes(cuda, mode, cl):
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(5)
    cases = [((2, 3, 540, 960), (128, 128)), ((1, 1, 256, 512), (64, 512)), ((1, 4, 333, 208), (56, 300)),
             ((3, 3, 200, 48), (33, 7)), ((1, 3, 1031, 400), (160, 90)), ((2, 1, 96, 4000), (31, 333))]
    for shape, osize in cases:
        x = torch.randint(0, 256, shape, dtype=torch.uint8, generator=g).to(cuda)
        if cl:
            x = x.contiguous(memory_format=torch.channels_last)
        if (shape[3] * (shape[1] if cl else 1)) % 16:
            continue  # TMA needs 16-byte row strides; AUTO falls back (covered by test_vmma_auto_fallback)
        for align in (False, True):
            _check(capi, x, osize, mode, align)


def test_vmma_large_scales_use_16_row_items(cuda):
    """Vertical scales above ~7x: a block of 32 output rows would span more than the 256 input rows one MMA tile holds,
    so the items shrink to 16 output rows (same kernel, upper two epilogue groups idle)."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(21)
    for shape, osize, mode in [((1, 3, 700, 256), (70, 50), "cubic"), ((2, 1, 1024, 1024), (128, 128), "cubic"),
                               ((1, 3, 1024, 512), (100, 77), "linear"), ((1, 4, 1200, 320), (83, 100), "nearest")]:
        x = torch.randint(0, 256, shape, dtype=torch.uint8, generator=g).to(cuda)
        _check(capi, x, osize, mode)
        _check(capi, x.contiguous(memory_format=torch.channels_last), osize, mode)
    # beyond what even 16-row items can hold: refused (AUTO falls back to the streaming kernel)
    x = torch.randint(0, 256, (1, 1, 2048, 256), dtype=torch.uint8, generator=g).to(cuda)
    with pytest.raises(capi.AAError):
        capi.resize_forward(x, (64, 64), "cubic", False, capi.FLAG_VMMA)
    _check(capi, x, (64, 64), "cubic", flags=capi.FLAG_AUTO)


def test_vmma_extreme_pixels(cuda):
    """All-255 / all-0 / checkerboard inputs: the int32 limb sums are at their largest magnitude."""
    from interpolate_antialiasing_b200 import capi
    for fill in (255, 0):
        x = torch.full((1, 3, 700, 256), fill, dtype=torch.uint8, device=cuda)
        _check(capi, x, (140, 50), "cubic")
        _check(capi, x, (100, 64), "linear")
    yy, xx = torch.meshgrid(torch.arange(700), torch.arange(256), indexing="ij")
    x = (((yy + xx) % 2) * 255).to(torch.uint8)[None, None].to(cuda)
    _check(capi, x, (140, 50), "cubic")


def test_vmma_is_auto_for_u8_downsampling_and_matches_stream(cuda):
    """AUTO routes uint8 >= 2x vertical downsampling to the tensor-core kernel; it agrees with the FP32-pipe streaming
    kernel to rounding, and both fused-uint8 outputs are within 1 LSB of the oracle after the same clamp + truncation."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(9)
    x = torch.randint(0, 256, (2, 3, 432, 768), dtype=torch.uint8, generator=g).to(cuda)
    for mode in ("linear", "cubic"):
        capi.launch_count(True)
        ya = capi.resize_forward(x, (96, 160), mode, False, capi.FLAG_AUTO)
        yv = capi.resize_forward(x, (96, 160), mode, False, capi.FLAG_VMMA)
        ys = capi.resize_forward(x, (96, 160), mode, False, capi.FLAG_FORCE_STREAM)
        torch.cuda.synchronize()
        capi.check_device(0)
        assert torch.equal(ya, yv)
        assert (ya - ys).abs().max().item() < 5e-4
        want = np.clip(O.forward(x.float().cpu().numpy(), (96, 160), mode), 0, 255).astype(np.uint8).astype(np.int32)
        yu = capi.resize_forward(x, (96, 160), mode, False, capi.FLAG_VMMA, out_u8=True)
        assert np.abs(yu.cpu().numpy().astype(np.int32) - want).max() <= 1


def test_vmma_auto_fallback(cuda):
    """Shapes the TMA path cannot take (row stride not a multiple of 16 bytes) still work through AUTO."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(10)
    x = torch.randint(0, 256, (1, 3, 300, 203), dtype=torch.uint8, generator=g).to(cuda)
    with pytest.raises(capi.AAError):
        capi.resize_forward(x, (60, 40), "cubic", False, capi.FLAG_VMMA)
    _check(capi, x, (60, 40), "cubic", flags=capi.FLAG_AUTO)


def test_vmma_batch_slices_and_planes(cuda):
    """Strided batch (a slice of a bigger tensor) and the (n, c) plane decomposition of the 4-D tensor map."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(11)
    big = torch.randint(0, 256, (6, 3, 256, 320), dtype=torch.uint8, generator=g).to(cuda)
    x = big[1:5]
    y = _check(capi, x, (50, 77), "cubic")
    y1 = _check(capi, big[2:3], (50, 77), "cubic")
    assert torch.equal(y[1:2], y1)


def test_vmma_decode_adjacent_epilogue(cuda):
    """HWC uint8 -> resize -> normalise -> CHW fp16 (aa_resize_forward_ex) on the tensor-core path."""
    from interpolate_antialiasing_b200 import capi
    from test_epilogue_gpu import affine_ref, assert_rounded, fast_eps, got64, ref_forward
    g = torch.Generator().manual_seed(12)
    x = torch.randint(0, 256, (2, 3, 480, 640), dtype=torch.uint8, generator=g).to(cuda).contiguous(memory_format=torch.channels_last)
    mean, std = [123.7, 116.3, 103.5], [58.4, 57.1, 57.4]
    scale = [1.0 / s for s in std]
    bias = [-m / s for m, s in zip(mean, std)]
    out = torch.empty((2, 3, 112, 112), dtype=torch.float16, device=cuda)
    capi.resize_forward_ex(x, (112, 112), "linear", out, scale, bias, flags=capi.FLAG_VMMA)
    torch.cuda.synchronize()
    capi.check_device(0)
    base = ref_forward(x.cpu().numpy(), (112, 112), "linear")
    want = affine_ref(base, scale, bias)
    assert_rounded(got64(out), want, fast_eps(base, want, scale), "f16", "vmma decode-adjacent fp16")
