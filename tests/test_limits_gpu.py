"""Past the launch and 32-bit limits: more than 65535 planes (the tile and band kernels launch in slabs of 65535 planes,
grid z + plane0, with one drain kernel behind the last slab) and tensors past 2^31 elements or 4 GiB (int64 plane
offsets, TMA maps over the whole tensor), checked against the oracle."""
import gc

import numpy as np
import pytest
import torch

from oracle import aa_oracle as O

pytestmark = pytest.mark.gpu

SLAB = 65535  # planes per launch of the tile / band kernels (aa_tile.cu, aa_band.cu)


@pytest.fixture(autouse=True)
def _release_device_memory():
    yield
    gc.collect()
    torch.cuda.empty_cache()


def _close(got, want, what):
    got = np.asarray(got, np.float64)
    wbad = ~np.isfinite(want)
    assert np.array_equal(~np.isfinite(got), wbad), (what, "non-finite placement")
    err = np.abs(got[~wbad] - want[~wbad])
    assert err.size == 0 or np.all(err <= 1e-3 + 1e-5 * np.abs(want[~wbad])), (what, float(err.max()))


def _nonfinite_past_first_slab(x, g):
    """NaN / +-Inf pixels only in planes >= SLAB (channels_first, one channel: plane = image)."""
    P, _, H, W = x.shape
    planes = [SLAB, SLAB + 1, P - 1] + torch.randint(SLAB + 2, P - 1, (20,), generator=g).tolist()
    for i, p in enumerate(planes):
        x[p, 0, int(torch.randint(0, H, (1,), generator=g)), int(torch.randint(0, W, (1,), generator=g))] = \
            (float("nan"), float("inf"), float("-inf"))[i % 3]
    return x


@pytest.mark.parametrize("shape,osize", [((70000, 1, 8, 8), (16, 16)),      # upsampling: tile kernel
                                         ((70000, 1, 16, 16), (12, 12))])   # 0.75x: band kernel
def test_more_than_65535_planes_forward(cuda, shape, osize):
    """Every plane against the oracle (planes 0, 65534, 65535, 65536 and the last among them), float and uint8 input.
    NaNs only in planes past the first slab: the drain after the slab loop must place them as the oracle does (its entries
    carry the absolute plane) and leave the planes of the first slab bit-identical to a run without the drain."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(51)
    x = torch.rand(shape, generator=g) * 255
    xu = x.to(torch.uint8)
    xn = _nonfinite_past_first_slab(x.clone(), g)
    for mode in ("linear", "cubic"):
        want = O.forward(xn.numpy(), osize, mode, False)
        assert np.isfinite(want[:SLAB]).all() and not np.isfinite(want[SLAB:]).all()
        xd = xn.to(cuda)
        y = capi.resize_forward(xd, osize, mode, False)
        ya = capi.resize_forward(xd, osize, mode, False, capi.FLAG_ASSUME_FINITE)
        torch.cuda.synchronize()
        _close(y.cpu().numpy(), want, (shape, osize, mode))
        assert torch.equal(y[:SLAB], ya[:SLAB]), (shape, osize, mode, "the drain wrote into the first slab")
        yu = capi.resize_forward(xu.to(cuda), osize, mode, False)
        torch.cuda.synchronize()
        _close(yu.cpu().numpy(), O.forward(xu.float().numpy(), osize, mode, False), (shape, osize, mode, "uint8"))


def test_more_than_65535_planes_backward(cuda):
    """The tile adjoint over 70000 planes ([70000,1,16,16] from (8,8)), non-finite grad_out only past the first slab."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(52)
    shape = (70000, 1, 16, 16)
    go = _nonfinite_past_first_slab(torch.rand((70000, 1, 8, 8), generator=g), g)
    for mode in ("linear", "cubic"):
        want = O.backward_adjoint(go.numpy(), shape, mode, False)
        gd = go.to(cuda)
        gi = capi.resize_backward(gd, shape, mode, False)
        gia = capi.resize_backward(gd, shape, mode, False, flags=capi.FLAG_ASSUME_FINITE)
        torch.cuda.synchronize()
        got = gi.cpu().numpy()
        gbad = ~np.isfinite(want)
        assert not gbad[:SLAB].any() and gbad[SLAB:].any()
        assert np.array_equal(~np.isfinite(got), gbad), (mode, "non-finite placement")
        np.testing.assert_allclose(got[~gbad], want[~gbad], rtol=1e-5, atol=4e-6)
        assert torch.equal(gi[:SLAB], gia[:SLAB]), (mode, "the drain wrote into the first slab")


# ---- tensors past 2^31 elements / 4 GiB -------------------------------------------------------------------------
def _need(nbytes):
    torch.cuda.empty_cache()
    free, _ = torch.cuda.mem_get_info()
    if free < nbytes:
        pytest.skip(f"needs {nbytes / 2**30:.1f} GiB of free device memory, {free / 2**30:.1f} GiB free")


def _images(n_images, per_image, boundary):
    """The first image, the one holding element (or byte) `boundary`, and the last."""
    return sorted({0, boundary // per_image, n_images - 1})


def _check_images(y, x, idx, osize, mode, what):
    for i in idx:
        want = O.forward(x[i:i + 1].float().cpu().numpy(), osize, mode, False)
        _close(y[i:i + 1].cpu().numpy(), want, what + (i,))


def test_cfg2_full_batch_past_4gib(cuda):
    """Full cfg2: [256,3,1080,1920] fp32 channels_last (6.4 GB) -> 224x224 bilinear, AUTO (streaming kernel) and TMA."""
    from interpolate_antialiasing_b200 import capi
    N, C, H, W = 256, 3, 1080, 1920
    _need(N * C * H * W * 4 + (1 << 30))
    gen = torch.Generator(device=cuda).manual_seed(61)
    x = torch.rand((N, H, W, C), generator=gen, device=cuda).mul_(255).permute(0, 3, 1, 2)
    idx = _images(N, C * H * W * 4, 1 << 32)
    assert len(idx) == 3
    for name, flags in (("auto", capi.FLAG_AUTO), ("tma", capi.FLAG_FORCE_STREAM | capi.FLAG_STREAM_TMA)):
        y = capi.resize_forward(x, (224, 224), "linear", False, flags)
        torch.cuda.synchronize()
        assert y.is_contiguous(memory_format=torch.channels_last)
        _check_images(y, x, idx, (224, 224), "linear", ("cfg2", name))


def test_cfg3_full_batch_past_2g_elements(cuda):
    """Full cfg3: [128,3,2160,3840] uint8 (3.2 G elements) -> 512x512 bicubic, tensor-core kernel and streaming kernel."""
    from interpolate_antialiasing_b200 import capi
    N, C, H, W = 128, 3, 2160, 3840
    _need(N * C * H * W + (1 << 30))
    gen = torch.Generator(device=cuda).manual_seed(62)
    x = torch.randint(0, 256, (N, C, H, W), generator=gen, device=cuda, dtype=torch.uint8)
    idx = _images(N, C * H * W, 1 << 31)
    for name, flags in (("vmma", capi.FLAG_VMMA), ("stream", capi.FLAG_FORCE_STREAM)):
        y = capi.resize_forward(x, (512, 512), "cubic", False, flags)
        torch.cuda.synchronize()
        capi.check_device(0)
        _check_images(y, x, idx, (512, 512), "cubic", ("cfg3", name))


def test_fp32_channels_first_past_2g_elements(cuda):
    """[360,3,1080,1920] fp32 channels_first (2.24 G elements) -> 224x224 bilinear."""
    from interpolate_antialiasing_b200 import capi
    N, C, H, W = 360, 3, 1080, 1920
    _need(N * C * H * W * 4 + (1 << 30))
    gen = torch.Generator(device=cuda).manual_seed(63)
    x = torch.rand((N, C, H, W), generator=gen, device=cuda).mul_(255)
    y = capi.resize_forward(x, (224, 224), "linear", False)
    torch.cuda.synchronize()
    _check_images(y, x, _images(N, C * H * W, 1 << 31), (224, 224), "linear", ("fp32 cf",))


def test_cfg4_backward_past_2g_elements(cuda):
    """The cfg4 backward at [2800,3,512,512] (2.2 G elements of grad_in) from 128x128 bilinear."""
    from interpolate_antialiasing_b200 import capi
    N, C, H, W = 2800, 3, 512, 512
    _need(N * C * (H * W + 128 * 128) * 4 + (1 << 30))
    gen = torch.Generator(device=cuda).manual_seed(64)
    go = torch.rand((N, C, 128, 128), generator=gen, device=cuda)
    gi = capi.resize_backward(go, (N, C, H, W), "linear", False)
    torch.cuda.synchronize()
    for i in _images(N, C * H * W, 1 << 31):
        want = O.backward_adjoint(go[i:i + 1].cpu().numpy(), (1, C, H, W), "linear", False)
        np.testing.assert_allclose(gi[i:i + 1].cpu().numpy(), want, rtol=1e-5, atol=4e-6, err_msg=str(i))
