"""The host-buffer entry point (aa_resize_forward_host: H2D / kernel / D2H pipelined inside the C ABI),
cache management and thread safety -- everything a non-torch host would exercise."""
import ctypes
import threading

import numpy as np
import pytest
import torch

from oracle import aa_oracle as O

pytestmark = pytest.mark.gpu


def _close(got, want, atol=1e-3, rtol=1e-5):
    err = np.abs(got.astype(np.float64) - want.astype(np.float64))
    assert np.all(err <= atol + rtol * np.abs(want)), err.max()


def test_host_entry_point(cuda):
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(3)
    for shape, osize, mode, cl, dt in [((7, 3, 120, 200), (30, 50), "linear", False, torch.float32),     # uneven chunks (7 images / 3 streams)
                                      ((5, 3, 96, 128), (48, 64), "cubic", True, torch.float32),
                                      ((4, 3, 200, 320), (25, 40), "cubic", False, torch.uint8),
                                      ((1, 1, 64, 64), (128, 128), "linear", False, torch.float32)]:
        x = (torch.rand(shape, generator=g) * 255).to(dt)
        if cl:
            x = x.contiguous(memory_format=torch.channels_last)
        want = O.forward(x.float().numpy(), osize, mode, False)
        for pinned in (False, True):
            xh = x.pin_memory() if pinned else x
            fmt = torch.channels_last if cl else torch.contiguous_format
            out = torch.empty((shape[0], shape[1]) + osize, dtype=torch.float32).contiguous(memory_format=fmt)
            if pinned:
                out = out.pin_memory()
            capi.resize_forward_host(xh, out, mode, False, device=0)
            _close(out.numpy(), want)
        # fused uint8 output through the host path
        out8 = torch.empty((shape[0], shape[1]) + osize, dtype=torch.uint8).contiguous(memory_format=fmt)
        capi.resize_forward_host(x, out8, mode, False, flags=capi.FLAG_ROUND_NEAREST, device=0)
        want8 = np.floor(np.clip(want, 0, 255) + 0.5)
        assert np.abs(out8.numpy().astype(np.float64) - want8).max() <= 1
    # empty batch: a no-op, not an error
    capi.resize_forward_host(torch.empty((0, 3, 8, 8)), torch.empty((0, 3, 4, 4)), "linear", False, device=0)
    # images that are not densely packed are refused with a status code
    xb = torch.rand((4, 3, 16, 16))[::2]
    with pytest.raises(capi.AAError):
        capi.resize_forward_host(xb, torch.empty((2, 3, 8, 8)), "linear", False, device=0)


def test_table_cache_clear_and_rebuild(cuda):
    from interpolate_antialiasing_b200 import capi
    x = torch.rand((1, 3, 50, 70), device=cuda) * 255
    a = capi.resize_forward(x, (20, 30), "cubic")
    n0 = capi.launch_count(reset=True)
    b = capi.resize_forward(x, (20, 30), "cubic")
    assert capi.launch_count(reset=True) == 2 and n0 >= 2          # warm cache: the kernel + the drain kernel behind it (aa_redo.cu)
    d = capi.resize_forward(x, (20, 30), "cubic", flags=capi.FLAG_ASSUME_FINITE)
    assert capi.launch_count(reset=True) == 1                      # ... which AA_FLAG_ASSUME_FINITE leaves out
    capi.resize_forward(x.byte(), (20, 30), "cubic")                 # (first uint8 call: derived tables of the tensor-core path)
    capi.launch_count(reset=True)
    capi.resize_forward(x.byte(), (20, 30), "cubic")
    assert capi.launch_count(reset=True) == 1                      # uint8 cannot hold a NaN: one launch
    assert torch.equal(b, d)
    assert capi.lib().aa_clear_table_cache() == 0
    c = capi.resize_forward(x, (20, 30), "cubic")
    assert capi.launch_count(reset=True) >= 3                        # tables rebuilt (fwd + adjoint kernels per axis) + the op
    torch.cuda.synchronize()
    assert torch.equal(a, b) and torch.equal(a, c)


def test_concurrent_callers_on_their_own_streams(cuda):
    """The library is stateless apart from the mutex-protected table / plan caches: threads on different
    streams with different shapes must not disturb each other (SURVEY 8(b) Threading)."""
    from interpolate_antialiasing_b200 import capi
    capi.lib().aa_clear_table_cache()
    errs = []

    def work(seed):
        try:
            g = torch.Generator().manual_seed(seed)
            s = torch.cuda.Stream()
            with torch.cuda.stream(s):
                for k in range(12):
                    h, w = 40 + 7 * seed + k, 64 + 5 * seed
                    x = (torch.rand((2, 3, h, w), generator=g) * 255)
                    osize = (h // 3 + 1, w // 2 + 1)
                    y = capi.resize_forward(x.to(cuda, non_blocking=False), osize, "linear" if k % 2 else "cubic")
                    s.synchronize()
                    want = O.forward(x.numpy(), osize, "linear" if k % 2 else "cubic", False)
                    _close(y.cpu().numpy(), want)
        except Exception as e:  # noqa: BLE001
            errs.append(repr(e))

    ts = [threading.Thread(target=work, args=(i,)) for i in range(4)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errs, errs


def test_host_entry_validates_before_touching_buffers(cuda):
    """ADVICE r1 (medium): dtype / strides are checked up front; a bad description never reaches the memcpy."""
    from interpolate_antialiasing_b200 import capi
    L = capi.lib()
    x = torch.rand((2, 3, 16, 16))
    o = torch.empty((2, 3, 8, 8))
    di, do = capi.desc(x, 0), capi.desc(o, 0)
    di.dtype = capi.F16  # would make the copy read past the buffer if it were sized from it
    assert L.aa_resize_forward_host(ctypes.byref(di), ctypes.byref(do), 1, 0, 0) == -1
    di = capi.desc(x, 0)
    di.stride_h = 32  # padded rows inside an image
    assert L.aa_resize_forward_host(ctypes.byref(di), ctypes.byref(do), 1, 0, 0) == -2
    di = capi.desc(x[:1], 0)
    di.stride_c = 999  # n == 1 used to skip every stride check
    assert L.aa_resize_forward_host(ctypes.byref(di), ctypes.byref(capi.desc(o[:1], 0)), 1, 0, 0) == -2
    assert L.aa_resize_forward_host(ctypes.byref(capi.desc(x, 0)), ctypes.byref(do), 7, 0, 0) == -1  # bad filter
    # mismatched memory formats
    xcl = x.contiguous(memory_format=torch.channels_last)
    assert L.aa_resize_forward_host(ctypes.byref(capi.desc(xcl, 0)), ctypes.byref(do), 1, 0, 0) == -2


def test_host_multi_device_runner(cuda):
    """aa_resize_forward_host_multi: one process, the batch sharded by image over the devices it is given; bit-identical
    to the single-device entry (SURVEY 8(e)).  With one GPU the device list [0] still exercises the sharded code path;
    with >= 2 GPUs the default list (all devices) is used as well."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(8)
    x = (torch.rand((9, 3, 150, 260), generator=g) * 255).pin_memory()
    for mode, osize in (("linear", (40, 70)), ("cubic", (33, 51))):
        want = torch.empty((9, 3) + osize).pin_memory()
        capi.resize_forward_host(x, want, mode, False, device=0)
        got = torch.empty((9, 3) + osize).pin_memory()
        capi.resize_forward_host_multi(x, got, mode, False, devices=[0])
        assert torch.equal(got, want)
        if torch.cuda.device_count() >= 2:
            got2 = torch.zeros((9, 3) + osize).pin_memory()
            capi.resize_forward_host_multi(x, got2, mode, False, devices=None)
            assert torch.equal(got2, want)
            got3 = torch.zeros((9, 3) + osize).pin_memory()
            capi.resize_forward_host_multi(x, got3, mode, False, devices=[1, 0])
            assert torch.equal(got3, want)
    with pytest.raises(capi.AAError):
        capi.resize_forward_host_multi(x, got, "linear", False, devices=[0, 0])


def test_table_cache_is_bounded_lru(cuda):
    """Variable-size pipelines (random-resized-crop) must not grow the cache without bound (ADVICE r1): more distinct
    sizes than AA_TABLE_CACHE_MAX (256 entries) go through, results stay right, and re-used early sizes still work."""
    from interpolate_antialiasing_b200 import capi
    capi.lib().aa_clear_table_cache()
    g = torch.Generator().manual_seed(13)
    x = (torch.rand((1, 1, 64, 700), generator=g) * 255).to(cuda)
    first = None
    for k in range(300):  # 300 distinct W tables + 1 H table > 256
        xs = x[:, :, :, : 380 + k].contiguous()
        y = capi.resize_forward(xs, (32, 100), "linear")
        if k == 0:
            first = y.clone()
    torch.cuda.synchronize()
    y0 = capi.resize_forward(x[:, :, :, :380].contiguous(), (32, 100), "linear")  # evicted by now: rebuilt
    torch.cuda.synchronize()
    assert torch.equal(y0, first)
    want = O.forward(x[:, :, :, :380].cpu().numpy(), (32, 100), "linear", False)
    _close(y0.cpu().numpy(), want)


def test_ragged_images_to_fixed_batch(cuda):
    """aa_resize_forward_ragged: decoded images of different sizes -> one [N,C,oH,oW] batch.  Images carved out of one
    pool at a constant distance and bound for consecutive slots share a launch; results equal per-image calls bit for bit
    and the oracle within tolerance."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(23)
    sizes = [(120, 160), (120, 160), (120, 160), (90, 200), (64, 64), (120, 160), (90, 200)]
    # images 0..2 are consecutive slices of one pool (one launch); the others are separate allocations
    pool = torch.randint(0, 256, (3, 120, 160, 3), dtype=torch.uint8, generator=g).to(cuda)
    imgs = [pool[0], pool[1], pool[2]] + [torch.randint(0, 256, (h, w, 3), dtype=torch.uint8, generator=g).to(cuda) for h, w in sizes[3:]]
    out, launches = capi.resize_forward_ragged(imgs, (48, 56), "linear")
    torch.cuda.synchronize()
    assert launches == 5 and out.shape == (7, 3, 48, 56) and out.is_contiguous(memory_format=torch.channels_last)
    for i, im in enumerate(imgs):
        x = im.permute(2, 0, 1)[None]  # channels_last NCHW view of the HWC image
        single = capi.resize_forward(x, (48, 56), "linear")
        assert torch.equal(out[i:i + 1], single), i
        want = O.forward(x.float().cpu().numpy(), (48, 56), "linear", False)
        _close(out[i:i + 1].cpu().numpy(), want)
    # planar float images, normalising epilogue into fp16
    fimgs = [(torch.rand((3, h, w), generator=g) * 255).to(cuda) for h, w in [(70, 90), (33, 47), (70, 90)]]
    o16 = torch.empty((3, 3, 32, 40), dtype=torch.float16, device=cuda)
    o16, launches = capi.resize_forward_ragged(fimgs, (32, 40), "cubic", out=o16, scale=[1 / 58.0] * 3, bias=[-2.0] * 3)
    torch.cuda.synchronize()
    assert launches == 3
    from test_epilogue_gpu import affine_ref, assert_rounded, fast_eps, got64, ref_forward
    for i, im in enumerate(fimgs):
        base = ref_forward(im[None].cpu().numpy(), (32, 40), "cubic")
        want = affine_ref(base, [1 / 58.0] * 3, [-2.0] * 3)
        assert_rounded(got64(o16[i:i + 1]), want, fast_eps(base, want, [1 / 58.0] * 3), "f16", ("ragged fp16", i))
