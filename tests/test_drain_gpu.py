"""The drain kernel (csrc/aa_redo.cu): a fast float kernel that stores a NaN/Inf reports its region to the stream's list,
and the drain launched right behind it recomputes the listed regions with in-window taps only, so that the set of
non-finite outputs is exactly the reference's.  These tests reach the drain's branches that ordinary non-finite inputs do
not: the overflow mode (more regions than the list holds: the whole output is recomputed), the list state a drain leaves
for the next call on the same stream, the generic-epilogue drain (fp16/bf16 outputs, normalisation, channels_last input
into a planar output), CUDA-graph replay, the ragged and host entry points.

Every result is checked against the oracle: the set of non-finite outputs must be the oracle's exactly, the finite ones
within the fast-path tolerance (forward 1e-3 + 1e-5 |want|, backward rtol 1e-5 / atol 4e-6)."""
import ctypes

import numpy as np
import pytest
import torch

from oracle import aa_oracle as O

pytestmark = pytest.mark.gpu

REDO_CAP = 2040      # entries of one list (kRedoCap, aa_common.cuh); past it the drain recomputes the whole output
TILE_ROWS, TILE_COLS = 64, 256  # the tile kernel's largest tile height and its flat tile width (aa_tile.cu)
BAND_COLS = 256      # the band kernel's flat column band (aa_band.cu)


def _placement(got, want, what):
    got = np.asarray(got, np.float64)
    wbad = ~np.isfinite(want)
    assert wbad.any() and not wbad.all(), what
    assert np.array_equal(~np.isfinite(got), wbad), (what, "non-finite placement", int((~np.isfinite(got)).sum()), int(wbad.sum()))
    w = want[~wbad].astype(np.float64)
    err = np.abs(got[~wbad] - w)
    assert np.all(err <= 1e-3 + 1e-5 * np.abs(w)), (what, float(err.max()))


def _placement_bwd(got, want, what):
    gbad = ~np.isfinite(want)
    assert gbad.any() and not gbad.all(), what
    assert np.array_equal(~np.isfinite(got), gbad), (what, "non-finite placement")
    np.testing.assert_allclose(got[~gbad], want[~gbad], rtol=1e-5, atol=4e-6, err_msg=str(what))


def _sprinkle(x, frac, g):
    """NaN, +Inf and -Inf at a fraction `frac` of the elements of the CPU tensor x (in place)."""
    flat = x.view(-1)
    idx = torch.randperm(flat.numel(), generator=g)[:max(1, int(flat.numel() * frac))]
    vals = torch.tensor([float("nan"), float("inf"), float("-inf")])[torch.randint(0, 3, (idx.numel(),), generator=g)]
    flat[idx] = vals
    return x


def _dev(x, cuda, cl):
    return x.to(cuda).contiguous(memory_format=torch.channels_last) if cl else x.to(cuda)


def _flat_cells(bad, cl, rows, cols):
    """Distinct (plane, row // rows, flat column // cols) cells holding a non-finite output, in the kernels' flat view
    (channels_first: one plane per channel; channels_last: one plane per image, columns x * C + c)."""
    N, C, H, W = bad.shape
    n, c, y, x = np.nonzero(bad)
    plane, f, nf = (n, x * C + c, W * C) if cl else (n * C + c, x, W)
    m = np.zeros((N * (1 if cl else C), -(-H // rows), -(-nf // cols)), bool)
    m[plane, y // rows, f // cols] = True
    return int(m.sum())


def _overflow_tile(g):
    """4x upsampling (tile kernel) with ~1 % non-finite pixels: their outputs fall in more tiles than one list holds."""
    return _sprinkle(torch.rand((16, 3, 256, 256), generator=g) * 255, 0.01, g), (1024, 1024), "cubic"


def test_overflow_mode_forward(cuda):
    """More flagged regions than the list holds: the drain recomputes the whole output (tile and band kernels)."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(41)
    band = _sprinkle(torch.rand((768, 3, 64, 512), generator=g) * 255, 0.01, g)    # 0.75x: band kernel
    for x, osize, mode, cells in [_overflow_tile(g) + (lambda bad, cl: _flat_cells(bad, cl, TILE_ROWS, TILE_COLS),),
                                  # a band CTA covers one column band of a plane over a run of row chunks: >= 1 entry per band
                                  (band, (48, 384), "linear", lambda bad, cl: _flat_cells(bad, cl, bad.shape[2], BAND_COLS))]:
        want = O.forward(x.numpy(), osize, mode, False)
        for cl in (False, True):
            n = cells(~np.isfinite(want), cl)
            assert n > 1.25 * REDO_CAP, (x.shape, cl, n)  # the list must overflow: the drain's whole-output branch runs
            y = capi.resize_forward(_dev(x, cuda, cl), osize, mode, False)
            torch.cuda.synchronize()
            _placement(y.cpu().numpy(), want, (tuple(x.shape), osize, cl))


def test_overflow_mode_backward(cuda):
    """The same on the tile adjoint: grad_out with ~1 % non-finite elements, grad_in of a 4x downsampling."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(42)
    shape = (16, 3, 1024, 1024)
    go = _sprinkle(torch.rand((16, 3, 256, 256), generator=g), 0.01, g)
    want = O.backward_adjoint(go.numpy(), shape, "linear", False)
    for cl in (False, True):
        n = _flat_cells(~np.isfinite(want), cl, TILE_ROWS, TILE_COLS)
        assert n > 1.25 * REDO_CAP, (cl, n)
        gi = capi.resize_backward(_dev(go, cuda, cl), shape, "linear", False)
        torch.cuda.synchronize()
        _placement_bwd(gi.cpu().numpy(), want, ("backward", cl))


def test_list_state_across_calls_on_one_stream(cuda):
    """The last CTA of a drain empties the list and clears the overflow flag for the next call on the stream: an
    overflow call, a call with one NaN (entries), a finite call (bit-identical to its run without the drain) and the
    overflow call again, in that order on one stream."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(43)
    big, bosize, bmode = _overflow_tile(g)
    bwant = O.forward(big.numpy(), bosize, bmode, False)
    one = torch.rand((2, 3, 64, 96), generator=g) * 255
    one[1, 2, 40, 50] = float("nan")
    owant = O.forward(one.numpy(), (128, 192), "cubic", False)
    fin = torch.rand((2, 3, 300, 400), generator=g) * 255
    fwant = O.forward(fin.numpy(), (75, 100), "cubic", False)
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        xb, xo, xf = big.to(cuda), one.to(cuda), fin.to(cuda)
        y1 = capi.resize_forward(xb, bosize, bmode, False)
        y2 = capi.resize_forward(xo, (128, 192), "cubic", False)
        y3 = capi.resize_forward(xf, (75, 100), "cubic", False)
        y3a = capi.resize_forward(xf, (75, 100), "cubic", False, capi.FLAG_ASSUME_FINITE)
        y4 = capi.resize_forward(xb, bosize, bmode, False)
        s.synchronize()
    _placement(y1.cpu().numpy(), bwant, "overflow call")
    _placement(y2.cpu().numpy(), owant, "one NaN after an overflow")
    assert torch.isfinite(y3).all() and torch.equal(y3, y3a), "finite call after a drain"
    err = np.abs(y3.cpu().numpy().astype(np.float64) - fwant)
    assert np.all(err <= 1e-3 + 1e-5 * np.abs(fwant))
    _placement(y4.cpu().numpy(), bwant, "overflow call again")


def test_generic_epilogue_drain(cuda):
    """Non-finite float input through aa_resize_forward_ex: fp32 / fp16 / bf16 outputs, with and without the per-channel
    affine map, channels_first and channels_last -> planar; AUTO (stream, band and tile kernels) and the forced streaming
    kernel where it takes the shape; then the ragged entry point with planar images that hold a NaN."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(44)
    x = torch.rand((2, 3, 120, 160), generator=g) * 255
    for (n, c, yy, xx), v in [((0, 0, 5, 7), float("nan")), ((0, 2, 119, 159), float("inf")), ((1, 1, 60, 53), float("-inf")),
                              ((1, 0, 0, 0), float("nan"))]:
        x[n, c, yy, xx] = v
    scale, bias = [1 / (255 * 0.229), 1 / (255 * 0.224), -1 / (255 * 0.225)], [-2.1, -2.0, 1.8]
    tols = {torch.float32: 1e-5, torch.float16: 1e-3, torch.bfloat16: 8e-3}
    ran = 0
    for osize in ((48, 64), (90, 120), (180, 240)):        # stream, band, tile
        base = O.forward(x.numpy(), osize, "cubic", False).astype(np.float64)
        for affine in (False, True):
            want = base * np.array(scale)[None, :, None, None] + np.array(bias)[None, :, None, None] if affine else base
            for odt, rtol in tols.items():
                for cl_in in (False, True):
                    xc = x.to(cuda)
                    xc = xc.permute(0, 2, 3, 1).contiguous().permute(0, 3, 1, 2) if cl_in else xc  # HWC -> planar output
                    for flags in (capi.FLAG_AUTO, capi.FLAG_FORCE_STREAM):
                        out = torch.empty((2, 3) + osize, dtype=odt, device=cuda)
                        try:
                            capi.resize_forward_ex(xc, osize, "cubic", out, scale if affine else None, bias if affine else None,
                                                   flags=flags)
                        except capi.AAError as e:
                            if "-2" in str(e) and flags == capi.FLAG_FORCE_STREAM:
                                continue
                            raise
                        torch.cuda.synchronize()
                        got = out.float().cpu().numpy().astype(np.float64)
                        what = (osize, affine, odt, cl_in, flags)
                        wbad = ~np.isfinite(want)
                        assert np.array_equal(~np.isfinite(got), wbad), what
                        err = np.abs(got[~wbad] - want[~wbad])
                        assert np.all(err <= 1e-3 + rtol * np.abs(want[~wbad])), (what, float(err.max()))
                        ran += 1
    assert ran >= 3 * 2 * 3 * 2
    # smallest case of a bug these checks found: a channels_first input got channel 0's scale / bias on every channel
    xs = torch.rand((1, 3, 8, 8), generator=g) * 255
    want = O.forward(xs.numpy(), (4, 4), "linear", False) * np.array(scale)[None, :, None, None] + np.array(bias)[None, :, None, None]
    for flags in (capi.FLAG_AUTO, capi.FLAG_FORCE_GENERAL):
        out = capi.resize_forward_ex(xs.to(cuda), (4, 4), "linear", torch.empty((1, 3, 4, 4), device=cuda), scale, bias, flags=flags)
        assert np.abs(out.cpu().numpy() - want).max() <= 1e-4, flags
    # ragged: planar float images of two sizes, NaN/Inf in some of them
    imgs = [torch.rand((3, 60, 80), generator=g) * 255, torch.rand((3, 90, 120), generator=g) * 255, torch.rand((3, 60, 80), generator=g) * 255]
    imgs[0][1, 10, 20] = float("nan")
    imgs[1][2, 89, 119] = float("inf")
    out, launches = capi.resize_forward_ragged([t.to(cuda) for t in imgs], (45, 60), "cubic")
    torch.cuda.synchronize()
    assert launches >= 2
    got = out.cpu().numpy()
    for i, t in enumerate(imgs):
        want = O.forward(t[None].numpy(), (45, 60), "cubic", False)[0]
        wbad = ~np.isfinite(want)
        assert np.array_equal(~np.isfinite(got[i]), wbad), ("ragged", i)
        assert np.all(np.abs(got[i][~wbad] - want[~wbad]) <= 1e-3 + 1e-5 * np.abs(want[~wbad])), ("ragged", i)


def test_cuda_graph_replay_repairs_nonfinite(cuda):
    """A forward + backward pair captured on finite data: replayed on NaN/Inf data, the captured drains place the
    non-finite outputs as the oracle does; replayed on finite data again, the outputs are finite and bit-identical to
    eager calls without the drain."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(45)
    x0 = torch.rand((1, 3, 438, 906), generator=g) * 255
    go0 = torch.rand((1, 3, 196, 320), generator=g)
    x, go = x0.to(cuda), go0.to(cuda)
    out = torch.empty((1, 3, 196, 320), device=cuda)
    gin = torch.empty_like(x)
    L = capi.lib()
    s = torch.cuda.Stream()
    with torch.cuda.stream(s):
        capi.check(L.aa_warm_tables(438, 906, 196, 320, capi.TRIANGLE, 0, capi.F32, 0, ctypes.c_void_p(s.cuda_stream)))
        capi.resize_forward(x, (196, 320), "linear", out=out)      # warm-up outside capture
        capi.resize_backward(go, x.shape, "linear", out=gin)
    s.synchronize()
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph, stream=s):
        capi.resize_forward(x, (196, 320), "linear", out=out)
        capi.resize_backward(go, x.shape, "linear", out=gin)
    xn, gon = x0.clone(), go0.clone()
    xn[0, 0, 100, 200] = float("nan"); xn[0, 2, 437, 905] = float("inf"); xn[0, 1, 0, 0] = float("-inf")
    gon[0, 1, 50, 60] = float("nan"); gon[0, 0, 195, 319] = float("-inf")
    x.copy_(xn); go.copy_(gon)
    graph.replay()
    torch.cuda.synchronize()
    _placement(out.cpu().numpy(), O.forward(xn.numpy(), (196, 320), "linear", False), "graph forward")
    _placement_bwd(gin.cpu().numpy(), O.backward_adjoint(gon.numpy(), x.shape, "linear", False), "graph backward")
    x.copy_(x0); go.copy_(go0)
    graph.replay()
    torch.cuda.synchronize()
    ye = capi.resize_forward(x, (196, 320), "linear", flags=capi.FLAG_ASSUME_FINITE)
    ge = capi.resize_backward(go, x.shape, "linear", flags=capi.FLAG_ASSUME_FINITE)
    torch.cuda.synchronize()
    assert torch.isfinite(out).all() and torch.isfinite(gin).all()
    assert torch.equal(out, ye) and torch.equal(gin, ge)


def test_host_entry_point_nonfinite(cuda):
    """aa_resize_forward_host: 7 images in chunks of 3 on three internal streams (each with its own list), non-finite
    pixels in every chunk."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(46)
    x = torch.rand((7, 3, 256, 384), generator=g) * 255
    for (n, c, yy, xx), v in [((0, 0, 10, 10), float("nan")), ((1, 2, 255, 383), float("inf")), ((4, 1, 128, 0), float("-inf")),
                              ((6, 0, 0, 200), float("nan"))]:
        x[n, c, yy, xx] = v
    for osize, mode in (((100, 150), "cubic"), ((384, 512), "linear")):   # stream, tile
        for cl in (False, True):
            fmt = torch.channels_last if cl else torch.contiguous_format
            xh = x.contiguous(memory_format=fmt)
            oh = torch.empty((7, 3) + osize, memory_format=fmt)
            capi.resize_forward_host(xh, oh, mode)
            _placement(oh.numpy(), O.forward(x.numpy(), osize, mode, False), (osize, mode, cl))
