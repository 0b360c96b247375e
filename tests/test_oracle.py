"""CPU tests pinning the oracle (oracle/aa_oracle.c) to the reference's own golden vectors and,
when the compiled reference is present, to the reference itself bit for bit."""
import hashlib
import random

import numpy as np
import pytest
import torch

from oracle import aa_oracle as O

SIZES = [(320, 196), (460, 220), (120, 96), (1200, 196), (120, 1200)]  # PIL (w, h): reference test.py:15-21
MODES = ["linear", "cubic", "nearest"]


def test_kat_notebook_table(golden):
    # notebooks/tensor_iterator_playground.ipynb:1202-1204, 1247-1255, 1274, 1416 (linear 64 -> 10)
    xmin, xsize, w = O.tables(64, 10, "linear")
    assert w.shape[1] == int(golden["kat_interp_size"]) == O.interp_size(64, 10, "linear")
    assert np.array_equal(xmin * 5, golden["kat_xmin_times_5"])
    assert xsize.tolist() == [10, 13, 12, 13, 13, 13, 13, 12, 13, 10]
    assert int(xsize[2]) == int(golden["kat_row2_xsize"])
    np.testing.assert_allclose(w[0, :10], golden["kat_row0"], rtol=0, atol=6e-7)  # notebook prints 6 digits
    np.testing.assert_allclose(w[2, :8], golden["kat_row2_head"], rtol=0, atol=6e-7)
    assert np.all(w[0, 10:] == 0)


def test_small_cases_bit_exact_vs_golden(golden):
    n = int(golden["n_cases"])
    assert n >= 16
    for i in range(n):
        x = golden[f"case{i}_x"]
        osize = tuple(int(v) for v in golden[f"case{i}_osize"])
        for mode in MODES:
            for align in (0, 1):
                want = golden[f"case{i}_{mode}_{align}"]
                got = O.forward(x, osize, mode, bool(align))
                assert np.array_equal(got, want), (i, mode, align)
                # channels_last strides in -> same values (SURVEY 8(b))
                xcl = np.ascontiguousarray(x.transpose(0, 2, 3, 1)).transpose(0, 3, 1, 2)
                assert np.array_equal(O.forward(xcl, osize, mode, bool(align)), want), (i, mode, align, "cl")
        for align in (0, 1):
            got = O.backward_nonaa(golden[f"case{i}_gout"], x.shape, bool(align))
            assert np.array_equal(got, golden[f"case{i}_linbwd_{align}"]), (i, align)


def test_photo_sha_and_golden_png(golden, photo):
    x = photo.transpose(2, 0, 1)[None].astype(np.float32)
    for (w, h) in SIZES:
        for mode in MODES:
            y = np.ascontiguousarray(O.forward(x, (h, w), mode))
            sha = hashlib.sha256(y.tobytes()).hexdigest()
            assert sha == str(golden[f"photo_sha_{mode}_{h}x{w}"]), (mode, h, w)
    # the reference's committed golden output: bilinear -> .byte() truncation (test.py:75, :381-385)
    y = O.forward(x, (196, 320), "linear")[0]
    assert np.array_equal(y.astype(np.uint8).transpose(1, 2, 0), golden["png_320x196"])


def test_photo_vs_pil(photo):
    """The reference's own acceptance check (test.py:360-379) applied to the oracle."""
    from PIL import Image
    img = Image.fromarray(photo)
    x = photo.transpose(2, 0, 1)[None].astype(np.float32)
    for (w, h) in SIZES:
        for mode, resample, max_tol in (("linear", Image.BILINEAR, 1.0 + 1e-5), ("cubic", Image.BICUBIC, 20.0)):
            pil = np.asarray(img.resize((w, h), resample=resample)).transpose(2, 0, 1).astype(np.float32)
            y = O.forward(x, (h, w), mode)[0]
            if mode == "cubic":
                y = np.clip(y, 0, 255)
            y = y.astype(np.uint8).astype(np.float32)
            assert np.abs(y - pil).mean() < 1.0
            assert np.abs(y - pil).max() < max_tol


def test_table_properties():
    rnd = random.Random(7)
    for _ in range(300):
        a, b = rnd.randint(1, 3000), rnd.randint(1, 2000)
        mode = rnd.choice(MODES)
        align = rnd.random() < 0.3
        xmin, xsize, w = O.tables(a, b, mode, align)
        assert np.all(xsize >= 1) and np.all(xsize <= w.shape[1])
        assert np.all(np.diff(xmin) >= 0) and np.all(np.diff(xmin + xsize) >= 0)
        assert np.all(xmin >= 0) and np.all(xmin + xsize <= a)
        np.testing.assert_allclose(w.sum(1), 1.0, atol=1e-5)


def test_adjoint_is_transpose_and_matches_torch_aa():
    g = torch.Generator().manual_seed(3)
    for shape, osize in [((2, 3, 37, 53), (11, 17)), ((1, 2, 16, 20), (33, 47)), ((1, 1, 40, 30), (13, 64))]:
        for mode, tmode in (("linear", "bilinear"), ("cubic", "bicubic")):
            go = torch.rand(shape[:2] + osize, generator=g, dtype=torch.float64)
            a = O.backward_adjoint(go.numpy(), shape, mode, False)
            Wh = O.dense_matrix(shape[2], osize[0], mode, False, np.float64)
            Ww = O.dense_matrix(shape[3], osize[1], mode, False, np.float64)
            d = np.einsum("oy,ncop,px->ncyx", Wh, go.numpy(), Ww)
            np.testing.assert_allclose(a, d, rtol=0, atol=1e-13)
            x = torch.rand(shape, generator=g, dtype=torch.float64, requires_grad=True)
            y = torch.nn.functional.interpolate(x, size=osize, mode=tmode, antialias=True, align_corners=False)
            (gt,) = torch.autograd.grad(y, x, go)
            np.testing.assert_allclose(a, gt.numpy(), rtol=0, atol=1e-12)


# ---- against the reference's own results (sha256 and strides in tests/golden/reference_checks_v1.npz) ----

def _sha(a):
    """sha256 of the values in C order; -0.0 counts as 0.0 (np.array_equal semantics)"""
    a = np.ascontiguousarray(a)
    return hashlib.sha256((a + a.dtype.type(0)).tobytes()).hexdigest()


def test_tables_bit_exact_vs_reference(golden):
    keys, shas = golden["tables_key"], golden["tables_sha256"]
    rnd = random.Random(1)
    cases = [(64, 10), (906, 320), (438, 196), (10, 64), (7, 7), (5, 1), (1, 5), (400, 3), (3, 400), (1920, 224), (1080, 224)]
    cases += [(rnd.randint(1, 400), rnd.randint(1, 400)) for _ in range(40)]
    k = 0
    for a, b in cases:
        for mode in MODES:
            for align in (False, True):
                for ndt, tdt in ((np.float32, torch.float32), (np.float64, torch.float64)):
                    assert str(keys[k]) == f"{a} {b} {mode} {align} {tdt}", (k, str(keys[k]))
                    assert _sha(O.dense_matrix(a, b, mode, align, ndt)) == str(shas[k]), (a, b, mode, align, ndt)
                    k += 1
    assert k == len(keys)


def test_forward_backward_bit_exact_vs_reference(golden):
    keys, shas, strides = golden["fb_key"], golden["fb_sha256"], golden["fb_stride"]
    g = torch.Generator().manual_seed(11)
    shapes = [((1, 3, 64, 96), (17, 40)), ((2, 4, 16, 20), (33, 47)), ((1, 1, 40, 30), (13, 64)), ((1, 3, 30, 50), (1, 1))]
    k = 0
    for shp, osz in shapes:
        for tdt in (torch.float32, torch.float64):
            for cl in (False, True):
                x = torch.rand(shp, generator=g, dtype=tdt) * 255
                if cl:
                    x = x.contiguous(memory_format=torch.channels_last)
                for mode in MODES:
                    for align in (False, True):
                        assert str(keys[k]) == f"fwd {shp} {osz} {tdt} cl={cl} {mode} {align}", (k, str(keys[k]))
                        o = O.forward(x.numpy(), osz, mode, align)
                        assert _sha(o) == str(shas[k]), (shp, osz, mode, align, tdt, cl)
                        assert tuple(strides[k]) == tuple(s // o.dtype.itemsize for s in o.strides) or min(o.shape) == 1
                        k += 1
            go = torch.rand(shp[:2] + osz, generator=g, dtype=tdt)
            for align in (False, True):
                assert str(keys[k]) == f"bwd {shp} {osz} {tdt} {align}", (k, str(keys[k]))
                assert _sha(O.backward_nonaa(go.numpy(), shp, align)) == str(shas[k])
                k += 1
    assert k == len(keys)


def test_scale_factors_knob_matches_torch_aa():
    """The oracle's `scale_factors` path (aa_interpolation_impl.h:735,740-742 -> compute_scales_value) against torch's
    own CPU anti-aliased interpolate called with scale_factor / recompute_scale_factor=False: same tables up to torch's
    different accumulation (tolerance as SURVEY Appendix C: a few 1e-4 on the 0..255 scale)."""
    import torch
    import torch.nn.functional as F
    g = torch.Generator().manual_seed(4)
    x = torch.rand((1, 2, 57, 83), generator=g) * 255
    for mode, tmode in (("linear", "bilinear"), ("cubic", "bicubic")):
        for sf in ((0.37, 0.37), (0.5, 0.81), (1.7, 0.4)):
            want = F.interpolate(x, scale_factor=sf, mode=tmode, antialias=True, recompute_scale_factor=False).numpy()
            osize = want.shape[-2:]
            got = O.forward(x.numpy(), osize, mode, False, scale_factors=sf)
            assert np.abs(got - want).max() < 5e-4, (mode, sf, np.abs(got - want).max())
            # and it differs from the in/out tables when floor(in*s)/in != s
            plain = O.forward(x.numpy(), osize, mode, False)
            if abs(osize[0] / 57 - sf[0]) > 1e-3 or abs(osize[1] / 83 - sf[1]) > 1e-3:
                assert np.abs(got - plain).max() > 1e-3


def test_reference_uint8_box_filter_is_unreachable(ref_ext):
    """The reference's code intends `nearest_forward` (box filter) to accept uint8 and return uint8
    (aa_interpolation_impl.h:566-570, :615-619), but compute_indices_weights overwrites interp_size (:210) before the
    `interp_size > 1` dispatch (:608), so the call raises for Byte.  Pinned so that the product's uint8 -> uint8 box
    filter is understood as an extension, not a parity claim."""
    import torch
    x = torch.randint(0, 256, (1, 2, 12, 16), dtype=torch.uint8)
    with pytest.raises(RuntimeError, match="not implemented for 'Byte'"):
        ref_ext.nearest_forward(x, (6, 8), False)
