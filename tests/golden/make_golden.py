"""Generates the committed golden fixtures in tests/golden/ from the UNMODIFIED reference.

Run in the build container only (needs /root/reference and the compiled oracle/_ref):
    python tests/golden/make_golden.py

What is written
  photo_438x906.npz      the reference's own fixture image data/test.png, RGBA->RGB exactly as
                         test.py:324 does, as a uint8 [438,906,3] array (pixels only, no code).
  golden_v1.npz          * `png_320x196`: data/proto_aa_interp_lin_step_two_output.png -- the
                           reference's committed golden output (bilinear 906x438 -> 320x196,
                           .byte()-truncated, test.py:381-385), uint8 [196,320,3].
                         * `kat_*`: the table known-answer vectors printed in
                           notebooks/tensor_iterator_playground.ipynb (linear 64->10), typed in
                           from the notebook output cells (:1202-1204, :1247-1255, :1274, :1416).
                         * `case{i}_*`: outputs of the reference extension (oracle/_ref) on small
                           seeded inputs: forward for 3 filters x align x memory format x
                           fp32/fp64, and the reference (non-AA) linear_backward.  The inputs
                           themselves are stored as shape, dtype and sha256 only; the `golden`
                           fixture (tests/conftest.py) draws them again from the same seed.
                         * `photo_sha_*`: sha256 of the fp32 bytes the reference produces on the
                           photo for test.py's 5 sizes (test.py:15-21) x 3 filters -- pins
                           bit-exactness at full size without storing 6 MB of floats.
  golden_v1_fp64.npz     the `case{i}_*` outputs of the fp64 cases (kept apart so that no file
                         exceeds 1 MB).
  reference_checks_v1.npz  what tests/test_oracle.py compares the oracle against (reference_checks()):
                         * `tables_key` / `tables_sha256`: the reference's dense weight matrix (an
                           identity resized along W) for 51 size pairs x 3 filters x align x fp32/fp64;
                         * `fb_key` / `fb_sha256` / `fb_stride`: the reference's forward outputs and
                           their strides, then its non-AA linear_backward, on seeded inputs.
                         The committed file was recorded through the oracle at the revision whose
                         test_tables_bit_exact_vs_reference and test_forward_backward_bit_exact_vs_reference
                         passed against the compiled reference on these same inputs (oracle/ and
                         tests/test_oracle.py unchanged since); main() regenerates it from the reference.
The tests never need /root/reference: they read these files and (optionally) the prebuilt _ref .so.
"""
import hashlib
import os
import sys

import numpy as np
import torch
from PIL import Image

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

from oracle.ref_ext import load_ref  # noqa: E402

REF_DATA = "/root/reference/data"
SIZES = [(320, 196), (460, 220), (120, 96), (1200, 196), (120, 1200)]  # PIL (w, h), test.py:15-21

# (shape, output_size) small cases: down, up, mixed, identity, out==1, in==1
CASES = [
    ((2, 3, 37, 53), (11, 17)),
    ((2, 4, 16, 20), (33, 47)),
    ((1, 1, 40, 30), (13, 64)),
    ((1, 3, 23, 64), (50, 9)),
    ((3, 2, 9, 9), (9, 9)),
    ((1, 3, 30, 50), (1, 1)),
    ((1, 2, 1, 1), (4, 5)),
    ((1, 3, 64, 96), (16, 24)),
]
MODES = ["linear", "cubic", "nearest"]


def _sha(a):
    """sha256 of the values in C order; -0.0 counts as 0.0 (the tests compared with np.array_equal)"""
    a = np.ascontiguousarray(a)
    return hashlib.sha256((a + a.dtype.type(0)).tobytes()).hexdigest()


def table_cases():
    """(a, b) size pairs of test_tables_bit_exact_vs_reference"""
    import random
    rnd = random.Random(1)
    cases = [(64, 10), (906, 320), (438, 196), (10, 64), (7, 7), (5, 1), (1, 5), (400, 3), (3, 400), (1920, 224), (1080, 224)]
    return cases + [(rnd.randint(1, 400), rnd.randint(1, 400)) for _ in range(40)]


def fb_cases():
    """(key, kind, x or grad_out, output size, input shape, mode, align) in the order of
    test_forward_backward_bit_exact_vs_reference's seeded draws"""
    g = torch.Generator().manual_seed(11)
    shapes = [((1, 3, 64, 96), (17, 40)), ((2, 4, 16, 20), (33, 47)), ((1, 1, 40, 30), (13, 64)), ((1, 3, 30, 50), (1, 1))]
    for shp, osz in shapes:
        for tdt in (torch.float32, torch.float64):
            for cl in (False, True):
                x = torch.rand(shp, generator=g, dtype=tdt) * 255
                if cl:
                    x = x.contiguous(memory_format=torch.channels_last)
                for mode in MODES:
                    for align in (False, True):
                        yield f"fwd {shp} {osz} {tdt} cl={cl} {mode} {align}", "fwd", x, osz, shp, mode, align
            go = torch.rand(shp[:2] + osz, generator=g, dtype=tdt)
            for align in (False, True):
                yield f"bwd {shp} {osz} {tdt} {align}", "bwd", go, osz, shp, "linear", align


def reference_checks(ref):
    """reference_checks_v1.npz from the reference module `ref`"""
    fwd = {"linear": ref.linear_forward, "cubic": ref.cubic_forward, "nearest": ref.nearest_forward}
    out = {"tables_key": [], "tables_sha256": [], "fb_key": [], "fb_sha256": [], "fb_stride": []}
    for a, b in table_cases():
        for mode in MODES:
            for align in (False, True):
                for tdt in (torch.float32, torch.float64):
                    dense = fwd[mode](torch.eye(a, dtype=tdt)[None, None], (a, b), align)[0, 0].T.numpy()
                    out["tables_key"].append(f"{a} {b} {mode} {align} {tdt}")
                    out["tables_sha256"].append(_sha(dense))
    for key, kind, t, osz, shp, mode, align in fb_cases():
        r = fwd[mode](t, osz, align) if kind == "fwd" else ref.linear_backward(t, osz, list(shp), align)
        out["fb_key"].append(key)
        out["fb_sha256"].append(_sha(r.numpy()))
        out["fb_stride"].append(list(r.stride()))
    return {k: np.array(v) for k, v in out.items()}


def main():
    ref = load_ref()
    assert ref is not None
    fwd = {"linear": ref.linear_forward, "cubic": ref.cubic_forward, "nearest": ref.nearest_forward}

    photo = np.asarray(Image.open(os.path.join(REF_DATA, "test.png")).convert("RGB")).copy()
    assert photo.shape == (438, 906, 3)
    np.savez_compressed(os.path.join(HERE, "photo_438x906.npz"), rgb=photo)

    out = {}
    out["png_320x196"] = np.asarray(Image.open(os.path.join(REF_DATA, "proto_aa_interp_lin_step_two_output.png"))).copy()
    assert np.array_equal(out["png_320x196"],
                          np.asarray(Image.open(os.path.join(REF_DATA, "proto_aa_interp_lin_step_one_output.png"))))

    # notebook known-answer vectors (linear 64 -> 10, element stride 5 in the notebook)
    out["kat_xmin_times_5"] = np.array([0, 15, 50, 80, 110, 145, 175, 210, 240, 270], np.int64)
    out["kat_row0"] = np.array([0.103352, 0.131285, 0.159218, 0.170391, 0.142458, 0.114525, 0.0865922,
                                0.0586592, 0.0307263, 0.0027933], np.float64)
    out["kat_row2_head"] = np.array([0.0220588, 0.0465686, 0.0710784, 0.0955882, 0.120098, 0.144608,
                                     0.144608, 0.120098], np.float64)
    out["kat_row2_xsize"] = np.array(12, np.int64)
    out["kat_interp_size"] = np.array(15, np.int64)

    out64 = {}
    g = torch.Generator().manual_seed(1234)
    idx = 0
    for shape, osize in CASES:
        for dt in (torch.float32, torch.float64):
            outs = out if dt == torch.float32 else out64
            x = torch.rand(shape, generator=g, dtype=dt) * 255
            out[f"case{idx}_shape"] = np.array(shape, np.int64)
            out[f"case{idx}_dtype"] = np.array(str(x.numpy().dtype))
            out[f"case{idx}_x_sha256"] = np.array(hashlib.sha256(x.numpy().tobytes()).hexdigest())
            out[f"case{idx}_osize"] = np.array(osize, np.int64)
            for mode, f in fwd.items():
                for align in (False, True):
                    y = f(x, osize, align)
                    ycl = f(x.contiguous(memory_format=torch.channels_last), osize, align)
                    assert torch.equal(y, ycl)  # SURVEY 8(b): formats give bit-identical values
                    outs[f"case{idx}_{mode}_{int(align)}"] = y.contiguous().numpy()
            gout = torch.rand(shape[:2] + osize, generator=g, dtype=dt)
            out[f"case{idx}_gout_sha256"] = np.array(hashlib.sha256(gout.numpy().tobytes()).hexdigest())
            for align in (False, True):
                outs[f"case{idx}_linbwd_{int(align)}"] = ref.linear_backward(gout, osize, list(shape), align).numpy()
            idx += 1
    out["n_cases"] = np.array(idx, np.int64)

    x = torch.from_numpy(photo.transpose(2, 0, 1).copy())[None].float()
    for (w, h) in SIZES:
        for mode, f in fwd.items():
            y = f(x, (h, w), False).contiguous().numpy()
            sha = hashlib.sha256(y.tobytes()).hexdigest()
            out[f"photo_sha_{mode}_{h}x{w}"] = np.array(sha)
            out[f"photo_sum_{mode}_{h}x{w}"] = np.array(y.astype(np.float64).sum())
    # the golden PNG is exactly the .byte()-truncated bilinear output (test.py:75)
    y = ref.linear_forward(x, (196, 320), False)[0].byte().permute(1, 2, 0).numpy()
    assert np.array_equal(y, out["png_320x196"]), "reference build does not reproduce its own golden PNG"

    np.savez_compressed(os.path.join(HERE, "golden_v1.npz"), **out)
    np.savez_compressed(os.path.join(HERE, "golden_v1_fp64.npz"), **out64)
    np.savez_compressed(os.path.join(HERE, "reference_checks_v1.npz"), **reference_checks(ref))
    for fn in ("photo_438x906.npz", "golden_v1.npz", "golden_v1_fp64.npz", "reference_checks_v1.npz"):
        print(fn, os.path.getsize(os.path.join(HERE, fn)), "bytes")


if __name__ == "__main__":
    main()
