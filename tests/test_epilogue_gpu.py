"""The fused output epilogue of the forward kernels (aa_store<true>, aa_common.cuh): the per-channel affine map
v*scale[c] + bias[c], float16 / bfloat16 / uint8 stores and planar (CHW) output from a channels_last (HWC) input, on the
tile, band, streaming and tensor-core kernels, the two-launch path, the general kernel and the entry points in front of
them (aa_resize_forward_ex, aa_resize_forward_ragged, decode_resize_normalize, resize_to_uint8).

The reference is computed in float64: the resize as exact sums over the float32 tables the kernels use, then the affine
map with the scale / bias values rounded to float32 (what the kernels receive), then the output type's own rounding rule.  Rounding is
monotone, so a fast kernel passes when round_T(ref - eps) <= got <= round_T(ref + eps) with
eps = (1e-3 + 1e-5 |pixel|) |scale[c]| + 2^-23 |ref| -- the fast-path tolerance carried through the affine map, plus the
float32 rounding of the fused multiply-add.  That accepts one output step only where the exact value lies within eps of a
rounding boundary, so a kernel that truncates instead of rounding, or is one step off, fails.  Rows whose sums and affine
maps are exact in float32 (identity resizes, box filters at integer factors) must equal the exact rounding outright.

Every case also records which kernels it launched (torch.profiler, CUDA activity) and asserts the family it exists for.
"""
import ctypes
import re
import warnings
from collections import Counter

import numpy as np
import pytest
import torch

from oracle import aa_oracle as O
from test_forward_gpu import _guarded, _untouched_outside

# ---- rounding rules of the output types (float64) ------------------------------------------------------------------
F16 = (10, -14, 65504.0)                            # mantissa bits, smallest normal exponent, largest finite value
BF16 = (7, -126, (2.0 - 2.0 ** -7) * 2.0 ** 127)


def rne(x, mantissa_bits, min_exp, max_finite):
    """Round-to-nearest-even of float64 values to a binary format with `mantissa_bits` stored bits, smallest normal
    exponent `min_exp` (below it the spacing stays 2^(min_exp - mantissa_bits): subnormals) and largest finite value
    `max_finite` (a result past it is +-inf, so ties at the overflow threshold go to inf like IEEE's)."""
    x = np.asarray(x, np.float64)
    ax = np.abs(x)
    with np.errstate(invalid="ignore", over="ignore"):
        _, e = np.frexp(ax)                                      # ax = m * 2^e, m in [0.5, 1)
        q = np.ldexp(1.0, np.maximum(e - 1, min_exp) - mantissa_bits)  # the spacing at ax: a power of two
        r = np.round(ax / q) * q                                 # ax / q and the product are exact; np.round: ties to even
        r = np.where(r > max_finite, np.inf, r)
    return np.copysign(r, x)


def to_u8(v, round_nearest):
    """The uint8 store: clamp to [0, 255], then truncate (.byte()) or add 0.5 first (FLAG_ROUND_NEAREST)."""
    v = np.clip(np.asarray(v, np.float64), 0.0, 255.0)
    return np.floor(v + 0.5) if round_nearest else np.floor(v)


KINDS = ("f32", "f16", "bf16", "u8", "u8r")   # u8: truncating store, u8r: FLAG_ROUND_NEAREST


def round_to(v, kind):
    if kind == "f16":
        return rne(v, *F16)
    if kind == "bf16":
        return rne(v, *BF16)
    if kind in ("u8", "u8r"):
        return to_u8(v, kind == "u8r")
    return np.asarray(v, np.float64)


def assert_rounded(got, ref, eps, kind, what):
    """got (any dtype, converted exactly to float64) against the float64 reference `ref`: |got - ref| <= eps for
    float32 outputs, round_T(ref - eps) <= got <= round_T(ref + eps) for the others; eps = 0 demands the exact rounding."""
    got = np.asarray(got, np.float64)
    ref = np.asarray(ref, np.float64)
    eps = np.broadcast_to(np.asarray(eps, np.float64), ref.shape)
    if kind == "f32":
        ok = np.abs(got - ref) <= eps
        lo, hi = ref - eps, ref + eps
    else:
        lo, hi = round_to(ref - eps, kind), round_to(ref + eps, kind)
        ok = (lo <= got) & (got <= hi)
    if not ok.all():
        bad = np.argwhere(~ok)
        i = tuple(bad[0])
        raise AssertionError(f"{what}: {len(bad)} of {ok.size} outputs outside the rounding window; first at {i}: "
                             f"got {got[i]!r}, ref {ref[i]!r}, window [{lo[i]!r}, {hi[i]!r}]")


def fast_eps(pixel, ref, scale=None):
    """eps of the acceptance rule for the resized values `pixel` [N, C, ...] mapped to `ref` with per-channel `scale`."""
    s = 1.0 if scale is None else np.abs(_f32(scale[:pixel.shape[1]]))[None, :, None, None]
    return (1e-3 + 1e-5 * np.abs(pixel)) * s + 2.0 ** -23 * np.abs(ref)


def _f32(v):
    return np.asarray(v, np.float32).astype(np.float64)


def ref_forward(x, osize, mode):
    """The resize in float64 over the float32 tables every kernel (and the reference implementation for float inputs)
    uses: out = Ah x Aw^T with exact sums.  Tables computed in float64 are not the operation the kernels perform: their
    window centres carry no float32 rounding, which moves outputs of large images by up to ~2e-3 -- more than the fast-path
    tolerance."""
    x = np.asarray(x, np.float64)
    ah = O.dense_matrix(x.shape[2], osize[0], mode, False, np.float32).astype(np.float64)
    aw = O.dense_matrix(x.shape[3], osize[1], mode, False, np.float32).astype(np.float64)
    return np.einsum("oh,nchw,pw->ncop", ah, x, aw, optimize=True)


def affine_ref(base, scale, bias):
    """base * scale[c] + bias[c] in float64, scale / bias rounded to float32 first (as the kernels receive them)."""
    if scale is None:
        return base
    C = base.shape[1]
    return base * _f32(scale[:C])[None, :, None, None] + _f32(bias[:C])[None, :, None, None]


def got64(t):
    return t.float().cpu().numpy().astype(np.float64) if t.dtype != torch.uint8 else t.cpu().numpy().astype(np.float64)


# ---- which kernels a call launched ----------------------------------------------------------------------------------
_KERNEL_FAMILY = re.compile(r"\b(aa_[A-Za-z0-9_]+?_kernel)\b")
_ROUTING = {}          # {"ok": bool, "why": str}: whether CUPTI traces kernels on this machine
ROUTES = {}            # case -> families seen (the routing report)


def _routing_available():
    if not _ROUTING:
        try:
            from torch.profiler import ProfilerActivity, profile
            x = torch.zeros(1024, device="cuda")
            torch.cuda.synchronize()
            with profile(activities=[ProfilerActivity.CUDA]) as prof:
                x.add_(1.0)
                torch.cuda.synchronize()
            n = sum(1 for e in prof.events() if getattr(e, "device_type", None) == torch.autograd.DeviceType.CUDA)
            _ROUTING.update(ok=n > 0, why="" if n else "torch.profiler recorded no CUDA kernel (CUPTI cannot trace here)")
        except Exception as e:  # noqa: BLE001 -- any profiler failure only disables the routing assertions
            _ROUTING.update(ok=False, why=f"torch.profiler with CUDA activity failed: {e!r}")
    return _ROUTING["ok"]


def launched(fn):
    """Runs fn() (and synchronises) -> (fn's result, Counter of the aa_*_kernel families it launched), or (result, None)
    when kernels cannot be traced here."""
    if not _routing_available():
        r = fn()
        torch.cuda.synchronize()
        return r, None
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        r = fn()
        torch.cuda.synchronize()
    fams = Counter()
    for e in prof.events():  # only CUDA activity is traced: the demangled kernel names
        m = _KERNEL_FAMILY.search(e.name)
        if m:
            fams[m.group(1)] += 1
    return r, fams


def assert_route(fams, expect, calls, what, fast=True):
    """Every family in `expect` ran at least `calls` times; a case meant for a fast kernel never reached aa_general_kernel."""
    ROUTES[what] = sorted(fams) if fams is not None else None
    if fams is None:
        warnings.warn(f"routing not checked for {what}: {_ROUTING.get('why')}")
        return
    for f in expect:
        assert fams[f] >= calls, (what, f"expected {f} x>={calls}", dict(fams))
    if fast:
        assert "aa_general_kernel" not in fams, (what, "fell back to the general kernel", dict(fams))


# ---- calls ------------------------------------------------------------------------------------------------------------
def _odtype(kind):
    return {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16, "u8": torch.uint8, "u8r": torch.uint8}[kind]


def _bits(t):
    return t.view({2: torch.int16, 4: torch.int32, 8: torch.int64}[t.element_size()]) if t.element_size() > 1 else t


def _fill_bits(fill, dtype):
    return _bits(torch.full((1,), fill, dtype=dtype)).item()


def _input(x, layout):
    return x.contiguous(memory_format=torch.channels_last) if layout in ("cl", "planar") else x.contiguous()


def run_ex(capi, x, osize, mode, kind, layout, flags, scale=None, bias=None, crop=None):
    """aa_resize_forward_ex through `out=` into a guarded view (crop: padded rows, base pointer one element past a row
    start).  Float outputs are canaried with NaN and compared as bits outside the view; uint8 outputs run with canary 0
    and 255, which must agree.  -> the output (a view)."""
    N, C = x.shape[:2]
    odt = _odtype(kind)
    fl = flags | (capi.FLAG_ROUND_NEAREST if kind == "u8r" else 0)
    outs = []
    for fill in ((0, 255) if odt == torch.uint8 else (float("nan"),)):
        buf, out = _guarded((N, C) + tuple(osize), odt, x.device, layout == "cl", fill, crop=crop)
        capi.resize_forward_ex(x, osize, mode, out, scale, bias, flags=fl)
        torch.cuda.synchronize()
        assert _untouched_outside(_bits(buf), _bits(out), _fill_bits(fill, odt)), (tuple(x.shape), osize, kind, layout, "wrote outside the output")
        outs.append(out)
    if len(outs) == 2:
        assert torch.equal(outs[0], outs[1]), (tuple(x.shape), osize, kind, layout, "an output byte was left unwritten")
    return outs[-1]


# per-channel maps that differ by sign and by large factors: a channel swap, or channel 0's map on every channel, misses
# by far more than eps
SCALE_F = [1 / 58.0, -3.0, 0.25, -40.0]
BIAS_F = [-2.0, 300.0, -17.5, 5000.0]
SCALE_U8 = [0.5, -1.0, 2.0, -0.25]      # uint8 outputs: spread over 0..255, clamped at both ends on channel 2
BIAS_U8 = [10.0, 255.0, -100.0, 80.0]

# The matrix: each case names the kernel family it exists for.  flags: per input dtype.
#   tile: upsampling.  band: 0.75x vertical (uint8 with FLAG_STREAM_LDG, which keeps AUTO off the tensor-core kernel), and
#   the identity.  stream: fp32 rows wider than 512 floats with 4-wide vectors under AUTO; uint8 rows of 8-byte vectors
#   under FLAG_FORCE_STREAM (AUTO sends uint8 downsampling to the tensor-core kernel).  vmma: uint8 4x vertical, rows a
#   multiple of 16 bytes (fp32 input takes the streaming kernel).  two_launch: 4x up in H (more output rows per input row
#   than the streaming kernel holds), 8x down in W: a streaming W pass into a temporary, then a tile H pass.
MATRIX = {
    "tile": ((24, 40), (50, 72), "linear", {}, {"u8": ["aa_tile_kernel"], "f32": ["aa_tile_kernel"]}),
    "band": ((48, 64), (36, 56), "linear", {"u8": "FLAG_STREAM_LDG"}, {"u8": ["aa_band_kernel"], "f32": ["aa_band_kernel"]}),
    "band_identity": ((40, 56), (40, 56), "linear", {}, {"u8": ["aa_band_kernel"], "f32": ["aa_band_kernel"]}),
    "stream": ((64, 544), (16, 136), "linear", {"u8": "FLAG_FORCE_STREAM"}, {"u8": ["aa_stream_kernel"], "f32": ["aa_stream_kernel"]}),
    "vmma": ((128, 544), (32, 136), "cubic", {}, {"u8": ["aa_vmma_kernel"], "f32": ["aa_stream_kernel"]}),
    "two_launch": ((16, 320), (64, 40), "linear", {}, {"u8": ["aa_stream_kernel", "aa_tile_kernel"],
                                                       "f32": ["aa_stream_kernel", "aa_tile_kernel"]}),
    "general": ((48, 64), (36, 56), "linear", {"u8": "FLAG_FORCE_GENERAL", "f32": "FLAG_FORCE_GENERAL"},
                {"u8": ["aa_general_kernel"], "f32": ["aa_general_kernel"]}),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(MATRIX))
def test_epilogue_matrix(cuda, case):
    """Each kernel x input uint8/fp32 x layout (channels_first -> channels_first through the per-channel split,
    channels_last -> channels_last, channels_last -> planar) x C in 1..4 x output fp32/fp16/bf16/uint8 truncate/uint8 round
    x affine map on/off, several epilogues in a row on one shape (the launch-plan caches key only on a 'generic' bit), all
    written through guarded views, dense and padded."""
    from interpolate_antialiasing_b200 import capi
    (H, W), osize, mode, flag_names, expect = MATRIX[case]
    g = torch.Generator().manual_seed(100 + list(MATRIX).index(case))
    ran = 0
    for C in (1, 2, 3, 4):
        x8 = torch.randint(0, 256, (2, C, H, W), dtype=torch.uint8, generator=g)
        xf = torch.rand((2, C, H, W), generator=g, dtype=torch.float64).float() * 255
        for dt, xs in (("u8", x8), ("f32", xf)):
            base = ref_forward(xs.numpy(), osize, mode)
            flags = getattr(capi, flag_names.get(dt, "FLAG_AUTO"))
            for layout in ("cf", "cl", "planar"):
                x = _input(xs.to(cuda), layout)
                planar = layout == "planar" and C > 1   # with one channel both formats are the same bytes
                variants = [(k, a) for a in (False, True) for k in KINDS]

                def run_all():
                    res = []
                    for i, (kind, affine) in enumerate(variants):
                        sc, bi = ((SCALE_U8, BIAS_U8) if kind in ("u8", "u8r") else (SCALE_F, BIAS_F)) if affine else (None, None)
                        crop = None if i % 2 == 0 else (1, 1, 2, 7)
                        res.append(run_ex(capi, x, osize, mode, kind, layout, flags, sc and sc[:C], bi and bi[:C], crop=crop))
                    return res
                outs, fams = launched(run_all)
                for (kind, affine), out in zip(variants, outs):
                    sc, bi = ((SCALE_U8, BIAS_U8) if kind in ("u8", "u8r") else (SCALE_F, BIAS_F)) if affine else (None, None)
                    ref = affine_ref(base, sc, bi)
                    assert_rounded(got64(out), ref, fast_eps(base, ref, sc), kind, (case, dt, layout, C, kind, affine))
                    ran += 1
                exp = expect[dt]
                fast = "aa_general_kernel" not in exp
                if case == "two_launch" and planar:  # the two-launch path has no planar epilogue: the general kernel
                    exp, fast = ["aa_general_kernel"], False
                assert_route(fams, exp, len(variants), (case, dt, layout, C), fast=fast)
    assert ran == 4 * 2 * 3 * 10


# ---- exact rows ---------------------------------------------------------------------------------------------------------
# scale / bias that keep every result exact in float32 and put a share of them on a tie of the output type: uint8 x*0.5
# (odd x), float16 2048 + x (the spacing there is 2), bfloat16 256 + x; the other channels differ in sign and factor
EXACT_MAPS = {
    "f32": ([1.0, -1.0, 2.0], [0.0, 1.0, -3.0]),
    "f16": ([1.0, -1.0, 2.0], [2048.0, -2048.0, 1024.0]),
    "bf16": ([1.0, -1.0, 2.0], [256.0, -256.0, 128.0]),
    "u8": ([0.5, -0.5, 0.25], [0.0, 255.0, 0.0]),
    "u8r": ([0.5, -0.5, 0.25], [0.0, 255.0, 0.0]),
}
# (name, input (H, W), output size, filter, flags per input dtype, kernel family per input dtype).  Identity: one tap of
# weight 1 (the neighbours' weights are exactly 0).  Box filter at 2x / 4x: weights exactly 1/2, 1/4; the sums of integer
# pixels are multiples of 1/4, 1/16 below 256: exact in float32 in any order.  The tensor-core kernel's vertical weights
# are base-256 digits of the float weight (aa_vmma.cu): 1, 1/2 and 1/4 are single digits, so its sums are exact too.
# The tile kernel takes upsampling only (2x / 4x box downsampling goes to the streaming kernel), so its rows are 2x
# upsamplings: box (one tap of weight 1) and linear (weights 3/4 and 1/4, sums multiples of 1/16).
EXACT_ROWS = [
    ("band identity", (40, 56), (40, 56), "linear", {}, {"u8": "aa_band_kernel", "f32": "aa_band_kernel"}),
    ("stream identity", (24, 544), (24, 544), "linear", {"u8": "FLAG_FORCE_STREAM", "f32": "FLAG_FORCE_STREAM"},
     {"u8": "aa_stream_kernel", "f32": "aa_stream_kernel"}),
    ("general identity", (40, 56), (40, 56), "linear", {"u8": "FLAG_FORCE_GENERAL", "f32": "FLAG_FORCE_GENERAL"},
     {"u8": "aa_general_kernel", "f32": "aa_general_kernel"}),
    ("vmma identity", (24, 544), (24, 544), "linear", {"u8": "FLAG_VMMA"}, {"u8": "aa_vmma_kernel"}),
    ("tile linear up 2x", (24, 136), (48, 272), "linear", {}, {"u8": "aa_tile_kernel", "f32": "aa_tile_kernel"}),
    ("tile box up 2x", (24, 136), (48, 272), "box", {}, {"u8": "aa_tile_kernel", "f32": "aa_tile_kernel"}),
    ("vmma box 2x", (64, 544), (32, 272), "box", {}, {"u8": "aa_vmma_kernel"}),
    ("vmma box 4x", (64, 544), (16, 136), "box", {}, {"u8": "aa_vmma_kernel"}),
    ("stream box 2x", (64, 544), (32, 272), "box", {"u8": "FLAG_FORCE_STREAM", "f32": "FLAG_FORCE_STREAM"},
     {"u8": "aa_stream_kernel", "f32": "aa_stream_kernel"}),
    ("stream box 4x", (64, 544), (16, 136), "box", {"u8": "FLAG_FORCE_STREAM", "f32": "FLAG_FORCE_STREAM"},
     {"u8": "aa_stream_kernel", "f32": "aa_stream_kernel"}),
    ("general box 4x", (64, 544), (16, 136), "box", {"u8": "FLAG_FORCE_GENERAL"}, {"u8": "aa_general_kernel"}),
]


def _ties(ref, kind):
    """Share of `ref` exactly halfway between two neighbours of the output type."""
    if kind in ("u8", "u8r"):
        v = ref[(ref > 0) & (ref < 255)]
        return float(np.mean(v - np.floor(v) == 0.5)) if v.size else 0.0
    if kind == "f32":
        return 0.0
    mb, me, _ = F16 if kind == "f16" else BF16
    _, e = np.frexp(np.abs(ref))
    q = np.ldexp(1.0, np.maximum(e - 1, me) - mb)
    return float(np.mean(np.abs(ref) / q % 1 == 0.5))


@pytest.mark.gpu
@pytest.mark.parametrize("row", [r[0] for r in EXACT_ROWS])
def test_exact_rows(cuda, row):
    """Sums and affine maps exact in float32: `got` must equal the exact rounding of the float64 result (no eps).  These
    rows tell round-half-even from round-half-up and truncation from rounding, on every kernel."""
    from interpolate_antialiasing_b200 import capi
    _, (H, W), osize, mode, flag_names, expect = next(r for r in EXACT_ROWS if r[0] == row)
    g = torch.Generator().manual_seed(7)
    x8 = torch.randint(0, 256, (2, 3, H, W), dtype=torch.uint8, generator=g)
    for dt in expect:
        xs = x8 if dt == "u8" else x8.float()            # fp32 input holding integers: the same exact sums
        base = ref_forward(xs.numpy(), osize, mode)
        flags = getattr(capi, flag_names.get(dt, "FLAG_AUTO"))
        for layout in ("cf", "cl", "planar"):
            x = _input(xs.to(cuda), layout)
            variants = [(k, a) for a in (False, True) for k in KINDS]

            def run_all():
                return [run_ex(capi, x, osize, mode, kind, layout, flags, *(EXACT_MAPS[kind] if affine else (None, None)),
                               crop=None if i % 2 else (1, 1, 2, 7)) for i, (kind, affine) in enumerate(variants)]
            outs, fams = launched(run_all)
            for (kind, affine), out in zip(variants, outs):
                ref = affine_ref(base, *(EXACT_MAPS[kind] if affine else (None, None)))
                if affine and kind != "f32":
                    assert _ties(ref, kind) > 0.02, (row, dt, kind, "too few ties to tell the rounding rules apart")
                assert_rounded(got64(out), ref, 0.0, kind, (row, dt, layout, kind, affine))
            assert_route(fams, [expect[dt]], len(variants), (row, dt, layout), fast=expect[dt] != "aa_general_kernel")


# ---- range edges ----------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_range_edges(cuda):
    """float16: an affine map per channel that lands in (65504, 65520) (rounds to 65504), at and past 65520 (inf), far
    past it, and across the subnormal boundary; uint8: maps that push values below 0 and above 255."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(9)
    sc16 = [0.125, -2.0 ** -20, 1000.0, -2.0 ** -24]
    bi16 = [65490.0, 0.0, 0.0, 2.0 ** -14]
    sc8 = [3.0, -2.0, 1.5, 1.0]
    bi8 = [-200.0, 300.0, -50.0, 100.0]
    seen = Counter()
    for name in ("tile", "band", "stream", "vmma", "general"):
        (H, W), osize, mode, flag_names, _ = MATRIX[name]
        x8 = torch.randint(0, 256, (2, 4, H, W), dtype=torch.uint8, generator=g)
        for dt, xs in (("u8", x8), ("f32", torch.rand((2, 4, H, W), generator=g) * 255)):
            base = ref_forward(xs.numpy(), osize, mode)
            flags = getattr(capi, flag_names.get(dt, "FLAG_AUTO"))
            for layout in ("cf", "planar"):
                x = _input(xs.to(cuda), layout)
                for kind, sc, bi in (("f16", sc16, bi16), ("u8", sc8, bi8), ("u8r", sc8, bi8)):
                    ref = affine_ref(base, sc, bi)
                    out = run_ex(capi, x, osize, mode, kind, layout, flags, sc, bi, crop=(1, 1, 2, 7))
                    assert_rounded(got64(out), ref, fast_eps(base, ref, sc), kind, ("range", name, dt, layout, kind))
                    if kind == "f16":
                        seen["(65504, 65520)"] += int(((ref > 65504) & (ref < 65520)).sum())
                        seen[">= 65520"] += int((ref >= 65520).sum())
                        seen["subnormal"] += int(((ref != 0) & (np.abs(ref) < 2.0 ** -14)).sum())
                    else:
                        seen["< 0"] += int((ref < 0).sum())
                        seen["> 255"] += int((ref > 255).sum())
    assert all(seen[k] > 0 for k in ("(65504, 65520)", ">= 65520", "subnormal", "< 0", "> 255")), dict(seen)


# ---- refusals --------------------------------------------------------------------------------------------------------------
def _rc(capi, fn_name, x, out, flags=0, scale=None, bias=None):
    L = capi.lib()
    di, do = capi.desc(x), capi.desc(out)
    st = capi._stream(x)
    if fn_name == "plain":
        return L.aa_resize_forward(ctypes.byref(di), ctypes.byref(do), capi.TRIANGLE, 0, flags, st)
    e = capi.Epilogue()
    e.normalize = 1 if scale is not None else 0
    for i in range(4):
        e.scale[i] = scale[i] if scale is not None and i < len(scale) else 1.0
        e.bias[i] = bias[i] if bias is not None and i < len(bias) else 0.0
    return L.aa_resize_forward_ex(ctypes.byref(di), ctypes.byref(do), capi.TRIANGLE, 0, flags, ctypes.byref(e), st)


@pytest.mark.gpu
def test_refusals_leave_output_untouched(cuda):
    """Combinations without a kernel return their documented status and do not write `out`."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(3)
    xf = (torch.rand((2, 3, 64, 544), generator=g) * 255).to(cuda)
    x5 = (torch.rand((1, 5, 32, 32), generator=g) * 255).to(cuda)
    xn = (torch.rand((1, 3, 32, 128), generator=g) * 255).to(cuda)        # 128 floats a row: the narrow streaming variant
    s3 = [0.5, 2.0, -1.0]

    def out(shape, dt, cl=False):
        t = torch.full(shape, 77, dtype=dt, device=cuda)
        return t.contiguous(memory_format=torch.channels_last) if cl else t
    cases = [
        ("fp16 output through aa_resize_forward", "plain", xf, out((2, 3, 16, 136), torch.float16), 0, None, -1),
        ("f64 input with the affine map", "ex", xf.double(), out((2, 3, 16, 136), torch.float64), 0, s3, -2),
        ("f64 input with fp16 output", "ex", xf.double(), out((2, 3, 16, 136), torch.float16), 0, None, -1),
        ("affine map with C = 5", "ex", x5, out((1, 5, 16, 16), torch.float32), 0, [1.0] * 4, -2),
        ("channels_first input into channels_last output", "ex", xf, out((2, 3, 16, 136), torch.float16, cl=True), 0, None, -2),
        ("FORCE_STREAM | STREAM_TMA with a generic epilogue", "ex", xf, out((2, 3, 16, 136), torch.float16),
         capi.FLAG_FORCE_STREAM | capi.FLAG_STREAM_TMA, None, -2),
        ("FORCE_STREAM without a generic streaming variant (narrow fp32 rows)", "ex", xn, out((1, 3, 8, 32), torch.float16),
         capi.FLAG_FORCE_STREAM, None, -2),
    ]
    for what, fn, x, o, flags, sc, want in cases:
        before = o.clone()
        rc = _rc(capi, fn, x, o, flags, sc, None if sc is None else [0.0] * len(sc))
        torch.cuda.synchronize()
        assert rc == want, (what, rc, capi.lib().aa_last_error().decode())
        assert torch.equal(_bits(o), _bits(before)), (what, "wrote the output")


# ---- entry points ------------------------------------------------------------------------------------------------------
@pytest.mark.gpu
def test_ragged_epilogue(cuda):
    """aa_resize_forward_ragged with an epilogue: HWC images -> planar fp16 / bf16 with the affine map, planar images with
    the affine map (the per-channel split runs inside each size-class group), uint8 output; launch counts."""
    from interpolate_antialiasing_b200 import capi
    g = torch.Generator().manual_seed(31)
    osize = (36, 48)
    pool = torch.randint(0, 256, (3, 60, 80, 3), dtype=torch.uint8, generator=g).to(cuda)
    hwc = [pool[0], pool[1], pool[2], torch.randint(0, 256, (90, 120, 3), dtype=torch.uint8, generator=g).to(cuda),
           torch.randint(0, 256, (24, 30, 3), dtype=torch.uint8, generator=g).to(cuda)]   # 3 launches: pool, then one each
    bases = [ref_forward(im.permute(2, 0, 1)[None].cpu().numpy(), osize, "cubic") for im in hwc]
    for kind in ("f16", "bf16", "f32"):
        o = torch.full((len(hwc), 3) + osize, float("nan"), dtype=_odtype(kind), device=cuda)
        o, launches = capi.resize_forward_ragged(hwc, osize, "cubic", out=o, scale=SCALE_F[:3], bias=BIAS_F[:3])
        torch.cuda.synchronize()
        assert launches == 3, (kind, launches)
        for i, b in enumerate(bases):
            ref = affine_ref(b, SCALE_F, BIAS_F)
            assert_rounded(got64(o[i:i + 1]), ref, fast_eps(b, ref, SCALE_F), kind, ("ragged hwc", kind, i))
    for kind in ("u8", "u8r"):   # HWC -> planar uint8, no affine map
        o = torch.zeros((len(hwc), 3) + osize, dtype=torch.uint8, device=cuda)
        o, launches = capi.resize_forward_ragged(hwc, osize, "cubic", out=o,
                                                 flags=capi.FLAG_ROUND_NEAREST if kind == "u8r" else 0)
        torch.cuda.synchronize()
        assert launches == 3
        for i, b in enumerate(bases):
            assert_rounded(got64(o[i:i + 1]), b, fast_eps(b, b), kind, ("ragged hwc", kind, i))
    # planar float images, affine map: two size classes, the first holds two images carved out of one pool
    ppool = (torch.rand((2, 3, 70, 90), generator=g) * 255).to(cuda)
    planar = [ppool[0], ppool[1], (torch.rand((3, 33, 47), generator=g) * 255).to(cuda)]
    for kind in ("f16", "bf16"):
        o = torch.full((3, 3) + osize, float("nan"), dtype=_odtype(kind), device=cuda)
        o, launches = capi.resize_forward_ragged(planar, osize, "linear", out=o, scale=SCALE_F[:3], bias=BIAS_F[:3])
        torch.cuda.synchronize()
        assert launches == 2, launches
        for i, im in enumerate(planar):
            b = ref_forward(im[None].cpu().numpy(), osize, "linear")
            ref = affine_ref(b, SCALE_F, BIAS_F)
            assert_rounded(got64(o[i:i + 1]), ref, fast_eps(b, ref, SCALE_F), kind, ("ragged planar", kind, i))


@pytest.mark.gpu
def test_decode_resize_normalize_and_resize_to_uint8(cuda):
    """The torch-facing entry points, one shape per kernel family.  decode_resize_normalize: HWC uint8 -> planar
    fp16/bf16/fp32 with (x/255 - mean)/std; 906*3-byte rows are 2-byte aligned (general kernel), 904*3 are 8-byte aligned
    (streaming kernel), 912*3 are 16-byte aligned (tensor-core kernel).  resize_to_uint8: uint8 and fp32 inputs."""
    import interpolate_antialiasing_b200 as aa
    g = torch.Generator().manual_seed(17)
    mean, std = [0.485, 0.456, 0.406], [0.229, 0.224, 0.225]
    scale = [1.0 / (255.0 * s) for s in std]
    bias = [-m / s for m, s in zip(mean, std)]
    dcases = [("tile", 120, 200, (240, 400), "bilinear", "aa_tile_kernel"),
              ("band", 120, 200, (100, 170), "bilinear", "aa_band_kernel"),   # 600 bytes a row: not 16-byte aligned
              ("stream", 96, 904, (24, 226), "bilinear", "aa_stream_kernel"),
              ("vmma", 96, 912, (24, 228), "bicubic", "aa_vmma_kernel"),
              ("general", 96, 906, (24, 226), "bicubic", "aa_general_kernel")]
    for name, H, W, osize, mode, fam in dcases:
        hwc = torch.randint(0, 256, (2, H, W, 3), dtype=torch.uint8, generator=g).to(cuda)
        base = ref_forward(hwc.permute(0, 3, 1, 2).cpu().numpy(), osize, {"bilinear": "linear", "bicubic": "cubic"}[mode])
        ref = affine_ref(base, scale, bias)
        for kind in ("f16", "bf16", "f32"):
            y, fams = launched(lambda: aa.decode_resize_normalize(hwc, osize, mean, std, mode, _odtype(kind)))
            assert y.shape == (2, 3) + osize and y.dtype == _odtype(kind) and y.is_contiguous()
            assert_rounded(got64(y), ref, fast_eps(base, ref, scale), kind, ("decode_resize_normalize", name, kind))
            assert_route(fams, [fam], 1, ("decode_resize_normalize", name, kind), fast=fam != "aa_general_kernel")
    ucases = [("tile", torch.uint8, False, (1, 3, 60, 80), (120, 150), "bilinear", "aa_tile_kernel"),
              ("band", torch.float32, True, (1, 3, 80, 100), (64, 80), "bilinear", "aa_band_kernel"),
              ("stream", torch.float32, False, (2, 3, 96, 640), (24, 160), "bicubic", "aa_stream_kernel"),
              ("vmma", torch.uint8, True, (2, 3, 128, 160), (32, 40), "bicubic", "aa_vmma_kernel"),
              ("general", torch.uint8, False, (1, 1, 96, 906), (24, 226), "bicubic", "aa_general_kernel")]  # 906-byte rows
    for name, dt, cl, shape, osize, mode, fam in ucases:
        xs = torch.randint(0, 256, shape, dtype=torch.uint8, generator=g).to(dt)
        base = ref_forward(xs.numpy(), osize, {"bilinear": "linear", "bicubic": "cubic"}[mode])
        x = _input(xs.to(cuda), "cl" if cl else "cf")
        for rn in (False, True):
            y, fams = launched(lambda: aa.resize_to_uint8(x, osize, mode, False, round_nearest=rn))
            assert y.dtype == torch.uint8
            assert_rounded(got64(y), base, fast_eps(base, base), "u8r" if rn else "u8", ("resize_to_uint8", name, rn))
            assert_route(fams, [fam], 1, ("resize_to_uint8", name, rn), fast=fam != "aa_general_kernel")


# ---- the rounding helper itself (no GPU) ---------------------------------------------------------------------------------
def test_rounding_helper():
    """rne() against numpy's float16 conversion (random doubles, every float16 midpoint, 65504 / 65520, the subnormal
    range) and torch's float32 -> bfloat16 conversion (float32-exact inputs); the two uint8 rules."""
    rng = np.random.default_rng(0)
    # float16: random doubles over the whole range, including subnormals and values past the largest finite one
    x = np.concatenate([rng.standard_normal(20000) * 10.0 ** rng.uniform(-9, 5.2, 20000),
                        rng.uniform(-70000, 70000, 20000), rng.uniform(-2.0 ** -14, 2.0 ** -14, 20000)])
    with np.errstate(over="ignore"):
        assert np.array_equal(rne(x, *F16), x.astype(np.float16).astype(np.float64))
    # every midpoint between neighbouring finite float16 values (subnormal ones included), both signs, and the overflow
    # threshold 65520 (midpoint of 65504 and 65536): ties go to the even neighbour, 65520 to inf
    h = np.arange(0, 0x7C00, dtype=np.uint16).view(np.float16).astype(np.float64)
    mids = np.concatenate([(h[:-1] + h[1:]) / 2, [65520.0, 65519.99999, 65504.0, 65505.0, 2.0 ** -25, 2.0 ** -26]])
    mids = np.concatenate([mids, -mids])
    with np.errstate(over="ignore"):
        want = mids.astype(np.float16).astype(np.float64)
    assert np.array_equal(rne(mids, *F16), want)
    assert rne(65520.0, *F16) == np.inf and rne(65519.99, *F16) == 65504.0 and rne(-65520.0, *F16) == -np.inf
    assert rne(2.0 ** -25, *F16) == 0.0 and rne(3 * 2.0 ** -25, *F16) == 2.0 ** -23   # subnormal ties to even
    # bfloat16: torch's float32 -> bfloat16 (round to nearest even) on float32-exact inputs: random bit patterns (finite),
    # and every bfloat16 midpoint of a sample of exponents (exactly representable in float32)
    bits = rng.integers(0, 2 ** 32, 200000, dtype=np.uint64).astype(np.uint32)
    f = bits.view(np.float32)
    f = f[np.isfinite(f)]
    b = np.arange(0, 0x7F80, 7, dtype=np.uint32)
    lo = (b << 16).view(np.float32).astype(np.float64)
    hi = ((b + 1) << 16).view(np.float32).astype(np.float64)
    f = np.concatenate([f, ((lo + hi) / 2).astype(np.float32), -((lo + hi) / 2).astype(np.float32),
                        np.float32([3.4028235e38, -3.4028235e38, 3.3895314e38, 1e-45, 1.1754942e-38])])
    want = torch.from_numpy(f).to(torch.bfloat16).to(torch.float64).numpy()
    assert np.array_equal(rne(f.astype(np.float64), *BF16), want)
    # uint8: clamp, then truncate or add 0.5 and truncate (halves round up)
    v = np.array([-3.0, -0.4, 0.0, 0.49999, 0.5, 1.5, 2.5, 127.99, 254.5, 254.9999, 255.0, 255.5, 300.0])
    assert np.array_equal(to_u8(v, False), [0, 0, 0, 0, 0, 1, 2, 127, 254, 254, 255, 255, 255])
    assert np.array_equal(to_u8(v, True), [0, 0, 0, 0, 1, 2, 3, 128, 255, 255, 255, 255, 255])
    # the acceptance window: one step either side only near a boundary
    assert_rounded(np.array([2048.0]), np.array([2049.0]), 0.0, "f16", "tie to even")
    with pytest.raises(AssertionError):
        assert_rounded(np.array([2050.0]), np.array([2049.0]), 0.0, "f16", "tie away from even")
    with pytest.raises(AssertionError):
        assert_rounded(np.array([1.0]), np.array([1.7]), 0.01, "u8r", "truncated instead of rounded")
