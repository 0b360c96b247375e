"""CPU-only checks of the boundary: the C-ABI library loads and exports every symbol the header
declares, host-only queries agree with the oracle, and argument errors come back as status codes
(no compute call is made here: there is no GPU in the build container and no CPU fallback)."""
import ctypes
import os
import random
import re

import numpy as np
import pytest

from oracle import aa_oracle as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _declared_functions():
    src = open(os.path.join(ROOT, "include", "aa_resize.h")).read()
    src = re.sub(r"/\*.*?\*/", "", src, flags=re.S)
    return sorted(set(re.findall(r"\b(aa_[a-z0-9_]+)\s*\(", src)))


def test_header_symbols_exported():
    from interpolate_antialiasing_b200 import capi
    L = capi.lib()
    names = _declared_functions()
    assert len(names) >= 11
    assert set(names) == set(capi.EXPORTS)
    for n in names:
        assert hasattr(L, n), f"{n} declared in include/aa_resize.h but not exported"
    assert L.aa_abi_version() == 2


def test_flag_constants_match_header():
    """The ctypes binding's flag values are the header's #defines (a drifted constant would silently select another path)."""
    from interpolate_antialiasing_b200 import capi
    src = open(os.path.join(ROOT, "include", "aa_resize.h")).read()
    flags = {m.group(1): int(m.group(2)) for m in re.finditer(r"#define\s+AA_FLAG_(\w+)\s+(\d+)u", src)}
    assert len(flags) >= 9
    for name, val in flags.items():
        assert getattr(capi, "FLAG_" + name) == val, name
    assert len(set(v for v in flags.values() if v)) == len([v for v in flags.values() if v])  # distinct bits


def test_no_oracle_in_product_path():
    """The product must not route through the oracle or any CPU fallback."""
    pkg = os.path.join(ROOT, "interpolate_antialiasing_b200")
    for dp, _, fs in os.walk(pkg):
        if "_build" in dp:
            continue
        for f in fs:
            if f.endswith((".py", ".cu", ".cuh", ".cpp", ".h")):
                txt = open(os.path.join(dp, f)).read()
                assert "aa_oracle" not in txt and "from oracle" not in txt and "import oracle" not in txt, f


def test_interp_size_matches_oracle():
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(9)
    for _ in range(2000):
        a, b = rnd.randint(1, 6000), rnd.randint(1, 6000)
        mode = rnd.choice(["linear", "cubic", "nearest"])
        align = rnd.random() < 0.5
        assert capi.interp_size(a, b, mode, align, capi.F32) == O.interp_size(a, b, mode, align, np.float32)
        assert capi.interp_size(a, b, mode, align, capi.F64) == O.interp_size(a, b, mode, align, np.float64)


def test_host_tables_match_oracle():
    """The host-side integer tables the launch planners use (aa_host_tables) are bit-identical to the oracle's
    restatement of aa_interpolation_impl.h:253-257, with and without a caller-provided scale factor."""
    from interpolate_antialiasing_b200 import capi
    rnd = random.Random(11)
    cases = [(906, 320), (438, 196), (1920, 224), (1080, 224), (3840, 512), (2160, 512), (512, 128), (64, 10), (1, 1), (5, 1), (1, 7)]
    cases += [(rnd.randint(1, 4000), rnd.randint(1, 3000)) for _ in range(300)]
    for a, b in cases:
        mode = rnd.choice(["linear", "cubic", "nearest"])
        align = rnd.random() < 0.3
        for code, ndt in ((capi.F32, np.float32), (capi.F64, np.float64)):
            for scale in (None, b / a * rnd.uniform(0.9, 1.1)):
                xm, xs = capi.host_tables(a, b, mode, align, code, scale)
                oxm, oxs, _ = O.tables(a, b, mode, align, ndt, scale)
                assert np.array_equal(xm, oxm) and np.array_equal(xs, oxs), (a, b, mode, align, code, scale)


def test_argument_errors_are_status_codes():
    from interpolate_antialiasing_b200 import capi
    L = capi.lib()
    k = ctypes.c_int32(0)
    assert L.aa_interp_size(0, 10, 1, 0, 1, ctypes.byref(k)) == -1
    assert b"bad arguments" in L.aa_last_error()
    assert L.aa_interp_size(10, 10, 9, 0, 1, ctypes.byref(k)) == -1
    d = capi.TensorDesc(None, capi.F32, 0, 1, 3, 0, 8, 0, 0, 0, 0)   # h == 0
    o = capi.TensorDesc(None, capi.F32, 0, 1, 3, 4, 4, 48, 16, 4, 1)
    assert L.aa_resize_forward(ctypes.byref(d), ctypes.byref(o), 1, 0, 0, None) == -1
    assert b"Non-empty 4D data tensor expected" in L.aa_last_error()
    assert L.aa_resize_forward(None, ctypes.byref(o), 1, 0, 0, None) == -1
    d = capi.TensorDesc(None, capi.F32, 0, 0, 3, 8, 8, 192, 64, 8, 1)   # empty batch: OK, no device touched
    o = capi.TensorDesc(None, capi.F32, 0, 0, 3, 4, 4, 48, 16, 4, 1)
    assert L.aa_resize_forward(ctypes.byref(d), ctypes.byref(o), 1, 0, 0, None) == 0
    assert L.aa_resize_backward(ctypes.byref(o), ctypes.byref(d), 1, 0, 0, None) == 0
    o = capi.TensorDesc(None, capi.F64, 0, 0, 3, 4, 4, 48, 16, 4, 1)    # dtype mismatch
    assert L.aa_resize_forward(ctypes.byref(d), ctypes.byref(o), 1, 0, 0, None) == -1


def test_product_fails_loudly_without_gpu():
    import torch
    import interpolate_antialiasing_b200 as aa
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        aa.linear_forward(torch.rand(1, 3, 8, 8), (4, 4), False)
    # the C ABI itself reports a CUDA error rather than computing on the host
    x = torch.rand(1, 3, 8, 8); y = torch.empty(1, 3, 4, 4)
    di, do = aa.capi.desc(x, 0), aa.capi.desc(y, 0)
    rc = aa.capi.lib().aa_resize_forward(ctypes.byref(di), ctypes.byref(do), 1, 0, 0, None)
    assert rc in (-3, -4) and b"CUDA error" in aa.capi.lib().aa_last_error()


def test_extension_exports_reference_names():
    import interpolate_antialiasing_b200 as aa
    m = aa.load()
    # /root/reference/step_two_dot_two/extension_interpolate.cpp:46-51
    for name in ("linear_forward", "nearest_forward", "cubic_forward", "linear_backward"):
        assert callable(getattr(m, name))


def test_stream_kernels_issue_row_loads_before_first_fma():
    """scripts/sass_lint.py on the built library: in every streaming-kernel instantiation the U input rows of
    a batch are requested before the first FMA (ptxas sinks loads when the register budget of a shape is too
    tight, which costs ~15 % on the headline config).  The 6-accumulator uint8 shape is the known exception."""
    import subprocess, sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "scripts", "sass_lint.py")], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    flagged = [l for l in r.stdout.splitlines() if "<--" in l]
    assert flagged and all(l.startswith("A=6 VEC=8 h") for l in flagged) or not flagged, "\n".join(flagged)
    assert any(l.startswith("A=3 VEC=4 f NT=256 U=4 GEN=0 PAD=0 PF=0: 4 data loads") for l in r.stdout.splitlines())
    assert any(l.startswith("A=3 VEC=4 f NT=256 U=4 GEN=0 PAD=0 PF=1: 4 data loads") for l in r.stdout.splitlines())


def test_sass_of_the_built_kernels():
    """What the built sm_100a library actually contains (cuobjdump on the .so, no GPU needed):
    the uint8 kernel issues tcgen05 MMAs (UTCIMMA), TMA tensor copies (UTMALDG) and TMEM loads (LDTM); the drain kernel
    that follows every fast float launch exists and waits on its programmatic dependency (ACQBULK = griddepcontrol.wait; the float
    tile kernels trigger it with PREEXIT = griddepcontrol.launch_dependents);
    the headline streaming instantiation keeps everything in registers (no local-memory loads or stores)."""
    import shutil, subprocess
    from interpolate_antialiasing_b200 import capi
    cuobjdump = shutil.which("cuobjdump") or os.path.join(os.environ.get("CUDA_HOME", "/usr/local/cuda"), "bin", "cuobjdump")
    out = subprocess.run([cuobjdump, "-sass", capi.LIB], capture_output=True, text=True, timeout=600, check=True).stdout
    funcs, cur = {}, None
    for line in out.splitlines():
        m = re.search(r"Function : (\S+)", line)
        if m:
            cur = m.group(1)
            funcs[cur] = []
        elif cur and re.match(r"\s+/\*[0-9a-f]{4}\*/", line):
            funcs[cur].append(line.split("*/", 1)[1].strip())
    vmma = [f for f in funcs if "aa_vmma_kernel" in f]
    assert vmma
    for f in vmma:
        text = "\n".join(funcs[f])
        assert "UTCIMMA" in text and "UTMALDG" in text and "LDTM" in text, f
    redo = [f for f in funcs if "aa_redo_kernel" in f]
    assert len(redo) == 2
    assert all(any(i.startswith("ACQBULK") for i in funcs[f]) for f in redo)                 # griddepcontrol.wait
    tile_f32 = [f for f in funcs if "aa_tile_kernel" in f and re.search(r"ELb0EfE", f)]
    assert tile_f32 and all(any(i.startswith("PREEXIT") for i in funcs[f]) for f in tile_f32)  # griddepcontrol.launch_dependents
    head = [f for f in funcs if re.search(r"aa_stream_kernelILi3ELi4EfLi256ELi4ELi4ELb0ELb0ELb0E", f)]
    assert len(head) == 1
    assert not any(i.startswith(("LDL", "STL")) for i in funcs[head[0]]), "the cfg2 streaming kernel spills"
