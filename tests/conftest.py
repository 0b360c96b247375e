import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

GOLDEN_DIR = os.path.join(ROOT, "tests", "golden")


def pytest_configure(config):
    config.addinivalue_line("markers", "gpu: needs a CUDA device (run on the B200 box with -m gpu)")


@pytest.fixture(scope="session")
def golden():
    """The stored golden vectors (see tests/golden/make_golden.py).  The seeded inputs of the small cases are not
    stored: they are drawn again here in the generator's order and must match the sha256 recorded with them."""
    import hashlib
    import torch
    g = {}
    for name in ("golden_v1.npz", "golden_v1_fp64.npz", "reference_checks_v1.npz"):
        with np.load(os.path.join(GOLDEN_DIR, name)) as z:
            g.update({k: z[k] for k in z.files})
    gen = torch.Generator().manual_seed(1234)
    for i in range(int(g["n_cases"])):
        shape, dt = tuple(int(v) for v in g[f"case{i}_shape"]), getattr(torch, str(g[f"case{i}_dtype"]))
        osize = tuple(int(v) for v in g[f"case{i}_osize"])
        for key, shp, scale in (("x", shape, 255), ("gout", shape[:2] + osize, 1)):
            a = (torch.rand(shp, generator=gen, dtype=dt) * scale).numpy()
            assert hashlib.sha256(a.tobytes()).hexdigest() == str(g[f"case{i}_{key}_sha256"]), (i, key)
            g[f"case{i}_{key}"] = a
    return g


@pytest.fixture(scope="session")
def photo():
    """The reference's fixture image (data/test.png as RGB), uint8 [438, 906, 3]."""
    return np.load(os.path.join(GOLDEN_DIR, "photo_438x906.npz"))["rgb"]


@pytest.fixture(scope="session")
def ref_ext():
    """The unmodified reference extension (oracle/_ref), or skip when the prebuilt .so is absent."""
    from oracle.ref_ext import load_ref
    m = load_ref(build_if_missing=os.path.exists("/root/reference"))
    if m is None:
        pytest.skip("oracle/_ref not built")
    return m


@pytest.fixture(scope="session")
def cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    return torch.device("cuda", 0)
