"""Randomised parity fuzz on a GPU box: random shapes / scales / layouts / dtypes / paths against the oracle.
usage: python scripts/fuzz_parity.py [seconds] [seed]"""
import os, sys, time, random
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch
from interpolate_antialiasing_b200 import capi
from oracle import aa_oracle as O

budget = float(sys.argv[1]) if len(sys.argv) > 1 else 120.0
seed = int(sys.argv[2]) if len(sys.argv) > 2 else 0
rnd = random.Random(seed)
g = torch.Generator().manual_seed(seed)
dev = torch.device("cuda", 0)
t0 = time.time()
n = fails = n_af = 0  # n_af: fast-path results compared bit for bit with their FLAG_ASSUME_FINITE run
paths = {"auto": capi.FLAG_AUTO, "stream": capi.FLAG_FORCE_STREAM, "tma": capi.FLAG_FORCE_STREAM | capi.FLAG_STREAM_TMA,
         "general": capi.FLAG_FORCE_GENERAL}
stats = {k: 0 for k in paths}
# Shared memory is not cleared between kernels: resizing all-NaN tensors through every fast kernel right before a
# case leaves NaNs behind, so any read of uninitialised shared memory (e.g. a zero weight times a stale value)
# shows up as a non-finite output instead of passing by luck.
poison = [torch.full((2, 3, 192, 256), float("nan"), device=dev), torch.full((2, 3, 192, 256), float("nan"), device=dev).contiguous(memory_format=torch.channels_last)]
def poison_smem():
    for pz in poison:
        for osz in ((24, 32), (150, 200), (300, 400)):       # stream, band, tile
            capi.resize_forward(pz, osz, "cubic", False)
        capi.resize_backward(pz, (2, 3, 768, 1024), "linear", False)   # tile (adjoint)
        capi.resize_backward(pz, (2, 3, 96, 128), "linear", False)     # stream (adjoint)
while time.time() - t0 < budget:
    C = rnd.choice([1, 1, 2, 3, 3, 4, 5])
    N = rnd.choice([1, 1, 2, 3])
    H = rnd.choice([rnd.randint(1, 40), rnd.randint(40, 300), rnd.randint(300, 700)])
    W = rnd.choice([rnd.randint(1, 40), rnd.randint(40, 300), rnd.randint(300, 1400), 4 * rnd.randint(10, 300), 8 * rnd.randint(10, 200)])
    def pick(n_in):
        s = rnd.choice([0.05, 0.125, 0.2, 0.25, 0.33, 0.5, 0.6, 0.75, 0.9, 1.0, 1.1, 1.5, 2.0, 3.0, rnd.uniform(0.03, 3.0)])
        return max(1, min(2000, round(n_in * s)))
    oH, oW = pick(H), pick(W)
    if N * C * (H * W + oH * oW) > 6e6:
        continue
    mode = rnd.choice(["linear", "linear", "cubic", "cubic", "nearest"])
    align = rnd.random() < 0.25
    cl = rnd.random() < 0.5
    dt = rnd.choice([torch.float32, torch.float32, torch.uint8, torch.float64])
    x = (torch.rand((N, C, H, W), generator=g, dtype=torch.float64) * 255).to(dt)
    nonfinite = dt == torch.float32 and rnd.random() < 0.3  # a few NaN/Inf pixels: their placement must be the oracle's
    if nonfinite:
        for _ in range(rnd.randint(1, 4)):
            x[rnd.randrange(N), rnd.randrange(C), rnd.randrange(H), rnd.randrange(W)] = rnd.choice([float("nan"), float("inf"), float("-inf")])
    ref_in = x.double().numpy() if dt == torch.float64 else x.float().numpy()
    want = O.forward(ref_in, (oH, oW), mode, align)
    xc = x.to(dev)
    if cl:
        xc = xc.contiguous(memory_format=torch.channels_last)
    for pname, fl in paths.items():
        if dt == torch.float64 and pname in ("stream", "tma"):
            continue
        if n % 4 == 0:
            poison_smem()
        try:
            y = capi.resize_forward(xc, (oH, oW), mode, align, fl)
            torch.cuda.synchronize()
        except capi.AAError as e:
            if "-2" in str(e) and pname in ("stream", "tma"):
                continue
            print("ERROR", pname, (N, C, H, W), (oH, oW), mode, align, cl, dt, e); fails += 1; continue
        got = y.cpu().numpy()
        n += 1; stats[pname] += 1
        if dt == torch.float32 and not nonfinite and pname != "general":
            # the drain kernel behind the fast float kernels recomputes whatever stored a NaN/Inf, so a stale NaN read from
            # shared memory would be repaired there: without it (FLAG_ASSUME_FINITE) the result must be the same bits
            poison_smem()
            ya = capi.resize_forward(xc, (oH, oW), mode, align, fl | capi.FLAG_ASSUME_FINITE)
            torch.cuda.synchronize()
            n_af += 1
            if not torch.equal(ya, y):
                fails += 1
                print("ASSUME_FINITE MISMATCH", pname, (N, C, H, W), (oH, oW), mode, align, cl, int((~torch.isfinite(ya)).sum()))
        if nonfinite:
            wbad = ~np.isfinite(want)
            ok = np.array_equal(~np.isfinite(got), wbad)
            if ok and pname == "general":
                ok = np.array_equal(got[~wbad], want[~wbad])
            elif ok:
                ok = bool(np.all(np.abs(got[~wbad].astype(np.float64) - want[~wbad]) <= 1e-3 + 1e-5 * np.abs(want[~wbad])))
            if not ok:
                fails += 1
                print("NONFINITE MISMATCH", pname, (N, C, H, W), (oH, oW), mode, align, cl, int((~np.isfinite(got)).sum()), int(wbad.sum()))
            continue
        if pname == "general":
            ok = np.array_equal(got, want)
        else:
            tol = (1e-3 + 1e-5 * np.abs(want)) if dt != torch.float64 else (1e-9 + 1e-12 * np.abs(want))
            ok = bool(np.all(np.abs(got.astype(np.float64) - want) <= tol))
        if not ok or not np.isfinite(got).all():
            fails += 1
            print("MISMATCH", pname, (N, C, H, W), (oH, oW), mode, align, cl, dt, float(np.abs(got.astype(np.float64) - want).max()))
    # backward (true adjoint) on a fraction of cases
    if dt != torch.uint8 and not nonfinite and rnd.random() < 0.4:
        go = torch.rand((N, C, oH, oW), generator=g, dtype=torch.float64).to(dt)
        gnf = dt == torch.float32 and rnd.random() < 0.3  # non-finite gradients: placement must be the oracle's
        if gnf:
            for _ in range(rnd.randint(1, 3)):
                go[rnd.randrange(N), rnd.randrange(C), rnd.randrange(oH), rnd.randrange(oW)] = rnd.choice([float("nan"), float("inf"), float("-inf")])
        wantg = O.backward_adjoint(go.numpy(), (N, C, H, W), mode, align)
        gc = go.to(dev)
        if cl:
            gc = gc.contiguous(memory_format=torch.channels_last)
        poison_smem()
        gi = capi.resize_backward(gc, (N, C, H, W), mode, align)
        torch.cuda.synchronize()
        n += 1
        if dt == torch.float32 and not gnf:
            poison_smem()
            gia = capi.resize_backward(gc, (N, C, H, W), mode, align, flags=capi.FLAG_ASSUME_FINITE)
            torch.cuda.synchronize()
            n_af += 1
            if not torch.equal(gia, gi):
                fails += 1
                print("BWD ASSUME_FINITE MISMATCH", (N, C, H, W), (oH, oW), mode, align, cl, int((~torch.isfinite(gia)).sum()))
        if gnf:
            gbad = ~np.isfinite(wantg)
            gnp = gi.cpu().numpy()
            if not np.array_equal(~np.isfinite(gnp), gbad) or not np.allclose(gnp[~gbad], wantg[~gbad], rtol=1e-5, atol=4e-6):
                fails += 1
                print("BWD NONFINITE MISMATCH", (N, C, H, W), (oH, oW), mode, align, cl, int((~np.isfinite(gnp)).sum()), int(gbad.sum()))
        elif not np.allclose(gi.cpu().numpy(), wantg, rtol=1e-5, atol=4e-6 if dt == torch.float32 else 1e-11):
            fails += 1
            print("BWD MISMATCH", (N, C, H, W), (oH, oW), mode, align, cl, dt, float(np.abs(gi.cpu().numpy() - wantg).max()))
print(f"fuzz: {n} checks in {time.time() - t0:.0f}s, {fails} failures, per path {stats}, {n_af} ASSUME_FINITE comparisons")
sys.exit(1 if fails else 0)
