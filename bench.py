#!/usr/bin/env python
"""bench.py -- the driver's benchmark contract for the anti-aliased resize hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--config cfg2|cfg3|cfg4] [--no-sub]
                    [--dump-outputs DIR]

One "step" = one pass of the hot path over one batch of synthetic images.  The headline workload
(BASELINE.json configs[1], "cfg2") is fp32 [256,3,1080,1920] channels_last -> (224,224) bilinear
antialias; each rank processes one such batch (weak scaling, no data-path collective; NCCL is used
only for the barrier and the max-over-ranks of the device time).

Prints ONE JSON line on rank 0:
  value     whole-job Mpix/s (pixels = N*(H*W + oH*oW), channels not counted) with inputs resident in HBM
  e2e       the same metric through the C ABI's host-buffer entry point (aa_resize_forward_host):
            pinned host input -> H2D -> kernel -> D2H of the result, all inside the timed region
  roofline  algorithmic bytes per launch / measured kernel time, against MEASURED_PEAKS.json hbm_gbs
  cpu_baseline  the UNMODIFIED reference extension (oracle/_ref) timed on this box's host cores on a
            bounded sample of the same workload (rank 0, N=1 only)

  sub       (default run only) the other BASELINE.json configs on the same box, same timing rules:
            cfg1 (launch-bound: eager + CUDA-graph replay + cold call for a never-seen size), cfg3 (uint8 bicubic, device
            + uint8 e2e), cfg4 (backward; "cold" rotates over 8 grad buffers so L2 cannot absorb the stream, "warm" reuses
            one), cfg5 (scale sweep: fp32 forward, mixed h/w pairs, uint8 input, backward), strong (the fixed 256-image
            cfg2 batch split over the N ranks) and, at N > 1, shard_equal (gathered shard outputs bitwise equal to rank 0
            recomputing the same images).

--impl reference times only the reference's CPU implementation (all host threads) and prints the
same line with "impl": "reference".

--dump-outputs DIR writes, on rank 0, what the timed path returned in its last step as DIR/<name>.npy (NCHW,
float32): "output" for a forward config, "grad_input" for cfg4.  Inputs are seeded, so two builds run with the
same arguments can be compared output for output.  An output above DUMP_BYTES keeps a fixed, seeded sample of
its images (the line's "dump" object says which).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

CONFIGS = {
    # name: (N, C, H, W, oH, oW, mode, in_dtype, channels_last, kind)
    "cfg1": dict(N=1, C=3, H=438, W=906, oH=196, oW=320, mode="linear", dtype="f32", cl=False, kind="forward",
                 workload="cfg1: fp32 [1,3,438,906] channels_first -> (196,320) bilinear antialias, forward (the README test)"),
    "cfg2": dict(N=256, C=3, H=1080, W=1920, oH=224, oW=224, mode="linear", dtype="f32", cl=True, kind="forward",
                 workload="cfg2: fp32 [256,3,1080,1920] channels_last -> (224,224) bilinear antialias, forward"),
    "cfg3": dict(N=128, C=3, H=2160, W=3840, oH=512, oW=512, mode="cubic", dtype="u8", cl=False, kind="forward",
                 workload="cfg3: uint8->fp32 [128,3,2160,3840] channels_first -> (512,512) bicubic antialias, forward"),
    "cfg4": dict(N=64, C=3, H=512, W=512, oH=128, oW=128, mode="linear", dtype="f32", cl=False, kind="backward",
                 workload="cfg4: backward of bilinear antialias [64,3,512,512] -> (128,128): grad_out [64,3,128,128] -> grad_in"),
}
METRIC = "Mpix/s (input+output pixels), AA bilinear/bicubic resize, and fraction of HBM peak"
DUMP_BYTES = 32 << 20


def mpix(cfg, n_images=None):
    n = cfg["N"] if n_images is None else n_images
    return n * (cfg["H"] * cfg["W"] + cfg["oH"] * cfg["oW"]) / 1e6


def algorithmic_bytes(cfg, n_images=None):
    """SURVEY 8(d): input read once + output written once (no temp, tables or halo)."""
    n = cfg["N"] if n_images is None else n_images
    ies = 1 if cfg["dtype"] == "u8" else 4
    if cfg["kind"] == "forward":
        return n * cfg["C"] * (cfg["H"] * cfg["W"] * ies + cfg["oH"] * cfg["oW"] * 4)
    return n * cfg["C"] * (cfg["oH"] * cfg["oW"] + cfg["H"] * cfg["W"]) * 4


def measured_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def recorded_traffic(name):
    """dram bytes per launch from the committed ncu --set full capture (profiles/traffic.json), or None."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    try:
        return json.load(open(p)).get(name, {}).get("dram_bytes_per_launch")
    except Exception:
        return None


class ClockSampler:
    """Samples nvidia-smi clocks / throttle reasons of one GPU while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.rows, self.proc, self.thr = index, [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thr = threading.Thread(target=self._read, daemon=True)
            self.thr.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            try:
                sm.append(float(r[0])); mx.append(float(r[1]))
                for n, v in zip(names, r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(n)
            except Exception:
                continue
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def bind_to_gpu_numa_node(torch, local_rank):
    """Pin this process to the CPU cores local to its GPU (sysfs local_cpulist) so that the pinned host
    buffers of the e2e leg are first-touched on the GPU's NUMA node.  Best effort; returns a note."""
    try:
        pr = torch.cuda.get_device_properties(local_rank)
        bus = "%04x:%02x:%02x.0" % (pr.pci_domain_id, pr.pci_bus_id, pr.pci_device_id)
        txt = open(f"/sys/bus/pci/devices/{bus}/local_cpulist").read().strip()
        cpus = set()
        for part in txt.split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if cpus:
            os.sched_setaffinity(0, cpus)
            return f"cpus {txt} (GPU {bus} local)"
    except Exception as e:  # noqa: BLE001
        return f"unbound ({type(e).__name__})"
    return "unbound"


def make_inputs(cfg, dev, torch, n_images=None):
    n = cfg["N"] if n_images is None else n_images
    g = torch.Generator(device=dev).manual_seed(0)
    if cfg["kind"] == "backward":
        return torch.rand((n, cfg["C"], cfg["oH"], cfg["oW"]), generator=g, device=dev)
    shape = (n, cfg["C"], cfg["H"], cfg["W"])
    if cfg["dtype"] == "u8":
        x = torch.randint(0, 256, shape, generator=g, device=dev, dtype=torch.uint8)
    else:
        x = torch.rand(shape, generator=g, device=dev) * 255
    if cfg["cl"]:
        x = x.contiguous(memory_format=torch.channels_last)
    return x


def dump_output(dirname, name, t):
    """Writes the [N,C,H,W] result `t` as dirname/<name>.npy; above DUMP_BYTES only a seeded sample of its images. -> dict"""
    import numpy as np
    import torch
    if t.dtype not in (torch.float32, torch.float64):
        t = t.float()
    n = t.shape[0]
    keep = min(n, max(1, DUMP_BYTES // (t[:1].numel() * t.element_size())))
    images = np.arange(n) if keep == n else np.sort(np.random.default_rng(0).permutation(n)[:keep])
    a = np.ascontiguousarray(t[torch.from_numpy(images).to(t.device)].cpu().numpy())
    os.makedirs(dirname, exist_ok=True)
    path = os.path.join(dirname, name + ".npy")
    np.save(path, a)
    return {"file": path, "shape": list(a.shape), "dtype": str(a.dtype), "images": images.tolist() if keep < n else "all"}


def cpu_reference_rate(cfg, seconds, torch, threads=None):
    """Times the UNMODIFIED reference extension (oracle/_ref) on a bounded sample of cfg. -> dict"""
    from oracle.ref_ext import load_ref
    ref = load_ref(build_if_missing=False)
    if ref is None:
        return None
    torch.set_num_threads(threads or len(os.sched_getaffinity(0)))
    cores = torch.get_num_threads()
    ns = 8 if cfg["H"] * cfg["W"] < 3e6 else 2
    g = torch.Generator().manual_seed(0)
    if cfg["kind"] == "backward":
        go = torch.rand((ns, cfg["C"], cfg["oH"], cfg["oW"]), generator=g)
        fn = lambda: ref.linear_backward(go, (cfg["oH"], cfg["oW"]), [ns, cfg["C"], cfg["H"], cfg["W"]], False)
        note = "reference linear_backward (non-AA arithmetic, SURVEY 0.2)"
    else:
        shape = (ns, cfg["C"], cfg["H"], cfg["W"])
        if cfg["dtype"] == "u8":
            xs = torch.randint(0, 256, shape, generator=g, dtype=torch.uint8)
        else:
            xs = torch.rand(shape, generator=g) * 255
        if cfg["cl"]:
            xs = xs.contiguous(memory_format=torch.channels_last)
        f = ref.linear_forward if cfg["mode"] == "linear" else ref.cubic_forward
        # uint8: the reference's caller casts first (test.py:55,67); that cast is part of its path
        fn = (lambda: f(xs.float(), (cfg["oH"], cfg["oW"]), False)) if cfg["dtype"] == "u8" else (lambda: f(xs, (cfg["oH"], cfg["oW"]), False))
        note = "reference %s_forward%s" % (cfg["mode"], " incl. .float()" if cfg["dtype"] == "u8" else "")
    fn()
    t0 = time.perf_counter(); fn(); t1 = time.perf_counter() - t0
    iters = max(2, min(200, int(seconds / max(t1, 1e-4))))
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    dt = (time.perf_counter() - t0) / iters
    return {"value": mpix(cfg, ns) / dt, "unit": "Mpix/s", "cores": cores, "kind": "reference",
            "sample": f"{ns} of {cfg['N']} images of the same workload, {iters} passes, {note}, "
                      f"torch.get_num_threads()={cores}, OMP_NUM_THREADS={os.environ.get('OMP_NUM_THREADS', 'unset')}, "
                      f"os.cpu_count()={os.cpu_count()}",
            "ms_per_pass": dt * 1e3, "images": ns}


def run_reference(args, cfg, rank, world):
    import torch
    if rank != 0:
        return
    line = {"metric": METRIC, "unit": "Mpix/s", "impl": "reference", "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": {"workload": cfg["workload"]}}
    from oracle.ref_ext import load_ref
    ref = load_ref(build_if_missing=False)
    if ref is None:
        line["unavailable"] = "oracle/_ref (compiled reference) is missing"
        print(json.dumps(line)); return
    # torchrun exports OMP_NUM_THREADS=1; the reference arm is meant to use every host thread it can
    torch.set_num_threads(len(os.sched_getaffinity(0)))
    cores = torch.get_num_threads()
    ns = 8 if cfg["H"] * cfg["W"] < 3e6 else 2
    g = torch.Generator().manual_seed(0)
    if cfg["kind"] == "backward":
        go = torch.rand((ns, cfg["C"], cfg["oH"], cfg["oW"]), generator=g)
        fn = lambda: ref.linear_backward(go, (cfg["oH"], cfg["oW"]), [ns, cfg["C"], cfg["H"], cfg["W"]], False)
    else:
        shape = (ns, cfg["C"], cfg["H"], cfg["W"])
        xs = torch.randint(0, 256, shape, generator=g, dtype=torch.uint8) if cfg["dtype"] == "u8" else torch.rand(shape, generator=g) * 255
        if cfg["cl"]:
            xs = xs.contiguous(memory_format=torch.channels_last)
        f = ref.linear_forward if cfg["mode"] == "linear" else ref.cubic_forward
        fn = (lambda: f(xs.float(), (cfg["oH"], cfg["oW"]), False)) if cfg["dtype"] == "u8" else (lambda: f(xs, (cfg["oH"], cfg["oW"]), False))
    for _ in range(args.warmup):
        fn()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        fn()
    dt = (time.perf_counter() - t0) / args.steps
    v = mpix(cfg, ns) / dt
    sample = (f"each step = {ns} of {cfg['N']} images of the workload through the unmodified reference extension "
              f"(oracle/_ref, -O3) on {cores} host threads; os.cpu_count()={os.cpu_count()}, "
              f"OMP_NUM_THREADS={os.environ.get('OMP_NUM_THREADS', 'unset')}")
    line.update({"value": v, "ms_per_step": dt * 1e3,
                 "cpu_baseline": {"value": v, "unit": "Mpix/s", "cores": cores, "kind": "reference", "sample": sample},
                 "e2e": {"value": v, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
    print(json.dumps(line))


def time_steps(torch, step, steps):
    """CUDA events on the launching (current) stream around each of `steps` back-to-back calls -> (total_ms, sorted per-step ms)"""
    evs = [torch.cuda.Event(enable_timing=True) for _ in range(steps + 1)]
    evs[0].record()
    for i in range(steps):
        step(i)
        evs[i + 1].record()
    torch.cuda.synchronize()
    return evs[0].elapsed_time(evs[-1]), sorted(evs[i].elapsed_time(evs[i + 1]) for i in range(steps))


def reduce_max(torch, dist, world, dev, v):
    if world <= 1:
        return v
    t = torch.tensor([v], device=dev, dtype=torch.float64)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def pinned_like(torch, cfg, x, out):
    if cfg["cl"]:
        xh = torch.empty((x.shape[0], cfg["H"], cfg["W"], cfg["C"]), dtype=x.dtype, pin_memory=True).permute(0, 3, 1, 2)
        oh = torch.empty((x.shape[0], cfg["oH"], cfg["oW"], cfg["C"]), dtype=out.dtype, pin_memory=True).permute(0, 3, 1, 2)
    else:
        xh = torch.empty(x.shape, dtype=x.dtype, pin_memory=True)
        oh = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
    return xh, oh


def measure_e2e(torch, dist, capi, cfg, x, out, dev, local_rank, world, barrier, steps, numa_note):
    """aa_resize_forward_host on pinned host buffers (copies inside the timed region) and, beside it, the ceiling: the same
    bytes moved by plain pinned cudaMemcpyAsync H2D + D2H with no kernel, all ranks concurrently."""
    xh, oh = pinned_like(torch, cfg, x, out)
    xh.copy_(x)
    for _ in range(2):
        capi.resize_forward_host(xh, oh, cfg["mode"], False, capi.FLAG_AUTO, device=local_rank)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        capi.resize_forward_host(xh, oh, cfg["mode"], False, capi.FLAG_AUTO, device=local_rank)
    torch.cuda.synchronize()
    dt = reduce_max(torch, dist, world, dev, time.perf_counter() - t0) / steps
    ok = bool(torch.allclose(oh.to(dev), out, rtol=1e-5, atol=1e-3))
    # ceiling probe: the copies alone
    xd = torch.empty_like(x)
    for _ in range(2):
        xd.copy_(xh, non_blocking=True); oh.copy_(out, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(max(2, steps // 2)):
        xd.copy_(xh, non_blocking=True)
        oh.copy_(out, non_blocking=True)
    torch.cuda.synchronize()
    ceil = reduce_max(torch, dist, world, dev, time.perf_counter() - t0) / max(2, steps // 2)
    h2d, d2h = xh.numel() * xh.element_size(), oh.numel() * oh.element_size()
    del xh, oh, xd
    return {"value": world * mpix(cfg, x.shape[0]) / dt, "unit": "Mpix/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
            "ms_per_step": dt * 1e3, "steps": steps, "api": "aa_resize_forward_host (C ABI, pinned host buffers)",
            "matches_device_result": ok, "host_affinity": numa_note,
            "h2d_ceiling_ms": ceil * 1e3, "h2d_ceiling_gbs_per_gpu": (h2d + d2h) / ceil / 1e9,
            "frac_of_copy_ceiling": ceil / dt,
            "ceiling_probe": "plain pinned cudaMemcpyAsync of the same H2D + D2H bytes, no kernel, all ranks concurrently"}


def sub_cfg1(torch, capi, dev, peak):
    """launch-bound: eager call, CUDA-graph replay, and the cold call for a size the table cache has never seen"""
    cfg = CONFIGS["cfg1"]
    x = make_inputs(cfg, dev, torch)
    osize = (cfg["oH"], cfg["oW"])
    out = capi.resize_forward(x, osize, cfg["mode"], False)
    for _ in range(5):
        capi.resize_forward(x, osize, cfg["mode"], False, out=out)
    torch.cuda.synchronize()
    tot, _ = time_steps(torch, lambda i: capi.resize_forward(x, osize, cfg["mode"], False, out=out), 200)
    eager_us = tot / 200 * 1e3
    graph_us = None
    try:
        s = torch.cuda.Stream()
        with torch.cuda.stream(s):
            g = torch.cuda.CUDAGraph()
            with torch.cuda.graph(g, stream=s):
                capi.resize_forward(x, osize, cfg["mode"], False, out=out)
            g.replay(); torch.cuda.synchronize()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record(s)
            for _ in range(200):
                g.replay()
            b.record(s)
            torch.cuda.synchronize()
            graph_us = a.elapsed_time(b) / 200 * 1e3
    except Exception as e:  # noqa: BLE001
        graph_us = f"graph capture failed: {type(e).__name__}"
    # cold call: sizes never used before in this process (table-cache miss + plan), wall clock until the call returns
    # and until the result is complete
    cold_ret, cold_done = [], []
    for k in range(5):
        xc = x[:, :, : 431 - 7 * k, : 901 - 11 * k].contiguous()
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        capi.resize_forward(xc, (190 + k, 310 + k), cfg["mode"], False)
        t1 = time.perf_counter()
        torch.cuda.synchronize()
        t2 = time.perf_counter()
        cold_ret.append((t1 - t0) * 1e6); cold_done.append((t2 - t0) * 1e6)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    capi.resize_forward(x, osize, cfg["mode"], False, out=out)
    t1 = time.perf_counter()
    torch.cuda.synchronize()
    warm_done = (time.perf_counter() - t0) * 1e6
    return {"workload": cfg["workload"], "eager_us_per_call": round(eager_us, 2), "graph_replay_us": graph_us if not isinstance(graph_us, float) else round(graph_us, 2),
            "hbm_bound_us": round(algorithmic_bytes(cfg) / peak / 1e3, 3),
            "cold_call_us": {"returns_after_median": round(statistics.median(cold_ret), 1), "complete_after_median": round(statistics.median(cold_done), 1),
                             "what": "first call for a never-seen (H,W)->(oH,oW): host-side table build + 2x2 table kernels + plan, no synchronisation"},
            "warm_call_us": {"returns_after": round((t1 - t0) * 1e6, 1), "complete_after": round(warm_done, 1)}}


def sub_forward(torch, dist, capi, name, dev, local_rank, world, barrier, peak, steps, with_e2e, numa_note):
    cfg = CONFIGS[name]
    x = make_inputs(cfg, dev, torch)
    osize = (cfg["oH"], cfg["oW"])
    out = capi.resize_forward(x, osize, cfg["mode"], False)
    for _ in range(3):
        capi.resize_forward(x, osize, cfg["mode"], False, out=out)
    barrier()
    capi.launch_count(reset=True)
    tot, per = time_steps(torch, lambda i: capi.resize_forward(x, osize, cfg["mode"], False, out=out), steps)
    launches = capi.launch_count()
    ms = reduce_max(torch, dist, world, dev, tot) / steps
    ab = algorithmic_bytes(cfg)
    r = {"workload": cfg["workload"], "ms": ms, "value": world * mpix(cfg) / (ms * 1e-3), "unit": "Mpix/s",
         "gpu_launches_per_step": launches / steps,
         "roofline": {"bound": "hbm", "achieved": ab / (tot / steps * 1e-3) / 1e9, "peak": peak, "unit": "GB/s",
                      "frac": ab / (tot / steps * 1e-3) / 1e9 / peak, "algorithmic_bytes_per_launch": ab, "median_step_ms": per[len(per) // 2],
                      "traffic": recorded_traffic(name), "traffic_kind": "recorded (ncu capture under profiles/, not this run)"}}
    if name == "cfg3":
        # the FP32-pipe streaming kernel beside the tensor-core one, same inputs (north_star prefers FP32 pipes; both reported)
        try:
            alt = capi.resize_forward(x, osize, cfg["mode"], False, capi.FLAG_FORCE_STREAM)
            for _ in range(2):
                capi.resize_forward(x, osize, cfg["mode"], False, capi.FLAG_FORCE_STREAM, out=alt)
            barrier()
            t2, _ = time_steps(torch, lambda i: capi.resize_forward(x, osize, cfg["mode"], False, capi.FLAG_FORCE_STREAM, out=alt), max(3, steps // 2))
            ms2 = t2 / max(3, steps // 2)
            r["alt_fp32_pipe_stream_kernel"] = {"ms": ms2, "frac": ab / (ms2 * 1e-3) / 1e9 / peak,
                                                "max_abs_diff_vs_default": float((alt - out).abs().max().item())}
            del alt
        except Exception as e:  # noqa: BLE001
            r["alt_fp32_pipe_stream_kernel"] = {"error": str(e)[:200]}
    if with_e2e:
        r["e2e"] = measure_e2e(torch, dist, capi, cfg, x, out, dev, local_rank, world, barrier, max(3, min(steps, 6)), numa_note)
    del x, out
    return r


def sub_cfg4(torch, dist, capi, dev, world, barrier, peak, steps):
    cfg = CONFIGS["cfg4"]
    ishape = (cfg["N"], cfg["C"], cfg["H"], cfg["W"])
    R = 8  # 8 x 201 MB of grad_in: the write stream cannot stay in the 126 MB L2
    gos = [make_inputs(cfg, dev, torch) + k for k in range(R)]
    gis = [torch.empty(ishape, device=dev) for _ in range(R)]
    ab = algorithmic_bytes(cfg)
    out = {"workload": cfg["workload"], "hbm_bound_us": round(ab / peak / 1e3, 2)}
    for label, nb in (("cold", R), ("warm", 1)):
        call = lambda i: capi.resize_backward(gos[i % nb], ishape, cfg["mode"], False, out=gis[i % nb])
        for i in range(max(3, nb)):
            call(i)
        barrier()
        tot, per = time_steps(torch, call, max(steps, 2 * R))
        n = max(steps, 2 * R)
        ms = reduce_max(torch, dist, world, dev, tot) / n
        out[label] = {"ms": ms, "median_ms": per[len(per) // 2], "frac": ab / (tot / n * 1e-3) / 1e9 / peak,
                      "buffers": nb, "value": world * mpix(cfg) / (ms * 1e-3)}
    out["note"] = ("cold: rotates over 8 grad_out/grad_in pairs (1.7 GB) so every launch streams from and to HBM; warm: one pair, the "
                   "214 MB working set is partly L2-resident between launches (the round-1 number)")
    del gos, gis
    return out


def sub_strong(torch, dist, capi, dev, rank, world, barrier, weak_ms, steps):
    """BASELINE configs[1] literally: the fixed 256-image batch sharded by image over the N ranks (no collective)."""
    from interpolate_antialiasing_b200.sharding import shard_bounds
    cfg = CONFIGS["cfg2"]
    b, e = shard_bounds(cfg["N"], world)[rank]
    x = make_inputs(cfg, dev, torch, n_images=e - b)
    osize = (cfg["oH"], cfg["oW"])
    out = capi.resize_forward(x, osize, cfg["mode"], False)
    for _ in range(3):
        capi.resize_forward(x, osize, cfg["mode"], False, out=out)
    barrier()
    tot, per = time_steps(torch, lambda i: capi.resize_forward(x, osize, cfg["mode"], False, out=out), steps)
    ms = reduce_max(torch, dist, world, dev, tot) / steps
    del x, out
    return {"N": world, "images_per_rank": e - b, "ms": ms, "value": mpix(cfg) / (ms * 1e-3), "unit": "Mpix/s",
            "efficiency_vs_this_box_1gpu_time": weak_ms / (world * ms),
            "note": "efficiency = (one rank's time for all 256 images, measured in this run as the weak-scaling step) / (N x sharded time)"}


def shard_equal(torch, dist, capi, dev, rank, world):
    """Bitwise check of the sharded path: every rank resizes its images of one seeded batch; the gathered result must equal
    rank 0 recomputing all of them (SURVEY 8(e): concat of shard outputs == single-GPU result, bit for bit)."""
    from interpolate_antialiasing_b200.sharding import gather_outputs, shard_bounds
    n = 2 * world + 1  # uneven on purpose
    g = torch.Generator(device=dev).manual_seed(77)
    full = (torch.rand((n, 3, 540, 960), generator=g, device=dev) * 255).contiguous(memory_format=torch.channels_last)
    res = {}
    for mode, osize in (("linear", (224, 224)), ("cubic", (97, 131))):
        b, e = shard_bounds(n, world)[rank]
        y = capi.resize_forward(full[b:e].contiguous(memory_format=torch.channels_last), osize, mode, False) if e > b else \
            torch.empty((0, 3) + osize, device=dev).contiguous(memory_format=torch.channels_last)
        got = gather_outputs(y.contiguous(), n)
        want = capi.resize_forward(full, osize, mode, False).contiguous()
        res[mode] = bool(torch.equal(got, want))
    t = torch.tensor([int(all(res.values()))], device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MIN)
    return bool(t.item()), res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", default="cfg2", choices=sorted(c for c in CONFIGS if c != "cfg1"))
    ap.add_argument("--images", type=int, default=None, help="override the batch size (debug only; invalidates the headline)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-sub", action="store_true", help="skip the sub-measurements (cfg1/3/4/5, strong scaling)")
    ap.add_argument("--sweep-quick", action="store_true", help="cfg5: every 7th point only")
    ap.add_argument("--cpu-seconds", type=float, default=12.0)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's result under DIR as .npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the GPU path's result; --impl reference times a CPU sample of other images")
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    cfg = dict(CONFIGS[args.config])
    if args.images:
        cfg["N"] = args.images
        cfg["workload"] += f" [DEBUG batch {args.images}]"

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference(args, cfg, rank, world)
        return

    import torch
    import torch.distributed as dist
    from interpolate_antialiasing_b200 import capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: this framework has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    peak, peak_src = measured_peak()
    numa_note = bind_to_gpu_numa_node(torch, local_rank) if world > 1 else "single process, unbound"
    t_start = time.time()

    x = make_inputs(cfg, dev, torch)
    osize = (cfg["oH"], cfg["oW"])
    if cfg["kind"] == "forward":
        out = capi.resize_forward(x, osize, cfg["mode"], False)
        step = lambda i: capi.resize_forward(x, osize, cfg["mode"], False, capi.FLAG_AUTO, out=out)
    else:
        ishape = (cfg["N"], cfg["C"], cfg["H"], cfg["W"])
        out = capi.resize_backward(x, ishape, cfg["mode"], False)
        step = lambda i: capi.resize_backward(x, ishape, cfg["mode"], False, out=out)
    for i in range(args.warmup):
        step(i)
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    capi.launch_count(reset=True)
    barrier()
    total_ms, per = time_steps(torch, step, args.steps)
    barrier()
    launches = capi.launch_count()
    capi.check_device(local_rank)
    total_ms_max = reduce_max(torch, dist, world, dev, total_ms)
    clocks = sampler.stop() if rank == 0 else None
    dump = None
    if args.dump_outputs and rank == 0:
        dump = dump_output(args.dump_outputs, "output" if cfg["kind"] == "forward" else "grad_input", out)

    # ---- e2e: host buffers through the C ABI, copies inside the timed region, with the copy ceiling beside it
    e2e = None
    if not args.no_e2e and cfg["kind"] == "forward":
        e2e = measure_e2e(torch, dist, capi, cfg, x, out, dev, local_rank, world, barrier, max(3, min(args.steps, 10)), numa_note)
    del x, out
    torch.cuda.empty_cache()

    # ---- the other configs (every rank takes part: reductions inside)
    sub = None
    if not args.no_sub and args.config == "cfg2" and not args.images:
        sub = {}
        try:
            if rank == 0:
                sub["cfg1"] = sub_cfg1(torch, capi, dev, peak)
            barrier()
            sub["cfg3"] = sub_forward(torch, dist, capi, "cfg3", dev, local_rank, world, barrier, peak, max(5, args.steps // 2),
                                      not args.no_e2e, numa_note)
            torch.cuda.empty_cache()
            sub["cfg4"] = sub_cfg4(torch, dist, capi, dev, world, barrier, peak, args.steps)
            torch.cuda.empty_cache()
            sys.path.insert(0, os.path.join(ROOT, "scripts"))
            import sweep_lib
            gen = torch.Generator(device=dev).manual_seed(1234 + rank)
            pts = [sweep_lib.run_point(p, torch, capi, dev, gen, peak, dist, world)
                   for p in sweep_lib.point_list(quick=args.sweep_quick)]
            sub["cfg5"] = sweep_lib.summarize(pts, peak)
            sub["cfg5"]["workload"] = ("cfg5: scale sweep of [N,C,1024,1024] (N per point sized for >= 1 GB of traffic): fwd = fp32 "
                                       "0.125x-2x, C in {1,3,4}, CF/CL, bilinear+bicubic; mixed = different h/w scales; uint8 = uint8 "
                                       "input; bwd = the adjoint; 2 warm-up + 5 timed calls per point, median, max over ranks")
            torch.cuda.empty_cache()
            sub["strong"] = sub_strong(torch, dist, capi, dev, rank, world, barrier, total_ms_max / args.steps, args.steps)
            if world > 1:
                ok, detail = shard_equal(torch, dist, capi, dev, rank, world)
                sub["shard_equal"] = ok
                sub["shard_equal_detail"] = detail
            capi.check_device(local_rank)
        except Exception as e:  # noqa: BLE001  (the headline line must still be printed)
            sub["error"] = f"{type(e).__name__}: {str(e)[:300]}"

    if rank == 0:
        ms_per_step = total_ms_max / args.steps
        ab = algorithmic_bytes(cfg)
        kern_ms = total_ms / args.steps  # one launch per step; events on the launching stream
        achieved = ab / (kern_ms * 1e-3) / 1e9
        line = {
            "metric": METRIC, "value": world * mpix(cfg) / (ms_per_step * 1e-3), "unit": "Mpix/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "u8" if cfg["dtype"] == "u8" else "f32", "data": "synthetic",
            "config": {"workload": cfg["workload"], "per_gpu_batch": cfg["N"], "sharding": "by image, no collective on the data path",
                       "l2": "inputs larger than L2 (%.2f GB read per step vs 126 MB L2)" % (ab / 1e9) if ab > 5e8 else
                             "working set fits L2: number is L2-warm, see DESIGN.md",
                       "path": "aa_resize_forward (C ABI)" if cfg["kind"] == "forward" else "aa_resize_backward (C ABI)"},
            "clocks": clocks, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": recorded_traffic(args.config), "traffic_kind": "recorded (ncu --set full capture under profiles/, not this run)",
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": ab, "kernel_ms": kern_ms,
                         "min_step_ms": per[0], "median_step_ms": per[len(per) // 2]},
        }
        if e2e:
            line["e2e"] = e2e
        if dump:
            line["dump"] = dump
        if sub is not None:
            line["sub"] = sub
        if world == 1 and not args.no_cpu_baseline:
            cb = cpu_reference_rate(cfg, args.cpu_seconds, torch)
            if cb:
                line["cpu_baseline"] = cb
        line["bench_wall_s"] = round(time.time() - t_start, 1)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
