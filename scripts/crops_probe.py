"""RandomResizedCrop + RandomHorizontalFlip of a training batch: aa_resize_crops against the two routes a caller has without it.

Workload: 256 seeded HWC uint8 images of ImageNet-like sizes (300-600 px per side); every step draws fresh
RandomResizedCrop(224) boxes (scale=(0.08, 1), ratio=(3/4, 4/3), torchvision's get_params algorithm) and 50 % flips; the
output is a normalised planar fp16 [256, 3, 224, 224] batch.  Three arms, timed alternately on the same boxes:
  (a) crops   aa_resize_crops: one launch
  (b) ragged  crop views through aa_resize_forward_ragged (normalised fp16 epilogue) + torch.flip of the flipped slots
  (c) tv      torchvision.transforms.v2.functional.resized_crop(antialias=True) per image on the GPU tensor, flip, normalise
Per arm: device time per batch (CUDA events around a repeat of the step's call, enqueued behind a spin kernel so that host
gaps do not count), host time per call (enqueue, no synchronisation), wall time per call (the step's first call, enqueue
to completion), launches per call (this library's counter and the CUDA activities torch.profiler records for one call),
and algorithmic bytes (box pixels read once + output written once) over device time as a fraction of the HBM peak.  The
peak is MEASURED_PEAKS.json's hbm_gbs when present, else a device-to-device copy of 4 GiB measured in the same run.
Prints one JSON line and writes it to --out when given.

    python scripts/crops_probe.py [--steps 30] [--warmup 5] [--out FILE.json]
"""
import argparse
import json
import math
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, OUT = 256, 224
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


def get_params(rnd, H, W, scale=(0.08, 1.0), ratio=(3 / 4, 4 / 3)):
    """torchvision.transforms.RandomResizedCrop.get_params on a Python RNG: (top, left, height, width)."""
    area = H * W
    log_ratio = (math.log(ratio[0]), math.log(ratio[1]))
    for _ in range(10):
        target = area * rnd.uniform(*scale)
        ar = math.exp(rnd.uniform(*log_ratio))
        w = int(round(math.sqrt(target * ar)))
        h = int(round(math.sqrt(target / ar)))
        if 0 < w <= W and 0 < h <= H:
            return rnd.randint(0, H - h), rnd.randint(0, W - w), h, w
    in_ratio = W / H
    if in_ratio < min(ratio):
        w, h = W, int(round(W / min(ratio)))
    elif in_ratio > max(ratio):
        h, w = H, int(round(H * max(ratio)))
    else:
        w, h = W, H
    return (H - h) // 2, (W - w) // 2, h, w


def gpu_info(index):
    try:
        r = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30)
        return r.stdout.strip()
    except Exception as e:  # noqa: BLE001
        return f"nvidia-smi unavailable: {e}"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()

    import torch
    from interpolate_antialiasing_b200 import capi
    if not torch.cuda.is_available():
        sys.exit("crops_probe needs a CUDA device")
    tvf = None
    try:
        import torchvision.transforms.v2.functional as tvf
    except Exception:  # noqa: BLE001
        pass
    dev = torch.device("cuda", 0)
    rnd = random.Random(0)
    g = torch.Generator(device=dev).manual_seed(0)
    images = [torch.randint(0, 256, (rnd.randint(300, 600), rnd.randint(300, 600), 3), generator=g, device=dev, dtype=torch.uint8)
              for _ in range(N)]
    scale = [1.0 / (255.0 * s) for s in STD]
    bias = [-m / s for m, s in zip(MEAN, STD)]
    outs = {k: torch.empty((N, 3, OUT, OUT), dtype=torch.float16, device=dev) for k in ("crops", "ragged", "tv")}
    mean_t = torch.tensor(MEAN, device=dev).view(1, 3, 1, 1) * 255
    std_t = torch.tensor(STD, device=dev).view(1, 3, 1, 1) * 255

    def arm_crops(boxes, flips):
        capi.resize_crops(images, boxes, (OUT, OUT), "bilinear", out=outs["crops"], hflip=flips, scale=scale, bias=bias)

    def arm_ragged(boxes, flips):
        views = [im[t:t + h, l:l + w] for im, (t, l, h, w) in zip(images, boxes)]
        o = outs["ragged"]
        capi.resize_forward_ragged(views, (OUT, OUT), "bilinear", out=o, scale=scale, bias=bias)
        idx = torch.tensor([i for i, f in enumerate(flips) if f], device=dev)
        o[idx] = o[idx].flip(-1)

    def arm_tv(boxes, flips):
        ys = []
        for im, (t, l, h, w), f in zip(images, boxes, flips):
            y = tvf.resized_crop(im.permute(2, 0, 1).float(), t, l, h, w, [OUT, OUT], antialias=True)
            ys.append(y.flip(-1) if f else y)
        outs["tv"].copy_(torch.stack(ys).sub_(mean_t).div_(std_t))

    arms = {"crops": arm_crops, "ragged": arm_ragged}
    if tvf is not None:
        arms["tv"] = arm_tv

    def draw():
        boxes = [get_params(rnd, im.shape[0], im.shape[1]) for im in images]
        return boxes, [rnd.random() < 0.5 for _ in images]

    # same boxes, same results up to fp16 rounding: (a) is the general kernel's arithmetic, (b) takes the fast kernels
    boxes, flips = draw()
    for f in arms.values():
        f(boxes, flips)
    torch.cuda.synchronize()
    check = {f"crops_vs_{k}_max_abs": float((outs["crops"].float() - outs[k].float()).abs().max()) for k in arms if k != "crops"}

    # launches per call: the library's own counter and every CUDA activity of one call
    launches = {}
    for name, f in arms.items():
        capi.launch_count(reset=True)
        f(boxes, flips)
        torch.cuda.synchronize()
        lib_n = capi.launch_count(reset=True)
        try:
            from torch.profiler import ProfilerActivity, profile
            with profile(activities=[ProfilerActivity.CUDA]) as p:
                f(boxes, flips)
                torch.cuda.synchronize()
            acts = sum(1 for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA)
        except Exception as e:  # noqa: BLE001
            acts = f"profiler unavailable: {e}"
        launches[name] = {"library_launches": lib_n, "cuda_activities": acts}

    # device time: the stream is held by a spin kernel long enough for the host to enqueue the whole call behind it, so the
    # events see the GPU's work without the host's gaps; wall time: the call from the host until its results are complete
    dev_ms = {k: [] for k in arms}
    host_us = {k: [] for k in arms}
    wall_ms = {k: [] for k in arms}
    bytes_ = []
    for step in range(args.warmup + args.steps):
        boxes, flips = draw()
        if step >= args.warmup:
            bytes_.append(sum(h * w * 3 for _, _, h, w in boxes) + N * 3 * OUT * OUT * 2)
        for name, f in arms.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            f(boxes, flips)
            t1 = time.perf_counter()
            torch.cuda.synchronize()
            t2 = time.perf_counter()
            hold_cycles = int(max(4 * (t1 - t0), 2e-3) * 2.5e9)  # >= 4x the enqueue time at up to 2.5 GHz
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda._sleep(hold_cycles)
            a.record()
            f(boxes, flips)
            b.record()
            torch.cuda.synchronize()
            if step >= args.warmup:
                dev_ms[name].append(a.elapsed_time(b))
                host_us[name].append((t1 - t0) * 1e6)
                wall_ms[name].append((t2 - t0) * 1e3)

    peak_src = "MEASURED_PEAKS.json hbm_gbs"
    try:
        peak = float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"])
    except Exception:  # noqa: BLE001
        src = torch.empty(1 << 32, dtype=torch.uint8, device=dev)
        dst = torch.empty_like(src)
        dst.copy_(src)
        torch.cuda.synchronize()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        for _ in range(10):
            dst.copy_(src)
        b.record()
        torch.cuda.synchronize()
        peak = 2 * src.numel() * 10 / (a.elapsed_time(b) * 1e-3) / 1e9
        peak_src = "device-to-device copy of 4 GiB in this run (read + write bytes)"
        del src, dst

    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    mean_bytes = sum(bytes_) / len(bytes_)
    res = {"gpu": gpu_info(0), "workload": f"{N} HWC uint8 images 300-600 px, RandomResizedCrop({OUT}) + 50% hflip -> "
                                            f"normalised planar fp16, bilinear", "steps": args.steps,
           "hbm_peak_gbs": round(peak, 1), "peak_source": peak_src, "algorithmic_bytes_mean": int(mean_bytes), "check": check,
           "arms": {}}
    for name in arms:
        d = med(dev_ms[name])
        res["arms"][name] = {"device_ms_median": round(d, 4), "device_ms_min": round(min(dev_ms[name]), 4),
                             "host_us_per_call_median": round(med(host_us[name]), 1),
                             "wall_ms_per_call_median": round(med(wall_ms[name]), 4), **launches[name],
                             "algorithmic_gbs": round(mean_bytes / (d * 1e-3) / 1e9, 1),
                             "frac_of_hbm_peak": round(mean_bytes / (d * 1e-3) / 1e9 / peak, 4)}
    for other in ("ragged", "tv"):
        if other in res["arms"]:
            for key in ("device_ms_median", "wall_ms_per_call_median"):
                res[f"ratio_{other}_over_crops_{key.split('_')[0]}"] = round(res["arms"][other][key] / res["arms"]["crops"][key], 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
