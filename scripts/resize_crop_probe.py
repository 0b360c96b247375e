"""Resize(256) + CenterCrop(224) and TenCrop(224) of an evaluation batch: aa_resize_crops_ex against the routes a caller has
without it.

Workload: the crops probe's images (scripts/crops_probe.py): 256 seeded HWC uint8 images of 300-600 px per side; the output
is a normalised planar fp16 batch, bilinear, torchvision v2 semantics (shorter side to 256, aspect ratio kept).  Arms:
  Resize(256) + CenterCrop(224) -> [256, 3, 224, 224]
    (a) crops_ex   aa.resize_center_crop: aa_resize_crops_ex, one launch, only the 224^2 windows computed
    (b) per_image  aa_resize_forward_ex per image to its resized size (normalised fp16 epilogue), then slice and stack
    (c) tv         torchvision.transforms.v2.functional resize(antialias=True) + center_crop per image on the GPU, normalise
  Resize(256) + TenCrop(224) -> [256, 10, 3, 224, 224]
    (d) crops_ex   aa.ten_crop: 2560 crops in ceil(2560 / 512) = 5 launches; the ten windows overlap, so this computes
                   each output pixel of the ten crops (5.7x the outputs of one resize of a 256x341 image)
    (e) per_image  aa_resize_forward_ex once per image, then ten slices / flips and a stack
Per arm: device time per batch (CUDA events around a repeat of the step's call, enqueued behind a spin kernel so that host
gaps do not count), wall time per call (enqueue to completion), launches per call (this library's counter and the CUDA
activities torch.profiler records for one call), and the largest difference from arm (a) / (d).  The card's name and power
limit are read in the same run.  Prints one JSON line and writes it to --out when given.

    python scripts/resize_crop_probe.py [--steps 30] [--warmup 5] [--out FILE.json]
"""
import argparse
import json
import os
import random
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

N, SIZE, CROP = 256, 256, 224
MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)


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
    import interpolate_antialiasing_b200 as aa
    from interpolate_antialiasing_b200 import capi
    if not torch.cuda.is_available():
        sys.exit("resize_crop_probe needs a CUDA device")
    tvf = None
    try:
        import torchvision.transforms.v2.functional as tvf
    except Exception:  # noqa: BLE001
        pass
    dev = torch.device("cuda", 0)
    rnd = random.Random(0)  # the crops probe's generator: the same 256 images
    g = torch.Generator(device=dev).manual_seed(0)
    images = [torch.randint(0, 256, (rnd.randint(300, 600), rnd.randint(300, 600), 3), generator=g, device=dev, dtype=torch.uint8)
              for _ in range(N)]
    scale = [1.0 / (255.0 * s) for s in STD]
    bias = [-m / s for m, s in zip(MEAN, STD)]
    mean_t = torch.tensor(MEAN, device=dev).view(1, 3, 1, 1) * 255
    std_t = torch.tensor(STD, device=dev).view(1, 3, 1, 1) * 255
    resized = [aa.resized_output_size(im.shape[0], im.shape[1], SIZE) for im in images]
    anchors = [(int(round((h - CROP) / 2.0)), int(round((w - CROP) / 2.0))) for h, w in resized]
    outs = {}

    def resize_each(o_list):
        for im, (h, w), o in zip(images, resized, o_list):
            capi.resize_forward_ex(im.permute(2, 0, 1).unsqueeze(0), (h, w), "bilinear", o, scale, bias)

    # preallocated per-image resize outputs of the per-image route (one size class each)
    per_image_buf = [torch.empty((1, 3, h, w), dtype=torch.float16, device=dev) for h, w in resized]

    def center_crops_ex():
        outs["center_crops_ex"] = aa.resize_center_crop(images, SIZE, CROP, mean=MEAN, std=STD)

    def center_per_image():
        resize_each(per_image_buf)
        outs["center_per_image"] = torch.cat([r[:, :, t:t + CROP, l:l + CROP] for r, (t, l) in zip(per_image_buf, anchors)])

    def center_tv():
        ys = [tvf.center_crop(tvf.resize(im.permute(2, 0, 1).float(), [SIZE], antialias=True), [CROP]) for im in images]
        outs["center_tv"] = torch.stack(ys).sub_(mean_t).div_(std_t).half()

    def ten_crops_ex():
        outs["ten_crops_ex"] = aa.ten_crop(images, SIZE, CROP, mean=MEAN, std=STD)

    def ten_per_image():
        resize_each(per_image_buf)
        ys = []
        for r in per_image_buf:
            five = [r[..., :CROP, :CROP], r[..., :CROP, -CROP:], r[..., -CROP:, :CROP], r[..., -CROP:, -CROP:]]
            H, W = r.shape[-2:]
            t, l = int(round((H - CROP) / 2.0)), int(round((W - CROP) / 2.0))
            five.append(r[..., t:t + CROP, l:l + CROP])
            f = r.flip(-1)
            five += [f[..., :CROP, :CROP], f[..., :CROP, -CROP:], f[..., -CROP:, :CROP], f[..., -CROP:, -CROP:],
                     f[..., t:t + CROP, l:l + CROP]]
            ys.append(torch.cat(five))
        outs["ten_per_image"] = torch.stack(ys)

    groups = {"center": {"crops_ex": center_crops_ex, "per_image": center_per_image},
              "ten": {"crops_ex": ten_crops_ex, "per_image": ten_per_image}}
    if tvf is not None:
        groups["center"]["tv"] = center_tv

    for arms in groups.values():
        for f in arms.values():
            f()
    torch.cuda.synchronize()
    check = {}
    for gname, arms in groups.items():
        ref = outs[f"{gname}_crops_ex"].float()
        for name in arms:
            if name != "crops_ex":
                check[f"{gname}_crops_ex_vs_{name}_max_abs"] = float((ref - outs[f"{gname}_{name}"].float().view_as(ref)).abs().max())

    launches = {}
    for gname, arms in groups.items():
        for name, f in arms.items():
            capi.launch_count(reset=True)
            f()
            torch.cuda.synchronize()
            lib_n = capi.launch_count(reset=True)
            try:
                from torch.profiler import ProfilerActivity, profile
                with profile(activities=[ProfilerActivity.CUDA]) as p:
                    f()
                    torch.cuda.synchronize()
                acts = sum(1 for e in p.events() if e.device_type == torch.autograd.DeviceType.CUDA)
            except Exception as e:  # noqa: BLE001
                acts = f"profiler unavailable: {e}"
            launches[f"{gname}_{name}"] = {"library_launches": lib_n, "cuda_activities": acts}

    # device time: the stream is held by a spin kernel long enough for the host to enqueue the whole call behind it, so the
    # events see the GPU's work without the host's gaps; wall time: the call from the host until its results are complete
    keys = [f"{gname}_{name}" for gname, arms in groups.items() for name in arms]
    dev_ms = {k: [] for k in keys}
    wall_ms = {k: [] for k in keys}
    for step in range(args.warmup + args.steps):
        for gname, arms in groups.items():
            for name, f in arms.items():
                k = f"{gname}_{name}"
                torch.cuda.synchronize()
                t0 = time.perf_counter()
                f()
                t1 = time.perf_counter()
                torch.cuda.synchronize()
                t2 = time.perf_counter()
                hold_cycles = int(max(4 * (t1 - t0), 2e-3) * 2.5e9)  # >= 4x the enqueue time at up to 2.5 GHz
                a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                torch.cuda._sleep(hold_cycles)
                a.record()
                f()
                b.record()
                torch.cuda.synchronize()
                if step >= args.warmup:
                    dev_ms[k].append(a.elapsed_time(b))
                    wall_ms[k].append((t2 - t0) * 1e3)

    med = lambda v: sorted(v)[len(v) // 2]  # noqa: E731
    res = {"gpu": gpu_info(0), "workload": f"{N} HWC uint8 images 300-600 px, Resize({SIZE}) + CenterCrop({CROP}) / "
                                            f"TenCrop({CROP}) -> normalised planar fp16, bilinear", "steps": args.steps,
           "check": check, "arms": {}}
    for k in keys:
        res["arms"][k] = {"device_ms_median": round(med(dev_ms[k]), 4), "device_ms_min": round(min(dev_ms[k]), 4),
                          "device_ms_max": round(max(dev_ms[k]), 4), "wall_ms_per_call_median": round(med(wall_ms[k]), 4),
                          **launches[k]}
    for gname, arms in groups.items():
        base = res["arms"][f"{gname}_crops_ex"]
        for name in arms:
            if name != "crops_ex":
                other = res["arms"][f"{gname}_{name}"]
                res[f"ratio_{gname}_{name}_over_crops_ex_device"] = round(other["device_ms_median"] / base["device_ms_median"], 2)
                res[f"ratio_{gname}_{name}_over_crops_ex_wall"] = round(other["wall_ms_per_call_median"] / base["wall_ms_per_call_median"], 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
