"""Padded batches: aa.resize_pad_batch (aa_resize_crops_pad) against the routes a caller has without it.

Workloads, bilinear, torchvision v2 resize(antialias=True) sizes, normalised planar fp16 output:
  (a) letterbox  the crops probe's 256 seeded HWC uint8 images of 300-600 px per side (scripts/crops_probe.py), each resized
                 so that its longer side is 640, centred on a 640x640 canvas filled with 114 (in the input's domain)
  (b) detection  16 seeded HWC uint8 images of mixed orientation from 480x640 to 1080x1920, Resize(800, max_size=1333), top
                 left of a canvas of the largest size rounded up to 32, zeros after normalisation (batch_images)
  (c) center     Resize(256) + CenterCrop(224) of the workload (a) images, where nothing needs padding: pad=True against
                 pad=False (the padded kernel is only used when a window leaves its resized image)
Arms of (a) and (b):
  pad_batch  aa.resize_pad_batch: one launch per 512 images
  per_image  the canvas filled by one copy from a pre-filled template, then aa_resize_forward_ex of each image (normalised
             fp16 epilogue) straight into its slice of the canvas
  tv         torchvision.transforms.v2.functional resize + pad per image on the GPU, stack, normalise
Per arm: device time per batch (CUDA events around a repeat of the call, enqueued behind a spin kernel so that host gaps do
not count), wall time per call (enqueue to completion), launches per call (this library's counter and the CUDA activities
torch.profiler records for one call), and the largest difference from the first arm of its workload.  The card's name and
power limit are read in the same run.  Prints one JSON line and writes it to --out when given.

    python scripts/resize_pad_probe.py [--steps 30] [--warmup 5] [--out FILE.json]
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

MEAN, STD = (0.485, 0.456, 0.406), (0.229, 0.224, 0.225)
LB, FILL = 640, 114


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
        sys.exit("resize_pad_probe needs a CUDA device")
    tvf = None
    try:
        import torchvision.transforms.v2.functional as tvf
    except Exception:  # noqa: BLE001
        pass
    dev = torch.device("cuda", 0)
    rnd = random.Random(0)  # the crops probe's generator: the same 256 images
    g = torch.Generator(device=dev).manual_seed(0)
    small = [torch.randint(0, 256, (rnd.randint(300, 600), rnd.randint(300, 600), 3), generator=g, device=dev, dtype=torch.uint8)
             for _ in range(256)]
    rnd = random.Random(1)
    det_sizes = [(480, 640), (720, 1280), (1080, 1920), (600, 800), (768, 1024), (900, 1600), (1024, 768), (1080, 1440)]
    big = []
    for k in range(16):
        h, w = det_sizes[k % len(det_sizes)]
        if k % 3 == 1:
            h, w = w, h  # portrait
        big.append(torch.randint(0, 256, (h, w, 3), generator=g, device=dev, dtype=torch.uint8))
    scale = [1.0 / (255.0 * s) for s in STD]
    bias = [-m / s for m, s in zip(MEAN, STD)]
    mean_t = torch.tensor(MEAN, device=dev).view(1, 3, 1, 1) * 255
    std_t = torch.tensor(STD, device=dev).view(1, 3, 1, 1) * 255

    def layout(images, size, max_size, canvas, align):
        return aa._pad_layout([im.shape[:2] for im in images], size, max_size, 32, canvas, align)

    work = {  # name: (images, size, max_size, canvas, align, fill, pad_value)
        "letterbox": (small, None, LB, (LB, LB), "center", FILL, None),
        "detection": (big, 800, 1333, None, "top_left", None, 0.0),
    }
    outs = {}
    groups = {}
    for wname, (images, size, max_size, canvas, align, fill, pad_value) in work.items():
        R, (Hc, Wc), place = layout(images, size, max_size, canvas, align)
        # the per-image route's canvas template: the fill after normalisation, or the stored pad value
        template = torch.empty((len(images), 3, Hc, Wc), dtype=torch.float16, device=dev)
        if fill is not None:
            template.copy_(((torch.full((1, 3, 1, 1), float(fill), device=dev) - mean_t) / std_t).expand(template.shape))
        else:
            template.fill_(pad_value)
        canvas_buf = torch.empty_like(template)

        def pad_batch(images=images, size=size, max_size=max_size, canvas=canvas, align=align, fill=fill, pad_value=pad_value,
                      wname=wname):
            outs[f"{wname}_pad_batch"] = aa.resize_pad_batch(images, size, max_size=max_size, canvas=canvas, align=align,
                                                             fill=fill, pad_value=pad_value, mean=MEAN, std=STD)[0]

        def per_image(images=images, place=place.tolist(), template=template, canvas_buf=canvas_buf, wname=wname):
            canvas_buf.copy_(template)
            for i, (im, (t, l, h, w)) in enumerate(zip(images, place)):
                capi.resize_forward_ex(im.permute(2, 0, 1).unsqueeze(0), (h, w), "bilinear",
                                       canvas_buf[i:i + 1, :, t:t + h, l:l + w], scale, bias)
            outs[f"{wname}_per_image"] = canvas_buf

        def tv(images=images, size=size, max_size=max_size, place=place.tolist(), Hc=Hc, Wc=Wc, fill=fill, wname=wname):
            if fill is not None:  # pad in the input's domain, then normalise
                ys = [tvf.pad(tvf.resize(im.permute(2, 0, 1).float(), size, max_size=max_size, antialias=True),
                              [l, t, Wc - w - l, Hc - h - t], fill=float(fill)) for im, (t, l, h, w) in zip(images, place)]
                outs[f"{wname}_tv"] = torch.stack(ys).sub_(mean_t).div_(std_t).half()
            else:  # normalise, then zeros
                ys = [tvf.resize(im.permute(2, 0, 1).float(), size, max_size=max_size, antialias=True) for im in images]
                batch = torch.zeros((len(images), 3, Hc, Wc), dtype=torch.float16, device=dev)
                for b, y in zip(batch, ys):
                    b[:, :y.shape[1], :y.shape[2]].copy_((y.unsqueeze(0) - mean_t).div_(std_t)[0])
                outs[f"{wname}_tv"] = batch

        groups[wname] = {"pad_batch": pad_batch, "per_image": per_image}
        if tvf is not None:
            groups[wname]["tv"] = tv

    def center(pad):
        def f():
            outs[f"center_pad_{str(pad).lower()}"] = aa.resize_center_crop(small, 256, 224, mean=MEAN, std=STD, pad=pad)
        return f

    groups["center"] = {"pad_false": center(False), "pad_true": center(True)}

    for arms in groups.values():
        for f in arms.values():
            f()
    torch.cuda.synchronize()
    check = {}
    for gname, arms in groups.items():
        names = list(arms)
        ref = outs[f"{gname}_{names[0]}"].float()
        for name in names[1:]:
            check[f"{gname}_{names[0]}_vs_{name}_max_abs"] = float((ref - outs[f"{gname}_{name}"].float().view_as(ref)).abs().max())

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
    res = {"gpu": gpu_info(0), "workload": {
        "letterbox": f"256 HWC uint8 images 300-600 px -> longer side {LB}, centred on {LB}x{LB}, fill {FILL}, normalised planar fp16",
        "detection": "16 HWC uint8 images 480x640-1080x1920 -> Resize(800, max_size=1333), top left, canvas rounded up to 32, "
                     "zeros after normalisation, planar fp16",
        "center": "the letterbox images, Resize(256) + CenterCrop(224), normalised planar fp16, pad=False vs pad=True"},
        "steps": args.steps, "check": check, "arms": {}}
    for k in keys:
        res["arms"][k] = {"device_ms_median": round(med(dev_ms[k]), 4), "device_ms_min": round(min(dev_ms[k]), 4),
                          "device_ms_max": round(max(dev_ms[k]), 4), "wall_ms_per_call_median": round(med(wall_ms[k]), 4),
                          **launches[k]}
    for gname, arms in groups.items():
        names = list(arms)
        base = res["arms"][f"{gname}_{names[0]}"]
        for name in names[1:]:
            other = res["arms"][f"{gname}_{name}"]
            res[f"ratio_{gname}_{name}_over_{names[0]}_device"] = round(other["device_ms_median"] / base["device_ms_median"], 2)
            res[f"ratio_{gname}_{name}_over_{names[0]}_wall"] = round(other["wall_ms_per_call_median"] / base["wall_ms_per_call_median"], 2)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, "w") as fh:
            fh.write(line + "\n")


if __name__ == "__main__":
    main()
