#!/usr/bin/env python
"""Time the post-network stage with rotation search (spg_postnet_rotated) on cuda:0 beside the same scales at angle 0.

usage: python tools/time_postnet_rotation.py [--iters 20] [--out FILE]

Two configurations of predict()'s loop after the forward pass (evaluate.py:90-161), stride 4, 48 channels used of 50:
  512: 32 images at 512 x 512, scale_search [0.5, 1, 2] (padded 256 / 512 / 1024, network output 64 / 128 / 256);
  128: 256 images at 128 x 128, scale_search [1] (network output 32 x 32);
each with rotation_search [-5, 0, 5] and with [0] only.  Network outputs are random float32 on the device (the stage's
time does not depend on the values).  Every working set exceeds the 126 MB L2.

Reported per configuration: ms per batch (CUDA events over --iters calls after 3 warm-up calls), the launches, the
algorithmic bytes -- network outputs read once (both images of each pair, 48 channels; tile halos not counted) plus the
output planes per launch (float64 sums written, read again by every launch after the first; float32 keypoint maps at
the end) -- and those bytes over the time as a fraction of the HBM bandwidth a 4 GiB device-to-device copy reaches in
the same run.  The card's name and power limit are read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch  # noqa: E402

from improved_body_parts_b200.grouping import Grouper  # noqa: E402

C_NET, C_USED, K, L = 50, 48, 18, 30


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def hbm_copy_gbs(dev, iters=20):
    """Bytes read + written by a 4 GiB device-to-device copy over its CUDA-event time."""
    a = torch.empty(1 << 30, dtype=torch.float32, device=dev)
    b = torch.empty_like(a)
    for _ in range(3):
        b.copy_(a)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        b.copy_(a)
    e1.record()
    torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / iters * 1e-3
    del a, b
    return 2 * 4 * (1 << 30) / s / 1e9


def launches_of(angles):
    """The launch schedule of spg_postnet(_rotated) for the stride-4 kernels: rotated items one launch each, runs of
    angle-0 items fused four to a launch."""
    if all(a == 0 for a in angles):
        return (len(angles) + 3) // 4
    n, t = 0, 0
    while t < len(angles):
        if angles[t] == 0:
            t1 = t
            while t1 < len(angles) and angles[t1] == 0:
                t1 += 1
            n += (t1 - t + 3) // 4
            t = t1
        else:
            n += 1
            t += 1
    return n


def alg_bytes(N, nets, angles_per_scale, H, W):
    items = [(hw, a) for hw in nets for a in angles_per_scale]
    net = sum(N * 2 * C_USED * h * w * 4 for (h, w), _ in items)
    n_launch = launches_of([a for _, a in items])
    px = N * H * W
    if len(items) == 1:
        out = px * (K * 4 + L * 4)  # single item: float32 planes written once
    elif n_launch == 1:
        out = px * (K * 4 + L * 8)  # the whole loop in one launch: sums in registers, planes written once
    else:
        out = n_launch * px * (K + L) * 8 + (n_launch - 1) * px * (K + L) * 8 + px * K * 4
    return net + out, n_launch


def run(g, N, image, scales, angles_per_scale, iters, dev):
    nets, crops = [], []
    for s in scales:
        crop = int(round(image * s))
        padded = (crop + 63) // 64 * 64
        nets.append((padded // 4, padded // 4))
        crops.append((crop, crop))
    tensors = [torch.rand((N, 2, C_NET, h, w), device=dev) for h, w in nets]
    outs, item_crops, angles = [], [], []
    for t, c in zip(tensors, crops):
        for a in angles_per_scale:
            outs.append(t)
            item_crops.append(c)
            angles.append(float(a))
    heat = torch.empty((N, K, image, image), dtype=torch.float32, device=dev)
    paf = torch.empty((N, L, image, image), dtype=torch.float32 if len(outs) == 1 else torch.float64, device=dev)
    rot = any(a != 0 for a in angles)

    def call():
        g.postnet(outs, item_crops, (image, image), heat_out=heat, paf_out=paf, paf_dtype=paf.dtype,
                  angles=angles if rot else None)
    for _ in range(3):
        call()
    torch.cuda.synchronize()
    l0 = g.launch_count
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        call()
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / iters
    launches = (g.launch_count - l0) // iters
    nbytes, predicted = alg_bytes(N, nets, angles_per_scale, image, image)
    assert launches == predicted, (launches, predicted)
    del tensors, outs
    return {"images": N, "image": image, "scales": scales, "angles": list(angles_per_scale), "items": len(angles),
            "net_hw": nets, "crops": crops, "launches": launches, "kernel": g.postnet_kernel(), "ms_per_batch": ms,
            "alg_bytes": nbytes, "alg_gbs": nbytes / (ms * 1e-3) / 1e9}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        sys.exit("time_postnet_rotation.py needs a CUDA device")
    dev = torch.device("cuda:0")
    res = {"card": card(), "hbm_copy_gbs": hbm_copy_gbs(dev), "configs": []}
    for N, image, scales in ((32, 512, [0.5, 1.0, 2.0]), (256, 128, [1.0])):
        g = Grouper(max_batch=N, max_h=image, max_w=image)
        try:
            for angles in ([-5.0, 0.0, 5.0], [0.0]):
                r = run(g, N, image, scales, angles, args.iters, dev)
                r["frac_of_copy_bw"] = r["alg_gbs"] / res["hbm_copy_gbs"]
                res["configs"].append(r)
                print(f"{N} x {image}^2 scales {scales} angles {angles}: {r['ms_per_batch']:.3f} ms/batch, "
                      f"{r['launches']} launches ({r['kernel']}), {r['alg_bytes'] / 1e9:.3f} GB, {r['alg_gbs']:.0f} GB/s = "
                      f"{r['frac_of_copy_bw']:.3f} of the copy bandwidth", flush=True)
        finally:
            g.close()
        torch.cuda.empty_cache()
    print(f"card: {res['card']}; device-to-device copy: {res['hbm_copy_gbs']:.0f} GB/s")
    if args.out:
        with open(args.out, "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
