#!/usr/bin/env python
"""Time the device pre-network stage (Grouper.prenet / spg_prenet) against the host chain dropin.predict runs by default.

usage: python tools/time_prenet.py [--iters 30] [--out-dir profiles/prenet]

One 480 x 640 uint8 BGR image with the reference's utils/config model parameters (boxsize 640, max_downsample 64,
padValue 128), three configurations of predict()'s loop before the forward pass (evaluate.py:89-116):
  scale_search [1] x rotation_search [0]  (the reference's default),
  [0.5, 1, 2] x [0],
  [0.5, 1, 2] x [-5, 0, 5].
Per configuration and image:
  device: upload of the uint8 image (pageable host memory, as predict() receives it) + one prenet per scale, host clock
          around the calls up to a device synchronise; and the prenet calls alone in CUDA events (image already on the
          device), with their launches and the bytes they must move (uint8 image read, padded uint8 written and read
          per angle, float32 pairs written);
  host:   cv2.resize -> pad -> np.float32(/ 255) -> cv2.warpAffine (angle != 0) -> mirror + concatenate -> pageable
          host-to-device copy of the pair, host clock up to a device synchronise -- dropin.predict's default path.
The CPUs of the host, cv2's version, thread count and IPP state, and the card's name and power limit are recorded in
the same run.  Writes time_prenet.json and time_prenet.txt under --out-dir.
"""
import argparse
import json
import os
import platform
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import cv2  # noqa: E402
import numpy as np  # noqa: E402
import torch  # noqa: E402

from improved_body_parts_b200.dropin import pad_right_down_corner  # noqa: E402
from improved_body_parts_b200.grouping import Grouper, prenet_size  # noqa: E402

BOXSIZE, MAX_DOWNSAMPLE, PAD_VALUE = 640, 64, 128
CONFIGS = [("[1] x [0]", [1.0], [0.0]), ("[0.5,1,2] x [0]", [0.5, 1.0, 2.0], [0.0]),
           ("[0.5,1,2] x [-5,0,5]", [0.5, 1.0, 2.0], [-5.0, 0.0, 5.0])]


def card():
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.SubprocessError):
        q = "nvidia-smi unavailable"
    return {"torch_name": torch.cuda.get_device_name(0), "nvidia_smi": q}


def host_cpus():
    model = platform.processor()
    try:
        with open("/proc/cpuinfo") as f:
            model = next(line.split(":", 1)[1].strip() for line in f if line.startswith("model name"))
    except (OSError, StopIteration):
        pass
    return {"model": model, "logical_cpus": os.cpu_count(), "usable_cpus": len(os.sched_getaffinity(0)),
            "cv2": cv2.__version__, "cv2_threads": cv2.getNumThreads(), "cv2_ipp": bool(cv2.ipp.useIPP())}


def host_chain(image, scales, angles, dev):
    for scale in scales:
        for angle in angles:
            resized = cv2.resize(image, (0, 0), fx=scale, fy=scale, interpolation=cv2.INTER_CUBIC)
            padded, _ = pad_right_down_corner(resized, MAX_DOWNSAMPLE, PAD_VALUE)
            x = np.float32(padded / 255)
            if angle != 0:
                x = cv2.warpAffine(x, cv2.getRotationMatrix2D((x.shape[0] / 2, x.shape[1] / 2), angle, 1), (0, 0))
            pair = np.concatenate((x[None, ...], x[:, ::-1, :].copy()[None, ...]), axis=0)
            torch.from_numpy(pair).to(dev)
    torch.cuda.synchronize()


def device_chain(g, image, scales, angles, dev, upload=True):
    img = torch.from_numpy(image).to(dev) if upload else image
    for scale in scales:
        g.prenet(img, scale, angles, max_downsample=MAX_DOWNSAMPLE, pad_value=PAD_VALUE)


def host_ms(fn, iters):
    fn()
    fn()
    t0 = time.perf_counter()
    for _ in range(iters):
        fn()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / iters * 1e3


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=30)
    ap.add_argument("--out-dir", default=os.path.join("profiles", "prenet"))
    args = ap.parse_args()
    assert torch.cuda.is_available(), "time_prenet.py measures on cuda:0"
    dev = torch.device("cuda:0")
    image = np.random.default_rng(0).integers(0, 256, size=(480, 640, 3), dtype=np.uint8)
    dimg = torch.from_numpy(image).to(dev)
    g = Grouper(max_batch=1, device=0)
    res = {"card": card(), "host": host_cpus(), "image_hw": [480, 640], "iters": args.iters, "configs": []}
    for name, search, angles in CONFIGS:
        scales = [x * BOXSIZE / image.shape[0] for x in search]
        sizes = [prenet_size(480, 640, s, MAX_DOWNSAMPLE) for s in scales]
        out_bytes = sum(len(angles) * 2 * hp * wp * 3 * 4 for _, (hp, wp) in sizes)
        moved = sum(480 * 640 * 3 + hp * wp * 3 * (1 + len(angles)) for _, (hp, wp) in sizes) + out_bytes
        n0 = g.launch_count
        device_chain(g, dimg, scales, angles, dev, upload=False)
        launches = g.launch_count - n0
        for _ in range(3):
            device_chain(g, dimg, scales, angles, dev, upload=False)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.iters):
            device_chain(g, dimg, scales, angles, dev, upload=False)
        e1.record()
        torch.cuda.synchronize()
        prenet_ms = e0.elapsed_time(e1) / args.iters
        dev_ms = host_ms(lambda: device_chain(g, image, scales, angles, dev), args.iters)
        hst_ms = host_ms(lambda: host_chain(image, scales, angles, dev), max(3, args.iters // 3))
        res["configs"].append({
            "config": name, "scales": scales, "angles": angles, "padded_hw": [list(p) for _, p in sizes],
            "items": len(scales) * len(angles), "launches": launches, "output_bytes": out_bytes, "bytes_moved": moved,
            "device_prenet_ms_events": prenet_ms, "device_prenet_gbs": moved / (prenet_ms * 1e-3) / 1e9,
            "device_upload_plus_prenet_ms_host_clock": dev_ms, "host_chain_ms_host_clock": hst_ms,
            "speedup_host_over_device": hst_ms / dev_ms})
    g.close()
    os.makedirs(args.out_dir, exist_ok=True)
    with open(os.path.join(args.out_dir, "time_prenet.json"), "w") as f:
        json.dump(res, f, indent=1)
    lines = [f"card: {res['card']['torch_name']} ({res['card']['nvidia_smi']})",
             f"host: {res['host']['model']}, {res['host']['usable_cpus']} usable of {res['host']['logical_cpus']} CPUs, "
             f"cv2 {res['host']['cv2']} ({res['host']['cv2_threads']} threads, IPP {'on' if res['host']['cv2_ipp'] else 'off'})",
             "480x640 image, boxsize 640, max_downsample 64, padValue 128; ms per image",
             f"{'scale x rotation':24s} {'items':>5s} {'launches':>8s} {'prenet (events)':>15s} {'GB/s':>7s} "
             f"{'upload+prenet':>13s} {'host chain':>10s} {'host/device':>11s}"]
    for c in res["configs"]:
        lines.append(f"{c['config']:24s} {c['items']:5d} {c['launches']:8d} {c['device_prenet_ms_events']:15.3f} "
                     f"{c['device_prenet_gbs']:7.0f} {c['device_upload_plus_prenet_ms_host_clock']:13.3f} "
                     f"{c['host_chain_ms_host_clock']:10.1f} {c['speedup_host_over_device']:10.0f}x")
    txt = "\n".join(lines) + "\n"
    with open(os.path.join(args.out_dir, "time_prenet.txt"), "w") as f:
        f.write(txt)
    print(txt, end="")


if __name__ == "__main__":
    main()
