#!/usr/bin/env python
"""bench.py -- grouping images/s on synthetic 128x128x(18+30) maps, 30 persons/image (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repo's CUDA path
    python bench.py --impl reference [--gpus N] ...                 # the reference's CPU algorithm (Python port)
    torchrun --nproc-per-node N ... bench.py --gpus N ...           # one rank per GPU, images sharded (weak scaling)
    python bench.py --config {p30,p10,f64,512}                      # the other single-GPU configurations (default p30)
    python bench.py --dump-outputs DIR                              # also write the last timed step's person lists to DIR

One pass = the hot path (peaks -> candidate scoring -> greedy matching -> person assembly + wire records, the window
/root/reference/evaluate.py:507-513 times plus the format_results payload) over one batch of images resident in HBM.
A "step" is `passes_per_step` passes, as many as make one step >= STEP_MS of device work, and `--steps K` times K
steps (every pass streams the whole input batch, which is larger than L2, from HBM).  At N > 1 every rank's assemble
kernel stores its wire records straight into rank 0's sink buffer over NVLink (sharding.PeerWireSink): the gather is
part of every pass.
One JSON line is printed by rank 0:

  value      whole-job images/s with the maps already resident in HBM, CUDA-event timed, max over ranks
  e2e        same metric through the C-ABI host entry point (spg_group_host): pinned HOST maps in, person lists
             back on the host, H2D/D2H inside the timed region
  roofline   the dominant kernel's algorithmic bytes / its CUDA-event time vs MEASURED_PEAKS.json's HBM peak
  kernels    per-kernel event times taken inside the timed steps
  cpu_baseline  the Python/numpy port of the reference's algorithm, one process, same batch (N=1 only)
"""
from __future__ import annotations

import argparse
import fcntl
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import threading
import time
import zlib

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

UNIT = "images/s"
STEP_MS = 5.0  # device time one step covers at least (the default 20 steps: >= 100 ms)
BASE_SEED = 20260921
CAP_ROWS = 64  # person-row capacity of the handles and of a wire record (<= 40 persons/image here; overflow trips the status assert)

# name -> workload.  p30 is the configuration the metric is quoted on (BASELINE configs[2]'s per-GPU shard).
CONFIGS = {
    "p30": dict(H=128, W=128, persons=30, batch=256, paf="f32", gen={},
                what="BASELINE configs[2] per-GPU shard: batch=256/GPU synthetic 128x128x(18+30) f32 maps, 30 persons/img"),
    "p10": dict(H=128, W=128, persons=10, batch=256, paf="f32", gen={},
                what="BASELINE configs[1]: batch=256 synthetic 128x128x(18+30) f32 maps, 10 persons/img, 1 GPU"),
    "f64": dict(H=128, W=128, persons=30, batch=256, paf="f64", gen={},
                what="configs[2]'s shard with float64 body-part maps -- the dtype predict() emits (evaluate.py:86,161)"),
    # pipeline configurations: the input is the NETWORK OUTPUT; the post-network stage (spg_postnet) is part of every pass
    "512": dict(H=512, W=512, persons=30, batch=32, paf="f64", gen={}, scales=(0.5, 1.0, 2.0), net_hw=(128, 128),
                what="BASELINE configs[3]: multi-scale x0.5/1/2 + flip-averaged maps -> grouping, 512x512 image, batch=32: network "
                     "outputs [32,2,50,{64,128,256}^2] f32 -> spg_postnet -> 512x512x(18 f32 + 30 f64) maps -> grouping, 30 persons/img"),
    "imhn": dict(H=512, W=512, persons=30, batch=8, paf="f32-as-f64", gen={}, scales=(1.0,), net_hw=(128, 128), imhn=True,
                 what="BASELINE configs[4] per-GPU shard: 8 images 512x512x3 (+ mirrored) -> 4-stack IMHN forward (random init as the "
                      "reference initialises it; bf16, channels-last, CUDA graph) -> [8,2,50,128,128] + injected synthetic maps (a "
                      "random-init network answers below thre1) -> spg_postnet -> 512x512 maps -> grouping, 30 persons/img"),
    "net128": dict(H=128, W=128, persons=30, batch=256, paf="f32-as-f64", gen={}, scales=(1.0,), net_hw=(32, 32),
                   what="configs[2]'s shard starting from the network output: [256,2,50,32,32] f32 -> spg_postnet (flip ensemble + x4 "
                        "bicubic) -> 128x128x(18+30) maps (f32 storage, the reference's f64 arithmetic) -> grouping, 30 persons/img"),
}


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", choices=["ours", "reference"], default="ours")
    ap.add_argument("--config", choices=sorted(CONFIGS), default="p30")
    ap.add_argument("--batch", type=int, default=0, help="images per GPU per pass (0 = the configuration's)")
    ap.add_argument("--persons", type=int, default=0, help="0 = the configuration's")
    ap.add_argument("--passes", type=int, default=0, help="passes per step (0 = as many as make a step >= STEP_MS)")
    ap.add_argument("--e2e-steps", type=int, default=0, help="0 = min(steps, 10)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-peer", action="store_true", help="N > 1: packed NCCL gather instead of NVLink peer stores")
    ap.add_argument("--trace", default="", help="write a per-rank CUDA-event timeline of 8 consecutive passes to this JSON file (rank 0)")
    ap.add_argument("--unfused", action="store_true", help="limb_match and assemble as two kernels instead of the fused match_assemble")
    ap.add_argument("--unmodified", action="store_true",
                    help="--impl reference only, build container only: time the UNMODIFIED reference functions (oracle/ref_loader)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="write the person lists the last timed step computed to DIR/<name>.npy (float64)")
    args = ap.parse_args()
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    cfg = CONFIGS[args.config]
    args.batch = args.batch or cfg["batch"]
    args.persons = args.persons or cfg["persons"]
    args.H, args.W, args.paf = cfg["H"], cfg["W"], cfg["paf"]
    if args.impl == "reference" and args.dump_outputs:
        raise SystemExit("--dump-outputs writes what the CUDA path computed: it does not apply to --impl reference")
    if args.impl == "reference" and "scales" in cfg:
        raise SystemExit("the reference arm times the grouping window (evaluate.py:507-513): use --config p30 / p10 / f64")
    return args


def metric_name(args):
    return f"grouping images/sec @{args.H}x{args.W} heatmaps, {args.persons} persons/img"


def workload_config(args, world, passes=None, gather=None):
    esz = 8 if args.paf == "f64" else 4
    mb = args.batch * (18 * 4 + 30 * esz) * args.H * args.W / 1e6
    c = {"workload": CONFIGS[args.config]["what"] if (args.batch, args.persons) == (CONFIGS[args.config]["batch"], CONFIGS[args.config]["persons"])
         else f"config {args.config} with batch={args.batch}/GPU, {args.persons} persons/img",
         "name": args.config, "batch_per_gpu": args.batch, "global_batch": args.batch * world, "persons": args.persons,
         "H": args.H, "W": args.W, "keypoint_channels": 18, "limb_channels": 30, "paf_dtype": args.paf,
         "capacities": {"max_peaks_per_part": 64, "max_cands_per_limb": 1024, "max_person_rows": CAP_ROWS, "wire_rows": CAP_ROWS},
         "parallelism": f"image-sharded x{world}" + (f"; person lists reach rank 0 by {gather}" if world > 1 else ""),
         "l2": f"inputs {mb:.0f} MB/GPU > 126 MB L2: every pass streams from HBM, no flush needed"}
    if passes is not None:
        c["passes_per_step"] = passes
        c["images_per_step"] = args.batch * world * passes
    return c


def make_shard(args, rank):
    from improved_body_parts_b200 import synth

    heat, paf = synth.make_batch(BASE_SEED + rank * args.batch, args.batch, args.H, args.W, args.persons, **CONFIGS[args.config]["gen"])
    if args.paf == "f64":  # as tests/golden/make_golden.py: values that are not f32-representable
        paf = paf.astype(np.float64) * (1.0 + 2.0 ** -30) + 2.0 ** -40
    return heat, paf


def build_once():
    """Every rank calls this; a file lock makes one of them compile while the others wait for the finished library.
    The lock lives in the temporary directory: the source tree may be read-only."""
    import __graft_entry__ as ge

    lock = os.path.join(tempfile.gettempdir(), f"spgroup-build-{zlib.crc32(ROOT.encode()):08x}.lock")
    with open(lock, "w") as fh:
        fcntl.flock(fh, fcntl.LOCK_EX)
        try:
            ge.build()
        finally:
            fcntl.flock(fh, fcntl.LOCK_UN)


def host_cpu_budget():
    """CPUs this process may actually use: affinity mask capped by the cgroup CPU quota (os.cpu_count() ignores both)."""
    affinity = len(os.sched_getaffinity(0))
    quota = None
    try:
        q, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = max(1, int(float(q) / float(period)))
    except (OSError, ValueError):
        pass
    usable = min(affinity, quota) if quota else affinity
    return {"os_cpu_count": os.cpu_count(), "affinity": affinity, "cgroup_quota_cpus": quota, "usable": usable}


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(dirname, views, B):
    """--dump-outputs: what a caller of the timed path receives -- person counts, keypoint coordinates, person scores and
    status flags -- as float64 ``DIR/<name>.npy``.  Rows at or beyond an image's person count are never written by the
    kernels and hold whatever an earlier pass left there, so they are stored as zeros.  Larger than DUMP_LIMIT_BYTES in
    all, a fixed seeded sample of the images is written, their indices in ``image_index.npy``."""
    out = {k: views[k][:B].cpu().numpy().astype(np.float64) for k in ("n_persons", "people_xy", "people_score", "status")}
    live = np.arange(out["people_score"].shape[1])[None, :] < out["n_persons"][:, None]
    out["people_xy"][~live] = 0.0
    out["people_score"][~live] = 0.0
    per_image = sum(v[0].nbytes for v in out.values()) + 8  # + its entry in image_index
    if B * per_image > DUMP_LIMIT_BYTES:
        idx = np.sort(np.random.default_rng(BASE_SEED).choice(B, DUMP_LIMIT_BYTES // per_image, replace=False))
        out = {k: v[idx] for k, v in out.items()}
        out["image_index"] = idx.astype(np.float64)
    os.makedirs(dirname, exist_ok=True)
    for k, v in out.items():
        np.save(os.path.join(dirname, k + ".npy"), v)


# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled in the background while the timed regions run."""
    Q = ("timestamp,index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.rows, self.proc, self.gpu = [], None, gpu_index
        self.windows = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._pump, daemon=True)
        self.thread.start()

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def window(self, t0, t1):
        self.windows.append((t0, t1))

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        time.sleep(0.12)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        inside = [r for t, r in self.rows if any(a - 0.03 <= t <= b + 0.03 for a, b in self.windows)]
        used, scope = (inside, "timed regions") if len(inside) >= 2 else ([r for _, r in self.rows], "whole run (timed regions shorter than the sampling period)")
        sm, smax, reasons = [], [], set()
        for r in used:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 10:
                continue
            try:
                sm.append(float(f[2])); smax.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[6:10]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "scope": scope}


# ------------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """--impl reference: the reference's CPU algorithm on the host cores this process may use, one image per task.

    The reference itself is pure Python and cannot travel to the GPU box, so the arm runs oracle/grouping_port.py --
    the Python/numpy port that is bit-pinned to reference-generated goldens.  Nothing of the product (no libspgroup.so,
    no CUDA) is loaded or built here.  With --unmodified (build container only) the UNMODIFIED reference functions are
    timed instead, single process as the README describes them."""
    if rank != 0:
        return
    from improved_body_parts_b200 import skeleton
    from oracle import grouping_port as gp

    cpus = host_cpu_budget()
    heat, paf = make_shard(args, 0)
    params = skeleton.default_params()
    extra = {}
    if args.unmodified:
        from oracle import ref_loader
        if not ref_loader.reference_available():
            raise SystemExit("--unmodified needs /root/reference (build container)")
        ref = ref_loader.Reference()
        n = min(args.batch, 4)
        hw = [np.ascontiguousarray(heat[i].transpose(1, 2, 0)) for i in range(n)]
        pw = [np.ascontiguousarray(paf[i].transpose(1, 2, 0)) for i in range(n)]
        ref.group(hw[0], pw[0], args.H, params)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            for i in range(n):
                ref.group(hw[i], pw[i], args.H, params)
        dt = time.perf_counter() - t0
        value, sample, cores, kind = n * args.steps / dt, n, 1, "reference"
        desc = f"{n} images per step through the UNMODIFIED evaluate.py functions (oracle/ref_loader.py), one process"
    else:
        workers = cpus["usable"]
        sample = min(args.batch, max(16, workers * 4))
        # single-process figure first (what the README describes), on a few images
        n1 = min(args.batch, 8)
        gp.group_image(heat[0], paf[0], args.H, params, skeleton.LIMBS)
        t0 = time.perf_counter()
        for i in range(n1):
            gp.group_image(heat[i], paf[i], args.H, params, skeleton.LIMBS)
        extra["single_process"] = {"value": n1 / (time.perf_counter() - t0), "unit": UNIT, "images": n1}
        pool, run = gp.make_pool(heat, paf, args.H, params, skeleton.LIMBS, workers=workers)
        try:
            for _ in range(max(args.warmup, 1)):
                run(range(sample))
            t0 = time.perf_counter()
            for _ in range(args.steps):
                run(range(sample))
            dt = time.perf_counter() - t0
        finally:
            pool.close()
            pool.join()
        value, cores, kind = sample * args.steps / dt, workers, "port"
        desc = (f"{sample} images of the batch per step, fork pool of {workers} processes (= usable CPUs: affinity "
                f"{cpus['affinity']}, cgroup quota {cpus['cgroup_quota_cpus']}, os.cpu_count {cpus['os_cpu_count']}), one image per task")
    try:
        import torch
        extra["torch_threads"] = torch.get_num_threads()
    except Exception:
        pass
    print(json.dumps({
        "impl": "reference", "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": f"{args.paf} maps; f64 coordinates", "data": "synthetic", "config": workload_config(args, world),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": desc, "cpus": cpus, **extra},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0}), flush=True)


# ------------------------------------------------------------------------------------------------------
def run_ours(args, rank, world, local_rank):
    import torch
    import torch.distributed as dist

    from improved_body_parts_b200 import skeleton, wire
    from improved_body_parts_b200.grouping import Grouper, GroupingError
    from improved_body_parts_b200.sharding import PackedGather, PeerWireSink

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the grouping path has no CPU fallback")
    if args.unfused:
        os.environ["SPG_FUSE_MA"] = "0"  # read once at spg_create: the host entry point then runs the two kernels too
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    H, W, B = args.H, args.W, args.batch
    heat_np, paf_np = make_shard(args, rank)
    params = skeleton.default_params()
    heat_pin = torch.from_numpy(heat_np).pin_memory()
    paf_pin = torch.from_numpy(paf_np).pin_memory()
    heat_d = heat_pin.to(dev, non_blocking=True)
    paf_d = paf_pin.to(dev, non_blocking=True)
    g = Grouper(max_batch=B, max_h=H, max_w=W, max_person_rows=CAP_ROWS, device=local_rank)
    views = g.device_tensors()
    rb = g.wire_record_bytes(CAP_ROWS)
    stream = torch.cuda.current_stream()

    # ---- where the wire records go: a local buffer at N = 1; rank 0's sink over NVLink at N > 1
    sink = pg = None
    local_wire = torch.zeros((B, rb), dtype=torch.uint8, device=dev)
    gather_how = None
    if world > 1:
        if not args.no_peer:
            try:
                sink = PeerWireSink(B, rb, local_rank, dst=0, slots=4)
                gather_how = "NVLink peer stores from the assemble kernel into rank 0's sink (CUDA IPC; no collective kernel)"
            except GroupingError as e:
                gather_how = f"packed NCCL gather (peer mapping unavailable: {e})"
        if sink is None:
            pg = PackedGather(B, rb, dev, dst=0)
            gather_how = gather_how or "one packed NCCL gather per pass (pre-allocated buffers)"
    cstream = torch.cuda.Stream(device=dev) if (sink is not None and rank == 0) else None
    pass_no = [0]
    stages = [lambda: g.nms_peaks(heat_d, params), lambda: g.limb_score(paf_d, H, params)]
    stages += [lambda: g.limb_match(B, params), lambda: g.assemble(B, params)] if args.unfused else [lambda: g.match_assemble(B, params)]
    n_stage = len(stages)

    def one_pass(evs=None):
        s = pass_no[0]
        pass_no[0] += 1
        if pg is not None:
            g.set_wire_output(pg.local.data_ptr(), 0, CAP_ROWS)
        elif sink is None:
            g.set_wire_output(local_wire.data_ptr(), 0, CAP_ROWS)
        for i, fn in enumerate(stages):
            if evs: evs[i].record(stream)
            if sink is not None and i == n_stage - 1:  # only the assemble stage needs the sink slot
                g.set_wire_output(sink.begin(s, stream), 0, CAP_ROWS)
                g.arm_wire_signal(sink.counter_address(s), s + 1)  # its last CTA publishes "step s landed" itself
            fn()
        if evs: evs[n_stage].record(stream)
        if sink is not None:
            if rank == 0:  # the consumer: waits for every rank's counters (stream memory ops), then frees the generation
                sink.collect(s, cstream)
                sink.release(s, cstream)
        elif pg is not None:
            pg.gather()
        if evs: evs[n_stage + 1].record(stream)

    def join_consumer():
        if cstream is not None:
            e = torch.cuda.Event()
            e.record(cstream)
            stream.wait_event(e)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    if sampler:
        sampler.start()

    n_ev = n_stage + 2
    for _ in range(3):
        one_pass()
    join_consumer()
    barrier()
    # ---- passes per step: enough that a step covers >= STEP_MS of device time (same number on every rank)
    passes = args.passes
    if passes <= 0:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for _ in range(4):
            one_pass()
        join_consumer()
        e1.record(stream)
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / 4], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MIN)
        passes = max(1, min(64, math.ceil(STEP_MS / float(t.item()))))
    for _ in range(max(args.warmup, 3)):
        for _ in range(passes):
            one_pass()
    join_consumer()
    barrier()
    # Per-kernel durations: CUDA events around every kernel of the FIRST pass of every step of the timed region (an event
    # between two kernels costs ~2.5 us of launch gap, so not every pass carries them); the region has its own two events.
    evs = [[torch.cuda.Event(enable_timing=True) for _ in range(n_ev)] for _ in range(args.steps)]
    ev_start, ev_end = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    l0 = g.launch_count
    w0 = time.time()
    ev_start.record(stream)
    for k in range(args.steps):
        for p in range(passes):
            one_pass(evs[k] if (p == 0 and passes > 1) or (passes == 1 and k % 5 == 0) else None)
    join_consumer()
    ev_end.record(stream)
    torch.cuda.synchronize()
    w1 = time.time()
    launches = g.launch_count - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, views, B)
    barrier()
    elapsed_ms = ev_start.elapsed_time(ev_end)
    used = [e for k, e in enumerate(evs) if passes > 1 or k % 5 == 0]
    stage_ms = [statistics.fmean(e[i].elapsed_time(e[i + 1]) for e in used) for i in range(n_ev - 1)]
    if sampler:
        sampler.window(w0, w1)
    t = torch.tensor([elapsed_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms = float(t.item())
    n_pass = args.steps * passes
    value = world * B * n_pass / (elapsed_ms / 1e3)

    # ---- optional timeline (nsys is not installed in this image): CUDA events around every stage of 8 consecutive passes
    if args.trace:
        barrier()
        tev = [[torch.cuda.Event(enable_timing=True) for _ in range(n_ev)] for _ in range(8)]
        for e in tev:
            one_pass(e)
        join_consumer()
        torch.cuda.synchronize()
        mine = [[tev[0][0].elapsed_time(x) for x in e] for e in tev]  # ms since the first pass started, per rank
        allr = [None] * world
        if world > 1:
            dist.all_gather_object(allr, mine)
        else:
            allr = [mine]
        if rank == 0:
            labels = ["nms_peaks", "limb_score"] + (["limb_match", "assemble"] if args.unfused else ["match_assemble"]) + ["publish/gather", "end"]
            json.dump({"what": "CUDA-event timestamps (ms since the rank's first pass began) at the start of each stage of 8 consecutive passes",
                       "labels": labels, "n_gpus": world, "gather": gather_how, "ranks": allr}, open(args.trace, "w"))
        barrier()

    # ---- correctness guards inside the bench: statuses clean, persons found, wire records = the device tables,
    # and at N > 1 what landed on rank 0 is byte for byte what every rank produced
    r_status = views["status"][:B].cpu().numpy()
    r_np = views["n_persons"][:B].cpu().numpy()
    assert (r_status == 0).all(), f"status flags set: {np.unique(r_status)}"
    assert r_np.min() > 0, "no persons found -- the timed path did no work"
    g.set_wire_output(local_wire.data_ptr(), 0, CAP_ROWS)
    stages[-1]()
    torch.cuda.synchronize()
    mine = local_wire.cpu().numpy()
    rec = wire.as_records(mine, 17, CAP_ROWS)
    assert np.array_equal(rec["n_persons"], r_np) and not rec["status"].any()
    xy, sc = views["people_xy"][:B].cpu().numpy(), views["people_score"][:B].cpu().numpy()
    for i in range(0, B, max(1, B // 16)):
        n = int(r_np[i])
        assert np.array_equal(rec[i]["rows"]["xy"][:n], xy[i, :n]) and np.array_equal(rec[i]["rows"]["score"][:n], sc[i, :n])
    gather_ok = None
    if world > 1:
        crc = zlib.crc32(mine.tobytes())
        crcs = [None] * world
        dist.all_gather_object(crcs, crc)
        if rank == 0:
            last = pass_no[0] - 1
            if sink is not None:
                landed = sink.collect(last, stream).cpu().numpy()  # already complete: only maps the generation of the last pass
            else:
                landed = pg.records().cpu().numpy()
            got = [zlib.crc32(landed[r * B:(r + 1) * B].tobytes()) for r in range(world)]
            gather_ok = got == crcs
            assert gather_ok, f"records on rank 0 differ from what the ranks produced: {got} vs {crcs}"

    # ---- e2e: HOST maps -> spg_group_host (H2D + kernels + D2H inside) -> person lists on the host
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    out = None

    def host_call(out):
        # at N > 1 the records of the call also travel to rank 0 (same sink, same hand-shakes as the device-resident passes)
        s = pass_no[0]
        pass_no[0] += 1
        if sink is not None:
            g.set_wire_output(sink.begin(s, stream), 0, CAP_ROWS)
            stream.synchronize()  # spg_group_host runs on the library's own streams: the slot must be free before it starts
        elif pg is not None:
            g.set_wire_output(pg.local.data_ptr(), 0, CAP_ROWS)
        else:
            g.set_wire_output(local_wire.data_ptr(), 0, CAP_ROWS)
        out = g.group_host(heat_pin.numpy(), paf_pin.numpy(), H, params, out)
        if sink is not None:
            sink.publish(s, stream)
            if rank == 0:
                sink.collect(s, cstream)
                sink.release(s, cstream)
        elif pg is not None:
            pg.gather()
        return out

    for _ in range(2):
        out = host_call(out)
    join_consumer()
    barrier()
    w0 = time.time()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        out = host_call(out)
    join_consumer()
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    w1 = time.time()
    if sampler:
        sampler.window(w0, w1)
    t = torch.tensor([e2e_s], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_s = float(t.item())
    e2e_value = world * B * e2e_steps / e2e_s
    assert np.array_equal(out["n_persons"], r_np), "host entry point disagrees with the device entry point"
    h2d = world * (heat_np.nbytes + paf_np.nbytes)
    d2h = world * sum(out[k].nbytes for k in ("n_persons", "people_xy", "people_score", "status"))
    clocks = sampler.stop() if sampler else None

    if sink is not None:
        sink.close()
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline of the dominant kernel (algorithmic bytes per launch / event time)
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        hbm_peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        hbm_peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
    names = [nme for nme in g.stage_kernels() if nme][:n_stage]  # the kernel variants that actually ran (ncu names)
    esz = 8 if args.paf == "f64" else 4
    alg_bytes = [B * 18 * H * W * 4, B * 30 * H * W * esz, None, None][:n_stage]  # DESIGN.md: K1 reads heat once, K2a reads the body-part maps once
    kernels = {}
    for i, nme in enumerate(names):
        kernels[nme] = {"ms": stage_ms[i], "algorithmic_GBps": (alg_bytes[i] / (stage_ms[i] * 1e-3) / 1e9) if alg_bytes[i] else None,
                        "frac_of_hbm_peak": (alg_bytes[i] / (stage_ms[i] * 1e-3) / 1e9 / hbm_peak) if alg_bytes[i] else None}
    if world > 1:
        kernels["gather"] = {"ms": stage_ms[n_stage], "note": gather_how}
    dom = max(range(n_stage), key=lambda i: stage_ms[i])
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and args.config == "p30":
        tr = {k.replace(" ", "").replace("spg::", ""): v for k, v in json.load(open(tpath)).items()}
        traffic = tr.get(names[dom].replace(" ", ""), tr.get(names[dom].split("<")[0]))  # ncu capture of the same kernel (template spelling may differ)
    path_bytes = B * (18 * 4 + 30 * esz) * H * W
    if alg_bytes[dom]:
        ach = alg_bytes[dom] / (stage_ms[dom] * 1e-3) / 1e9
        roofline = {"kernel": names[dom], "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": alg_bytes[dom]}
    else:
        ach = path_bytes / (stage_ms[dom] * 1e-3) / 1e9
        roofline = {"kernel": names[dom], "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s",
                    "frac": ach / hbm_peak, "traffic": traffic, "peak_source": peak_src,
                    "algorithmic_bytes_per_launch": path_bytes,
                    "note": "serial, latency-bound kernel; bytes are the whole path's per-image figure x batch"}
    roofline["limb_score_frac"] = kernels[names[1]]["frac_of_hbm_peak"]
    roofline["nms_peaks_frac"] = kernels[names[0]]["frac_of_hbm_peak"]
    ms_per_pass = elapsed_ms / n_pass
    roofline["whole_path_frac"] = path_bytes / (ms_per_pass * 1e-3) / 1e9 / hbm_peak

    result = {
        "metric": metric_name(args), "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": elapsed_ms / args.steps, "ms_per_pass": ms_per_pass, "timed_region_ms": elapsed_ms,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": f"{args.paf} body-part maps, f32 keypoint maps; f64 coordinates/scores", "data": "synthetic",
        "config": workload_config(args, world, passes, gather_how),
        "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "steps": e2e_steps, "api": "spg_group_host (C ABI, pinned host maps in, person lists out); one call per step"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kernels,
        "kernel_timing": f"CUDA events around every kernel of {len(used)} passes inside the timed region ({n_pass} passes)",
        "persons_found_per_image": float(r_np.mean()), "gather_verified": gather_ok,
    }

    if world == 1 and not args.no_cpu_baseline:
        from oracle import grouping_port as gp
        from oracle import spg_oracle as so

        n_cpu = min(B, 256 if H * W <= 128 * 128 else 8)
        gp.group_image(heat_np[0], paf_np[0], H, params, skeleton.LIMBS)
        t0 = time.perf_counter()
        found = [gp.group_image(heat_np[i], paf_np[i], H, params, skeleton.LIMBS)[3].shape[0] for i in range(n_cpu)]
        dt = time.perf_counter() - t0
        assert found == [int(v) for v in r_np[:n_cpu]], "CPU port and CUDA path disagree on person counts"
        result["cpu_baseline"] = {"value": n_cpu / dt, "unit": UNIT, "cores": 1, "kind": "port",
                                  "sample": f"first {n_cpu} images of the same batch, Python/numpy port of the reference "
                                            f"(oracle/grouping_port.py), one process, {dt:.1f} s"}
        t0 = time.perf_counter()
        so.group_batch(heat_np, paf_np, skeleton.LIMBS, H, params, threads=1)
        dt1 = time.perf_counter() - t0
        nt = min(so.max_threads(), host_cpu_budget()["usable"])
        t0 = time.perf_counter()
        so.group_batch(heat_np, paf_np, skeleton.LIMBS, H, params, threads=nt)
        dtn = time.perf_counter() - t0
        result["cpu_checker_c"] = {"single_thread": B / dt1, "all_threads": B / dtn, "threads": nt, "unit": UNIT,
                                   "note": "oracle/spg_oracle.c, a C rewrite used as test checker (not the reference's implementation)"}
    print(json.dumps(result), flush=True)
    if world > 1:
        dist.destroy_process_group()


# ------------------------------------------------------------------------------------------------------
def make_network_outputs(args):
    """Per scale: [B, 2, 50, h, w] float32 network outputs of the same synthetic people (synth.make_network_output)."""
    from improved_body_parts_b200 import synth
    cfg = CONFIGS[args.config]
    bh, bw = cfg["net_hw"]
    outs, crops = [], []
    for f in cfg["scales"]:
        h, w = int(round(bh * f)), int(round(bw * f))
        outs.append(np.stack([synth.make_network_output(BASE_SEED + i, h, w, args.persons, body_scale=f, base_hw=(bh, bw))
                              for i in range(args.batch)]))
        crops.append((4 * h, 4 * w))  # no padding: the scaled image is a multiple of max_downsample
    return outs, crops


def run_pipeline(args, local_rank):
    """Configurations whose input is the network output: one pass = spg_postnet (evaluate.py:126-161) + the grouping path."""
    import torch

    from improved_body_parts_b200 import skeleton
    from improved_body_parts_b200.grouping import Grouper

    if not torch.cuda.is_available():
        raise SystemExit("bench.py (impl=ours) needs a CUDA device: the grouping path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    H, W, B = args.H, args.W, args.batch
    cfg = CONFIGS[args.config]
    params = skeleton.default_params()
    outs_np, crops = make_network_outputs(args)
    outs_pin = [torch.from_numpy(o).pin_memory() for o in outs_np]
    outs_d = [o.to(dev, non_blocking=True) for o in outs_pin]
    single = len(outs_d) == 1
    g = Grouper(max_batch=B, max_h=H, max_w=W, max_person_rows=CAP_ROWS, device=local_rank)
    views = g.device_tensors()
    heat_d = torch.empty((B, 18, H, W), dtype=torch.float32, device=dev)
    paf_d = torch.empty((B, 30, H, W), dtype=torch.float32 if single else torch.float64, device=dev)
    local_wire = torch.zeros((B, g.wire_record_bytes(CAP_ROWS)), dtype=torch.uint8, device=dev)
    g.set_wire_output(local_wire.data_ptr(), 0, CAP_ROWS)
    stream = torch.cuda.current_stream()
    runner = None
    if cfg.get("imhn"):
        from improved_body_parts_b200.imhn import IMHN, Runner
        runner = Runner(IMHN().init_like_reference_(0), device=dev)
        imgs_pin = torch.rand((B, 4 * cfg["net_hw"][0], 4 * cfg["net_hw"][1], 3), generator=torch.Generator().manual_seed(7)).pin_memory()
        imgs_d = imgs_pin.to(dev, non_blocking=True)
        pair_d = torch.empty((2 * B,) + tuple(imgs_d.shape[1:]), device=dev)
        inject = outs_d[0]            # the synthetic maps, added to what the random-init network answers
        outs_d = [torch.empty_like(inject)]

        def forward(src):
            pair_d[0::2].copy_(src)                      # image, mirrored image interleaved: [B,2,...] after the view (evaluate.py:116-121)
            pair_d[1::2].copy_(src.flip(2))
            raw = runner(pair_d)                         # [2B,50,h,w] float32 = output_tuple[-1][0]
            torch.add(raw.view(B, 2, 50, raw.shape[2], raw.shape[3]), inject, out=outs_d[0])
    stages = ([("imhn_forward", lambda: forward(imgs_d))] if runner else []) + [
              ("postnet_kernel", lambda: g.postnet(outs_d, crops, (H, W), heat_out=heat_d, paf_out=paf_d)),
              ("nms", lambda: g.nms_peaks(heat_d, params)),
              ("score", lambda: g.limb_score(paf_d, H, params, paf_as_f64=single)),
              ("match_assemble", lambda: g.match_assemble(B, params))]
    n_pre = len(stages) - 3       # stages in front of the three grouping kernels

    def one_pass(evs=None, first=0):
        for i, (_, fn) in enumerate(stages[first:]):
            if evs: evs[i].record(stream)
            fn()
        if evs: evs[len(stages) - first].record(stream)

    sampler = ClockSampler(local_rank)
    sampler.start()
    for _ in range(3):
        one_pass()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for _ in range(4):
        one_pass()
    e1.record(stream)
    torch.cuda.synchronize()
    passes = args.passes or max(1, min(64, math.ceil(STEP_MS / (e0.elapsed_time(e1) / 4))))
    for _ in range(max(args.warmup, 3) * passes):
        one_pass()
    torch.cuda.synchronize()

    def timed(first):
        evs = [[torch.cuda.Event(enable_timing=True) for _ in range(len(stages) + 1)] for _ in range(args.steps)]
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        w0 = time.time()
        a.record(stream)
        for k in range(args.steps):
            for p in range(passes):
                one_pass(evs[k] if p == 0 else None, first)
        b.record(stream)
        torch.cuda.synchronize()
        sampler.window(w0, time.time())
        ms = [statistics.fmean(e[i].elapsed_time(e[i + 1]) for e in evs) for i in range(len(stages) - first)]
        return a.elapsed_time(b), ms

    l0 = g.launch_count
    elapsed_ms, stage_ms = timed(0)          # value: post-network stage + grouping
    launches = g.launch_count - l0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, views, B)
    group_ms, _ = timed(n_pre)               # the grouping stages alone on the resident maps
    n_pass = args.steps * passes
    value = B * n_pass / (elapsed_ms / 1e3)
    r_status = views["status"][:B].cpu().numpy()
    r_np = views["n_persons"][:B].cpu().numpy()
    assert (r_status == 0).all(), f"status flags set: {np.unique(r_status)}"
    assert r_np.min() > 0, "no persons found -- the timed path did no work"

    # ---- e2e: pinned HOST network outputs -> H2D -> postnet -> grouping -> person lists on the host, every step
    e2e_steps = args.e2e_steps or min(args.steps, 10)
    host_out = {k: torch.empty_like(views[k][:B], device="cpu").pin_memory() for k in ("n_persons", "people_xy", "people_score", "status")}
    stage_in = [torch.empty_like(o) for o in outs_d]
    img_in = torch.empty_like(imgs_d) if runner else None

    def host_call():
        if runner:
            img_in.copy_(imgs_pin, non_blocking=True)
            forward(img_in)
            g.postnet(outs_d, crops, (H, W), heat_out=heat_d, paf_out=paf_d)
        else:
            for dst, src in zip(stage_in, outs_pin):
                dst.copy_(src, non_blocking=True)
            g.postnet(stage_in, crops, (H, W), heat_out=heat_d, paf_out=paf_d)
        g.group_device(heat_d, paf_d, H, params, paf_as_f64=single)
        for k, t in host_out.items():
            t.copy_(views[k][:B], non_blocking=True)
        torch.cuda.synchronize()

    for _ in range(2):
        host_call()
    w0 = time.time()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        host_call()
    e2e_s = time.perf_counter() - t0
    sampler.window(w0, time.time())
    assert np.array_equal(host_out["n_persons"].numpy(), r_np)
    h2d = imgs_pin.numel() * 4 if runner else sum(o.nbytes for o in outs_np)
    d2h = sum(t.numel() * t.element_size() for t in host_out.values())
    clocks = sampler.stop()

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        hbm_peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (of measured)"
    else:
        hbm_peak, peak_src = 6650.0, "B200_PROFILING.md fallback 6.65 TB/s (of fallback)"
    esz = 4 if single else 8
    ns = len(outs_d)
    net_read = sum(B * 2 * 48 * o.shape[3] * o.shape[4] * 4 for o in outs_d)
    plane = B * H * W
    if single:
        post_bytes = net_read + plane * (18 * 4 + 30 * 4)
    else:
        # the scale loop runs inside the kernel (groups of 4 scales): network outputs read once, float32 keypoint maps and
        # float64 body-part maps written once; a further group of scales re-reads and re-writes the float64 sums
        # (48 planes: the keypoint sums live in a float64 scratch until the last group)
        groups = (ns + 3) // 4
        post_bytes = net_read + plane * (18 * 4 + 30 * 8) + (groups - 1) * plane * 48 * 8 * 2
    alg = [None] * n_pre + [plane * 18 * 4, plane * 30 * esz, None]
    alg[n_pre - 1] = post_bytes
    names = [g.postnet_kernel() if nme == "postnet_kernel" else nme for nme, _ in stages[:n_pre]] + [n for n in g.stage_kernels() if n][:3]
    kernels = {}
    for i, nme in enumerate(names):
        kernels[nme] = {"ms": stage_ms[i], "algorithmic_GBps": alg[i] / (stage_ms[i] * 1e-3) / 1e9 if alg[i] else None,
                        "frac_of_hbm_peak": alg[i] / (stage_ms[i] * 1e-3) / 1e9 / hbm_peak if alg[i] else None}
        if nme.startswith("postnet") and ns > 4:
            kernels[nme]["launches_per_pass"] = (ns + 3) // 4
        if nme == "imhn_forward":
            kernels[nme]["note"] = "cuDNN/cuBLAS library kernels inside one CUDA graph (imhn.Runner); not a kernel of this repo"
    dom = max(range(n_pre - 1, len(names)), key=lambda i: stage_ms[i])  # dominant kernel of THIS repo (the network is library code)
    ach = (alg[dom] or sum(a for a in alg if a)) / (stage_ms[dom] * 1e-3) / 1e9
    traffic = None   # ncu capture of the same kernel on the same configuration (profiles/traffic.json), if there is one
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and args.config in ("net128", "512"):
        tr = json.load(open(tpath))
        suffix = "@512" if args.config == "512" else ""
        hits = [v for k, v in tr.items() if k.split("<")[0] == names[dom].split("<")[0] and k.endswith(suffix) and ("@" in k) == bool(suffix)]
        traffic = hits[-1] if hits else None
    roofline = {"kernel": names[dom], "bound": "hbm", "achieved": ach, "peak": hbm_peak, "unit": "GB/s", "frac": ach / hbm_peak,
                "traffic": traffic, "peak_source": peak_src, "algorithmic_bytes_per_launch": alg[dom]}
    result = {
        "metric": metric_name(args) + (" (from the images: network + post-network stage + grouping)" if runner else " (from the network output)"), "value": value, "unit": UNIT, "n_gpus": 1, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": elapsed_ms / args.steps, "ms_per_pass": elapsed_ms / n_pass,
        "timed_region_ms": elapsed_ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": f"f32 network output; {cfg['paf']} body-part maps, f32 keypoint maps; f64 coordinates/scores", "data": "synthetic",
        "config": dict(workload_config(args, 1, passes), network_output=[list(o.shape) for o in outs_d], crops=crops),
        "grouping_only": {"value": B * n_pass / (group_ms / 1e3), "unit": UNIT, "ms_per_pass": group_ms / n_pass,
                          "note": "the three grouping kernels alone on the resident maps the post-network stage produced"},
        "e2e": {"value": B * e2e_steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": e2e_steps,
                "api": "Grouper.postnet + Grouper.group_device on pinned host network outputs, person lists copied back; one call per step"},
        "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline, "kernels": kernels,
        "persons_found_per_image": float(r_np.mean()),
    }
    if not args.no_cpu_baseline and not runner:
        from oracle import grouping_port as gp
        from oracle import postnet_port as pp
        n_cpu = 2 if H > 128 else 16
        t0 = time.perf_counter()
        found = []
        for i in range(n_cpu):
            ha, pa = np.zeros((H, W, 18)), np.zeros((H, W, 30))
            for o, (ch, cw) in zip(outs_np, crops):
                hm, pf = pp.post_network_scale(o[i], 4, (ch, cw), [0, 0, 0, 0], (H, W), 30, 48, skeleton.FLIP_PAF_ORD, skeleton.FLIP_HEAT_ORD[:18])
                ha, pa = pp.accumulate(ha, hm, ns), pp.accumulate(pa, pf, ns)
            found.append(gp.group_image(np.ascontiguousarray(ha.transpose(2, 0, 1)).astype(np.float32),
                                        np.ascontiguousarray(pa.transpose(2, 0, 1)), H, params, skeleton.LIMBS)[3].shape[0])
        dt = time.perf_counter() - t0
        assert found == [int(v) for v in r_np[:n_cpu]], f"CPU pipeline and CUDA pipeline disagree on person counts: {found} vs {r_np[:n_cpu]}"
        result["cpu_baseline"] = {"value": n_cpu / dt, "unit": UNIT, "cores": 1, "kind": "port",
                                  "sample": f"first {n_cpu} images: oracle/postnet_port.py + oracle/grouping_port.py (Python/numpy ports "
                                            f"of evaluate.py:126-161 and :169-498), one process, {dt:.1f} s"}
    print(json.dumps(result), flush=True)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if world == 1 and args.gpus > 1 and args.impl == "ours":
        raise SystemExit(f"--gpus {args.gpus} needs `python -m torch.distributed.run --nproc-per-node {args.gpus} bench.py ...`")
    if args.impl == "reference":
        run_reference(args, rank, world)  # pure Python: builds and loads nothing of the product
    elif "scales" in CONFIGS[args.config]:
        if world > 1:
            raise SystemExit("the pipeline configurations are single-GPU configurations")
        build_once()
        run_pipeline(args, local_rank)
    else:
        build_once()
        run_ours(args, rank, world, local_rank)


if __name__ == "__main__":
    main()
