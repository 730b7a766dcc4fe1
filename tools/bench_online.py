"""Online augmentation from a device-resident dataset against the engine's other two ways of being fed, in one process.

Workload: bench.py's c3 shape (256-scan batches of 120 000-point KITTI-shape scans, 112 x 1440 range image, 1024 yaw
candidates, 10 objects per scan) from a store of 1024 distinct scans: bench.py's 32 c3 scenes, each in 32 variants whose
intensities are redrawn (2.2 GB of points + labels: larger than L2, so the gather reads HBM).

    python tools/bench_online.py [--batches 20] [--warmup 2] [--depth 3] [--out DIR]            rates
    python tools/bench_online.py --profile [--out DIR]                                           kernel times + copies
    python tools/bench_online.py --targets [--world-aug] [--rounds 3] [--out DIR]                 variants A/B

Rates (scans/s, host clock around work that ends in a device synchronise):
  * online     OnlineAugmenter.epochs over the store, a new epoch each pass (gather + device schedule draw + run), and
               the same with one OnlineAugmenter.epoch call per epoch (the look-ahead restarts at every epoch);
  * resident   the same engines' reset(from_raw_points=True) + run loop (bench.py's device-resident definition);
  * host       load + run of a batch staged in pinned host buffers (Real3DEngine.stage, outside the timed loop).
--profile: torch.profiler over a few online batches: device time of k_gather_points and k_draw_schedule, the gather's
bytes per second against a device-to-device copy measured in the same run, and every host-to-device copy of a batch.
--targets / --world-aug: the online rate of plain batches, of batches with detection targets (targets_device) and, with
--world-aug, of batches with targets and world augmentation, alternating the variants round by round on the same
engines; with --profile, the kernel times of a plain epoch and of an epoch with the variant's options, in one process.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_STORE = 1024
BATCH = 256


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return q.stdout.strip().splitlines()[0] if q.returncode == 0 and q.stdout.strip() else "unknown"


TARGETS = ["Car", "Pedestrian", "Cyclist"]


def setup(depth, targets=False, world_aug=None):
    import bench
    from pcl_augmentation_b200.engine import scan_input_from_case
    from pcl_augmentation_b200.online import OnlineAugmenter, ResidentDataset
    w = bench.WORKLOADS["c3"]
    base = bench.build_cases("c3", 0)[:w["distinct"]]
    scans = []
    for j in range(N_STORE):
        s = scan_input_from_case(base[j % len(base)])
        if j >= len(base):
            s.xyzi = s.xyzi.copy()
            s.xyzi[:, 3] = np.random.default_rng(j).uniform(0.0, 1.0, len(s.xyzi)).astype(np.float32)
        scans.append(s)
    store = ResidentDataset.from_scans("od", scans)
    kw = bench.engine_kwargs("c3", base)
    kw.pop("max_scans"), kw.pop("map_data")
    c0 = base[0]
    aug = OnlineAugmenter("od", c0.config, c0.db, store, batch_size=BATCH, seed=2024, depth=depth,
                          target_classes=TARGETS if targets else None, world_aug=world_aug, **kw)
    return aug, store, scans


def set_variant(aug, targets, world_aug):
    """Switch an augmenter built with targets between the variants (its target buffers stay allocated)."""
    aug.target_classes = TARGETS if targets else None
    aug.world_aug = world_aug
    for e in aug.engines:
        e.set_world_aug(world_aug)


def variants(args):
    import torch
    from pcl_augmentation_b200.online import WorldAug
    aug, store, _ = setup(args.depth, targets=True)
    names = {"online": (False, None), "online_targets": (True, None)}
    if args.world_aug:
        names["online_targets_world"] = (True, WorldAug())
    per_epoch = N_STORE // BATCH
    n_epochs = -(-args.batches // per_epoch)
    out = {"card": card(), "store_scans": N_STORE, "batch": BATCH, "rounds": args.rounds}
    for name, (t, w) in names.items():                  # warm every variant
        set_variant(aug, t, w)
        for _ in aug.epochs(range(10_000, 10_000 + -(-args.warmup // per_epoch))):
            pass
    torch.cuda.synchronize()
    rates_by = {k: [] for k in names}
    epoch = 0
    for _ in range(args.rounds):
        for name, (t, w) in names.items():
            set_variant(aug, t, w)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            n = 0
            for _, b in aug.epochs(range(epoch, epoch + n_epochs)):
                n += len(b.indices)
            torch.cuda.synchronize()
            rates_by[name].append(n / (time.perf_counter() - t0))
            epoch += n_epochs
    for name, r in rates_by.items():
        out[name + "_scans_per_s"] = r
        out[name + "_median"] = float(np.median(r))
    for name in names:
        out[name + "_over_online"] = out[name + "_median"] / out["online_median"]
    aug.close()
    return out


def rates(args):
    import torch
    aug, store, scans = setup(args.depth)
    out = {"card": card(), "store_scans": N_STORE, "batch": BATCH, "store_bytes": int(store.h_point_offsets[-1]) * 18}
    per_epoch = N_STORE // BATCH
    n_epochs = -(-args.batches // per_epoch)
    for _ in aug.epochs(range(10_000, 10_000 + -(-args.warmup // per_epoch))):
        pass
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = 0
    for _, b in aug.epochs(range(n_epochs)):         # one pipeline across the epochs
        n += len(b.indices)
    torch.cuda.synchronize()
    out["online_scans_per_s"] = n / (time.perf_counter() - t0)
    out["online_batches"] = n // BATCH
    t0 = time.perf_counter()
    n = 0
    for e in range(n_epochs):                         # epoch by epoch: the pipeline drains at each boundary
        for b in aug.epoch(e):
            n += len(b.indices)
    torch.cuda.synchronize()
    out["online_per_epoch_loop_scans_per_s"] = n / (time.perf_counter() - t0)
    # the same engines, each re-running the batch it holds from the raw resident points
    engines = aug.engines
    for e in engines:
        e.sync()
    t0 = time.perf_counter()
    steps = n_epochs * per_epoch
    for k in range(steps):
        engines[k % len(engines)].reset(from_raw_points=True)
        engines[k % len(engines)].run()
    for e in engines:
        e.sync()
    out["resident_scans_per_s"] = steps * BATCH / (time.perf_counter() - t0)
    # pinned host buffers -> device -> run (the stage() packing itself is outside the loop)
    staged = engines[0].stage(scans[:BATCH])
    for e in engines:
        e.load(staged); e.run()
    for e in engines:
        e.sync()
    t0 = time.perf_counter()
    for k in range(steps):
        engines[k % len(engines)].load(staged)
        engines[k % len(engines)].run()
    for e in engines:
        e.sync()
    out["host_load_scans_per_s"] = steps * BATCH / (time.perf_counter() - t0)
    out["online_over_resident"] = out["online_scans_per_s"] / out["resident_scans_per_s"]
    aug.close()
    return out


def profile(args):
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    from pcl_augmentation_b200.online import WorldAug
    aug, store, _ = setup(args.depth, targets=args.targets)
    set_variant(aug, False, None)
    for _ in aug.epoch(99):
        pass
    torch.cuda.synchronize()
    # copy peak of this card: a device-to-device copy of 2 GiB (read + write)
    src = torch.empty(1 << 31, dtype=torch.uint8, device="cuda")
    dst = torch.empty_like(src)
    dst.copy_(src)
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(10):
        dst.copy_(src)
    ev1.record()
    torch.cuda.synchronize()
    copy_bps = 10 * 2 * src.numel() / (ev0.elapsed_time(ev1) * 1e-3)
    del src, dst
    n_batches = 0
    with tprofile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        for b in aug.epoch(0):
            n_batches += 1
        torch.cuda.synchronize()
    trace = os.path.join(tempfile.mkdtemp(), "online.pt.trace.json")
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    kern = {}
    h2d = []
    for ev in events:
        name, cat = ev.get("name", ""), ev.get("cat", "")
        if cat == "kernel":
            for k in KERNELS:
                if k in name:
                    kern.setdefault(k, []).append(float(ev.get("dur", 0.0)))
        elif cat == "gpu_memcpy" and "HtoD" in name:
            h2d.append({"name": name, "bytes": int(ev.get("args", {}).get("bytes", -1))})
    pts = int(store.h_point_offsets[-1]) / store.n_scans * BATCH             # points gathered per batch
    gather_us = float(np.mean(kern["k_gather_points"]))
    out = {"card": card(), "batches": n_batches,
           "kernels_us_per_launch": {k: {"mean": float(np.mean(v)), "launches": len(v)} for k, v in kern.items()},
           "gather_bytes_per_batch": int(pts * 38),                             # 18 B read + 20 B written per point
           "gather_bytes_per_s": pts * 38 / (gather_us * 1e-6), "copy_peak_bytes_per_s": copy_bps,
           "h2d_copies_per_batch": len(h2d) / max(n_batches, 1), "h2d_copies": h2d[:16]}
    out["gather_over_copy_peak"] = out["gather_bytes_per_s"] / copy_bps
    if args.targets or args.world_aug:                 # the same epoch with the variant's options, same process
        set_variant(aug, args.targets, WorldAug() if args.world_aug else None)
        for _ in aug.epoch(98):
            pass
        torch.cuda.synchronize()
        kern_on, _ = kernel_times(aug, 0)
        out["variant"] = {"targets": args.targets, "world_aug": args.world_aug}
        out["variant_kernels_us_per_launch"] = {k: {"mean": float(np.mean(v)), "launches": len(v)} for k, v in kern_on.items()}
    aug.close()
    return out


KERNELS = ("k_gather_points", "k_draw_schedule", "k_gather_boxes", "k_gather_scan_meta", "k_inserted_targets", "k_draw_world",
           "k_gt_targets", "k_out_write")


def kernel_times(aug, epoch):
    """Device time per launch of KERNELS over one online epoch (torch.profiler), and the host-to-device copies."""
    import torch
    from torch.profiler import ProfilerActivity, profile as tprofile
    n_batches = 0
    with tprofile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        for _ in aug.epoch(epoch):
            n_batches += 1
        torch.cuda.synchronize()
    trace = os.path.join(tempfile.mkdtemp(), "online.pt.trace.json")
    prof.export_chrome_trace(trace)
    with open(trace) as f:
        events = json.load(f)["traceEvents"]
    kern = {}
    for ev in events:
        if ev.get("cat", "") == "kernel":
            for k in KERNELS:
                if k in ev.get("name", ""):
                    kern.setdefault(k, []).append(float(ev.get("dur", 0.0)))
    return kern, n_batches


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batches", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--depth", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--targets", action="store_true", help="detection targets for every batch (see the module doc)")
    ap.add_argument("--world-aug", action="store_true", help="world flip / rotation / scaling (WorldAug defaults)")
    ap.add_argument("--rounds", type=int, default=3, help="--targets: alternations of the variants")
    ap.add_argument("--out", default=None, help="directory for the JSON result (printed either way)")
    args = ap.parse_args()
    import __graft_entry__  # noqa: F401  (puts the repository on sys.path)
    from pcl_augmentation_b200 import _lib
    _lib.require_cuda()
    if args.world_aug and not args.targets and not args.profile:
        ap.error("--world-aug is measured as online + targets + world aug: pass --targets too")
    res = profile(args) if args.profile else variants(args) if args.targets else rates(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        name = "bench_online_profile" if args.profile else "bench_online"
        name += "_targets" if args.targets else ""
        name += "_world" if args.world_aug else ""
        with open(os.path.join(args.out, name + ".json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
