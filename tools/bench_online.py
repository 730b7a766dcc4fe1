"""Online augmentation from a device-resident dataset against the engine's other two ways of being fed, in one process.

Workload: bench.py's c3 shape (256-scan batches of 120 000-point KITTI-shape scans, 112 x 1440 range image, 1024 yaw
candidates, 10 objects per scan) from a store of 1024 distinct scans: bench.py's 32 c3 scenes, each in 32 variants whose
intensities are redrawn (2.2 GB of points + labels: larger than L2, so the gather reads HBM).

    python tools/bench_online.py [--batches 20] [--warmup 2] [--depth 3] [--out DIR]            rates
    python tools/bench_online.py --profile [--out DIR]                                           kernel times + copies

Rates (scans/s, host clock around work that ends in a device synchronise):
  * online     OnlineAugmenter.epochs over the store, a new epoch each pass (gather + device schedule draw + run), and
               the same with one OnlineAugmenter.epoch call per epoch (the look-ahead restarts at every epoch);
  * resident   the same engines' reset(from_raw_points=True) + run loop (bench.py's device-resident definition);
  * host       load + run of a batch staged in pinned host buffers (Real3DEngine.stage, outside the timed loop).
--profile: torch.profiler over a few online batches: device time of k_gather_points and k_draw_schedule, the gather's
bytes per second against a device-to-device copy measured in the same run, and every host-to-device copy of a batch.
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


def setup(depth):
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
    aug = OnlineAugmenter("od", c0.config, c0.db, store, batch_size=BATCH, seed=2024, depth=depth, **kw)
    return aug, store, scans


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
    aug, store, _ = setup(args.depth)
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
            for k in ("k_gather_points", "k_draw_schedule", "k_gather_boxes", "k_gather_scan_meta", "k_inserted_targets"):
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
    aug.close()
    return out


def main():
    ap = argparse.ArgumentParser(description=__doc__, formatter_class=argparse.RawDescriptionHelpFormatter)
    ap.add_argument("--batches", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=4)
    ap.add_argument("--depth", type=int, default=3)
    ap.add_argument("--profile", action="store_true")
    ap.add_argument("--out", default=None, help="directory for the JSON result (printed either way)")
    args = ap.parse_args()
    import __graft_entry__  # noqa: F401  (puts the repository on sys.path)
    from pcl_augmentation_b200 import _lib
    _lib.require_cuda()
    res = profile(args) if args.profile else rates(args)
    line = json.dumps(res)
    print(line)
    if args.out:
        os.makedirs(args.out, exist_ok=True)
        with open(os.path.join(args.out, "bench_online_profile.json" if args.profile else "bench_online.json"), "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
