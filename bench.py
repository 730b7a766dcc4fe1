"""bench.py — augmented scans/sec of the Real3D-Aug hot path on B200 (BASELINE.json metric).

  python bench.py --gpus N --steps K --warmup W            (N > 1: launched by torchrun, one rank per GPU)
  python bench.py --impl reference --gpus N --steps K --warmup W
  python bench.py --config c2|c4|c5 ...                     (the other BASELINE.json configurations as the headline)
  python bench.py --dump-outputs DIR ...                    (+ the results of the last timed step as DIR/<name>.npy)

Headline workload (BASELINE.json configs[2], "c3", the one the metric is quoted on): a batch of 256 synthetic
KITTI-shape HDL-64 scans (120 000 points each, 112 x 1440 range image), 10 cut pedestrians / cyclists to insert per
scan, 1024 yaw candidates per cut object, sharded by scan: every rank owns its own batch of 256 (weak scaling, no
collective on the data path).  One step = one pass of the WHOLE device path over the rank's batch, starting from the
raw float4 points: spherical ingest + spatial indices + first range image (streaming kernels), the per-scan walker
(placement search + occlusion + insertion for every slot of every scan), output compaction.

  value   : scans/s with the raw points already resident in HBM (CUDA events on the engine streams); the K steps
            are dealt to `--resident-depth` engines so that one engine's streaming kernels overlap another's walker
  serial  : the same step alone on ONE engine (`single_batch_ms`), and the per-kernel CUDA-event times of exactly
            that mode (`kernels`): they add up to the serial step
  e2e     : scans/s through the public API (ScanPipeline) with HOST (pinned) buffers: H2D of every scan + the step +
            D2H of the augmented clouds inside the timed region; `copy_only` = the same bytes moved with no kernels
  roofline: the kernel with the largest share of the serial step.  Streaming kernels: algorithmic bytes (DESIGN.md §4)
            / measured time.  The walker is latency / issue bound and has no streaming model: its `achieved` is the
            ncu-measured DRAM traffic of one launch over the measured duration, with ncu's sm / issue utilisation
  cpu_baseline: the numpy oracle port of the reference timed on one host core on a bounded sample (rank 0, N = 1)
  configs : short runs of the other BASELINE.json configurations (c2 semseg, c4 128-beam, c5 4541-scan stream)
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "augmented scans/sec (120k-pt KITTI scan, placement + occlusion + insertion)"

# name -> workload (BASELINE.json `configs`, in order c1 .. c5)
WORKLOADS = {
    "c1": dict(task="od", shape="KITTI", scans=1, objects=10, yaw=360, rows=112, cols=1440, distinct=1,
               text="one KITTI-shape HDL-64 scan (120000 pts, 112x1440 range image), 10 cut pedestrians/cyclists, 360 yaw "
                    "candidates per object"),
    "c2": dict(task="ss", shape="SEMKITTI", scans=256, objects=20, yaw=360, rows=64, cols=2048, distinct=8, resident=10,
               text="batch of 256 SemanticKITTI-shape scans per GPU (124992 pts, 64x2048 range image), 20 rare-class objects "
                    "per scan placed on the rich_map road / sidewalk, 360 yaw candidates per object"),
    "c3": dict(task="od", shape="KITTI", scans=256, objects=10, yaw=1024, rows=112, cols=1440, distinct=32,
               text="batch of 256 KITTI-shape scans per GPU (120000 pts, 112x1440 range image), 10 cut "
                    "pedestrians/cyclists per scan, 1024 yaw candidates per object, sharded by scan"),
    "c4": dict(task="od", shape="OS128", scans=128, objects=50, yaw=360, rows=128, cols=2048, distinct=4, resident=6,
               text="batch of 128 OS1-128-shape scans per GPU (262144 pts, 128x2048 range image), 50 inserted objects per "
                    "scan, 360 yaw candidates per object"),
    "c5": dict(task="ss", shape="SEMKITTI", scans=256, objects=10, yaw=360, rows=112, cols=1440, distinct=8, stream=4541, resident=6,
               text="SemanticKITTI-sequence-sized stream of 4541 scans (124992 pts, 112x1440 range image, 10 objects per "
                    "scan) in batches of 256, sharded by scan over the GPUs, end to end incl. host<->device transfer"),
}


def workload_config(name, n_gpus):
    w = WORKLOADS[name]
    from pcl_augmentation_b200 import synth
    shape = getattr(synth, w["shape"] + "_SHAPE")
    pts = shape.beams * shape.az_steps
    return {"workload": w["text"], "name": name, "task": w["task"], "scans_per_gpu": w["scans"], "points_per_scan": pts,
            "objects_per_scan": w["objects"], "yaw_candidates": w["yaw"], "range_image": [w["rows"], w["cols"]],
            "parallelism": f"scan-sharded x{n_gpus}", "distinct_scans": w["distinct"],
            "l2": f"inputs larger than L2 ({w['scans'] * pts * 20 / 1e6:.0f} MB of points per batch, no flush needed)"
                  if w["scans"] * pts * 20 > 200e6 else
                  f"NOT flushed: the {w['scans'] * pts * 20 / 1e6:.1f} MB of a step stay L2-resident (single-scan latency case, not a throughput figure)"}


def build_cases(name, rank):
    """`distinct` different synthetic scans per rank, tiled to `scans` with different schedules / object draws."""
    from pcl_augmentation_b200 import synth
    w = WORKLOADS[name]
    shape = getattr(synth, w["shape"] + "_SHAPE")
    seed0 = {"c1": 9000, "c2": 7300, "c3": 9000, "c4": 7600, "c5": 7900}[name] + rank * 1000
    base = [synth.make_case(w["task"], seed0 + i, shape=shape, number_of_object=w["objects"]) for i in range(w["distinct"])]
    if w["task"] == "ss":                    # one engine = one sequence map: every scan uses the first pose / map
        for c in base[1:]:
            c.pose, c.map_data = base[0].pose, base[0].map_data
    cases = []
    for j in range(w["scans"]):
        c = base[j % w["distinct"]]
        classes = c.config["insertion"]["classes"]
        sched = synth.make_schedule(50000 + seed0 + j, len(classes), w["objects"], [len(c.db[k]) for k in classes])
        cc = synth.Case(c.task, c.config, c.pcl5, c.box_lines, c.db, sched, maps=c.maps, cars=c.cars)
        cc.pose, cc.map_data = c.pose, c.map_data
        cases.append(cc)
    return cases


def engine_kwargs(name, cases):
    w = WORKLOADS[name]
    return dict(max_scans=w["scans"], max_points=max(len(c.pcl5) for c in cases), rows=w["rows"], cols=w["cols"],
                yaw_steps=w["yaw"], max_events=w["objects"] + 1, max_boxes=128, map_data=cases[0].map_data)


class ClockSampler:
    """SM clock / throttle reasons of this rank's GPU, sampled through NVML every 10 ms from a background thread
    while the timed regions run (the quantities of the profiling recipe's nvidia-smi line: clocks.sm, clocks.max.sm,
    power.draw, clocks_event_reasons.*).  `mark(True/False)` brackets the timed regions; only samples taken inside
    them are summarised."""

    REASONS = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown"), ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown"),
               ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown"), ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap"),
               ("hw_power_brake", "nvmlClocksEventReasonHwPowerBrakeSlowdown"))

    def __init__(self, cuda_index, period_s=0.01):
        self.period, self.samples, self.inside, self.stop_flag, self.thread = period_s, [], False, False, None
        self.nv, self.handle, self.error = None, None, None
        try:
            import pynvml
            import torch
            pynvml.nvmlInit()
            uuid = str(torch.cuda.get_device_properties(cuda_index).uuid)
            self.handle = pynvml.nvmlDeviceGetHandleByUUID(("GPU-" + uuid) if not uuid.startswith("GPU-") else uuid)
            self.nv = pynvml
        except Exception as exc:                      # reported in the JSON line, never silently dropped
            self.error = f"NVML unavailable: {exc!r}"

    def start(self):
        if self.nv is None:
            return
        self.thread = threading.Thread(target=self._loop, daemon=True)
        self.thread.start()

    def mark(self, inside):
        self.inside = inside

    def _loop(self):
        nv, h = self.nv, self.handle
        while not self.stop_flag:
            try:
                sm = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    mask = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:
                    mask = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                pw = nv.nvmlDeviceGetPowerUsage(h) / 1000.0
                self.samples.append((self.inside, sm, mask, pw))
            except Exception as exc:
                self.error = f"NVML sample failed: {exc!r}"
                return
            time.sleep(self.period)

    def stop(self):
        if self.nv is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.error or "NVML unavailable"], "samples": 0}
        self.stop_flag = True
        self.thread.join(timeout=2)
        nv = self.nv
        mx = nv.nvmlDeviceGetMaxClockInfo(self.handle, nv.NVML_CLOCK_SM)
        timed = [s for s in self.samples if s[0]]
        reasons = set()
        for _, _, mask, _ in timed:
            for name, attr in self.REASONS:
                if mask & getattr(nv, attr, 0):
                    reasons.add(name)
        out = {"sm_mhz": statistics.median(s[1] for s in timed) if timed else None, "sm_max_mhz": float(mx),
               "sm_min_mhz": min(s[1] for s in timed) if timed else None,
               "power_w_max": round(max(s[3] for s in timed), 1) if timed else None,
               "reasons": sorted(reasons), "samples": len(timed), "samples_total": len(self.samples),
               "source": "NVML, 10 ms period, samples inside the timed regions (device-resident + e2e)"}
        if self.error:
            out["error"] = self.error
        return out


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def ncu_record(kernel):
    """What the committed `ncu --set full` capture of this workload says about a bench kernel (profiles/ncu_traffic.json,
    written by tools/ncu_summary.py): DRAM bytes per launch, sm / issue utilisation; or None."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    if not os.path.exists(path):
        return None
    with open(path) as f:
        return json.load(f).get(kernel)


def index_fractions(cases, eng):
    """Fractions of the points that go into the all-points (collision) grid and into the surface (road-level) grid."""
    fa, fg, n = 0.0, 0.0, 0
    surface = eng.surface_labels()
    for c in cases[:8]:
        lab = c.pcl5[:, 4].astype(np.int64)
        fa += float(np.sum(lab != eng.road_label)) if eng.task == "od" else float(len(lab))
        fg += float(np.sum(np.isin(lab, surface) & (c.pcl5[:, 2] > -3.0)))
        n += len(lab)
    return fa / n, fg / n


def algorithmic_bytes_per_scan(kernel, cases, eng):
    """Bytes ONE scan's share of a streaming kernel's launch has to move by its own formulation (DESIGN.md §4).
    None for kernels without a streaming model (the walker)."""
    n = float(np.mean([len(c.pcl5) for c in cases]))
    hw = eng.rows * eng.cols
    g2 = (2 * eng.grid_half) ** 2
    if kernel == "ingest_spherical":          # xyzi 16 + label 4 in; r 8 + el 8 + col 2 + alive 1 out; z-buffer clear
        return 39 * n + 8 * hw
    if kernel == "scatter_project":           # xyzi, label, col, el, r in; pix + column index out; 16 B per grid entry; z atomics
        fa, fg = index_fractions(cases, eng)
        return (38 + 8 + 16 * (fa + fg)) * n + 8 * hw
    if kernel == "index_build":               # three exclusive scans (read + write) + the distance transform
        return 8 * (2 * g2 + eng.cols + 1) + 5 * g2
    if kernel == "close_fill_full":           # SURVEY 8d: 16 B per pixel
        return 16 * hw
    if kernel == "compact_output":            # SURVEY 8d: 40 B per point
        return 40 * n
    if kernel == "project_zbuffer_full":
        return 20 * n + 8 * hw
    if kernel == "clear_images_full":
        return 8 * hw
    return None


def copy_only_probe(h2d_bytes, d2h_bytes, steps, barrier):
    """The PCIe ceiling of the e2e leg: the same bytes per step, pinned host <-> device on two streams, no kernels."""
    import torch
    src_h = torch.empty(int(h2d_bytes), dtype=torch.uint8, pin_memory=True)
    dst_d = torch.empty(int(h2d_bytes), dtype=torch.uint8, device="cuda")
    src_d = torch.empty(int(d2h_bytes), dtype=torch.uint8, device="cuda")
    dst_h = torch.empty(int(d2h_bytes), dtype=torch.uint8, pin_memory=True)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    for _ in range(2):
        with torch.cuda.stream(s1):
            dst_d.copy_(src_h, non_blocking=True)
        with torch.cuda.stream(s2):
            dst_h.copy_(src_d, non_blocking=True)
    barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        with torch.cuda.stream(s1):
            dst_d.copy_(src_h, non_blocking=True)
        with torch.cuda.stream(s2):
            dst_h.copy_(src_d, non_blocking=True)
    barrier()
    return time.perf_counter() - t0


def oracle_scan_seconds(case, w):
    from oracle import real3d_oracle as orc            # checker / baseline only
    t0 = time.perf_counter()
    orc.augment_scan(case.task, case.pcl5, case.box_lines, case.db, case.schedule.counts, case.schedule.perms, case.config,
                     maps=case.maps, map_data=case.map_data, transform_matrix=case.pose, mode="closed",
                     yaw_steps=w["yaw"], num_row=w["rows"], num_column=w["cols"])
    return time.perf_counter() - t0


def cpu_baseline_sample(name, budget_s):
    """The numpy oracle port of the reference (oracle/real3d_oracle.py) on ONE host core on whole scans of the same
    workload until ~budget_s of CPU work is spent (at least one scan)."""
    from pcl_augmentation_b200 import synth
    w = WORKLOADS[name]
    shape = getattr(synth, w["shape"] + "_SHAPE")
    t_total, n = 0.0, 0
    while t_total < budget_s and n < 4:
        case = synth.make_case(w["task"], 9000 + n, shape=shape, number_of_object=w["objects"])
        t_total += oracle_scan_seconds(case, w)
        n += 1
    return {"value": n / t_total, "unit": "scans/s", "cores": 1, "kind": "port",
            "sample": f"{n} whole scan(s) of the {name} workload through oracle/real3d_oracle.py, {t_total:.1f} s",
            "host_cpus": os.cpu_count()}


def _ref_worker(arg):
    name, seed = arg
    from pcl_augmentation_b200 import synth
    w = WORKLOADS[name]
    case = synth.make_case(w["task"], seed, shape=getattr(synth, w["shape"] + "_SHAPE"), number_of_object=w["objects"])
    return oracle_scan_seconds(case, w)


REF_OBJECTS_PER_SAMPLE = 1           # objects the reference inserts into each sampled scan (the workload asks for w["objects"])


def _ref_real_worker(arg):
    """One bounded sample of the workload through the UNMODIFIED reference (oracle/_ref, `oracle/build_ref.py`): its own
    `insertion.py` executed as `__main__` on a one-frame dataset written in its on-disk formats, inserting
    REF_OBJECTS_PER_SAMPLE objects instead of the workload's w["objects"] (a whole 120k-point scan takes the
    reference 1-2 minutes).  Returns (seconds inside the reference, objects it inserted)."""
    name, seed = arg
    import random
    import shutil
    import tempfile
    os.environ["R3D_REFERENCE_ROOT"] = os.path.join(ROOT, "oracle", "_ref")
    from oracle import shim                                       # baseline leg only
    from pcl_augmentation_b200 import synth, synth_io
    shim.REFERENCE_ROOT = os.environ["R3D_REFERENCE_ROOT"]
    w = WORKLOADS[name]
    case = synth.make_case(w["task"], seed, shape=getattr(synth, w["shape"] + "_SHAPE"), number_of_object=w["objects"])
    classes = case.config["insertion"]["classes"]
    counts = [0] * len(classes)
    counts[seed % len(classes)] = REF_OBJECTS_PER_SAMPLE
    root = tempfile.mkdtemp(prefix="r3d_refarm_")
    try:
        if w["task"] == "od":
            cwd, out, _ = synth_io.write_od_dataset([case], root, fixed_counts=counts)
            inputs = []
        else:
            cwd, out, _ = synth_io.write_ss_dataset([case], root, fixed_counts=counts)
            inputs = ["1", "0", "no"]
        random.seed(seed)
        np.random.seed(seed % (2 ** 31))
        t0 = time.perf_counter()
        shim.run_main(w["task"], cwd, inputs=inputs)
        dt = time.perf_counter() - t0
        added = os.path.join(out, "added_objects", "000000.txt")
        inserted = len([l for l in open(added).read().splitlines() if l.strip()]) if os.path.exists(added) else 0
        return dt, inserted
    finally:
        shutil.rmtree(root, ignore_errors=True)


def run_reference(args, json_out):
    """--impl reference: the reference's own CPU implementation of the path on all host cores.  With `oracle/_ref`
    present (the unmodified reference files, copied there by `oracle/build_ref.py` in the build container) every step runs
    the reference's `insertion.py` itself on one scan per worker process, bounded to REF_OBJECTS_PER_SAMPLE inserted
    objects per scan (`kind: "reference"`); the per-scan figure scales that by the workload's objects per scan — the
    reference's cost is per object slot (projection + closing of the scene, the yaw loop, the occlusion loop), nothing
    of it is per scan.  Without `oracle/_ref`: the numpy oracle port on whole scans (`kind: "port"`, ~20x faster than
    the reference)."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    from oracle import build_ref                                   # baseline leg only
    real = build_ref.available() and os.environ.get("R3D_REFERENCE_ARM", "reference") != "port"
    w = WORKLOADS[args.config]
    cores = max(1, min(os.cpu_count() or 1, 32))
    worker = _ref_real_worker if real else _ref_worker
    ctx = mp.get_context("fork")
    inserted = 0
    with ctx.Pool(cores) as pool:
        if args.warmup:
            pool.map(worker, [(args.config, 9000 + i) for i in range(cores)])      # one warm-up wave is enough for a CPU path
        t0 = time.perf_counter()
        done = 0.0
        for s in range(args.steps):
            res = pool.map(worker, [(args.config, 9100 + s * cores + i) for i in range(cores)])
            if real:
                inserted += sum(r[1] for r in res)
                done += cores * REF_OBJECTS_PER_SAMPLE / w["objects"]
            else:
                done += cores
        dt = time.perf_counter() - t0
    value = done / dt
    if real:
        kind = "reference"
        sample = (f"{cores} scans per step (one per worker process) through the unmodified reference insertion.py (oracle/_ref), "
                  f"{REF_OBJECTS_PER_SAMPLE} of the {w['objects']} objects per scan each = {REF_OBJECTS_PER_SAMPLE}/{w['objects']} scan; "
                  f"{args.steps} steps, {inserted} objects inserted; the reference's yaw loop is fixed at 360 candidates "
                  f"(find_spot.py:263) whatever the workload's yaw_candidates")
    else:
        kind = "port"
        sample = f"{cores} whole scans per step (one per worker process) through oracle/real3d_oracle.py, {args.steps} steps"
    print(file=json_out, flush=True, *[json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "scans/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": workload_config(args.config, args.gpus),
        "cpu_baseline": {"value": value, "unit": "scans/s", "cores": cores, "kind": kind, "sample": sample},
        "e2e": {"value": value, "unit": "scans/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0})])


def run_side(args, json_out):
    """SURVEY 8f rows 3-4: GPU numbers of an offline tool (tools/bench_*.py) + its CPU baseline (bench.py is the only
    place besides tests/ that executes oracle/)."""
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    if args.side == "rich_map_od":
        import bench_rich_map as tool
        from oracle import rich_map_oracle as rmo                  # CPU baseline leg only
        res, clouds = tool.gpu_bench(256, 10)
        t0, k = time.perf_counter(), 0
        while time.perf_counter() - t0 < 5.0:
            rmo.rich_map_od(clouds[k % len(clouds)], 40)
            k += 1
        unit, cpu, sample = "frames/s", k / (time.perf_counter() - t0), f"{k} frames"
    elif args.side == "rich_map_ss":
        import bench_rich_map_ss as tool
        from oracle import rich_map_oracle as rmo                  # CPU baseline leg only
        res, (frames, labels_cfg) = tool.gpu_bench(256, 10)
        t0 = time.perf_counter()
        rmo.rich_map_ss([(np.hstack((p.astype(np.float64), l.reshape(-1, 1).astype(np.float64))), T) for p, l, T in frames],
                        labels_cfg)
        unit, cpu, sample = "frames/s", len(frames) / (time.perf_counter() - t0), f"a {len(frames)}-frame sequence"
    else:
        import bench_cut_objects as tool
        from oracle import cut_objects_oracle as coo               # CPU baseline leg only
        res, (frames, cfg) = tool.gpu_bench(64, 10)
        t0 = time.perf_counter()
        for f in frames:
            coo.cut_objects_ss(np.hstack((f[0].astype(np.float64), f[1].reshape(-1, 1).astype(np.float64))), f[2], cfg, f[3], f[4])
        unit, cpu, sample = "frames/s", len(frames) / (time.perf_counter() - t0), f"{len(frames)} frames"
    res["cpu_baseline"] = {"value": round(cpu, 2), "unit": unit, "cores": 1, "kind": "port", "sample": sample}
    print(json.dumps(res), file=json_out, flush=True)


DUMP_BYTES = 60 * 10 ** 6          # --dump-outputs: bytes of all arrays at most (under 64 MB with the .npy headers)


class Bench:
    """One workload on this rank's GPU: engines, the staged (pinned) batch and the three measurements."""

    def __init__(self, name, rank, world, args, barrier, max_over_ranks):
        from pcl_augmentation_b200.engine import Real3DEngine, scan_input_from_case
        from pcl_augmentation_b200.pipeline import ScanPipeline
        self.name, self.rank, self.world, self.args = name, rank, world, args
        self.barrier, self.max_over_ranks = barrier, max_over_ranks
        self.w = WORKLOADS[name]
        self.cases = build_cases(name, rank)
        self.n_scans = len(self.cases)
        kw = engine_kwargs(name, self.cases)
        c0 = self.cases[0]
        # engines of the e2e pipeline: --depth, more for the semseg workloads (a batch's walker ends with a few long scans:
        # more batches in flight keep the device busy while the copies of the others run)
        self.depth = max(args.depth, self.w.get("e2e_depth", 0))
        self.pipe = ScanPipeline(self.w["task"], c0.config, c0.db, depth=self.depth, **kw)
        # engines the device-resident leg deals its steps to: --resident-depth, or the workload's own figure when the
        # flag is left at its default (semseg scans differ a lot in the tries they need — the walker of one batch ends
        # with a few long scans, which more resident batches fill)
        self.res_depth = max(1, args.resident_depth if args.resident_depth > 0 else self.w.get("resident", 3))
        self.extra = [Real3DEngine(self.w["task"], c0.config, c0.db, **kw) for _ in range(self.res_depth - self.depth)]
        self.res_engines = (self.pipe.engines + self.extra)[:self.res_depth]
        self.eng = self.pipe.engines[0]
        self.staged = self.eng.stage([scan_input_from_case(c) for c in self.cases])

    def close(self):
        self.pipe.close()
        for e in self.extra:
            e.close()

    # ---- device-resident: K steps dealt round-robin to the resident engines (own host thread, own stream) --------
    def _resident_steps(self, n_steps):
        errors = []
        engines = self.res_engines

        def worker(w):
            try:
                for _ in range(w, n_steps, len(engines)):
                    engines[w].reset(from_raw_points=True)      # the WHOLE device path: ingest + indices included
                    engines[w].run()
            except BaseException as exc:
                errors.append(exc)
        threads = [threading.Thread(target=worker, args=(w,), daemon=True) for w in range(len(engines))]
        for t in threads:
            t.start()
        for t in threads:
            t.join()
        if errors:
            raise errors[0]

    def resident(self, steps, warmup, sampler=None):
        import torch
        for e in self.res_engines:
            e.load(self.staged)
            e.sync()
        self._resident_steps(max(warmup, len(self.res_engines)))
        for e in self.res_engines:
            e.sync()
        streams = [e.cuda_stream() for e in self.res_engines]
        ev0 = torch.cuda.Event(enable_timing=True)
        ev_end = [torch.cuda.Event(enable_timing=True) for _ in streams]
        self.barrier()
        launches0 = self.eng.launch_count()
        if sampler:
            sampler.mark(True)
        ev0.record(streams[0])              # every engine stream is idle here (barrier = device synchronize)
        self._resident_steps(steps)
        for ev, es in zip(ev_end, streams):
            ev.record(es)
        for e in self.res_engines:
            e.sync()
        if sampler:
            sampler.mark(False)
        self.barrier()
        dev_ms = self.max_over_ranks(max(ev0.elapsed_time(ev) for ev in ev_end))
        return dev_ms, self.eng.launch_count() - launches0

    def dump_outputs(self, steps, out_dir):
        """Write what the last device-resident step computed, as a caller receives it (Real3DEngine.unpack), to
        `out_dir/<name>.npy` (float32 / float64): status, output sizes and inserted objects of every scan, and the
        clouds of a sample of the scans, taken in a seeded order for as long as the dump stays within DUMP_BYTES (so
        two builds whose outputs have the same sizes dump the same scans)."""
        eng = self.res_engines[(steps - 1) % len(self.res_engines)]      # _resident_steps deals step i to engine i % n
        res = eng.unpack(eng.fetch_raw(), raise_on_error=False)
        ss = self.w["task"] == "ss"
        obj_id = {name: i for i, name in enumerate(eng.obj_names)}
        ins = [(s, obj_id[name], rot, eng.classes.index(cls), vis, box) for s, r in enumerate(res)
               for (name, rot, cls), vis, box in zip(r.inserted, r.visible, r.boxes)]
        f64 = lambda rows, cols: np.array(rows, dtype=np.float64).reshape(-1, cols)
        out = {"status": f64([r.status for r in res], 1)[:, 0],
               "points_per_scan": f64([len(r.velodyne) for r in res], 1)[:, 0],
               "check_rows_per_scan": f64([len(r.check) for r in res], 1)[:, 0],
               # scan, object index in the cut-object database, rotation step, class index, visible points
               "inserted": f64([i[:5] for i in ins], 5),
               # center x y z, rotation quaternion x y z w, length, width, height
               "inserted_boxes": f64([[*b["center"].values(), *b["rotation"].values(), b["length"], b["width"], b["height"]]
                                      for *_, b in ins], 10)}
        # float32 velodyne + check rows, float64 labels; 8 B per scan reserved for `sample_scans`
        cloud_bytes = lambda r: 4 * r.velodyne.size + 4 * r.check.size + (8 * len(r.velodyne) if ss else 0)
        budget = DUMP_BYTES - sum(a.nbytes for a in out.values()) - 8 * self.n_scans
        pick = []
        for s in np.random.default_rng(0).permutation(self.n_scans):
            budget -= cloud_bytes(res[s])
            if budget < 0:
                break
            pick.append(int(s))
        pick.sort()
        out["sample_scans"] = np.array(pick, dtype=np.float64)
        out["velodyne"] = np.concatenate([np.zeros((0, 4), np.float32)] + [res[s].velodyne for s in pick]).astype(np.float32)
        out["check"] = np.concatenate([np.zeros((0, 5 if ss else 4), np.float32)] + [res[s].check for s in pick]).astype(np.float32)
        if ss:
            out["labels"] = np.concatenate([np.zeros(0)] + [res[s].labels for s in pick]).astype(np.float64)
        os.makedirs(out_dir, exist_ok=True)
        for name, a in out.items():
            np.save(os.path.join(out_dir, name + ".npy"), a)

    # ---- one step alone on one engine + the per-kernel CUDA-event times of exactly that mode -------------------
    def serial(self, steps):
        import torch
        eng, stream = self.eng, self.eng.cuda_stream()
        eng.load(self.staged)
        eng.reset(from_raw_points=True); eng.run(); eng.sync()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record(stream)
        for _ in range(steps):
            eng.reset(from_raw_points=True); eng.run()
        ev1.record(stream)
        eng.sync()
        serial_ms = ev0.elapsed_time(ev1) / steps
        eng.profile(True)                       # CUDA events around every launch; same engine, same serial order
        for _ in range(steps):
            eng.reset(from_raw_points=True); eng.run()
        eng.sync()
        prof, stats = eng.profile_read(), eng.stats()
        stats["walk_profile"] = eng.walk_profile()           # (cycles, tries) per scan of the last step
        eng.profile(False)
        results = eng.unpack(eng.fetch_raw())
        return serial_ms, prof, stats, results

    # ---- end to end through the public API with host buffers ----------------------------------------------------
    def e2e(self, steps, sampler=None, stream_scans=None):
        st = self.staged
        self.pipe.warmup(st)
        self.pipe.warmup(st)
        if stream_scans is None:
            n_batches = steps
        else:                                   # the stream is sharded by scan over the ranks, batches of n_scans
            per_rank = -(-stream_scans // self.world)
            n_batches = -(-per_rank // self.n_scans)
        self.barrier()
        if sampler:
            sampler.mark(True)
        t0 = time.perf_counter()
        out_bytes = self.pipe.process([st] * n_batches)
        self.barrier()
        secs = self.max_over_ranks(time.perf_counter() - t0)
        if sampler:
            sampler.mark(False)
        h2d = sum(st[k].nbytes for k in ("xyzi", "labels", "boxes", "perms", "counts") if k in st)
        h2d += st["maps"].nbytes if "maps" in st else st["poses"].nbytes
        d2h = sum(out_bytes) / n_batches
        return {"seconds": secs, "batches": n_batches, "h2d": int(h2d), "d2h": int(d2h)}


def kernel_table(bench, prof, steps, peak):
    total = sum(v["ms"] for v in prof.values())
    table = {}
    for name, v in sorted(prof.items(), key=lambda kv: -kv[1]["ms"]):
        if not v["launches"]:
            continue
        ms_step = v["ms"] / steps
        entry = {"ms_per_step": round(ms_step, 4), "launches_per_step": v["launches"] / steps,
                 "share": round(v["ms"] / max(total, 1e-9), 4)}
        per_scan = algorithmic_bytes_per_scan(name, bench.cases, bench.eng)
        rec = ncu_record(name) if bench.name == "c3" else None
        if per_scan is not None:
            gbs = per_scan * bench.n_scans / (ms_step / 1e3) / 1e9
            entry.update(bound="hbm", algorithmic_bytes_per_scan=int(per_scan), achieved_gbs=round(gbs, 1), frac=round(gbs / peak, 4))
        else:
            entry.update(bound="latency / issue (no streaming model)")
        if rec:
            entry["ncu"] = rec
        table[name] = entry
    return table, total / steps


NOMINAL_HBM_GBS = 8000.0           # B200 HBM3e, nominal (SURVEY 8d; B200_PROFILING.md quotes ~7.7 TB/s for this part)


def roofline_of(name, entry, bench, peak, peak_src):
    """The JSON `roofline` object of one kernel-table entry."""
    rec = entry.get("ncu")
    launch_ms = entry["ms_per_step"] / max(entry["launches_per_step"], 1)
    out = {"kernel": name, "bound": "hbm", "peak": peak, "unit": "GB/s", "peak_source": peak_src,
           "avg_launch_ms": round(launch_ms, 4), "share_of_serial_step": entry["share"],
           "traffic": rec["bytes_per_launch"] if rec else None, "traffic_source": rec["source"] if rec else None}
    if "achieved_gbs" in entry:
        out.update(achieved=entry["achieved_gbs"], frac=entry["frac"],
                   bytes_per_launch=int(entry["algorithmic_bytes_per_scan"] * bench.n_scans / max(entry["launches_per_step"], 1)),
                   bytes_source="algorithmic (DESIGN.md section 4)")
    elif rec:
        # latency-bound kernel without a streaming model: the DRAM bytes ncu measured for one launch of this workload
        gbs = rec["bytes_per_launch"] / (launch_ms / 1e3) / 1e9
        out.update(achieved=round(gbs, 1), frac=round(gbs / peak, 4), bytes_per_launch=rec["bytes_per_launch"],
                   bytes_source="ncu dram__bytes_read.sum + dram__bytes_write.sum (no streaming model: the kernel is "
                                "latency / issue bound)",
                   limiter={k: rec[k] for k in ("sm_throughput_pct", "issue_active_pct", "warps_active_pct") if k in rec})
    else:
        out.update(achieved=None, frac=None, bytes_source="no ncu capture committed for this kernel")
    # SURVEY 8(d): both denominators — the copy bandwidth measured on this pod (`peak`) and the nominal HBM3e figure
    out["frac_of_nominal"] = round(out["achieved"] / NOMINAL_HBM_GBS, 4) if out.get("achieved") is not None else None
    out["nominal_peak"] = NOMINAL_HBM_GBS
    return out


def walk_spread(stats, clocks):
    """Spread of the walker CTA lifetimes over the scans of one step (ms): what makes one batch alone tail bound."""
    cyc, tries = stats["walk_profile"]
    mhz = (clocks.get("sm_mhz") or 1965.0) * 1e3
    ms = np.sort(cyc / mhz)
    pick = lambda q: round(float(ms[min(len(ms) - 1, int(q * len(ms)))]), 3)
    return {"p50": pick(0.5), "p90": pick(0.9), "p99": pick(0.99), "max": round(float(ms[-1]), 3),
            "tries_p50": int(np.sort(tries)[len(tries) // 2]), "tries_max": int(tries.max())}


WALK_CTAS_PER_SM = {"od": 3, "ss": 2}          # csrc/r3d_engine_kernels.cuh: walk_od 384 x 3, walk_ss 512 x 2


def timed_mode_model(task, n_scans, table, cyc, prof_steps, clocks, ms_per_step, sm_count=None):
    """Device time one step HOLDS when several resident batches overlap (the timed mode of `value`): a streaming kernel
    fills the device for its serial duration, the walker holds n_scans CTA lifetimes spread over the CTA slots of the
    device.  The two add up to about the measured step: the device is full, and the streaming kernels are the larger part."""
    if sm_count is None:
        import torch
        sm_count = torch.cuda.get_device_properties(torch.cuda.current_device()).multi_processor_count
    slots = sm_count * WALK_CTAS_PER_SM[task]
    cta_ms = cyc.get("total", 0) / max(prof_steps * n_scans, 1) / ((clocks.get("sm_mhz") or 1965.0) * 1e3)
    walker = n_scans * cta_ms / slots
    streaming = sum(v["ms_per_step"] for k, v in table.items() if k != "scan_walk")
    return {"walker_cta_slots": slots, "walker_slot_ms_per_step": round(walker, 4), "streaming_kernels_ms_per_step": round(streaming, 4),
            "sum_ms": round(walker + streaming, 4), "measured_ms_per_step": round(ms_per_step, 4)}


def measure_side_config(name, rank, world, args, barrier, max_over_ranks, sum_over_ranks, peak):
    """A short run of another BASELINE.json configuration: device-resident value, serial step + dominant kernel, e2e."""
    b = Bench(name, rank, world, args, barrier, max_over_ranks)
    try:
        steps = max(4, args.steps // 4, 2 * b.res_depth)
        dev_ms, _ = b.resident(steps, 2)
        serial_ms, prof, stats, results = b.serial(3)
        table, _ = kernel_table(b, prof, 3, peak)
        top = next(iter(table))
        e = b.e2e(steps, stream_scans=b.w.get("stream"))
        scans_e2e = world * b.n_scans * e["batches"]
        out = {"config": workload_config(name, world), "value": world * b.n_scans * steps / (dev_ms / 1e3), "unit": "scans/s",
               "ms_per_step": dev_ms / steps, "steps": steps, "resident_engines": b.res_depth, "single_batch_ms": serial_ms,
               "e2e": {"value": scans_e2e / e["seconds"], "unit": "scans/s", "h2d_bytes_per_step": e["h2d"],
                       "d2h_bytes_per_step": e["d2h"], "batches": e["batches"], "pipeline_depth": b.depth,
                       "pcie_gbs_each_way": round(max(e["h2d"], e["d2h"]) * e["batches"] / e["seconds"] / 1e9, 1)},
               "dominant_kernel": {top: table[top]},
               "streaming_kernels": {k: {"ms_per_step": v["ms_per_step"], "frac": v["frac"]} for k, v in table.items() if "frac" in v},
               "objects_inserted_per_scan": sum_over_ranks(sum(len(r.inserted) for r in results)) / (world * b.n_scans),
               "steps_per_scan_max": stats["max_steps_per_scan"], "walker_cta_ms": walk_spread(stats, {})}
        if b.w.get("stream"):
            out["stream_scans"] = scans_e2e
        return out
    finally:
        b.close()


def main():
    # Libraries (NCCL's version banner, for one) write to fd 1: keep the real stdout for the ONE JSON line and send
    # everything else written to fd 1 during the run to stderr
    json_out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default="c3", choices=sorted(WORKLOADS), help="headline workload (default: the one the metric is quoted on)")
    ap.add_argument("--side-configs", default="c1,c2,c4,c5",
                    help="comma-separated other configurations measured briefly into the `configs` block ('' = none)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--resident-depth", type=int, default=0,
                    help="engines (each with its own HBM-resident batch) the device-resident leg deals the steps to: one "
                         "engine's streaming kernels overlap another's walker (0 = the workload's default: 3, semseg 6-8)")
    ap.add_argument("--depth", type=int, default=4, help="engines (streams) the e2e leg pipelines batches through")
    ap.add_argument("--side", default=None, choices=["rich_map_od", "rich_map_ss", "cut_objects"],
                    help="instead of the headline bench: one of the offline tools either side of the path (SURVEY 8f rows "
                         "3-4), GPU numbers from tools/bench_*.py plus the CPU baseline (numpy oracle port, one host core)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one computed (rank 0's batch) to DIR/<name>.npy, so "
                         "that two builds can be compared output for output on the same seeded inputs")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and (args.side or args.impl != "b200"):
        ap.error("--dump-outputs applies to the headline B200 path only (not to --side or --impl reference)")
    if args.side:
        run_side(args, json_out)
        return
    if args.impl == "reference":
        run_reference(args, json_out)
        return

    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    assert torch.cuda.is_available(), "bench.py needs a CUDA device (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    from pcl_augmentation_b200 import sharding
    numa_cpus = sharding.bind_to_gpu_numa_node(local_rank) if (world > 1 and os.environ.get("R3D_NUMA_BIND", "1") != "0") else None
    if world > 1:
        # NCCL_DEBUG output goes to fd 1, which was redirected to stderr above: the JSON line keeps the real stdout
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        return sharding.all_reduce_scalar(x, "max", "cuda")

    def sum_over_ranks(x):
        return sharding.all_reduce_scalar(x, "sum", "cuda")

    peak, peak_src = peaks()
    name = args.config
    b = Bench(name, rank, world, args, barrier, max_over_ranks)
    n_scans = b.n_scans
    sampler = ClockSampler(local_rank)
    sampler.start()

    # ---- device-resident throughput ("value"): the whole device path from the raw points, steps overlapped ----------
    dev_ms, launches = b.resident(args.steps, args.warmup, sampler)
    value = world * n_scans * args.steps / (dev_ms / 1000.0)
    if args.dump_outputs and rank == 0:
        b.dump_outputs(args.steps, args.dump_outputs)
    # ---- the same step alone on one engine, and the per-kernel times of exactly that mode ---------------------------
    prof_steps = max(3, min(args.steps, 10))
    serial_ms, prof, stats, results = b.serial(prof_steps)
    table, kernel_sum_ms = kernel_table(b, prof, prof_steps, peak)
    dominant = next(iter(table))
    roofline = roofline_of(dominant, table[dominant], b, peak, peak_src)
    streaming = [k for k, v in table.items() if "achieved_gbs" in v]
    roofline_streaming = roofline_of(streaming[0], table[streaming[0]], b, peak, peak_src) if streaming else None
    # consistency of the serial mode: the kernels add up to the step and none is longer than it
    consistency = {"serial_step_ms": round(serial_ms, 4), "sum_of_kernels_ms": round(kernel_sum_ms, 4),
                   "dominant_kernel_ms": table[dominant]["ms_per_step"],
                   "ok": bool(table[dominant]["ms_per_step"] <= serial_ms * 1.02 and 0.85 * serial_ms <= kernel_sum_ms <= 1.1 * serial_ms)}
    # measured DRAM traffic of one whole step (ncu, profiles/r2_step_traffic.json) over the timed step
    step_traffic = None
    tp = os.path.join(ROOT, "profiles", "r2_step_traffic.json")
    if name == "c3" and os.path.exists(tp):
        with open(tp) as f:
            t = json.load(f)
        gbs = t["dram_bytes_per_step"] / (dev_ms / args.steps / 1e3) / 1e9
        step_traffic = {"dram_bytes_per_step": t["dram_bytes_per_step"], "source": t["source"],
                        "achieved_gbs": round(gbs, 1), "frac_of_peak": round(gbs / peak, 4)}

    # ---- end to end through the public API with host buffers ("e2e") ------------------------------------------------
    e = b.e2e(args.steps, sampler, stream_scans=b.w.get("stream"))
    e2e_value = world * n_scans * e["batches"] / e["seconds"]
    copy_s = max_over_ranks(copy_only_probe(e["h2d"], e["d2h"], args.steps, barrier))
    copy_only = {"scans_per_s": world * n_scans * args.steps / copy_s,
                 "gbs_each_way_per_gpu": round(max(e["h2d"], e["d2h"]) * args.steps / copy_s / 1e9, 1),
                 "what": "the same H2D + D2H bytes per step from / to pinned host memory on two streams, no kernels, all ranks "
                         "at once: the PCIe / host-memory ceiling of the e2e leg"}
    clocks = sampler.stop()
    inserted_all = sum_over_ranks(sum(len(r.inserted) for r in results))

    # ---- CPU baseline (rank 0, N = 1 only) and the other configurations -----------------------------------------------
    cpu = None
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        cpu = cpu_baseline_sample(name, 20.0)
    res_depth, b_depth, b_task = b.res_depth, b.depth, b.w["task"]
    b.close()
    configs = {}
    for side in [s for s in args.side_configs.split(",") if s and s != name]:
        configs[side] = measure_side_config(side, rank, world, args, barrier, max_over_ranks, sum_over_ranks, peak)
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            configs[side]["cpu_baseline"] = cpu_baseline_sample(side, 6.0)
    if rank == 0:
        cyc = stats.get("walker_cycles", {})
        print(file=json_out, flush=True, *[json.dumps({
            "metric": METRIC, "value": value, "unit": "scans/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": dev_ms / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": dict(workload_config(name, world),
                           steps_in_flight=f"{res_depth} resident engines, one {n_scans}-scan step each (`single_batch_ms` is a step alone)"),
            "roofline": roofline, "roofline_streaming": roofline_streaming, "step_traffic": step_traffic,
            "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": "scans/s", "h2d_bytes_per_step": e["h2d"], "d2h_bytes_per_step": e["d2h"],
                    "pipeline_depth": b_depth, "ms_per_step": 1000.0 * e["seconds"] / e["batches"],
                    "pcie_gbs_each_way": round(max(e["h2d"], e["d2h"]) * e["batches"] / e["seconds"] / 1e9, 1),
                    "copy_only": copy_only, "of_copy_only": round(e2e_value / copy_only["scans_per_s"], 3),
                    "timed": "H2D of the staged batch (pinned), ingest + walker + compaction, D2H of the augmented clouds into "
                             "pinned buffers; packing scans into the staged batch (the dataset reader's job) is outside"},
            "gpu_launches": int(launches), "clocks": clocks, "resident_engines": res_depth,
            "single_batch_ms": serial_ms, "single_batch_scans_per_s": n_scans / (serial_ms / 1000.0),
            "numa_bound_cpus": numa_cpus,
            "kernel_times": "CUDA events around every launch of the serial mode (one engine, one step at a time); `share` = of "
                            "the sum of kernel times",
            "kernels": table, "consistency": consistency,
            "walker": {"steps_per_scan_max": stats["max_steps_per_scan"],
                       "tries_per_scan": stats["tried_objects"] / max(prof_steps * n_scans, 1),
                       "candidate_windows_per_try": stats["candidate_windows"] / max(stats["tried_objects"], 1),
                       "exact_occlusion_counts_per_try": stats["exact_occlusion_counts"] / max(stats["tried_objects"], 1),
                       "cta_ms_mean": round(cyc.get("total", 0) / max(prof_steps * n_scans, 1) / ((clocks.get("sm_mhz") or 1965.0) * 1e3), 4),
                       "cta_ms_percentiles": walk_spread(stats, clocks),
                       "timed_mode_model": timed_mode_model(b_task, n_scans, table, cyc, prof_steps, clocks, dev_ms / args.steps),
                       "phase_share_of_cta_time": {k: round(v / max(cyc.get("total", 1), 1), 4) for k, v in cyc.items() if k != "total"}},
            "objects_inserted_per_scan": inserted_all / (world * n_scans),
            "configs": configs, "engine_stats": {k: v for k, v in stats.items() if k not in ("walker_cycles", "walk_profile")}})])
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
