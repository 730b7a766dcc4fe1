"""CPU tier: the pieces of bench.py that shape the ONE JSON line (no GPU, no timing): workloads of BASELINE.json,
roofline objects for a streaming kernel and for the latency-bound walker, the walker's CTA-lifetime spread."""
import json
import os

import numpy as np
import pytest

import bench

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_workloads_cover_the_baseline_configs():
    with open(os.path.join(ROOT, "BASELINE.json")) as f:
        base = json.load(f)
    assert len(base["configs"]) == 5 and sorted(bench.WORKLOADS) == ["c1", "c2", "c3", "c4", "c5"]
    c3 = bench.workload_config("c3", 8)
    assert c3["scans_per_gpu"] == 256 and c3["yaw_candidates"] == 1024 and c3["points_per_scan"] == 120000
    assert c3["range_image"] == [112, 1440] and c3["parallelism"] == "scan-sharded x8" and "larger than L2" in c3["l2"]
    assert bench.workload_config("c2", 1)["range_image"] == [64, 2048] and bench.workload_config("c4", 1)["points_per_scan"] == 262144
    assert bench.WORKLOADS["c5"]["stream"] == 4541
    assert "NOT flushed" in bench.workload_config("c1", 1)["l2"]            # the single-scan case says so


class _FakeBench:
    n_scans = 256


def test_roofline_objects_have_the_contract_keys():
    streaming = {"ms_per_step": 0.62, "launches_per_step": 1.0, "share": 0.13, "bound": "hbm", "algorithmic_bytes_per_scan": 8730240,
                 "achieved_gbs": 3600.0, "frac": 0.55}
    r = bench.roofline_of("scatter_project", streaming, _FakeBench(), 6551.7, "measured")
    for k in ("kernel", "bound", "achieved", "peak", "unit", "frac", "traffic"):
        assert k in r
    assert r["frac"] <= 1.0 and r["bytes_per_launch"] == 8730240 * 256
    assert r["nominal_peak"] == 8000.0 and abs(r["frac_of_nominal"] - 3600.0 / 8000.0) < 1e-4      # SURVEY 8d: both denominators
    walker = {"ms_per_step": 2.8, "launches_per_step": 1.0, "share": 0.6, "bound": "latency / issue (no streaming model)",
              "ncu": {"bytes_per_launch": 432000000, "source": "profiles/x.csv", "sm_throughput_pct": 15.6, "issue_active_pct": 28.8,
                      "warps_active_pct": 29.7}}
    r = bench.roofline_of("scan_walk", walker, _FakeBench(), 6551.7, "measured")
    assert r["traffic"] == 432000000 and 0 < r["frac"] < 0.1 and r["limiter"]["issue_active_pct"] == 28.8
    r = bench.roofline_of("scan_walk", {k: v for k, v in walker.items() if k != "ncu"}, _FakeBench(), 6551.7, "measured")
    assert r["achieved"] is None and r["frac"] is None and r["frac_of_nominal"] is None and "no ncu capture" in r["bytes_source"]


def test_walk_spread_percentiles():
    cyc = np.arange(1, 257, dtype=np.int64) * 19650            # 0.01 .. 2.56 ms at 1965 MHz
    tries = np.full(256, 11, dtype=np.int32); tries[-1] = 15
    s = bench.walk_spread({"walk_profile": (cyc, tries)}, {"sm_mhz": 1965.0})
    assert s["max"] == 2.56 and abs(s["p50"] - 1.29) < 0.02 and s["tries_max"] == 15 and s["tries_p50"] == 11


def test_committed_profile_records_are_consistent():
    """What bench.py reads from profiles/: the step traffic derived from the ncu launch list and the per-kernel records."""
    with open(os.path.join(ROOT, "profiles", "r2_step_traffic.json")) as f:
        t = json.load(f)
    assert t["dram_bytes_per_step"] == sum(k["dram_bytes"] for k in t["kernels"].values())
    assert abs(sum(k["share_of_device_time"] for k in t["kernels"].values()) - 1.0) < 0.01
    assert max(t["kernels"], key=lambda k: t["kernels"][k]["us"]) == "k_scan_walk"
    with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
        n = json.load(f)
    for name in ("scan_walk", "scatter_project", "ingest_spherical", "close_fill_full", "compact_output"):
        assert n[name]["bytes_per_launch"] > 0 and n[name]["source"].startswith("profiles/r2_")
        assert os.path.exists(os.path.join(ROOT, n[name]["source"].split(" ")[0]))


def test_timed_mode_model_adds_walker_slot_time_and_streaming_kernels():
    """256 CTAs of 1.44 ms over 148 x 3 slots = 0.83 ms of device time next to 1.9 ms of streaming kernels."""
    table = {"scan_walk": {"ms_per_step": 2.9}, "scatter_project": {"ms_per_step": 0.62}, "ingest_spherical": {"ms_per_step": 0.48},
             "compact_output": {"ms_per_step": 0.30}, "close_fill_full": {"ms_per_step": 0.30}, "index_build": {"ms_per_step": 0.19}}
    cyc = {"total": int(1.44e-3 * 1965e6) * 256 * 10}
    m = bench.timed_mode_model("od", 256, table, cyc, 10, {"sm_mhz": 1965.0}, 2.95, sm_count=148)
    assert m["walker_cta_slots"] == 444
    assert abs(m["walker_slot_ms_per_step"] - 256 * 1.44 / 444) < 1e-3
    assert abs(m["streaming_kernels_ms_per_step"] - 1.89) < 1e-9
    assert abs(m["sum_ms"] - (m["walker_slot_ms_per_step"] + 1.89)) < 1e-3 and m["measured_ms_per_step"] == 2.95
    assert bench.timed_mode_model("ss", 256, table, cyc, 10, {}, 13.0, sm_count=148)["walker_cta_slots"] == 296


@pytest.mark.parametrize("task", ["od", "ss"])
def test_dump_outputs_writes_the_last_steps_results(tmp_path, monkeypatch, task):
    """--dump-outputs: the engine that ran the last timed step, float32 / float64 files only, per-scan records of every
    scan, and the clouds of the scans that fit the byte budget in the seeded order."""
    from types import SimpleNamespace
    from pcl_augmentation_b200.engine import ScanResult
    ss = task == "ss"
    rng = np.random.default_rng(5)
    box = {"center": {"x": 1.0, "y": 2.0, "z": 3.0}, "rotation": {"x": 0.0, "y": 0.0, "z": 0.6, "w": 0.8},
           "length": 4.0, "width": 5.0, "height": 6.0, "class": "Cyclist"}

    def engine(tag):
        res = [ScanResult(velodyne=rng.normal(size=(10 + s, 4)).astype(np.float32),
                          labels=rng.integers(0, 260, 10 + s).astype(np.uint32) if ss else np.zeros(0, np.uint32),
                          check=np.full((s % 3, 5 if ss else 4), tag, np.float32), inserted=[("b.npz", 7 * s, "Cyclist")] * (s % 2),
                          lines=[], boxes=[box] * (s % 2), visible=[s] * (s % 2), status=tag) for s in range(40)]
        return SimpleNamespace(obj_names=["a.npz", "b.npz"], classes=["Pedestrian", "Cyclist"],
                               fetch_raw=lambda: None, unpack=lambda buffers, raise_on_error: res, res=res)
    engines = [engine(0), engine(1), engine(2)]
    fake = SimpleNamespace(res_engines=engines, w={"task": task}, n_scans=40)
    monkeypatch.setattr(bench, "DUMP_BYTES", 8000)
    bench.Bench.dump_outputs(fake, 5, str(tmp_path))                    # steps 0..4 dealt to engines 0 1 2 0 1
    got = {p.stem: np.load(p) for p in tmp_path.iterdir()}
    assert all(a.dtype in (np.float32, np.float64) for a in got.values())
    assert sum(a.nbytes for a in got.values()) <= 8000
    res = engines[1].res
    assert np.all(got["status"] == 1) and got["points_per_scan"].tolist() == [10.0 + s for s in range(40)]
    assert got["check_rows_per_scan"].tolist() == [float(s % 3) for s in range(40)]
    np.testing.assert_array_equal(got["inserted"], [[s, 1, 7 * s, 1, s] for s in range(1, 40, 2)])
    np.testing.assert_array_equal(got["inserted_boxes"], [[1, 2, 3, 0, 0, 0.6, 0.8, 4, 5, 6]] * 20)
    # the longest prefix of the seeded scan order whose clouds fit next to the per-scan records
    left, want = 8000 - 3360 - 8 * 40, []
    for s in np.random.default_rng(0).permutation(40):
        left -= (10 + s) * (24 if ss else 16) + (s % 3) * (20 if ss else 16)
        if left < 0:
            break
        want.append(s)
    pick = got["sample_scans"].astype(int)
    assert len(want) >= 3 and pick.tolist() == sorted(want)
    np.testing.assert_array_equal(got["velodyne"], np.concatenate([res[s].velodyne for s in pick]))
    assert got["check"].shape == (sum(s % 3 for s in pick), 5 if ss else 4)
    if ss:
        np.testing.assert_array_equal(got["labels"], np.concatenate([res[s].labels for s in pick]))
    else:
        assert "labels" not in got


@pytest.mark.parametrize("extra", [["--side", "cut_objects"], ["--impl", "reference"], ["--steps", "0"]])
def test_arguments_the_headline_path_cannot_honour_are_refused(tmp_path, extra):
    import subprocess
    import sys
    p = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--dump-outputs", str(tmp_path / "d")] + extra,
                       capture_output=True, text=True, timeout=120)
    assert p.returncode == 2 and "error" in p.stderr and not (tmp_path / "d").exists()
