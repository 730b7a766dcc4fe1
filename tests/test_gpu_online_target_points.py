"""GPU tier: points of the augmented clouds inside their detection targets (r3d_engine_target_points_device): counts,
first-hit assignment and the min-points filter against the host reference oracle/target_points.py."""
import math

import numpy as np
import pytest

from oracle.target_points import filter_min_points, near_faces, points_in_boxes, target_points
from pcl_augmentation_b200 import _lib
from pcl_augmentation_b200.engine import scan_input_from_case
from pcl_augmentation_b200.online import OnlineAugmenter, WorldAug
from tests.test_gpu_online_targets import MODES, POLICY, TARGETS, make_cases, make_engine, make_store, target_buffers

pytestmark = pytest.mark.gpu

IDX = [3, 0, 7, 3, 11, 5]                     # store index 3 twice


def buffers(eng, store, n, m=None):
    import torch
    out = target_buffers(n, m or store.max_kept_boxes(TARGETS) + eng.max_events - 1)
    out["gt_points"] = torch.full(out["gt_classes"].shape, 7, dtype=torch.int32, device="cuda")
    return out


def point_gt_buffer(eng):
    import torch
    return torch.full((eng.max_scans * (eng.max_points + eng.max_inserted + 16),), 7, dtype=torch.int32, device="cuda")


def host(out):
    return {k: v.cpu().numpy() for k, v in out.items()}


def run_batch(cases, store, staged=False, world_aug=None, idx=IDX, **kw):
    eng = make_engine(cases, staged_rounds=staged, **kw)
    eng.set_world_aug(world_aug)
    eng.set_target_classes(TARGETS)
    eng.load_resident(store, idx, 1234, 5)
    eng.run()
    return eng


def points_and_targets(eng, store, n, min_points):
    """Targets, then target points with min_points: (outputs, targets before the call, targets after, point_gt)."""
    out = buffers(eng, store, n)
    pg = point_gt_buffer(eng)
    eng.targets_device(store, out)
    eng.sync()
    before = host(out)
    eng.target_points_device(out, min_points, pg)
    eng.sync()
    o = eng.outputs_on_device()
    total = int(o["offsets"][n])
    return o, before, host(out), pg[:total].cpu().numpy()


def check_against_reference(o, before, after, pg, n, k):
    """Every scan: kept set, counts, compaction, zero padding and point_gt as the reference computes them."""
    xyz = o["xyzi"].cpu().numpy()[:, :3]
    off = o["offsets"]
    near_total, dropped = 0, 0
    for s in range(n):
        rows = xyz[off[s]:off[s + 1]]
        m = int(before["n_gt"][s])
        boxes = before["gt_boxes"][s, :m]
        near_total += int(near_faces(rows, boxes).sum())
        kept, counts, gt = filter_min_points(rows, boxes, k)
        mk = len(kept)
        dropped += m - mk
        assert after["n_gt"][s] == mk
        np.testing.assert_array_equal(after["gt_boxes"][s, :mk], boxes[kept])
        np.testing.assert_array_equal(after["gt_classes"][s, :mk], before["gt_classes"][s, kept])
        np.testing.assert_array_equal(after["gt_points"][s, :mk], counts)
        assert not after["gt_boxes"][s, mk:].any() and not after["gt_classes"][s, mk:].any()
        assert not after["gt_points"][s, mk:].any()
        np.testing.assert_array_equal(pg[off[s]:off[s + 1]], gt)
    # rows on a face (cut objects reach their box's top face): compared above all the same, and reported
    print(f"points within 1e-9 m of a face: {near_total}; targets dropped: {dropped}")
    assert near_total <= 1e-4 * len(xyz)
    return dropped


# ------------------------------------------------------------------ counts and point_gt against the reference
@pytest.mark.parametrize("world_aug", [None, POLICY], ids=["plain", "world"])
@pytest.mark.parametrize("staged", MODES)
def test_counts_and_point_gt(staged, world_aug):
    cases = make_cases("od")
    store = make_store(cases)
    eng = run_batch(cases, store, staged, world_aug)
    o, before, after, pg = points_and_targets(eng, store, len(IDX), 0)
    assert eng.fetch_raw()["n_inserted"].sum() > 0
    assert check_against_reference(o, before, after, pg, len(IDX), 0) == 0
    assert (pg >= 0).any() and (pg < 0).any()
    eng.close()


# ------------------------------------------------------------------ the min-points filter
@pytest.mark.parametrize("staged", MODES)
def test_min_points_filter(staged):
    cases = make_cases("od")
    store = make_store(cases)
    eng = run_batch(cases, store, staged, POLICY)
    n = len(IDX)
    _, before, counted, _ = points_and_targets(eng, store, n, 0)
    raw = eng.fetch_raw()
    scene = [int(before["n_gt"][s] - raw["n_inserted"][s]) for s in range(n)]
    ins_counts = [int(counted["gt_points"][s, t]) for s in range(n) for t in range(scene[s], int(before["n_gt"][s]))]
    k_ins = min(ins_counts) + 1                   # drops at least one inserted target
    for k in (1, 40, k_ins):
        o, before_k, after, pg = points_and_targets(eng, store, n, k)
        np.testing.assert_array_equal(before_k["gt_boxes"], before["gt_boxes"])
        dropped = check_against_reference(o, before_k, after, pg, n, k)
        if k == k_ins:
            assert dropped > 0
    eng.close()


def test_k0_and_off_leave_targets_and_rows_unchanged():
    cases = make_cases("od")
    store = make_store(cases)
    eng = run_batch(cases, store, False, POLICY)
    n = len(IDX)
    rows_off = eng.outputs_on_device()["xyzi"].cpu().numpy().copy()
    out = buffers(eng, store, n)
    eng.targets_device(store, out)
    eng.sync()
    plain = host(out)
    eng.target_points_device(out, 0, point_gt_buffer(eng))
    eng.sync()
    after = host(out)
    for key in ("gt_boxes", "gt_classes", "n_gt"):
        assert after[key].tobytes() == plain[key].tobytes()
    assert eng.outputs_on_device()["xyzi"].cpu().numpy().tobytes() == rows_off.tobytes()
    eng.close()


# ------------------------------------------------------------------ scans with more than 32 and 64 targets
def crowded_lines(xyz, count, rng):
    """``count`` Car lines (KITTI camera frame) around points of the scan, overlapping one another."""
    lines = []
    for p in xyz[rng.choice(len(xyz), count, replace=False)]:
        h, w, l = 1.5, 1.6, 3.9
        cam_x, cam_z, cam_y = -p[1], p[0] - 0.27, -(p[2] - h / 2) - 0.08
        ry = rng.uniform(-math.pi, math.pi)
        lines.append(f"Car 0.00 0 0.00 100.00 120.00 150.00 220.00 {h:.2f} {w:.2f} {l:.2f} {cam_x:.2f} {cam_y:.2f} {cam_z:.2f} {ry:.2f}")
    return lines


@pytest.mark.parametrize("staged", MODES)
def test_more_than_32_and_64_targets(staged):
    cases = make_cases("od", 4)
    scans = [scan_input_from_case(c) for c in cases]
    rng = np.random.default_rng(5)
    for s, extra in ((0, 40), (1, 90)):
        scans[s].box_lines = list(scans[s].box_lines) + crowded_lines(scans[s].xyzi[:, :3], extra, rng)
    store = make_store(cases, scans)
    idx = [0, 1, 2, 1]
    eng = run_batch(cases, store, staged, None, idx=idx, n_scans=4, max_boxes=160)
    for k in (0, 3):
        o, before, after, pg = points_and_targets(eng, store, len(idx), k)
        assert before["n_gt"][0] > 32 and before["n_gt"][1] > 64
        check_against_reference(o, before, after, pg, len(idx), k)
    eng.close()


# ------------------------------------------------------------------ why: occlusion empties scene targets
def test_scene_targets_lose_points_to_occlusion():
    cases = make_cases("od")
    store = make_store(cases)
    idx = list(range(12))
    eng = run_batch(cases, store, False, None, idx=idx)
    o, before, after, _ = points_and_targets(eng, store, len(idx), 0)
    raw = eng.fetch_raw()
    fewer = 0
    for s, j in enumerate(idx):
        k = int(before["n_gt"][s] - raw["n_inserted"][s])
        boxes = before["gt_boxes"][s, :k]
        raw_counts = points_in_boxes(scan_input_from_case(cases[j]).xyzi[:, :3], boxes).sum(axis=0)
        fewer += int((after["gt_points"][s, :k] < raw_counts).sum())
    print(f"scene targets with fewer points after augmentation: {fewer}")
    assert fewer >= 1
    eng.close()


# ------------------------------------------------------------------ errors before anything is enqueued
def test_errors_before_enqueue():
    cases = make_cases("od", 6)
    store = make_store(cases)
    eng = make_engine(cases, n_scans=6)
    eng.set_target_classes(TARGETS)
    lib = _lib.load()
    idx = [0, 4, 5]
    out = buffers(eng, store, len(idx))
    pg = point_gt_buffer(eng)
    m = int(out["gt_boxes"].shape[1])

    def call(max_targets=m, k=0, null=None):
        ptrs = [out["gt_boxes"].data_ptr(), out["gt_classes"].data_ptr(), out["n_gt"].data_ptr(), out["gt_points"].data_ptr(),
                pg.data_ptr()]
        if null is not None:
            ptrs[null] = None
        return lib.r3d_engine_target_points_device(eng.handle, max_targets, ptrs[0], ptrs[1], ptrs[2], k, ptrs[3], ptrs[4])

    def refused(**kw):
        before = lib.r3d_launch_count()
        assert call(**kw) != 0
        assert lib.r3d_launch_count() == before

    eng.load_resident(store, idx, 3, 0)
    refused()                                          # not run yet
    eng.run()
    refused()                                          # no targets for this batch yet
    eng.targets_device(store, out)
    for null in range(5):
        refused(null=null)
    refused(k=-1)
    refused(max_targets=0)
    before = lib.r3d_launch_count()
    assert call(k=1) == 0 and lib.r3d_launch_count() > before
    eng.augment_batch([scan_input_from_case(c) for c in cases[:2]])   # a host batch
    refused()
    with pytest.raises(_lib.Real3DError):
        eng.target_points_device(out, -1, pg)
    eng.close()
    ss = make_cases("ss", 2)
    se = make_engine(ss, n_scans=2)
    ss_store = make_store(ss)
    se.load_resident(ss_store, [0, 1], 3, 0)
    se.run()
    refused_ss = lib.r3d_engine_target_points_device(se.handle, m, out["gt_boxes"].data_ptr(), out["gt_classes"].data_ptr(),
                                                     out["n_gt"].data_ptr(), 0, out["gt_points"].data_ptr(), pg.data_ptr())
    assert refused_ss != 0
    se.close()


# ------------------------------------------------------------------ lifetime with two batches in flight
def test_depth2_buffers_stay_valid_while_next_is_enqueued():
    import torch
    cases = make_cases("od", 12)
    store = make_store(cases)
    aug = OnlineAugmenter("od", cases[0].config, cases[0].db, store, batch_size=4, seed=11, depth=2,
                          target_classes=TARGETS, world_aug=WorldAug(), target_points=1)
    consumer = torch.cuda.Stream()
    seen = 0
    with torch.cuda.stream(consumer):
        for batch in aug.epoch(0):
            torch.cuda._sleep(20_000_000)                 # a slow training step in front of the read
            snap = {k: getattr(batch, k).clone() for k in ("xyzi", "gt_boxes", "n_gt", "gt_points", "point_gt")}
            consumer.synchronize()
            h = {k: v.cpu().numpy() for k, v in snap.items()}
            n = len(batch.indices)
            assert h["gt_points"].shape == (n, aug.max_targets) and len(h["point_gt"]) == len(h["xyzi"])
            for s in range(n):
                a, b = batch.offsets[s], batch.offsets[s + 1]
                m = int(h["n_gt"][s])
                counts, first = target_points(h["xyzi"][a:b, :3], h["gt_boxes"][s, :m])
                assert (counts >= 1).all()
                np.testing.assert_array_equal(h["gt_points"][s, :m], counts)
                np.testing.assert_array_equal(h["point_gt"][a:b], first)
            seen += n
    assert seen == 12
    aug.close()
