"""GPU tier: detection targets of online batches (r3d_engine_targets_device) and the per-scan world augmentation
(r3d_engine_set_world_aug) against host restatements of their formulas."""
import ctypes as C
import math
from types import SimpleNamespace

import numpy as np
import pytest
from scipy import stats

from oracle.online_draws import world_boxes, world_points
from pcl_augmentation_b200 import _lib
from pcl_augmentation_b200 import boxes as bx
from pcl_augmentation_b200.engine import Real3DEngine, ScanInput, scan_input_from_case
from pcl_augmentation_b200.online import OnlineAugmenter, ResidentDataset, WorldAug, epoch_batches
from tests.helpers import case_from_spec

pytestmark = pytest.mark.gpu

MODES = [pytest.param(False, id="walker"), pytest.param(True, id="staged")]
COUNTS = {"od": [2, 1], "ss": [1, 1, 0, 1, 0, 1]}
SEEDS = {"od": list(range(301, 313)), "ss": list(range(401, 413))}
P_MIN = 1e-4
TARGETS = ["Car", "Pedestrian", "Cyclist"]
POLICY = WorldAug(flip_x_prob=0.5, flip_y_prob=0.5, rot_max=math.pi, scale_lo=0.9, scale_hi=1.1)


# ------------------------------------------------------------------ fixtures (as in tests/test_gpu_online.py)
def make_cases(task, n=12):
    cases = [case_from_spec(dict(task=task, seed=s, counts=COUNTS[task], n_cars=1 + i % 5)) for i, s in enumerate(SEEDS[task][:n])]
    for c in cases[1:]:                      # one semseg sequence: one pose / rich map
        c.pose, c.map_data = cases[0].pose, cases[0].map_data
    return cases


def make_store(cases, scans=None):
    scans = scans or [scan_input_from_case(c) for c in cases]
    return ResidentDataset.from_scans(cases[0].task, scans, map_data=cases[0].map_data)


def make_engine(cases, n_scans=12, **kw):
    c = cases[0]
    kw.setdefault("max_points", max(len(x.pcl5) for x in cases))
    return Real3DEngine(c.task, c.config, c.db, max_scans=n_scans, map_data=c.map_data, **kw)


def host_path(cases, idx, counts, perms, **kw):
    """The same scans through ScanInput -> augment_batch with the given schedule tables."""
    scans = []
    for i, j in enumerate(idx):
        s = scan_input_from_case(cases[j])
        scans.append(ScanInput(xyzi=s.xyzi, labels=s.labels, box_lines=s.box_lines, counts=counts[i], perms=perms[i],
                               maps=s.maps, pose=s.pose))
    eng = make_engine(cases, **kw)
    out = eng.augment_batch(scans)
    eng.close()
    return out


# ------------------------------------------------------------------ host restatements
def angle_diff(a, b):
    return np.abs(bx.wrap_pi(np.asarray(a, np.float64) - np.asarray(b, np.float64)))


def obj_dims(eng, obj):
    s = eng.obj_strings[obj]
    items = (s.item() if hasattr(s, "item") else str(s)).split(" ")
    return np.float32(items[10]), np.float32(items[9]), np.float32(items[8])


def target_buffers(n, m):
    import torch
    return {"gt_boxes": torch.full((n, m, 7), 7.0, device="cuda"), "gt_classes": torch.full((n, m), 7, dtype=torch.int32, device="cuda"),
            "n_gt": torch.zeros(n, dtype=torch.int32, device="cuda")}


def targets(eng, store, n):
    m = store.max_kept_boxes(TARGETS) + eng.max_events - 1
    out = target_buffers(n, m)
    eng.targets_device(store, out)
    eng.sync()
    return out["gt_boxes"].cpu().numpy(), out["gt_classes"].cpu().numpy(), out["n_gt"].cpu().numpy()


def outputs(eng):
    eng.sync()
    o = eng.outputs_on_device()
    return {k: (v.cpu().numpy() if hasattr(v, "cpu") else v) for k, v in o.items()}


def world(eng):
    eng.sync()
    return eng.world_device().cpu().numpy()


# ------------------------------------------------------------------ 1 + 2: targets with the policy off
@pytest.mark.parametrize("staged", MODES)
def test_targets_policy_off(staged):
    cases = make_cases("od")
    store = make_store(cases)
    idx = [3, 0, 7, 3, 11, 5]
    eng = make_engine(cases, staged_rounds=staged)
    eng.set_target_classes(TARGETS)
    eng.load_resident(store, idx, 1234, 5)
    eng.run()
    gb, gc, ng = targets(eng, store, len(idx))
    raw = eng.fetch_raw()
    counts, perms = eng.schedule_read()
    want = host_path(cases, idx, counts, perms, staged_rounds=staged)
    assert raw["n_inserted"].sum() > 0
    for s, j in enumerate(idx):
        sb, sc = bx.targets_from_lines_od(cases[j].box_lines, TARGETS)
        k, ni = len(sc), int(raw["n_inserted"][s])
        assert ng[s] == k + ni
        np.testing.assert_array_equal(gb[s, :k], sb)                   # scene rows: bit for bit
        np.testing.assert_array_equal(gc[s, :k], sc)
        for t in range(ni):
            obj, _, ci, _ = (int(v) for v in raw["inserted"][s, t])
            q = raw["inserted_box"][s, t]
            l, w, h = obj_dims(eng, obj)                               # float32 in the ABI
            row = gb[s, k + t]
            np.testing.assert_array_equal(row[:6], np.array([q[0], q[1], q[2] + np.float64(h) * 0.5, l, w, h], np.float64).astype(np.float32))
            head = np.float32(bx.wrap_pi(np.arctan2(q[4], q[3]) - np.pi / 2))
            assert abs(row[6] - head) <= np.spacing(np.abs(head)), (row[6], head)
            assert gc[s, k + t] == TARGETS.index(eng.classes[ci]) + 1
        assert not gb[s, ng[s]:].any() and not gc[s, ng[s]:].any()
        # the reference's annotation lines of the same objects, read with the scene formula (2-decimal rounding)
        r = want[s]
        assert len(r.lines) == ni
        if ni:
            ref, _ = bx.scene_targets_od([line.rstrip("\n") for line in r.lines])
            got = gb[s, k:k + ni].astype(np.float64)
            np.testing.assert_allclose(got[:, :3], ref[:, :3], rtol=0, atol=0.005 + 1e-6)
            np.testing.assert_array_equal(got[:, 3:6], ref[:, 3:6].astype(np.float32))
            assert (angle_diff(got[:, 6], ref[:, 6]) <= 0.005 + 1e-6).all()
    eng.close()


# ------------------------------------------------------------------ 3: world augmentation, off versus on
def check_world_outputs(off, on, w, n):
    for s in range(n):
        a, b = off["offsets"][s], off["offsets"][s + 1]
        assert on["offsets"][s + 1] - on["offsets"][s] == b - a
        x0, x1 = off["xyzi"][a:b], on["xyzi"][on["offsets"][s]:on["offsets"][s + 1]]
        np.testing.assert_array_equal(x1[:, :3], world_points(w[s], x0))
        np.testing.assert_array_equal(x1[:, 3], x0[:, 3])
        np.testing.assert_array_equal(on["labels"][on["offsets"][s]:on["offsets"][s + 1]], off["labels"][a:b])
        ca, cb = off["check_offsets"][s], off["check_offsets"][s + 1]
        c0, c1 = off["check"][ca:cb], on["check"][on["check_offsets"][s]:on["check_offsets"][s + 1]]
        assert len(c0) == len(c1)
        np.testing.assert_array_equal(c1[:, :3], world_points(w[s], c0))
        np.testing.assert_array_equal(c1[:, 3:], c0[:, 3:])


@pytest.mark.parametrize("staged", MODES)
def test_world_aug_od(staged):
    cases = make_cases("od")
    store = make_store(cases)
    idx = [3, 0, 7, 3, 11, 5, 9, 1]
    eng = make_engine(cases, staged_rounds=staged)
    eng.set_target_classes(TARGETS)
    eng.load_resident(store, idx, 77, 2)
    eng.run()
    off = outputs(eng)
    t_off = targets(eng, store, len(idx))
    eng.set_world_aug(POLICY)
    eng.load_resident(store, idx, 77, 2)
    eng.run()
    on = outputs(eng)
    w = world(eng)
    t_on = targets(eng, store, len(idx))
    assert len(off["check"]) > 0
    check_world_outputs(off, on, w, len(idx))
    np.testing.assert_array_equal(t_on[2], t_off[2])
    np.testing.assert_array_equal(t_on[1], t_off[1])
    for s in range(len(idx)):
        n = int(t_off[2][s])
        want = world_boxes(w[s], t_off[0][s, :n])
        got = t_on[0][s, :n]
        np.testing.assert_array_equal(got[:, :6], want[:, :6])
        assert (angle_diff(got[:, 6], want[:, 6]) <= 2e-6).all()
        assert not t_on[0][s, n:].any()
    eng.close()


@pytest.mark.parametrize("staged", MODES)
def test_world_aug_semseg(staged):
    import torch
    cases = make_cases("ss")
    store = make_store(cases)
    idx = [2, 6, 6, 0, 10]
    eng = make_engine(cases, staged_rounds=staged)
    eng.load_resident(store, idx, 5, 1)
    eng.run()
    off = outputs(eng)
    eng.set_world_aug(POLICY)
    eng.load_resident(store, idx, 5, 1)
    eng.run()
    on = outputs(eng)
    w = world(eng)
    check_world_outputs(off, on, w, len(idx))
    with pytest.raises(_lib.Real3DError):
        eng.targets_device(store, target_buffers(len(idx), 16))
    # the C call refuses a semseg engine too, before any launch
    lib = _lib.load()
    buf = target_buffers(len(idx), 16)
    before = lib.r3d_launch_count()
    dummy = torch.zeros(16 * 7, device="cuda")
    rc = lib.r3d_engine_targets_device(eng.handle, C.byref(store.abi), dummy.data_ptr(), dummy.data_ptr(), 16,
                                       buf["gt_boxes"].data_ptr(), buf["gt_classes"].data_ptr(), buf["n_gt"].data_ptr())
    assert rc != 0 and lib.r3d_launch_count() == before
    eng.close()


# ------------------------------------------------------------------ 4: independence of batching and sharding
def test_world_params_independent_of_batching():
    cases = make_cases("od")
    store = make_store(cases)
    eng = make_engine(cases)
    eng.set_world_aug(POLICY)
    eng.load_resident(store, list(range(12)), 9, 3)
    full = world(eng)
    for sub in ([7, 2, 5, 7], [5], [11, 0, 11, 3, 3]):
        eng.load_resident(store, sub, 9, 3)
        np.testing.assert_array_equal(world(eng), full[sub])
    for rank in (0, 1):
        for b in epoch_batches(12, 4, rank=rank, world=2, seed=9, epoch=3):
            eng.load_resident(store, b, 9, 3)
            np.testing.assert_array_equal(world(eng), full[b])
    for seed, epoch in ((9, 4), (10, 3)):
        eng.load_resident(store, list(range(12)), seed, epoch)
        other = world(eng)
        assert (other[:, 2] != full[:, 2]).sum() >= 11 and (other[:, 5] != full[:, 5]).sum() >= 11
    eng.close()


# ------------------------------------------------------------------ 5: distributions
def test_world_param_distributions():
    cases = make_cases("od")
    store = make_store(cases)
    eng = make_engine(cases)
    pol = WorldAug(flip_x_prob=0.3, flip_y_prob=0.5, rot_max=0.7, scale_lo=0.9, scale_hi=1.2)
    eng.set_world_aug(pol)
    draws = []
    for epoch in range(350):
        eng.load_resident(store, list(range(12)), 31, epoch)
        draws.append(world(eng))
    w = np.concatenate(draws).astype(np.float64)
    n = len(w)
    assert n >= 4096
    r = np.float64(np.float32(pol.rot_max))
    assert stats.kstest(w[:, 2], "uniform", args=(-r, 2 * r)).pvalue > P_MIN
    lo, hi = np.float64(np.float32(pol.scale_lo)), np.float64(np.float32(pol.scale_hi))
    assert stats.kstest(w[:, 5], "uniform", args=(lo, hi - lo)).pvalue > P_MIN
    assert set(np.unique(w[:, :2])) <= {0.0, 1.0}
    assert stats.binomtest(int(w[:, 0].sum()), n, 0.3).pvalue > P_MIN
    assert stats.binomtest(int(w[:, 1].sum()), n, 0.5).pvalue > P_MIN
    np.testing.assert_allclose(w[:, 3], np.cos(w[:, 2]), rtol=0, atol=2e-7)
    np.testing.assert_allclose(w[:, 4], np.sin(w[:, 2]), rtol=0, atol=2e-7)
    assert (w[:, 6:] == 0).all()
    eng.set_world_aug(WorldAug(flip_x_prob=0.0, flip_y_prob=0.0, rot_max=0.0, scale_lo=1.0, scale_hi=1.0))
    for epoch in range(20):
        eng.load_resident(store, list(range(12)), 31, epoch)
        w0 = world(eng)
        assert (w0[:, :2] == 0).all() and (w0[:, 2] == 0).all() and (w0[:, 3] == 1).all() and (w0[:, 4] == 0).all()
        assert (w0[:, 5] == 1).all()
    eng.close()


# ------------------------------------------------------------------ 6: the host path is untouched
def test_host_path_never_transformed():
    cases = make_cases("od", 6)
    store = make_store(cases)
    scans = [scan_input_from_case(c) for c in cases]
    eng = make_engine(cases, n_scans=6)
    eng.set_world_aug(POLICY)
    eng.load_resident(store, [0, 1, 2], 3, 0)
    eng.run()
    eng.sync()
    got = eng.augment_batch(scans)
    with pytest.raises(_lib.Real3DError):
        eng.world_device()
    eng.close()
    fresh = make_engine(cases, n_scans=6)
    want = fresh.augment_batch(scans)
    fresh.close()
    for a, b in zip(got, want):
        np.testing.assert_array_equal(a.velodyne, b.velodyne)
        np.testing.assert_array_equal(a.check, b.check)
        assert a.inserted == b.inserted and a.lines == b.lines


# ------------------------------------------------------------------ 7: errors before anything is enqueued
def test_errors_before_enqueue():
    cases = make_cases("od", 6)
    store = make_store(cases)
    eng = make_engine(cases, n_scans=6)
    lib = _lib.load()
    for bad in (dict(flip_x_prob=1.5), dict(flip_y_prob=-0.1), dict(rot_max=3.5), dict(rot_max=-1.0), dict(scale_lo=0.0),
                dict(scale_lo=1.2, scale_hi=1.1), dict(scale_hi=float("inf")), dict(flip_x_prob=float("nan"))):
        p = dict(flip_x_prob=0.5, flip_y_prob=0.5, rot_max=0.5, scale_lo=0.95, scale_hi=1.05)
        p.update(bad)
        with pytest.raises(_lib.Real3DError):
            eng.set_world_aug(SimpleNamespace(**p))                  # past WorldAug's own checks, to the C validation
    eng.set_target_classes(TARGETS)
    m = store.max_kept_boxes(TARGETS) + eng.max_events - 1
    idx = [0, 4, 5]
    eng.load_resident(store, idx, 3, 0)
    before = lib.r3d_launch_count()
    with pytest.raises(_lib.Real3DError):                            # not run yet
        eng.targets_device(store, target_buffers(len(idx), m))
    assert lib.r3d_launch_count() == before
    eng.run()
    before = lib.r3d_launch_count()
    with pytest.raises(_lib.Real3DError):                            # max_targets too small for the fullest scan
        eng.targets_device(store, target_buffers(len(idx), m - 1))
    assert lib.r3d_launch_count() == before
    eng.targets_device(store, target_buffers(len(idx), m))
    eng.augment_batch([scan_input_from_case(c) for c in cases[:2]])   # a host batch
    before = lib.r3d_launch_count()
    with pytest.raises(_lib.Real3DError):
        eng.targets_device(store, target_buffers(2, m))
    assert lib.r3d_launch_count() == before
    eng.close()
    ss = make_cases("ss", 2)
    with pytest.raises(_lib.Real3DError):
        make_engine(ss, n_scans=2).set_target_classes(TARGETS)


# ------------------------------------------------------------------ 8: lifetime of a batch's targets and parameters
def test_depth2_targets_stay_valid_while_next_is_enqueued():
    import torch
    cases = make_cases("od", 12)
    store = make_store(cases)
    aug = OnlineAugmenter("od", cases[0].config, cases[0].db, store, batch_size=4, seed=11, depth=2,
                          target_classes=TARGETS, world_aug=POLICY)
    ref = make_engine(cases, n_scans=4)
    ref.set_world_aug(POLICY)
    consumer = torch.cuda.Stream()
    seen = 0
    with torch.cuda.stream(consumer):
        for k, batch in enumerate(aug.epoch(0)):
            torch.cuda._sleep(20_000_000)                 # a slow training step in front of the read
            boxes, classes, n_gt, w = batch.gt_boxes.clone(), batch.gt_classes.clone(), batch.n_gt.clone(), batch.world.clone()
            consumer.synchronize()
            n = len(batch.indices)
            assert boxes.shape == (n, aug.max_targets, 7) and classes.shape == (n, aug.max_targets)
            ref.load_resident(store, batch.indices, 11, 0)
            np.testing.assert_array_equal(w.cpu().numpy(), world(ref))
            eng = aug.engines[k % 2]                      # still holds batch k: its targets again, into fresh buffers
            again = target_buffers(n, aug.max_targets)
            eng.targets_device(store, again)
            eng.sync()
            np.testing.assert_array_equal(boxes.cpu().numpy(), again["gt_boxes"].cpu().numpy())
            np.testing.assert_array_equal(classes.cpu().numpy(), again["gt_classes"].cpu().numpy())
            np.testing.assert_array_equal(n_gt.cpu().numpy(), again["n_gt"].cpu().numpy())
            for s, j in enumerate(batch.indices):
                sb, _ = bx.targets_from_lines_od(cases[j].box_lines, TARGETS)
                got = boxes[s, :len(sb)].cpu().numpy()
                np.testing.assert_array_equal(got[:, :6], world_boxes(w[s].cpu().numpy(), sb)[:, :6])
            seen += n
    assert seen == 12
    ref.close()
    aug.close()
