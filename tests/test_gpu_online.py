"""GPU tier: online augmentation from a device-resident dataset (r3d_engine_load_resident, online.OnlineAugmenter)
against the host path (ScanInput -> augment_batch) fed the schedule tables the device drew."""
import numpy as np
import pytest
from scipy import stats

from pcl_augmentation_b200 import _lib
from pcl_augmentation_b200.engine import Real3DEngine, ScanInput, scan_input_from_case
from pcl_augmentation_b200.online import OnlineAugmenter, ResidentDataset
from tests.helpers import case_from_spec

pytestmark = pytest.mark.gpu

MODES = [pytest.param(False, id="walker"), pytest.param(True, id="staged")]
COUNTS = {"od": [2, 1], "ss": [1, 1, 0, 1, 0, 1]}
SEEDS = {"od": list(range(301, 313)), "ss": list(range(401, 413))}
P_MIN = 1e-4


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


def resident_run(eng, store, idx, seed, epoch):
    eng.load_resident(store, idx, seed, epoch)
    eng.run()
    return eng.unpack(eng.fetch_raw())


def assert_same(a, b):
    np.testing.assert_array_equal(a.velodyne, b.velodyne)
    np.testing.assert_array_equal(a.labels, b.labels)
    np.testing.assert_array_equal(a.check, b.check)
    assert a.inserted == b.inserted and a.visible == b.visible and a.lines == b.lines


@pytest.mark.parametrize("staged", MODES)
@pytest.mark.parametrize("task", ["od", "ss"])
def test_resident_equals_host_path(task, staged):
    cases = make_cases(task)
    store = make_store(cases)
    idx = [3, 0, 7, 3, 11, 5]
    eng = make_engine(cases, staged_rounds=staged)
    got = resident_run(eng, store, idx, seed=1234, epoch=5)
    counts, perms = eng.schedule_read()
    eng.close()
    assert perms.shape[1] == eng.max_events
    want = host_path(cases, idx, counts, perms, staged_rounds=staged)
    assert sum(len(r.inserted) for r in got) > 0
    for a, b in zip(got, want):
        assert a.status == 0
        assert_same(a, b)
    assert_same(got[0], got[3])                  # the duplicate: same store scan, same draws


def test_independent_of_batching():
    cases = make_cases("od", 8)
    store = make_store(cases)
    eng = make_engine(cases, n_scans=8)
    full = resident_run(eng, store, list(range(8)), seed=9, epoch=3)
    c_full, p_full = eng.schedule_read()
    part = resident_run(eng, store, [7, 2, 5], seed=9, epoch=3)
    c_part, p_part = eng.schedule_read()
    alone = resident_run(eng, store, [5], seed=9, epoch=3)
    for i, j in enumerate([7, 2, 5]):
        assert_same(part[i], full[j])
        np.testing.assert_array_equal(c_part[i], c_full[j])
        np.testing.assert_array_equal(p_part[i], p_full[j])
    assert_same(alone[0], full[5])
    for seed, epoch in ((9, 4), (10, 3)):
        eng.load_resident(store, list(range(8)), seed, epoch)
        c, p = eng.schedule_read()
        assert sum(not np.array_equal(p[i], p_full[i]) for i in range(8)) >= 7
    eng.close()


@pytest.mark.parametrize("tries", [20, 128])
def test_schedule_distribution(tries):
    cases = make_cases("od", 12)
    store = make_store(cases)
    eng = make_engine(cases, max_tries=tries)
    n_c = len(cases[0].db["Pedestrian"])
    nobj = int(cases[0].config["insertion"]["number_of_object"])
    counts, heads = [], []
    for epoch in range(200):
        eng.load_resident(store, list(range(12)), 77, epoch)
        c, p = eng.schedule_read()
        counts.append(c)
        heads.append(p.reshape(-1, tries))
    counts, heads = np.concatenate(counts), np.concatenate(heads)
    assert (counts.sum(axis=1) == nobj).all()
    totals = counts.sum(axis=0)
    assert stats.chisquare(totals).pvalue > P_MIN
    k = min(tries, n_c)
    assert (heads[:, :k] >= 0).all() and (heads[:, :k] < n_c).all() and (heads[:, k:] == -1).all()
    srt = np.sort(heads[:, :k], axis=1)
    assert (np.diff(srt, axis=1) > 0).all()                    # distinct entries
    for pos in (0, k - 1):
        assert stats.chisquare(np.bincount(heads[:, pos], minlength=n_c)).pvalue > P_MIN
    eng.close()


def test_fixed_counts():
    cases = make_cases("od", 4)
    cfg = dict(cases[0].config)
    cfg["insertion"] = dict(cfg["insertion"], random=False, number_of_classes=[2, 1])
    eng = Real3DEngine("od", cfg, cases[0].db, max_scans=4, max_points=len(cases[0].pcl5))
    eng.load_resident(make_store(cases), [0, 1, 2, 3], 1, 0)
    c, _ = eng.schedule_read()
    assert (c == [2, 1]).all()
    eng.close()


@pytest.mark.parametrize("task", ["od", "ss"])
def test_augmented_batch_boxes(task):
    cases = make_cases(task, 8)
    store = make_store(cases)
    aug = OnlineAugmenter(task, cases[0].config, cases[0].db, store, batch_size=8, seed=5, depth=1)
    idx = [6, 1, 4, 4, 0]
    batch = aug.augment(idx, epoch=2)
    eng = aug.engines[0]
    counts, perms = eng.schedule_read()
    want = host_path(cases, idx, counts, perms)
    n_ins = batch.n_inserted.cpu().numpy()
    boxes, obj = batch.boxes.cpu().numpy(), batch.object_id.cpu().numpy()
    vis, cls = batch.visible.cpu().numpy(), batch.class_index.cpu().numpy()
    assert n_ins.sum() > 0
    for s, r in enumerate(want):
        assert n_ins[s] == len(r.inserted)
        for j, ((name, rot, c), b) in enumerate(zip(r.inserted, r.boxes)):
            assert eng.obj_names[obj[s, j]] == name and eng.classes[cls[s, j]] == c and vis[s, j] == r.visible[j]
            assert batch.rotation[s, j].item() == rot
            m = b["_matrix"]
            ref = np.array([b["center"]["x"], b["center"]["y"], b["center"]["z"], b["length"], b["width"], b["height"],
                            np.arctan2(m[1, 0], m[0, 0])], dtype=np.float64)
            np.testing.assert_allclose(boxes[s, j], ref.astype(np.float32), rtol=0, atol=1e-6)
        assert not boxes[s, len(r.inserted):].any()
        a, b = batch.offsets[s], batch.offsets[s + 1]
        np.testing.assert_array_equal(batch.xyzi[a:b].cpu().numpy(), r.velodyne)
    np.testing.assert_array_equal(batch.indices, idx)
    aug.close()


def test_errors_before_any_launch():
    cases = make_cases("od", 4)                      # 1, 2, 3, 4 scene boxes
    scans = [scan_input_from_case(c) for c in cases]
    for i in (0, 3):                                 # two short scans: 1 and 4 scene boxes
        scans[i].xyzi, scans[i].labels = scans[i].xyzi[:5000], scans[i].labels[:5000]
    store = make_store(cases, scans)
    kw = dict(n_scans=4, max_points=5000, max_boxes=3)
    eng = make_engine(cases, **kw)
    lib = _lib.load()
    # index out of range (both sides), a scan over max_points, a scan with too many scene boxes
    for bad in ([0, 4], [0, -1], [0, 2], [0, 3]):
        before = lib.r3d_launch_count()
        with pytest.raises(_lib.Real3DError):
            eng.load_resident(store, bad, 3, 0)
        assert lib.r3d_launch_count() == before
    eng.load_resident(store, [0], 3, 0)
    eng.run()
    got = eng.unpack(eng.fetch_raw(), raise_on_error=False)
    eng.close()
    fresh = make_engine(cases, **kw)
    fresh.load_resident(store, [0], 3, 0)
    fresh.run()
    want = fresh.unpack(fresh.fetch_raw(), raise_on_error=False)
    fresh.close()
    assert got[0].status == want[0].status
    assert_same(got[0], want[0])


def test_depth2_batches_stay_valid_while_next_is_enqueued():
    import torch
    cases = make_cases("od", 12)
    store = make_store(cases)
    aug = OnlineAugmenter("od", cases[0].config, cases[0].db, store, batch_size=4, seed=11, depth=2)
    consumer = torch.cuda.Stream()
    seen = 0
    with torch.cuda.stream(consumer):
        for k, batch in enumerate(aug.epoch(0)):
            torch.cuda._sleep(20_000_000)                 # a slow training step in front of the read
            copy = batch.xyzi.clone()                      # read on the consumer stream; batch k + 1 is already enqueued
            boxes = batch.boxes.clone()
            eng = aug.engines[k % 2]
            raw = eng.fetch_raw()
            consumer.synchronize()
            rows = int(batch.offsets[-1])
            np.testing.assert_array_equal(copy.cpu().numpy(), raw["xyzi"][:rows])
            n = len(batch.indices)
            assert (boxes[:, :, 0].cpu().numpy()[np.arange(aug.max_events)[None, :] >= raw["n_inserted"][:n, None]] == 0).all()
            seen += n
    assert seen == 12
    aug.close()
