"""GPU tier: the online path's draws (k_draw_schedule, k_draw_world) entry for entry against the numpy restatement
oracle/online_draws.py, across class-list lengths around max_tries and the warp width, empty classes, 16 classes with up
to 301 events, fixed counts, Lemire rejections, max_tries past 1024, and seeds / epochs of 2^32 and more; and the
detection targets (k_gt_targets) of scans with more than 32 scene boxes and more than 32 inserted objects."""
import copy
import ctypes as C
import math

import numpy as np
import pytest

from oracle import online_draws as od
from pcl_augmentation_b200 import _lib
from pcl_augmentation_b200 import boxes as bx
from pcl_augmentation_b200.engine import Real3DEngine, scan_input_from_case
from pcl_augmentation_b200.online import ResidentDataset, WorldAug
from tests.helpers import case_from_spec

pytestmark = pytest.mark.gpu

KEYS = [(1234, 5), (2**64 - 1, 2**32 + 5), (2**32, 7), (0, 2**32)]
IDX = [3, 0, 7, 3, 11, 5, 0, 9]                      # duplicates draw the same as their first occurrence


# ------------------------------------------------------------------ fixtures
@pytest.fixture(scope="module")
def base():
    return case_from_spec(dict(task="od", seed=301, counts=[2, 1], n_cars=2))


@pytest.fixture(scope="module")
def store(base):
    """32 store scans; the draws depend on the store index only, so they may all hold the same scan."""
    return ResidentDataset.from_scans("od", [scan_input_from_case(base)] * 32)


def draw_config(base, n_classes, nobj=0, fixed=None):
    names = [f"K{c}" for c in range(n_classes)]
    cfg = copy.deepcopy(base.config)
    cfg["insertion"].update(classes=names, min_points={n: 40 for n in names}, placement={n: "Road" for n in names},
                            labels_shortcut={n: n for n in names}, random=fixed is None, number_of_object=nobj,
                            number_of_classes=list(fixed) if fixed is not None else [0] * n_classes)
    return cfg


def draw_engine(base, list_lens, T, nobj=0, fixed=None, n_scans=12):
    """An engine that only draws: class c holds list_lens[c] reused DB samples under new names."""
    samples = [s for _, s in base.db["Pedestrian"]]
    cfg = draw_config(base, len(list_lens), nobj, fixed)
    db = {n: [(f"{n}_{j:06d}", samples[j % len(samples)]) for j in range(m)]
          for n, m in zip(cfg["insertion"]["classes"], list_lens)}
    return Real3DEngine("od", cfg, db, max_scans=n_scans, max_points=len(base.pcl5), max_tries=T, max_inserted=4096)


def check_draws(eng, store, list_lens, idx=IDX, keys=KEYS, nobj=0, fixed=None):
    """Counts and heads of every (seed, epoch) equal to the reference's; returns the words the reference rejected."""
    rejected = 0
    for seed, epoch in keys:
        eng.load_resident(store, idx, seed, epoch)
        counts, perms = eng.schedule_read()
        want_c, want_h, rej = od.draw_schedule(idx, seed, epoch, eng.max_events, list_lens, eng.max_tries,
                                               random=fixed is None, number_of_object=nobj, fixed=fixed)
        np.testing.assert_array_equal(counts, want_c, err_msg=f"counts, key {seed, epoch}")
        np.testing.assert_array_equal(perms, want_h, err_msg=f"heads, key {seed, epoch}")
        rejected += rej
    return rejected


# ------------------------------------------------------------------ schedule draws
@pytest.mark.parametrize("T", [1, 31, 32, 33, 100])
def test_heads_around_max_tries(base, store, T):
    """n_c in {1, T - 1, T, T + 1, 3 T}: heads shorter than, as long as and cut from the shuffle; T - 1 = 0 at T = 1 is
    an empty class, whose heads are all -1."""
    lens = [1, T - 1, T, T + 1, 3 * T]
    eng = draw_engine(base, lens, T, nobj=6)
    check_draws(eng, store, lens, nobj=6)
    eng.close()


@pytest.mark.parametrize("nobj", [0, 1, 127, 128, 129, 300])
def test_sixteen_classes(base, store, nobj):
    """C = 16 with up to 301 events: stream ids up to 1 + 300 * 16 + 15, counts past four words of a round."""
    lens = [0 if c == 5 else 1 + (c * 13) % 40 for c in range(16)]
    eng = draw_engine(base, lens, 8, nobj=nobj)
    assert eng.max_events == nobj + 1
    check_draws(eng, store, lens, nobj=nobj)
    eng.close()


def test_fixed_counts_with_zeros(base, store):
    lens, fixed = [5, 40, 0, 33], [0, 3, 0, 2]
    eng = draw_engine(base, lens, 32, fixed=fixed)
    assert eng.max_events == 6
    check_draws(eng, store, lens, fixed=fixed)
    eng.close()


def test_head_rejections(base, store):
    """One class of 129971 objects at T = 1024: Lemire's method rejects a word with probability (2^32 mod r) / 2^32,
    about 0.0155 rejected words per head, so 2048 heads meet some.  The object DB is tiled on the ABI directly (four
    points per object), which is much faster than 130k objects through the Python DB preparation."""
    n_c, T = 129971, 1024
    eng = draw_engine(base, [100], T, nobj=15, n_scans=32)
    pts = np.ascontiguousarray(eng._db_points[:4])
    keep = [np.ascontiguousarray(np.tile(pts, (n_c, 1))), np.arange(n_c + 1, dtype=np.int64) * 4,
            np.ascontiguousarray(np.tile(eng._db_boxes[:1], (n_c, 1))), np.zeros(n_c, dtype=np.int32),
            np.array([0, n_c], dtype=np.int32), np.arange(n_c, dtype=np.int32)]
    db = _lib.ObjectDb()
    db.n_objects = n_c
    db.points5, db.point_offsets, db.boxes, db.class_index, db.class_list_offsets, db.class_list = (a.ctypes.data for a in keep)
    _lib.check(eng.lib.r3d_engine_set_objects(eng.handle, C.byref(db)), "set_objects")
    rejected = check_draws(eng, store, [n_c], idx=list(range(32)), nobj=15)
    assert rejected >= 5, rejected                   # the comparison covered redrawn words
    eng.close()


@pytest.mark.parametrize("T", [1025, 4096])
def test_max_tries_past_1024(base, store, T):
    """More than 48 KiB of dynamic shared memory per block for the draw kernel."""
    lens = [T + 1, 2 * T]
    eng = draw_engine(base, lens, T, nobj=2)
    check_draws(eng, store, lens, keys=KEYS[:2], nobj=2)
    eng.close()


def test_max_tries_beyond_device_bound(base, store):
    """max_tries above 4266 is refused by load_resident before anything is enqueued; the host path still takes it."""
    T = 4267
    eng = Real3DEngine("od", base.config, base.db, max_scans=4, max_points=len(base.pcl5), max_tries=T)
    lib = _lib.load()
    before = lib.r3d_launch_count()
    with pytest.raises(_lib.Real3DError):
        eng.load_resident(store, [0, 1], 1, 0)
    assert lib.r3d_launch_count() == before
    got = eng.augment_batch([scan_input_from_case(base)])[0]
    eng.close()
    fresh = Real3DEngine("od", base.config, base.db, max_scans=4, max_points=len(base.pcl5), max_tries=T)
    want = fresh.augment_batch([scan_input_from_case(base)])[0]
    fresh.close()
    assert got.status == 0 and len(got.inserted) > 0
    np.testing.assert_array_equal(got.velodyne, want.velodyne)
    assert got.inserted == want.inserted and got.lines == want.lines


# ------------------------------------------------------------------ world draw
WORLD_POLICIES = [
    WorldAug(flip_x_prob=0.0, flip_y_prob=1.0, rot_max=0.0, scale_lo=1.0, scale_hi=1.0),
    WorldAug(flip_x_prob=1.0, flip_y_prob=0.0, rot_max=math.pi, scale_lo=0.9, scale_hi=1.1),
    WorldAug(flip_x_prob=0.3, flip_y_prob=0.5, rot_max=0.7, scale_lo=0.95, scale_hi=0.95),
]


def within_ulps(got, want64, n):
    return np.abs(got.astype(np.float64) - want64) <= n * np.spacing(np.abs(want64).astype(np.float32)).astype(np.float64)


@pytest.mark.parametrize("pol", WORLD_POLICIES, ids=["no_rotation", "rot_pi", "fixed_scale"])
def test_world_params_bit_exact(base, store, pol):
    eng = Real3DEngine("od", base.config, base.db, max_scans=32, max_points=len(base.pcl5))
    eng.set_world_aug(pol)
    idx = list(range(30)) + [5, 0]
    for seed, epoch in KEYS:
        eng.load_resident(store, idx, seed, epoch)
        eng.sync()
        w = eng.world_device().cpu().numpy()
        fx, fy, theta, k = od.draw_world(idx, seed, epoch, pol.flip_x_prob, pol.flip_y_prob, pol.rot_max,
                                         pol.scale_lo, pol.scale_hi)
        np.testing.assert_array_equal(w[:, 0], fx)
        np.testing.assert_array_equal(w[:, 1], fy)
        np.testing.assert_array_equal(w[:, 2], theta)
        np.testing.assert_array_equal(w[:, 5], k)
        t64 = theta.astype(np.float64)                 # cosf / sinf: within 2 ulp (CUDA C Programming Guide)
        assert within_ulps(w[:, 3], np.cos(t64), 2).all(), (w[:, 3], np.cos(t64))
        assert within_ulps(w[:, 4], np.sin(t64), 2).all(), (w[:, 4], np.sin(t64))
        assert (w[:, 6:] == 0).all()
    eng.close()


# ------------------------------------------------------------------ targets past 32 rows
TARGETS = ["Car", "Pedestrian"]                      # Cyclist, an insertion class, is not a target
NOBJ = 48


def crowded_case(seed, n_cars):
    """Scene lines renamed so that non-targets sit between targets: every 4th a Van, every 7th a DontCare."""
    case = case_from_spec(dict(task="od", seed=seed, counts=[NOBJ // 2, NOBJ // 2], n_cars=n_cars))
    lines = []
    for i, line in enumerate(case.box_lines):
        name = "Van" if i % 4 == 1 else "DontCare" if i % 7 == 3 else "Car"
        lines.append(name + line[len("Car"):])
    case.box_lines = lines
    return case


@pytest.fixture(scope="module")
def crowded():
    cases = [crowded_case(501, 60), crowded_case(502, 0), crowded_case(503, 1), crowded_case(504, 58)]
    store = ResidentDataset.from_scans("od", [scan_input_from_case(c) for c in cases])
    return cases, store


def set_targets_dropping_cyclist(eng):
    """set_target_classes refuses a list without every insertion class, so this calls the C entry point with class
    id 0 (dropped) for Cyclist."""
    dims = np.zeros((len(eng.obj_strings), 3), dtype=np.float32)
    for i, s in enumerate(eng.obj_strings):
        items = (s.item() if hasattr(s, "item") else str(s)).split(" ")
        dims[i] = (float(items[10]), float(items[9]), float(items[8]))
    ids = np.array([TARGETS.index(c) + 1 if c in TARGETS else 0 for c in eng.classes], dtype=np.int32)
    assert ids[eng.classes.index("Cyclist")] == 0
    _lib.check(eng.lib.r3d_engine_set_object_targets(eng.handle, dims.ctypes.data, ids.ctypes.data), "set_object_targets")
    eng.target_classes = TARGETS
    return ids


def run_targets(eng, store, idx, seed, epoch):
    import torch
    eng.load_resident(store, idx, seed, epoch)
    eng.run()
    m = store.max_kept_boxes(TARGETS) + eng.max_events - 1
    out = {"gt_boxes": torch.full((len(idx), m, 7), 7.0, device="cuda"),
           "gt_classes": torch.full((len(idx), m), 7, dtype=torch.int32, device="cuda"),
           "n_gt": torch.zeros(len(idx), dtype=torch.int32, device="cuda")}
    eng.targets_device(store, out)
    eng.sync()
    return out["gt_boxes"].cpu().numpy(), out["gt_classes"].cpu().numpy(), out["n_gt"].cpu().numpy()


def test_targets_past_32(crowded):
    cases, store = crowded
    idx = [0, 1, 2, 3, 1]
    cfg = copy.deepcopy(cases[0].config)
    cfg["insertion"]["number_of_object"] = NOBJ
    eng = Real3DEngine("od", cfg, cases[0].db, max_scans=len(idx), max_points=max(len(c.pcl5) for c in cases), max_boxes=128)
    assert eng.max_events == NOBJ + 1
    ids = set_targets_dropping_cyclist(eng)
    gb, gc, ng = run_targets(eng, store, idx, 77, 2**32 + 3)
    raw = eng.fetch_raw()
    kept_scene = [len(bx.targets_from_lines_od(cases[j].box_lines, TARGETS)[1]) for j in idx]
    assert max(kept_scene) > 32 and max(len(cases[j].box_lines) for j in idx) >= 40
    n_ins = raw["n_inserted"][:len(idx)]
    assert n_ins.max() > 32, n_ins                  # a scan inserted more objects than one ballot covers
    classes = raw["inserted"][:len(idx), :, 2]
    assert any((classes[s, :n_ins[s]] == eng.classes.index("Cyclist")).any() for s in range(len(idx)))
    for s, j in enumerate(idx):
        sb, sc = bx.targets_from_lines_od(cases[j].box_lines, TARGETS)
        k = len(sc)
        np.testing.assert_array_equal(gb[s, :k], sb)
        np.testing.assert_array_equal(gc[s, :k], sc)
        row = k
        for t in range(int(n_ins[s])):
            obj, _, ci, _ = (int(v) for v in raw["inserted"][s, t])
            if ids[ci] == 0:
                continue
            q = raw["inserted_box"][s, t]
            items = str(eng.obj_strings[obj]).split(" ")
            l, w, h = np.float32(items[10]), np.float32(items[9]), np.float32(items[8])
            np.testing.assert_array_equal(gb[s, row, :6], np.array([q[0], q[1], q[2] + np.float64(h) * 0.5, l, w, h],
                                                                   np.float64).astype(np.float32))
            head = np.float32(bx.wrap_pi(np.arctan2(q[4], q[3]) - np.pi / 2))
            assert abs(gb[s, row, 6] - head) <= np.spacing(np.abs(head)), (gb[s, row, 6], head)
            assert gc[s, row] == ids[ci]
            row += 1
        assert ng[s] == row
        assert not gb[s, row:].any() and not gc[s, row:].any()
    # world augmentation on: the same rows through the scan's transform
    eng.set_world_aug(WorldAug(flip_x_prob=0.5, flip_y_prob=0.5, rot_max=math.pi, scale_lo=0.9, scale_hi=1.1))
    wb, wc, wn = run_targets(eng, store, idx, 77, 2**32 + 3)
    w = eng.world_device().cpu().numpy()
    np.testing.assert_array_equal(wn, ng)
    np.testing.assert_array_equal(wc, gc)
    for s in range(len(idx)):
        want = od.world_boxes(w[s], gb[s, :ng[s]])
        np.testing.assert_array_equal(wb[s, :ng[s], :6], want[:, :6])
        assert (np.abs(bx.wrap_pi(wb[s, :ng[s], 6].astype(np.float64) - want[:, 6])) <= 2e-6).all()
        assert not wb[s, ng[s]:].any()
    eng.close()
