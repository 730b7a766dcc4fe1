"""CPU tier: host-side logic of the offline-tool drop-ins (SURVEY §8f rows 3-4) — label parsing, label -> map class
precedence, camera record, filter_objects bookkeeping — against the oracle restatement and the reference goldens.
No CUDA call is made here."""
import os
import pytest
import json

import numpy as np

from oracle import cut_objects_oracle as coo
from oracle import rich_map_oracle as rmo
from pcl_augmentation_b200 import cut_objects as co
from pcl_augmentation_b200.object_detection.cut_object import object_cut_out as oco
from pcl_augmentation_b200.semantic_segmentation.cut_object import cut_out, filter_objects
from pcl_augmentation_b200.semantic_segmentation.rich_map import drivable_area_map as srm
from tests.helpers import KITTI_CALIB_LINES, KITTI_IMAGE_SHAPE, cut_object_cases, load_golden
from tests.test_oracle_cut_objects import golden_samples


def test_od_label_boxes_match_the_oracle_parse():
    cases = cut_object_cases("od")
    n = 0
    for line in cases[0].box_lines:
        cls, occluded, base, expand, cx, cy = oco.label_boxes(line + "\n")
        w_cls, w_occ, w_base, w_expand, w_cx, w_cy = coo.od_boxes(line + "\n")
        assert (cls, occluded, cx, cy) == (w_cls, w_occ, w_cx, w_cy)
        for got, want in ((base, w_base), (expand, w_expand)):
            assert got["center"] == want["center"] and got["rotation"] == want["rotation"]
            assert (got["length"], got["width"], got["height"]) == (want["length"], want["width"], want["height"])
        n += 1
    assert n >= 10


def test_ss_line_box_matches_the_oracle_parse():
    case = cut_object_cases("ss")[0]
    for line in case.box_lines:
        box, x, y = cut_out.line_box(line + "\n")
        items = line.split(" ")
        assert (x, y) == (float(items[1]), float(items[2]))
        assert (box["length"], box["width"], box["height"]) == (float(items[6]), float(items[5]), float(items[4]))   # ss/co:124-139


def test_surface_table_precedence_matches_the_oracle():
    labels = {1: [40, 44, 60], 2: [48, 70, 44], 3: [44, 48, 72]}        # 44: class 1 wins; 48: class 3 wins over 2
    labs, cls = srm.surface_table(labels)
    assert dict(zip(labs.tolist(), cls.tolist())) == rmo.surface_classes(labels) == {40: 1, 44: 1, 60: 1, 48: 3, 70: 2, 72: 3}


def test_camera_record_holds_the_float32_products_of_the_reference(tmp_path):
    (tmp_path / "calib.txt").write_text("\n".join(KITTI_CALIB_LINES) + "\n")
    calib = co.read_kitti_calib(str(tmp_path / "calib.txt"))
    want = coo.read_calib(str(tmp_path / "calib.txt"))
    for k in ("P2", "R0", "Tr_velo2cam"):
        assert calib[k].dtype == np.float32
        np.testing.assert_array_equal(calib[k], want[k])
    rec = co.camera_record(calib, KITTI_IMAGE_SHAPE)
    m1 = np.dot(want["Tr_velo2cam"].T, want["R0"].T)                    # cutout.py:80, a float32 product
    assert m1.dtype == np.float32
    np.testing.assert_array_equal(rec[:12], m1.astype(np.float64).ravel())
    np.testing.assert_array_equal(rec[12:24], want["P2"].astype(np.float64).ravel())
    assert list(rec[24:]) == [375.0, 1242.0, 1.0]
    # the field-of-view flags the oracle derives from these matrices: points ahead are seen, points behind are not
    pts = np.array([[10.0, 0.0, -1.0], [-10.0, 0.0, -1.0], [10.0, 30.0, -1.0]])
    assert coo.fov_flag(pts, want, KITTI_IMAGE_SHAPE).tolist() == [True, False, False]


def test_filter_objects_bookkeeping_matches_reference_run():
    g = load_golden("cut_objects_ss")
    cfg = cut_object_cases("ss")[0].config
    removed = 0
    for cls in cfg["insertion"]["classes"]:
        folder = cfg["labels"][cls]
        samples = golden_samples(g, folder)
        kept = set(samples)
        for d in range(100):
            bucket = [(n, a, len(p)) for n, (a, p) in samples.items() if n.endswith(f"_{d:03d}_m")]
            if bucket:
                drop = filter_objects.to_delete(bucket)
                assert drop == coo.filter_objects(bucket)
                kept -= set(drop)
        assert sorted(kept) == json.loads(str(g[folder + "_kept"]))
        removed += len(samples) - len(kept)
    assert removed >= 10


def test_reference_arm_recipe_lists_existing_reference_files():
    """oracle/build_ref.py (the recipe behind `bench.py --impl reference`, kind "reference"): every file it names exists
    in the reference tree, and the copy under oracle/_ref is byte-identical (skipped where the original project's source
    tree, build_ref.SRC, is absent: the repository does not carry those source files)."""
    import filecmp
    from oracle import build_ref
    if not os.path.isdir(build_ref.SRC):
        pytest.skip("the original project's source tree (oracle/build_ref.py SRC) is not present")
    assert build_ref.build(verbose=False)
    for rel in build_ref.FILES:
        src = os.path.join(build_ref.SRC, rel)
        assert os.path.isfile(src), rel
        assert filecmp.cmp(src, os.path.join(build_ref.DST, rel), shallow=False), rel


def _label_lines(n, seed):
    from pcl_augmentation_b200 import synth
    rng = np.random.default_rng(seed)
    od, ss = [], []
    for i in range(n):
        yaw = rng.uniform(-np.pi, np.pi) if i % 7 else rng.choice([0.0, np.pi / 2, -np.pi / 2, np.pi, -np.pi, 1e-9])
        dims, c = rng.uniform(0.4, 8, 3), rng.uniform(-60, 60, 3)
        od.append(synth.od_label_line("Car", tuple(c), yaw, tuple(dims)) + "\n")
        ss.append(synth.ss_label_line(18, tuple(c), yaw, tuple(dims)) + "\n")
    return od, ss


def test_batched_box_records_equal_the_per_line_path():
    """read_label_line (od/fs:175-224, ss/fs:155-189) + the quaternion -> matrix step of cut_bounding_box (cb:28) for a
    whole batch in one scipy call: every one of the 16 doubles per box bit-identical to the per-line path."""
    from pcl_augmentation_b200 import boxes as bx
    od, ss = _label_lines(400, 11)
    for lines, is_ss, read in ((od, False, bx.read_label_line_od), (ss, True, bx.read_label_line_ss)):
        want = np.array([bx.box_record(read(line)) for line in lines])
        np.testing.assert_array_equal(bx.box_records_from_lines(lines, is_ss), want)
        np.testing.assert_array_equal(bx.box_records_from_lines(lines[:1], is_ss), want[:1])
    assert bx.box_records_from_lines([], False).shape == (0, 16)


def test_stage_packs_scene_boxes_of_line_and_dictionary_scans():
    """Real3DEngine.stage on the CPU (pageable buffers without a GPU): box offsets and records of a batch that mixes scans
    with annotation lines, with box dictionaries and without boxes; labels as one Road bit per point for object detection."""
    from types import SimpleNamespace
    from pcl_augmentation_b200 import boxes as bx
    from pcl_augmentation_b200.engine import Real3DEngine, ScanInput
    od, _ = _label_lines(9, 12)
    rng = np.random.default_rng(3)

    def scan(n_pts, lines=None, dicts=None):
        maps = {k: {"map": np.ones((4, 5), np.uint8), "min_x": np.array(-2), "min_y": np.array(-3)} for k in ("Road", "Sidewalk")}
        return ScanInput(xyzi=rng.normal(size=(n_pts, 4)).astype(np.float32), labels=rng.choice([40, 1, 48], n_pts).astype(np.uint32),
                         box_lines=lines or [], box_dicts=dicts, counts=np.array([1, 0]), perms=np.zeros((2, 2, 100), np.int32), maps=maps)
    scans = [scan(50, od[:4]), scan(30), scan(20, dicts=[bx.read_label_line_od(l) for l in od[4:6]]), scan(10, od[6:])]
    eng = SimpleNamespace(max_scans=8, task="od", classes=["Pedestrian", "Cyclist"], max_events=3, max_tries=100, road_label=40)
    st = Real3DEngine.stage(eng, scans)
    assert list(st["box_off"]) == [0, 4, 4, 6, 9] and list(st["pt_off"]) == [0, 50, 80, 100, 110]
    np.testing.assert_array_equal(st["boxes"], np.array([bx.box_record(bx.read_label_line_od(l)) for l in od]))
    road = np.concatenate([s.labels == 40 for s in scans])
    np.testing.assert_array_equal(np.unpackbits(st["labels"], bitorder="little")[:110].astype(bool), road)
    np.testing.assert_array_equal(st["xyzi"][50:80], scans[1].xyzi)


def test_batched_placed_box_dictionaries_equal_the_per_box_path():
    from pcl_augmentation_b200 import boxes as bx
    rng = np.random.default_rng(2)
    recs = []
    for _ in range(200):
        a = rng.uniform(-np.pi, np.pi)
        recs.append([*rng.uniform(-50, 50, 3), np.cos(a), np.sin(a), *rng.uniform(0.5, 8, 3)])
    for cls, ss in (("Cyclist", False), ("18", True)):
        one = [bx.placed_box_dictionary(r, cls, ss) for r in recs]
        many = bx.placed_box_dictionaries(recs, [cls] * len(recs), ss)
        for a, b in zip(one, many):
            assert a["rotation"] == b["rotation"] and a["center"] == b["center"] and a["class"] == b["class"]
            assert (a["length"], a["width"], a["height"]) == (b["length"], b["width"], b["height"])
            np.testing.assert_array_equal(a["_matrix"], b["_matrix"])
    assert bx.placed_box_dictionaries([], [], False) == []
