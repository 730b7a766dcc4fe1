"""GPU tier, SURVEY §8f row 4: cut-object database building against the files the unmodified reference scripts wrote
(golden) and against the oracle on full-size frames; names, annotation strings and point rows bit-exact."""
import json
import os

import numpy as np
import pytest
import yaml

from oracle import cut_objects_oracle as coo
from oracle import real3d_oracle as orc
from pcl_augmentation_b200 import cut_objects as co
from pcl_augmentation_b200 import synth, synth_io
from tests.helpers import (KITTI_CALIB_LINES, KITTI_IMAGE_SHAPE, cut_object_cases, load_golden, read_sample_dir,
                           write_kitti_camera_files)
from tests.test_oracle_cut_objects import frame_points, golden_samples

pytestmark = pytest.mark.gpu


def assert_same_samples(got, want):
    assert sorted(got) == sorted(want)
    for name, (anno, pcl) in want.items():
        assert got[name][0] == anno
        assert got[name][1].dtype == np.float64 and got[name][1].shape == pcl.shape
        np.testing.assert_array_equal(got[name][1], pcl)


def test_od_script_writes_the_reference_files(tmp_path):
    from pcl_augmentation_b200.object_detection.cut_object import object_cut_out as oco
    g = load_golden("cut_objects_od")
    cases = cut_object_cases("od")
    _, _, cfg = synth_io.write_od_dataset(cases, str(tmp_path))
    write_kitti_camera_files(str(tmp_path), len(cases))
    cfg["path"]["sample_path"] = str(tmp_path / "cut")
    os.makedirs(cfg["path"]["sample_path"])
    n = oco.generate_samples(cfg, batch_size=2, log=lambda *a: None)
    total = 0
    for cls in cfg["insertion"]["classes"]:
        want = golden_samples(g, cls)
        assert_same_samples(read_sample_dir(tmp_path / "cut" / cls), want)
        total += len(want)
    assert n == total >= 10


def test_ss_scripts_write_the_reference_files(tmp_path):
    from pcl_augmentation_b200.semantic_segmentation.cut_object import cut_out, filter_objects
    g = load_golden("cut_objects_ss")
    cases = cut_object_cases("ss")
    _, _, cfg = synth_io.write_ss_dataset(cases, str(tmp_path))
    cfg["path"]["bbox_path"] = str(tmp_path / "cut")
    cut_out.generate_samples(cfg, "00", batch_size=2, log=lambda *a: None)
    folders = [cfg["labels"][c] for c in cfg["insertion"]["classes"]]
    for folder in folders:
        assert_same_samples(read_sample_dir(tmp_path / "cut" / folder), golden_samples(g, folder))
    removed = filter_objects.filter_samples(cfg, log=lambda *a: None)
    assert removed >= 10
    for folder in folders:
        assert sorted(read_sample_dir(tmp_path / "cut" / folder)) == json.loads(str(g[folder + "_kept"]))


def test_full_size_frames_vs_oracle(tmp_path):
    from pcl_augmentation_b200.object_detection.cut_object import object_cut_out as oco
    from pcl_augmentation_b200.semantic_segmentation.cut_object import cut_out
    (tmp_path / "calib.txt").write_text("\n".join(KITTI_CALIB_LINES) + "\n")
    calib = coo.read_calib(str(tmp_path / "calib.txt"))
    for task in ("od", "ss"):
        cases = cut_object_cases(task, shape=synth.KITTI_SHAPE)
        cfg = cases[0].config
        # frame 1 gets > 64 boxes (every line three times), frame 2 is cut short (ragged), a last frame has no box
        cases[1].box_lines = list(cases[1].box_lines) * 3
        cases[2].pcl5 = cases[2].pcl5[7:]
        frames, want = [], []
        for i, case in enumerate(cases):
            pts = frame_points(case)
            lines = [l + "\n" for l in case.box_lines]
            xyzi, labels = pts[:, :4].astype(np.float32), pts[:, 4].astype(np.uint32)
            if task == "od":
                frames.append((xyzi, labels, lines, calib, KITTI_IMAGE_SHAPE, f"{i:06d}"))
                want.append(coo.cut_objects_od(pts, lines, calib, KITTI_IMAGE_SHAPE, cfg, f"{i:06d}"))
            else:
                frames.append((xyzi, labels, lines, "00", f"{i:06d}"))
                want.append(coo.cut_objects_ss(pts, lines, cfg, "00", f"{i:06d}"))
        empty = (frames[0][0][:100], frames[0][1][:100], []) + frames[0][3:]
        frames.append(empty)
        want.append([])
        got = (oco if task == "od" else cut_out).cut_frames(frames, cfg)
        assert len(got) == len(want)
        n = 0
        for g_frame, w_frame in zip(got, want):
            assert [(a, b, c) for a, b, c, _ in g_frame] == [(a, b, c) for a, b, c, _ in w_frame]
            for (_, _, _, gp), (_, _, _, wp) in zip(g_frame, w_frame):
                assert gp.dtype == np.float64
                np.testing.assert_array_equal(gp, wp)
                n += 1
        assert n >= 20, (task, n)


def test_tilted_boxes_counts_and_indices_vs_cut_bounding_box(tmp_path):
    """General (non yaw-only) quaternions, overlapping boxes, emitted indices and the field-of-view count."""
    from scipy.spatial.transform import Rotation as R
    pcl, labels = synth.make_scan(95, synth.KITTI_SHAPE, synth.make_scene_cars(95, 5))
    labels = labels & 0xFFFF
    pts5 = np.hstack((pcl.astype(np.float64), labels.reshape(-1, 1).astype(np.float64)))
    rng = np.random.default_rng(95)
    boxes = []
    for _ in range(70):
        q = R.from_euler("zyx", [rng.uniform(-3, 3), rng.uniform(-0.3, 0.3), rng.uniform(-0.3, 0.3)]).as_quat()
        c = rng.uniform(-25, 25, 2)
        boxes.append({'center': {'x': c[0], 'y': c[1], 'z': rng.uniform(-2.2, -1.2)},
                      'rotation': {'x': q[0], 'y': q[1], 'z': q[2], 'w': q[3]},
                      'length': rng.uniform(1, 6), 'width': rng.uniform(1, 6), 'height': rng.uniform(0.5, 3), 'class': 0})
    boxes.append(dict(boxes[0]))                                   # a duplicate: a point may belong to several boxes
    # beyond the kernel's pruning grid (+-81.92 m): clusters at 100 - 140 m with their boxes, and a box far from everything
    far = []
    for cx, cy in ((101.0, -93.0), (-120.0, 5.0), (3.0, 139.0)):
        far.append(np.c_[rng.uniform(-1.5, 1.5, (300, 2)) + [cx, cy], rng.uniform(-1.5, 0.5, 300), rng.uniform(0, 1, 300)])
        boxes.append({'center': {'x': cx, 'y': cy, 'z': -1.0}, 'rotation': {'x': 0.0, 'y': 0.0, 'z': 0.38268343, 'w': 0.92387953},
                      'length': 2.0, 'width': 2.2, 'height': 1.2, 'class': 0})
    boxes.append({'center': {'x': 500.0, 'y': 500.0, 'z': 0.0}, 'rotation': {'x': 0.0, 'y': 0.0, 'z': 0.0, 'w': 1.0},
                  'length': 2.0, 'width': 2.0, 'height': 2.0, 'class': 0})
    far = np.vstack(far).astype(np.float32)
    pcl = np.vstack((pcl, far))
    labels = np.concatenate((labels, np.full(len(far), 7, dtype=labels.dtype)))
    pts5 = np.hstack((pcl.astype(np.float64), labels.reshape(-1, 1).astype(np.float64)))
    (tmp_path / "calib.txt").write_text("\n".join(KITTI_CALIB_LINES) + "\n")
    calib = coo.read_calib(str(tmp_path / "calib.txt"))
    cam = co.camera_record(calib, KITTI_IMAGE_SHAPE)
    cuts = co.cut_boxes_batch([(pcl, labels)], [boxes], [[co.EMIT_ANY] * len(boxes)], cameras=[cam], want_index=True)[0]
    hits = 0
    for b, cut in zip(boxes, cuts):
        mask = orc.cut_bounding_box_mask(pts5, b)
        idx = np.nonzero(mask)[0]
        assert cut.count_inside == len(idx)
        np.testing.assert_array_equal(cut.index, idx)
        np.testing.assert_array_equal(cut.xyzi, pcl[idx])
        np.testing.assert_array_equal(cut.labels, labels[idx])
        assert cut.count_fov == int(coo.fov_flag(pts5[idx, :3], calib, KITTI_IMAGE_SHAPE).sum())
        hits += len(idx)
    assert hits > 2000
    assert all(c.count_inside > 20 for c in cuts[-4:-1]) and cuts[-1].count_inside == 0
