"""CPU tier: the host reference of the points-in-targets test (oracle/target_points.py) against an independent
point-in-polygon formulation, the min-points filter restated, and the validation of OnlineAugmenter(target_points=)."""
import math

import numpy as np
import pytest

from oracle.target_points import filter_min_points, near_faces, points_in_boxes, target_points
from pcl_augmentation_b200.online import OnlineAugmenter


def polygon_inside(points, box):
    """Inside the box's four xy corners (strictly, by the signs of the edge cross products) and its closed z slab."""
    p = np.asarray(points, dtype=np.float32).astype(np.float64)
    cx, cy, cz, dx, dy, dz, h = (float(v) for v in np.asarray(box, dtype=np.float32))
    c, s = math.cos(h), math.sin(h)
    local = [(dx / 2, dy / 2), (-dx / 2, dy / 2), (-dx / 2, -dy / 2), (dx / 2, -dy / 2)]     # counter-clockwise
    corners = [(cx + c * a - s * b, cy + s * a + c * b) for a, b in local]
    inside = np.abs(p[:, 2] - cz) <= dz / 2
    for k in range(4):
        (x0, y0), (x1, y1) = corners[k], corners[(k + 1) % 4]
        inside &= (x1 - x0) * (p[:, 1] - y0) - (y1 - y0) * (p[:, 0] - x0) > 0
    return inside


def random_boxes(rng, m):
    b = np.zeros((m, 7), dtype=np.float32)
    b[:, 0:2] = rng.uniform(-30, 30, (m, 2))
    b[:, 2] = rng.uniform(-2, 1, m)
    b[:, 3] = rng.uniform(0.5, 6, m)
    b[:, 4] = rng.uniform(0.5, 3, m)
    b[:, 5] = rng.uniform(1, 3, m)
    b[:, 6] = rng.uniform(-math.pi, math.pi, m)
    return b


def points_around(rng, boxes, per_box):
    out = []
    for b in boxes:
        local = rng.uniform(-0.7, 0.7, (per_box, 3)) * b[3:6]
        c, s = math.cos(b[6]), math.sin(b[6])
        out.append(np.stack([b[0] + c * local[:, 0] - s * local[:, 1], b[1] + s * local[:, 0] + c * local[:, 1],
                             b[2] + local[:, 2]], axis=1))
    return np.concatenate(out).astype(np.float32)


@pytest.mark.parametrize("turn", [0.0, 2 * math.pi, -2 * math.pi])
def test_reference_matches_polygon_test(turn):
    rng = np.random.default_rng(7)
    boxes = random_boxes(rng, 40)
    pts = points_around(rng, boxes, 500)
    boxes[:, 6] = (boxes[:, 6].astype(np.float64) + turn).astype(np.float32)
    ref = points_in_boxes(pts, boxes)
    near = near_faces(pts, boxes)
    assert near.sum() == 0
    for j in range(len(boxes)):
        np.testing.assert_array_equal(ref[:, j], polygon_inside(pts, boxes[j]))
    assert 0.2 < ref.any(axis=1).mean() < 0.9            # both sides of the faces are exercised


def test_points_on_faces():
    box = np.array([[1.0, 2.0, -1.0, 4.0, 2.0, 1.5, 0.0]], dtype=np.float32)      # heading 0: the faces are exact
    on_z = [[1.0, 2.0, -1.75], [1.0, 2.0, -0.25], [2.5, 2.5, -0.25]]              # closed z bound: inside
    on_x = [[3.0, 2.0, -1.0], [-1.0, 2.0, -1.0], [3.0, 2.5, -0.25]]              # open x bound: outside
    on_y = [[1.0, 3.0, -1.0], [1.0, 1.0, -1.0]]                                   # open y bound: outside
    just_in = [[np.nextafter(np.float32(3.0), np.float32(0)), 2.0, -1.0], [1.0, np.nextafter(np.float32(1.0), np.float32(2)), -1.0]]
    beyond_z = [[1.0, 2.0, np.nextafter(np.float32(-0.25), np.float32(1))]]
    pts = np.array(on_z + on_x + on_y + just_in + beyond_z, dtype=np.float32)
    got = points_in_boxes(pts, box)[:, 0]
    np.testing.assert_array_equal(got, [True] * 3 + [False] * 5 + [True] * 2 + [False])
    np.testing.assert_array_equal(got, polygon_inside(pts, box[0]))
    assert near_faces(pts, box)[:8].all()                # on a face: left out of the device comparisons


def test_counts_and_first_hit_with_overlaps():
    boxes = np.array([[0, 0, 0, 4, 4, 2, 0], [1, 0, 0, 4, 4, 2, 0], [10, 0, 0, 2, 2, 2, 0]], dtype=np.float32)
    pts = np.array([[0.5, 0, 0], [-1.5, 0, 0], [2.5, 0, 0], [10, 0, 0], [20, 0, 0]], dtype=np.float32)
    counts, first = target_points(pts, boxes)
    np.testing.assert_array_equal(counts, [2, 2, 1])        # the point in both overlapping boxes counts in both
    np.testing.assert_array_equal(first, [0, 0, 1, 2, -1])


def filter_loop(points, boxes, k):
    """The filter as a trainer would write it, box by box and point by point."""
    inside = points_in_boxes(points, boxes)
    kept = [j for j in range(len(boxes)) if inside[:, j].sum() >= k]
    gt = [next((n for n, j in enumerate(kept) if inside[i, j]), -1) for i in range(len(points))]
    return np.array(kept, dtype=np.int64), inside[:, kept].sum(axis=0).astype(np.int32), np.array(gt, dtype=np.int32)


def test_filter_keeps_order_and_reassigns_dropped_points():
    boxes = np.array([[0, 0, 0, 2, 2, 2, 0],      # 1 point, which is also in box 2: dropped with K = 2
                      [5, 0, 0, 2, 2, 2, 0],      # 3 points
                      [0.5, 0, 0, 4, 2, 2, 0],    # 3 points (one shared with box 0)
                      [9, 9, 0, 1, 1, 1, 0]],     # empty
                     dtype=np.float32)
    pts = np.array([[0, 0, 0], [1.5, 0, 0], [2, 0, 0], [5, 0, 0], [5.5, 0, 0], [4.5, 0, 0], [30, 0, 0]], dtype=np.float32)
    kept, counts, gt = filter_min_points(pts, boxes, 2)
    np.testing.assert_array_equal(kept, [1, 2])
    np.testing.assert_array_equal(counts, [3, 3])
    np.testing.assert_array_equal(gt, [1, 1, 1, 0, 0, 0, -1])   # point 0 was box 0's: now the kept box 2 (index 1)
    kept0, counts0, gt0 = filter_min_points(pts, boxes, 0)
    np.testing.assert_array_equal(kept0, [0, 1, 2, 3])
    np.testing.assert_array_equal(gt0, target_points(pts, boxes)[1])


@pytest.mark.parametrize("k", [0, 1, 5, 40, 10_000])
def test_filter_against_loop(k):
    rng = np.random.default_rng(11 + k)
    boxes = random_boxes(rng, 70)
    boxes[35:, :3] = boxes[:35, :3] + rng.uniform(-1, 1, (35, 3)).astype(np.float32)     # overlapping pairs
    pts = np.concatenate([points_around(rng, boxes[:20], 60), points_around(rng, boxes[20:], 3)])
    for got, want in zip(filter_min_points(pts, boxes, k), filter_loop(pts, boxes, k)):
        np.testing.assert_array_equal(got, want)


@pytest.mark.parametrize("kw", [dict(target_points=-1, target_classes=["Car"]), dict(target_points=1),
                                dict(target_points=1.5, target_classes=["Car"]), dict(target_points=True, target_classes=["Car"])])
def test_augmenter_refuses_bad_target_points(kw):
    with pytest.raises(ValueError):
        OnlineAugmenter("od", None, None, None, batch_size=1, seed=0, **kw)
