"""CPU tier: detection targets from KITTI lines, the world transform restated in numpy, and the validation of the
world-augmentation and target-class settings."""
import math

import numpy as np
import pytest

from pcl_augmentation_b200 import boxes as bx
from pcl_augmentation_b200 import _lib
from pcl_augmentation_b200.online import WorldAug


def kitti(name, h, w, l, x, y, z, ry):
    return f"{name} 0.00 0 0.00 100.00 120.00 150.00 220.00 {h:.2f} {w:.2f} {l:.2f} {x:.2f} {y:.2f} {z:.2f} {ry:.2f}"


def world_points(w, xyz):
    """The point transform of r3d_world_aug in float32: flip, rotate, scale (no contraction)."""
    fx, fy, _, c, s, k = (np.float32(v) for v in w[:6])
    x, y, z = (xyz[:, i].astype(np.float32) for i in range(3))
    x1 = -x if fy else x
    y1 = -y if fx else y
    return np.stack([(c * x1 - s * y1) * k, (s * x1 + c * y1) * k, z * k], axis=1)


def world_boxes(w, b7):
    """The box transform: centre as the points, dimensions * k, heading flipped / rotated and wrapped."""
    out = np.array(b7, dtype=np.float32, copy=True)
    out[:, :3] = world_points(w, out[:, :3])
    out[:, 3:6] *= np.float32(w[5])
    h = out[:, 6].astype(np.float64)
    if w[0]:
        h = -h
    if w[1]:
        h = -(h + np.pi)
    out[:, 6] = bx.wrap_pi(h + np.float64(np.float32(w[2]))).astype(np.float32)
    return out


def params(fx, fy, theta, k):
    theta = np.float32(theta)
    return np.array([fx, fy, theta, np.cos(theta), np.sin(theta), k, 0, 0], dtype=np.float32)


def test_targets_from_lines_formula_and_filtering():
    lines = [kitti("Car", 1.5, 1.6, 3.9, 2.43, 1.65, 41.57, 1.52),
             kitti("DontCare", 1.0, 1.0, 1.0, 0.0, 1.0, 5.0, 0.0),
             kitti("Pedestrian", 1.8, 0.6, 0.8, -3.0, 1.7, 12.0, -0.5),
             kitti("Tram", 3.0, 2.5, 12.0, 1.0, 1.0, 30.0, 0.0),
             kitti("Car", 1.4, 1.7, 4.2, 5.0, 1.6, 20.0, 1.5707963267948966 + 0.1) + "\n"]
    b7, cls = bx.targets_from_lines_od(lines, ["Car", "Pedestrian", "Cyclist"])
    assert b7.dtype == np.float32 and cls.dtype == np.int32
    np.testing.assert_array_equal(cls, [1, 2, 1])
    want = np.array([41.57 + 0.27, -2.43, (-1.65 - 0.08) + 1.5 / 2, 3.9, 1.6, 1.5, -1.52 - np.pi / 2], dtype=np.float64)
    np.testing.assert_array_equal(b7[0], want.astype(np.float32))
    assert b7[1, 3] == np.float32(0.8) and b7[1, 4] == np.float32(0.6) and b7[1, 5] == np.float32(1.8)
    # -ry - pi/2 = -1.67 - pi/2 wraps to pi - (1.67 + pi/2 - pi) ... i.e. into [-pi, pi)
    h = -1.67 - np.pi / 2
    assert h < -np.pi and b7[2, 6] == np.float32(h + 2 * np.pi)
    assert (b7[:, 6] >= -np.float32(np.pi)).all() and (b7[:, 6] < np.float32(np.pi)).all()


def test_wrap_pi_edges():
    np.testing.assert_array_equal(bx.wrap_pi([-np.pi, np.pi, 0.0, 3 * np.pi]), [-np.pi, -np.pi, 0.0, -np.pi])
    assert bx.wrap_pi(np.pi - 1e-9) < np.pi


def test_empty_and_unknown_only():
    b7, cls = bx.targets_from_lines_od([kitti("DontCare", 1, 1, 1, 0, 0, 5, 0)], ["Car"])
    assert b7.shape == (0, 7) and cls.shape == (0,)
    b7, cls = bx.targets_from_lines_od([], ["Car"])
    assert b7.shape == (0, 7)


def test_world_transform_order_and_flips():
    rng = np.random.default_rng(0)
    xyz = rng.uniform(-40, 40, (64, 3)).astype(np.float32)
    x, y, z = (xyz[:, i].astype(np.float64) for i in range(3))
    # OpenPCDet's random_flip_along_x: y = -y, heading = -heading; random_flip_along_y: x = -x, heading = -(heading + pi)
    np.testing.assert_array_equal(world_points(params(1, 0, 0.0, 1.0), xyz), np.stack([x, -y, z], 1).astype(np.float32))
    np.testing.assert_array_equal(world_points(params(0, 1, 0.0, 1.0), xyz), np.stack([-x, y, z], 1).astype(np.float32))
    # flip, then rotate (global_rotation about z), then scale (global_scaling)
    theta, k = 0.3, 1.04
    got = world_points(params(1, 0, theta, k), xyz).astype(np.float64)
    c, s = math.cos(theta), math.sin(theta)
    want = np.stack([(c * x - s * -y) * k, (s * x + c * -y) * k, z * k], 1)
    np.testing.assert_allclose(got, want, rtol=0, atol=1e-4)
    rotate_first = np.stack([(c * x - s * y) * k, -(s * x + c * y) * k, z * k], 1)
    assert np.abs(got - rotate_first).max() > 1e-2          # flips do not commute with a rotation


@pytest.mark.parametrize("fx,fy", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_box_and_interior_points_stay_consistent(fx, fy):
    box = np.array([[12.0, -3.0, -0.9, 4.2, 1.7, 1.5, 0.7]], dtype=np.float32)
    rng = np.random.default_rng(1)
    local = rng.uniform(-0.45, 0.45, (200, 3)) * box[0, 3:6]
    ch, sh = math.cos(box[0, 6]), math.sin(box[0, 6])
    pts = np.stack([box[0, 0] + ch * local[:, 0] - sh * local[:, 1], box[0, 1] + sh * local[:, 0] + ch * local[:, 1],
                    box[0, 2] + local[:, 2]], 1).astype(np.float32)
    w = params(fx, fy, -0.6, 0.97)
    nb = world_boxes(w, box)[0].astype(np.float64)
    npt = world_points(w, pts).astype(np.float64)
    d = npt - nb[:3]
    ch, sh = math.cos(nb[6]), math.sin(nb[6])
    u, v = ch * d[:, 0] + sh * d[:, 1], -sh * d[:, 0] + ch * d[:, 1]
    want = local * np.float32(0.97)
    if fx != fy:                                              # a mirror image: the box's own y axis turns around
        want[:, 1] *= -1
    np.testing.assert_allclose(np.stack([u, v, d[:, 2]], 1), want, rtol=0, atol=1e-4)


def test_world_aug_validation():
    WorldAug()
    WorldAug(flip_x_prob=0.0, flip_y_prob=1.0, rot_max=math.pi, scale_lo=1.0, scale_hi=1.0)
    for bad in (dict(flip_x_prob=-0.1), dict(flip_y_prob=1.5), dict(rot_max=-0.1), dict(rot_max=3.2),
                dict(scale_lo=0.0), dict(scale_lo=1.1, scale_hi=1.0), dict(scale_hi=float("inf")),
                dict(flip_x_prob=float("nan"))):
        with pytest.raises(ValueError):
            WorldAug(**bad)


def test_set_target_classes_validation():
    from pcl_augmentation_b200.engine import Real3DEngine

    class Stub:
        task, classes, obj_strings = "od", ["Cyclist", "Pedestrian"], []
    with pytest.raises(_lib.Real3DError):
        Real3DEngine.set_target_classes(Stub(), ["Car", "Pedestrian"])          # Cyclist is inserted but not a target
    Stub.task = "ss"
    with pytest.raises(_lib.Real3DError):
        Real3DEngine.set_target_classes(Stub(), ["Car", "Pedestrian", "Cyclist"])
