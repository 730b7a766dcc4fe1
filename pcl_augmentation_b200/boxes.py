"""Host-side annotation handling: the reference's box dictionaries, label-line parsing and KITTI line writing.

These are the small pure-Python pieces of the operator interface (a handful of scalars per box); everything that
touches points runs in CUDA.  Function names / argument meaning follow the reference:
``make_dictionary`` / ``dictionary2array`` (od/fs:44-68, ss/fs:15-39), ``read_label_line`` (od/fs:175-224,
ss/fs:155-189), ``create_annotation_line`` (od/ins:227-265).
"""
from __future__ import annotations

import math

import numpy as np
from scipy.spatial.transform import Rotation as R


def make_dictionary(annotation_array, ss=False):
    center = {'x': annotation_array[0][0], 'y': annotation_array[0][1], 'z': annotation_array[0][2]}
    rotation = {'x': annotation_array[1][0], 'y': annotation_array[1][1], 'z': annotation_array[1][2],
                'w': annotation_array[1][3]}
    return {'center': center, 'rotation': rotation, 'length': annotation_array[2][0], 'width': annotation_array[2][1],
            'height': annotation_array[2][2], 'class': annotation_array[3] if ss else annotation_array[3][0]}


def dictionary2array(d, ss=False):
    return [[d['center']['x'], d['center']['y'], d['center']['z']],
            [d['rotation']['x'], d['rotation']['y'], d['rotation']['z'], d['rotation']['w']],
            [d['length'], d['width'], d['height']], d['class'] if ss else [d['class']]]


def _yaw_quaternion(z_rot):
    rot_matrix = [[math.cos(z_rot), -1 * math.sin(z_rot), 0], [math.sin(z_rot), math.cos(z_rot), 0], [0, 0, 1]]
    return R.from_matrix(rot_matrix).as_quat()


def read_label_line_od(line):
    """KITTI ``label_2`` line -> lidar-frame box dictionary; ``center.z`` is the box bottom (od/fs:175-224)."""
    items = line.split(' ')
    height, width, length = float(items[8]), float(items[9]), float(items[10])
    x, y, z = float(items[11]), float(items[12]), float(items[13])
    q = _yaw_quaternion(float(items[14]) * -1)
    return make_dictionary([[float(z) + 0.27, float(x) * -1, float(y) * -1 - 0.08], [q[0], q[1], q[2], q[3]],
                            [width + 0.1, length + 0.1, height + 0.1], [items[0]]])


def wrap_pi(h):
    """Angle(s) wrapped to [-pi, pi), in float64 (the arithmetic of the device's ``wrap_pi``)."""
    h = np.asarray(h, dtype=np.float64)
    return h - 2.0 * np.pi * np.floor((h + np.pi) * (1.0 / (2.0 * np.pi)))


def scene_targets_od(lines):
    """Every KITTI ``label_2`` line as a detection target box in the engine's lidar frame (the fixed-offset frame of
    ``read_label_line_od``), computed in float64: (float64 [n, 7] x, y, z_center, dx, dy, dz, heading; names [n]).
    ``dx, dy, dz`` are the unpadded KITTI ``l, w, h`` and ``heading = -rotation_y - pi/2``, measured from +x toward +y."""
    out = np.zeros((len(lines), 7), dtype=np.float64)
    names = []
    for i, line in enumerate(lines):
        items = line.split(' ')
        height, width, length = float(items[8]), float(items[9]), float(items[10])
        x, y, z = float(items[11]), float(items[12]), float(items[13])
        out[i] = (z + 0.27, x * -1, (y * -1 - 0.08) + height / 2, length, width, height, -float(items[14]) - np.pi / 2)
        names.append(items[0])
    out[:, 6] = wrap_pi(out[:, 6])
    return out, names


def targets_from_lines_od(lines, target_classes):
    """KITTI lines -> OpenPCDet-style ``gt_boxes`` (float32 [n, 7]: x, y, z_center, dx, dy, dz, heading) and 1-based
    class ids into ``target_classes`` (int32 [n]); lines whose name is not in ``target_classes`` (``DontCare``
    included) are dropped, as OpenPCDet drops them."""
    boxes, names = scene_targets_od(lines)
    ids = np.array([list(target_classes).index(n) + 1 if n in target_classes else 0 for n in names], dtype=np.int32)
    keep = ids > 0
    return boxes[keep].astype(np.float32), ids[keep]


def read_label_line_ss(line):
    """Semseg bbox line ``cls x y z h w l yaw`` -> box dictionary (ss/fs:155-189)."""
    items = line.split(' ')
    q = _yaw_quaternion(float(items[7]))
    return make_dictionary([[float(items[1]), float(items[2]), float(items[3])], [q[0], q[1], q[2], q[3]],
                            [float(items[6]), float(items[5]), float(items[4])], [items[0]]], ss=True)


def rotation_matrix(annotation):
    if '_matrix' in annotation:
        return np.asarray(annotation['_matrix'], dtype=np.float64)
    r = annotation['rotation']
    return R.from_quat([r['x'], r['y'], r['z'], r['w']]).as_matrix()


def box_record(annotation, annotation_move=(0, 0, 0)):
    """Box dictionary -> the 16-double record of the C ABI: centre (z = bottom), 3x3 matrix, L, W, H, reach."""
    m = rotation_matrix(annotation)
    out = np.zeros(16, dtype=np.float64)
    out[0] = annotation['center']['x'] - annotation_move[0]
    out[1] = annotation['center']['y'] - annotation_move[1]
    out[2] = annotation['center']['z'] - annotation_move[2]
    out[3:12] = m.reshape(-1)
    out[12], out[13], out[14] = annotation['length'], annotation['width'], annotation['height']
    yaw_only = abs(m[2][2]) > 0.999999
    out[15] = 0.5 * math.hypot(out[12], out[13]) + 0.05 if yaw_only else 0.5 * math.hypot(out[12], out[13]) + out[14] + 0.05
    return out


def box_records_from_lines(lines, ss=False):
    """``box_record(read_label_line_*(line))`` for many annotation lines at once -> float64 [n, 16].

    The two scipy conversions per box (yaw matrix -> quaternion in ``read_label_line``, quaternion -> matrix in
    ``cut_bounding_box``, od/fs:213, cb:28) dominate the per-line path (~0.2 ms per box); scipy runs the same per-rotation
    arithmetic over a stack of rotations, so one call for the whole batch gives bit-identical records
    (``tests/test_host_tools.py::test_batched_box_records_equal_the_per_line_path``)."""
    n = len(lines)
    out = np.zeros((n, 16), dtype=np.float64)
    if n == 0:
        return out
    z_rot = np.empty(n, dtype=np.float64)
    for i, line in enumerate(lines):
        items = line.split(' ')
        if ss:                                                           # ss/fs:161-173
            out[i, 0], out[i, 1], out[i, 2] = float(items[1]), float(items[2]), float(items[3])
            out[i, 12], out[i, 13], out[i, 14] = float(items[6]), float(items[5]), float(items[4])
            z_rot[i] = float(items[7])
        else:                                                            # od/fs:181-211
            height, width, length = float(items[8]), float(items[9]), float(items[10])
            x, y, z = float(items[11]), float(items[12]), float(items[13])
            out[i, 0], out[i, 1], out[i, 2] = float(z) + 0.27, float(x) * -1, float(y) * -1 - 0.08
            out[i, 12], out[i, 13], out[i, 14] = width + 0.1, length + 0.1, height + 0.1
            z_rot[i] = float(items[14]) * -1
    mats = np.zeros((n, 3, 3), dtype=np.float64)
    for i in range(n):                                                   # math.cos / math.sin as in _yaw_quaternion
        c, sn = math.cos(z_rot[i]), math.sin(z_rot[i])
        mats[i] = [[c, -1 * sn, 0], [sn, c, 0], [0, 0, 1]]
    m = R.from_quat(R.from_matrix(mats).as_quat()).as_matrix()
    out[:, 3:12] = m.reshape(n, 9)
    half_diag = np.array([0.5 * math.hypot(out[i, 12], out[i, 13]) for i in range(n)])
    yaw_only = np.abs(m[:, 2, 2]) > 0.999999
    out[:, 15] = np.where(yaw_only, half_diag + 0.05, half_diag + out[:, 14] + 0.05)
    return out


def object_box_record(annotation):
    """Cut-object box -> (cx, cy, cz, R0[0][0], R0[1][0], L, W, H) for ``r3d_object_db.boxes``."""
    m = rotation_matrix(annotation)
    return np.array([annotation['center']['x'], annotation['center']['y'], annotation['center']['z'], m[0][0], m[1][0],
                     annotation['length'], annotation['width'], annotation['height']], dtype=np.float64)


def placed_box_dictionary(rec, cls, ss=False):
    """(cx, cy, cz, m00, m10, L, W, H) of an inserted object -> box dictionary (with its matrix attached)."""
    cx, cy, cz, m00, m10, length, width, height = (float(v) for v in rec)
    m = np.array([[m00, -m10, 0.0], [m10, m00, 0.0], [0.0, 0.0, 1.0]])
    q = R.from_matrix(m).as_quat()
    d = make_dictionary([[cx, cy, cz], [q[0], q[1], q[2], q[3]], [length, width, height], [cls]], ss=ss)
    d['_matrix'] = m
    return d


def placed_box_dictionaries(recs, classes, ss=False):
    """``placed_box_dictionary`` for many inserted objects with one scipy call (same per-rotation arithmetic)."""
    recs = np.asarray(recs, dtype=np.float64).reshape(-1, 8)
    if len(recs) == 0:
        return []
    mats = np.zeros((len(recs), 3, 3), dtype=np.float64)
    mats[:, 0, 0], mats[:, 0, 1], mats[:, 1, 0], mats[:, 1, 1], mats[:, 2, 2] = recs[:, 3], -recs[:, 4], recs[:, 4], recs[:, 3], 1.0
    quats = R.from_matrix(mats).as_quat()
    out = []
    for rec, m, q, cls in zip(recs, mats, quats, classes):
        cx, cy, cz, _, _, length, width, height = (float(v) for v in rec)
        d = make_dictionary([[cx, cy, cz], [q[0], q[1], q[2], q[3]], [length, width, height], [cls]], ss=ss)
        d['_matrix'] = m
        out.append(d)
    return out


def create_annotation_line(original_string, new_annotation_dict, rotation):
    """KITTI line of an inserted object (od/ins:227-265)."""
    rotation = np.deg2rad(rotation)
    cx, cy, cz = (new_annotation_dict['center'][k] for k in 'xyz')
    original_string = original_string.item() if hasattr(original_string, 'item') else str(original_string)
    items = original_string.split(' ')
    rotation_y = float(items[14]) - rotation
    if rotation_y < -np.pi:
        rotation_y += 2 * np.pi
    elif rotation_y > np.pi:
        rotation_y -= 2 * np.pi
    assert -np.pi <= rotation_y <= np.pi, f'Error in range of sample_rotation_y = {rotation_y}'
    alpha = (np.arctan2((cy * -1), cx - 0.27) * -1) + rotation_y
    if alpha < -np.pi:
        alpha += 2 * np.pi
    elif alpha > np.pi:
        alpha -= 2 * np.pi
    assert -np.pi <= alpha <= np.pi, f'Error in range of alpha = {alpha}'
    return (f"{new_annotation_dict['class']} {items[1]} 3 {alpha:.02f} {items[4]} {items[5]} {items[6]} {items[7]} "
            f"{items[8]} {items[9]} {items[10]} {(cy * -1):.02f} {(cz * -1) - 0.08:.02f} {cx - 0.27:.02f} "
            f"{rotation_y:.02f}\n")


def search_radii():
    """radius**2 of the road-level search (od/fs:149-160): 0.1 grown by repeated += 0.1, and whether the pass still
    satisfies ``radius <= 5`` after its own increment."""
    r2, ok = [], []
    radius = 0.1
    for _ in range(50):
        r2.append(radius ** 2)
        radius += 0.1
        ok.append(0 if radius > 5 else 1)
    return np.array(r2, dtype=np.float64), np.array(ok, dtype=np.int32)


def yaw_tables(yaw_steps):
    """cos / sin of k * (360 / yaw_steps) degrees, k = 0..yaw_steps (the reference's K = 360 gives whole degrees)."""
    ang = np.deg2rad(np.arange(yaw_steps + 1) * (360.0 / yaw_steps))
    return np.ascontiguousarray(np.cos(ang)), np.ascontiguousarray(np.sin(ang))
