"""Host reference of r3d_engine_target_points_device (include/real3d_b200.h): which output rows of a scan lie inside
which detection target, per-target point counts, the first-hit assignment of every row and the min-points filter."""
import numpy as np


def box_frame(points, boxes):
    """(dz, lx, ly) float64 [N, M]: each point (x, y, z) relative to each box (cx, cy, cz, dx, dy, dz, h), every step
    rounded once in float64 on the float32 values: u = x - cx, v = y - cy, lx = c u + s v, ly = -s u + c v."""
    p = np.asarray(points, dtype=np.float32).astype(np.float64)
    b = np.asarray(boxes, dtype=np.float32).astype(np.float64)
    c, s = np.cos(b[:, 6]), np.sin(b[:, 6])
    u = p[:, 0:1] - b[None, :, 0]
    v = p[:, 1:2] - b[None, :, 1]
    lx = c * u + s * v
    ly = -(s * u) + c * v
    return p[:, 2:3] - b[None, :, 2], lx, ly


def points_in_boxes(points, boxes):
    """bool [N, M]: OpenPCDet's points_in_boxes test, |z - cz| <= dz / 2 and |lx| < dx / 2 and |ly| < dy / 2."""
    dz, lx, ly = box_frame(points, boxes)
    half = np.asarray(boxes, dtype=np.float32).astype(np.float64)[:, 3:6] * 0.5
    return (np.abs(dz) <= half[:, 2]) & (np.abs(lx) < half[:, 0]) & (np.abs(ly) < half[:, 1])


def near_faces(points, boxes, eps=1e-9):
    """bool [N]: points whose inside test against some box is decided by less than ``eps`` m in float64 (one bound
    within eps and none of the others clearly false); the device's cos / sin may differ from numpy's in the last bit."""
    dz, lx, ly = box_frame(points, boxes)
    half = np.asarray(boxes, dtype=np.float32).astype(np.float64)[:, 3:6] * 0.5
    margins = [half[:, 2] - np.abs(dz), half[:, 0] - np.abs(lx), half[:, 1] - np.abs(ly)]
    clearly_out = np.zeros(dz.shape, dtype=bool)
    close = np.zeros(dz.shape, dtype=bool)
    for m in margins:
        clearly_out |= m <= -eps
        close |= np.abs(m) < eps
    return (close & ~clearly_out).any(axis=1) if dz.shape[1] else np.zeros(len(dz), dtype=bool)


def target_points(points, boxes):
    """(counts int32 [M], point_gt int32 [N]): points inside each box, and the first box containing each point or -1."""
    inside = points_in_boxes(points, boxes)
    counts = inside.sum(axis=0).astype(np.int32)
    first = np.where(inside.any(axis=1), inside.argmax(axis=1), -1).astype(np.int32) if inside.shape[1] else \
        np.full(len(inside), -1, dtype=np.int32)
    return counts, first


def filter_min_points(points, boxes, min_points):
    """(kept indices int64 [K], counts of the kept boxes, point_gt into the kept boxes): drop every box with fewer than
    ``min_points`` points, keep the order, and assign each point to the first kept box that contains it."""
    inside = points_in_boxes(points, boxes)
    counts = inside.sum(axis=0)
    kept = np.flatnonzero(counts >= min_points)
    inside = inside[:, kept]
    first = np.where(inside.any(axis=1), inside.argmax(axis=1), -1).astype(np.int32) if len(kept) else \
        np.full(len(inside), -1, dtype=np.int32)
    return kept, counts[kept].astype(np.int32), first
