"""GPU tier: engine lifetime through the C ABI.  A create that fails releases everything it made, and destroy releases
the whole engine.  Measured as device-wide free memory, so the tolerance stays well above what other processes on a
shared GPU move and well below one engine of this size (about 1 GiB)."""
import ctypes as C

import pytest

from pcl_augmentation_b200 import _lib

pytestmark = pytest.mark.gpu

R3D_ERR_CAPACITY = -5
TOLERANCE = 512 << 20


def semseg_cfg(second_class_labels):
    """Two semseg classes of 8 surface labels each: 64 scans of 131072 points, a 112 x 1440 image."""
    cfg = _lib.EngineCfg()
    cfg.task = 1
    cfg.rows, cfg.cols, cfg.yaw_steps, cfg.max_tries = 112, 1440, 360, 100
    cfg.n_classes = 2
    cfg.max_scans, cfg.max_points, cfg.max_inserted = 64, 131072, 4096
    cfg.max_boxes, cfg.max_events = 64, 11
    cfg.map_window, cfg.grid_half, cfg.grid_cell = 512, 120, 0.5
    for c, labels in enumerate([range(1, 9), second_class_labels]):
        cfg.classes[c].min_points = 10
        cfg.classes[c].n_surface = 8
        for i, v in enumerate(labels):
            cfg.classes[c].surface[i] = v
    return cfg


def free_bytes():
    import torch
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info()[0]


def test_failed_create_releases_everything():
    lib = _lib.load()
    cfg = semseg_cfg(range(9, 17))                   # 16 distinct surface labels: more than the 15 the engine takes
    before = free_bytes()
    for _ in range(3):
        handle = C.c_void_p()
        assert lib.r3d_engine_create(C.byref(cfg), C.byref(handle)) == R3D_ERR_CAPACITY
        assert b"surface labels" in lib.r3d_last_error()
        assert not handle
    assert abs(free_bytes() - before) < TOLERANCE


def test_destroy_releases_everything():
    lib = _lib.load()
    cfg = semseg_cfg(range(1, 9))
    before = free_bytes()
    for _ in range(3):
        handle = C.c_void_p()
        _lib.check(lib.r3d_engine_create(C.byref(cfg), C.byref(handle)), "r3d_engine_create")
        assert before - free_bytes() > TOLERANCE     # the engine's memory is visible to this measurement
        _lib.check(lib.r3d_engine_destroy(handle), "r3d_engine_destroy")
    assert abs(free_bytes() - before) < TOLERANCE
