"""ctypes binding of ``libreal3d_b200.so`` (C ABI in ``include/real3d_b200.h``).

There is NO CPU fallback: importing works without a GPU (so the CPU test tier can check that the library loads and
exports every declared symbol), but every compute call needs a CUDA device and raises otherwise, and a missing
library raises ``ImportError`` with the build command.
"""
from __future__ import annotations

import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libreal3d_b200.so")

R3D_MAX_CLASSES = 16
R3D_MAX_SURFACE = 8
R3D_NUM_RADII = 50
R3D_BOX_DOUBLES = 16

ERRORS = {-1: "CUDA error", -2: "bad argument", -3: "AssertionError in the reference (projection bin out of range)",
          -4: "IndexError in the reference (sample list shorter than MAX_NUM_TRIES)", -5: "capacity exceeded"}


class ClassCfg(C.Structure):
    _fields_ = [("min_points", C.c_int32), ("map_sel", C.c_int32), ("map_ok_mask", C.c_uint32),
                ("pedestrian", C.c_int32), ("n_surface", C.c_int32), ("surface", C.c_int32 * R3D_MAX_SURFACE)]


class EngineCfg(C.Structure):
    _fields_ = [("task", C.c_int32), ("rows", C.c_int32), ("cols", C.c_int32), ("yaw_steps", C.c_int32),
                ("max_tries", C.c_int32), ("n_classes", C.c_int32), ("max_scans", C.c_int32),
                ("max_points", C.c_int32), ("max_inserted", C.c_int32), ("max_boxes", C.c_int32),
                ("max_events", C.c_int32), ("road_label", C.c_int32), ("n_road_indexes", C.c_int32),
                ("road_indexes", C.c_int32 * R3D_MAX_SURFACE), ("map_window", C.c_int32),
                ("grid_half", C.c_int32), ("grid_cell", C.c_double), ("flags", C.c_int32),
                ("radii_sq", C.c_double * R3D_NUM_RADII), ("radii_ok", C.c_int32 * R3D_NUM_RADII),
                ("classes", ClassCfg * R3D_MAX_CLASSES)]


class ObjectDb(C.Structure):
    _fields_ = [("n_objects", C.c_int32), ("point_offsets", C.c_void_p), ("points5", C.c_void_p),
                ("boxes", C.c_void_p), ("class_index", C.c_void_p), ("class_list_offsets", C.c_void_p),
                ("class_list", C.c_void_p)]


class Batch(C.Structure):
    _fields_ = [("n_scans", C.c_int32), ("point_offsets", C.c_void_p), ("xyzi", C.c_void_p), ("labels", C.c_void_p),
                ("box_offsets", C.c_void_p), ("boxes", C.c_void_p), ("map_offsets", C.c_void_p), ("maps", C.c_void_p),
                ("map_dims", C.c_void_p), ("poses", C.c_void_p), ("counts", C.c_void_p), ("perms", C.c_void_p),
                ("n_events", C.c_int32), ("labels16", C.c_void_p), ("labels1", C.c_void_p)]


class BatchResult(C.Structure):
    _fields_ = [("out_offsets", C.c_void_p), ("out_xyzi", C.c_void_p), ("out_labels", C.c_void_p),
                ("capacity_points", C.c_int64), ("check_offsets", C.c_void_p), ("check_xyzil", C.c_void_p),
                ("capacity_check", C.c_int64), ("n_inserted", C.c_void_p), ("inserted", C.c_void_p),
                ("inserted_box", C.c_void_p), ("status", C.c_void_p), ("rounds", C.c_void_p), ("out_labels16", C.c_void_p)]


class ResidentStore(C.Structure):
    _fields_ = [("n_scans", C.c_int32), ("xyzi", C.c_void_p), ("labels", C.c_void_p), ("point_offsets", C.c_void_p),
                ("boxes", C.c_void_p), ("box_offsets", C.c_void_p), ("maps", C.c_void_p), ("map_offsets", C.c_void_p),
                ("map_dims", C.c_void_p), ("poses", C.c_void_p), ("h_point_offsets", C.c_void_p),
                ("h_box_offsets", C.c_void_p)]


class WorldAug(C.Structure):
    _fields_ = [("flip_x_prob", C.c_float), ("flip_y_prob", C.c_float), ("rot_max", C.c_float), ("scale_lo", C.c_float),
                ("scale_hi", C.c_float)]


# name -> (restype, argtypes); must list every symbol declared in include/real3d_b200.h
PROTOTYPES = {
    "r3d_version": (C.c_int, []),
    "r3d_last_error": (C.c_char_p, []),
    "r3d_launch_count": (C.c_int64, []),
    "r3d_fill_spherical": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "r3d_project_zbuffer": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_int, C.c_double, C.c_double, C.c_int,
                                      C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_close_fill": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_cut_bounding_box": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_transform_points": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_double, C.c_double, C.c_double, C.c_void_p]),
    "r3d_road_level": (C.c_int, [C.c_void_p, C.c_int64, C.c_int, C.c_int, C.c_void_p, C.c_int, C.c_double, C.c_double,
                                 C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_double), C.POINTER(C.c_int32),
                                 C.c_void_p]),
    "r3d_adjust_map": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_int64, C.c_void_p, C.c_int,
                                 C.c_void_p, C.c_int, C.c_int, C.c_void_p]),
    "r3d_place_candidates": (C.c_int, [C.c_void_p, C.c_int64, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                       C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64, C.c_void_p, C.c_uint32, C.c_void_p,
                                       C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_obb_collide": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int32, C.c_void_p, C.c_int64, C.c_int32, C.c_void_p,
                                  C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "r3d_occlude_mask": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p,
                                   C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_compact_insert": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                     C.c_void_p, C.c_int64, C.c_void_p]),
    "r3d_engine_walk_profile": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int]),
    "r3d_engine_probe_places": (C.c_int, [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p,
                                          C.c_void_p, C.c_int, C.POINTER(C.c_int32)]),
    "r3d_engine_create": (C.c_int, [C.POINTER(EngineCfg), C.POINTER(C.c_void_p)]),
    "r3d_engine_destroy": (C.c_int, [C.c_void_p]),
    "r3d_engine_set_yaw_tables": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_engine_set_objects": (C.c_int, [C.c_void_p, C.POINTER(ObjectDb)]),
    "r3d_engine_set_ss_map": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64]),
    "r3d_engine_load_batch": (C.c_int, [C.c_void_p, C.POINTER(Batch)]),
    "r3d_engine_reset_batch": (C.c_int, [C.c_void_p]),
    "r3d_engine_run": (C.c_int, [C.c_void_p]),
    "r3d_engine_fetch": (C.c_int, [C.c_void_p, C.POINTER(BatchResult)]),
    "r3d_rich_map_od_extents": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p]),
    "r3d_rich_map_od_build": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_uint32, C.c_void_p, C.c_void_p,
                                        C.c_int64, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_rich_map_ss_extents": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int32, C.c_void_p,
                                          C.c_void_p, C.c_void_p]),
    "r3d_rich_map_ss_raster": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p,
                                         C.c_void_p, C.c_int32, C.c_int64, C.c_int64, C.c_int32, C.c_int32, C.c_int64,
                                         C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_rich_map_ss_finalize": (C.c_int, [C.c_void_p, C.c_int64, C.c_void_p, C.c_void_p]),
    "r3d_cut_objects_count": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p, C.c_int32,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_cut_objects_write": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_int32, C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p,
                                        C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_engine_output_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                           C.c_void_p, C.c_void_p]),
    "r3d_engine_sync": (C.c_int, [C.c_void_p]),
    "r3d_engine_set_sub_batches": (C.c_int, [C.c_void_p, C.c_int]),
    "r3d_engine_run_until": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "r3d_engine_output_rows": (C.c_int, [C.c_void_p, C.POINTER(C.c_int64), C.POINTER(C.c_int64)]),
    "r3d_engine_profile_enable": (C.c_int, [C.c_void_p, C.c_int]),
    "r3d_engine_profile_read": (C.c_int, [C.c_void_p, C.c_char_p, C.c_int, C.c_void_p, C.c_void_p, C.c_int,
                                          C.POINTER(C.c_int)]),
    "r3d_engine_stats": (C.c_int, [C.c_void_p, C.c_void_p]),
    "r3d_engine_stats_ex": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int]),
    "r3d_engine_rearm_batch": (C.c_int, [C.c_void_p, C.c_int]),
    "r3d_engine_stream": (C.c_void_p, [C.c_void_p]),
    "r3d_engine_debug_image": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p]),
    "r3d_engine_debug_candidates": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_engine_debug_col_index": (C.c_int, [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_engine_set_schedule_policy": (C.c_int, [C.c_void_p, C.c_int32, C.c_int32, C.c_void_p]),
    "r3d_engine_load_resident": (C.c_int, [C.c_void_p, C.POINTER(ResidentStore), C.c_void_p, C.c_int32, C.c_uint64, C.c_uint64]),
    "r3d_engine_set_ss_map_device": (C.c_int, [C.c_void_p, C.c_void_p, C.c_int32, C.c_int32, C.c_int64, C.c_int64]),
    "r3d_engine_schedule_read": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p, C.POINTER(C.c_int32)]),
    "r3d_engine_inserted_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p),
                                             C.POINTER(C.c_void_p)]),
    "r3d_engine_set_world_aug": (C.c_int, [C.c_void_p, C.POINTER(WorldAug)]),
    "r3d_engine_world_device": (C.c_int, [C.c_void_p, C.POINTER(C.c_void_p)]),
    "r3d_engine_set_object_targets": (C.c_int, [C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_engine_targets_device": (C.c_int, [C.c_void_p, C.POINTER(ResidentStore), C.c_void_p, C.c_void_p, C.c_int32,
                                            C.c_void_p, C.c_void_p, C.c_void_p]),
    "r3d_engine_target_points_device": (C.c_int, [C.c_void_p, C.c_int32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_int32,
                                                  C.c_void_p, C.c_void_p]),
}

_lib = None


def load():
    """Load the shared library (once) and bind the prototypes."""
    global _lib
    if _lib is not None:
        return _lib
    path = os.environ.get("R3D_LIB_PATH", LIB_PATH)         # tuning aid: a variant build of the same sources
    if not os.path.exists(path):
        raise ImportError(
            f"{path} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(nvcc -gencode arch=compute_100a,code=sm_100a).  There is no CPU fallback.")
    lib = C.CDLL(path)
    for name, (res, args) in PROTOTYPES.items():
        fn = getattr(lib, name)          # AttributeError if the .so does not export a declared symbol
        fn.restype = res
        fn.argtypes = args
    _lib = lib
    return lib


class Real3DError(RuntimeError):
    pass


def check(rc, what=""):
    if rc == 0:
        return
    msg = load().r3d_last_error().decode(errors="replace")
    kind = ERRORS.get(rc, f"error {rc}")
    if rc == -3:
        raise AssertionError(f"{what}: {kind}: {msg}")
    if rc == -4:
        raise IndexError(f"{what}: {kind}: {msg}")
    raise Real3DError(f"{what}: {kind}: {msg}")


def require_cuda():
    import torch
    if not torch.cuda.is_available():
        raise Real3DError("real3d_b200 needs a CUDA device (sm_100a); there is no CPU fallback")
    return torch
