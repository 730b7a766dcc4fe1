"""Batched, device-resident driver of the Real3D-Aug per-scan loop (``augment_batch``).

The reference runs one scan at a time through nested Python loops (od/ins:321-628, ss/ins:317-599).  Here a whole
batch of scans is resident in HBM and advanced in lock-step rounds by ``libreal3d_b200.so``; this module only
prepares the host-side tables (class configuration from the YAML, parsed boxes, yaw and radius tables, the cut-object
database, the pre-drawn schedules) and unpacks the results into the reference's output records
(``save_data`` od/ds:76-95, ss/ds:72-91; ``create_annotation_line`` od/ins:227-265; ``added_objects/<frame>.txt``).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field

import numpy as np

from . import _lib
from . import boxes as bx

ROAD_INDEXES = [40, 44, 48]          # od/fs:14, used by the semseg addjust_map_2 (ss/ins:209)
MAX_NUM_TRIES = 100                  # od/ins:24


@dataclass
class ScanInput:
    """One scan in the layouts the reference's dataset adapters hand to insertion.py."""
    xyzi: np.ndarray                  # N x 4 float32 (velodyne/*.bin)
    labels: np.ndarray                # N uint32 (semantic label & 0xFFFF)
    box_lines: list                   # scene annotation lines (label_2/*.txt or bbox/*.txt)
    counts: np.ndarray                # objects to insert per class (generate_seed)
    perms: np.ndarray                 # int32 [events, classes, tries]: pre-drawn random.shuffle results
    maps: dict | None = None          # OD: {'Road': {...}, 'Sidewalk': {...}} (npz payloads)
    pose: np.ndarray | None = None    # semseg: 4x4 lidar->world
    box_dicts: list | None = None     # scene annotations already parsed to box dictionaries (instead of box_lines)


@dataclass
class ScanResult:
    velodyne: np.ndarray              # N' x 4 float32  (velodyne/<frame>.bin)
    labels: np.ndarray                # N' uint32       (labels/<frame>.label, semseg)
    check: np.ndarray                 # V x 4 (OD) / V x 5 (semseg) float32 (check/<frame>.bin)
    inserted: list                    # [(object name, rotation, class)]  -> added_objects/<frame>.txt
    lines: list                       # OD: KITTI annotation lines of the inserted objects
    boxes: list                       # box dictionaries of the inserted objects
    visible: list                     # visible points per inserted object
    status: int = 0
    extra: dict = field(default_factory=dict)


def _cuda_tensor(ptr, shape, typestr, dtype):
    """CUDA tensor that aliases ``prod(shape)`` elements of library-owned device memory at ``ptr`` (no copy)."""
    import torch
    dev = torch.device("cuda", torch.cuda.current_device())
    if shape[0] == 0:
        return torch.empty(shape, dtype=dtype, device=dev)

    class _View:
        def __init__(self):
            self.__cuda_array_interface__ = {"shape": shape, "typestr": typestr, "data": (int(ptr), False), "version": 3,
                                             "strides": None}
    return torch.as_tensor(_View(), device=dev)


def _pinned(shape, dtype):
    """numpy array backed by page-locked host memory (owned by a torch tensor kept alive on the array)."""
    import torch
    tdt = {np.float32: torch.float32, np.float64: torch.float64, np.int32: torch.int32, np.int64: torch.int64, np.int16: torch.int16,
           np.uint8: torch.uint8}[np.dtype(dtype).type]
    pin = torch.cuda.is_available()
    t = torch.empty(tuple(int(s) for s in np.atleast_1d(shape)), dtype=tdt, pin_memory=pin)
    return t.numpy()


class Real3DEngine:
    """One engine per process / GPU.  ``task`` is 'od' (KITTI) or 'ss' (SemanticKITTI)."""

    def __init__(self, task, config, db, *, max_scans, max_points, rows=112, cols=1440, yaw_steps=360,
                 max_tries=MAX_NUM_TRIES, max_inserted=None, max_boxes=64, max_events=None, map_data=None,
                 map_window=512, road_indexes=None, grid_cell=0.5, grid_half=120, force_full_projection=False,
                 sub_batches=0, fetch_labels=None, round_graphs=True, candidate_window=True, staged_rounds=False):
        _lib.require_cuda()
        self.lib = _lib.load()
        self.task = task
        self.config = config
        self.classes = list(config['insertion']['classes'])
        self.rows, self.cols, self.yaw_steps, self.max_tries = rows, cols, yaw_steps, max_tries
        self.max_scans, self.max_points = int(max_scans), int(max_points)
        self.grid_half, self.grid_cell = int(grid_half), float(grid_cell)
        self.road_label = int(config['labels']['Road']) if task == 'od' else 0
        ins = config['insertion']
        # slots per scan: the pre-drawn class counts sum to number_of_object (random) or to sum(number_of_classes)
        nobj = int(ins.get('number_of_object', 10)) if ins.get('random', True) else int(np.sum(ins['number_of_classes']))
        self.max_events = int(max_events if max_events is not None else nobj + 1)
        self._prepare_db(db)
        if max_inserted is None:
            max_inserted = max(4096, self.max_events * self.max_obj_points)
        self.max_inserted, self.max_boxes = int(max_inserted), int(max_boxes)
        cfg = _lib.EngineCfg()
        cfg.task = 0 if task == 'od' else 1
        cfg.rows, cfg.cols, cfg.yaw_steps, cfg.max_tries = rows, cols, yaw_steps, max_tries
        cfg.n_classes = len(self.classes)
        cfg.max_scans, cfg.max_points, cfg.max_inserted = self.max_scans, self.max_points, self.max_inserted
        cfg.max_boxes, cfg.max_events = self.max_boxes, self.max_events
        cfg.road_label = int(config['labels']['Road']) if task == 'od' else 0
        if road_indexes is None:         # config key (shipped waymo.yaml), else the reference's constant (od/fs:14)
            road_indexes = config['insertion'].get('road_indexes', ROAD_INDEXES)
        self.road_indexes = [int(v) for v in road_indexes]
        cfg.n_road_indexes = len(road_indexes)
        for i, v in enumerate(road_indexes):
            cfg.road_indexes[i] = int(v)
        cfg.map_window = int(map_window)
        cfg.grid_half, cfg.grid_cell = int(grid_half), float(grid_cell)
        # bit 0: full re-projection every slot; bit 1: no round graphs; bit 2: no ordered early-out window; bit 3: the
        # staged round kernels instead of the per-scan persistent walker (needed by debug_candidates, which wants every
        # candidate of a try evaluated); bits 8-12: concurrent sub-batches of the staged rounds (0 = library default)
        self.staged_rounds = bool(staged_rounds) or not candidate_window
        cfg.flags = ((1 if force_full_projection else 0) | (0 if round_graphs else 2) | (0 if candidate_window else 4)
                     | (8 if self.staged_rounds else 0) | ((int(sub_batches) & 31) << 8))
        r2, ok = bx.search_radii()
        for i in range(50):
            cfg.radii_sq[i] = float(r2[i])
            cfg.radii_ok[i] = int(ok[i])
        for ci, cls in enumerate(self.classes):
            cc = cfg.classes[ci]
            cc.min_points = int(config['insertion']['min_points'][cls])
            if task == 'od':
                placement = config['insertion']['placement'][cls]
                assert placement in ('Road', 'Sidewalk'), f'unrecognized placement area for {cls}'    # od/ins:443
                cc.map_sel = 0 if placement == 'Road' else 1
                cc.pedestrian = 1 if cls == 'Pedestrian' else 0
                cc.n_surface = 1
                cc.surface[0] = int(config['labels']['Road'])                                        # od/fs:154
            else:
                ok_map_surface = config['insertion']['placement'][cls]                               # ss/fs:221
                mask = 0
                surf = []
                for v in ok_map_surface:
                    mask |= 1 << int(v)
                    surf += list(config['insertion']['placement_labels'][v])                         # ss/fs:223-226
                cc.map_ok_mask = mask
                cc.n_surface = len(surf)
                assert len(surf) <= _lib.R3D_MAX_SURFACE
                for i, v in enumerate(surf):
                    cc.surface[i] = int(v)
        handle = C.c_void_p()
        _lib.check(self.lib.r3d_engine_create(C.byref(cfg), C.byref(handle)), "r3d_engine_create")
        self.handle = handle
        cos_k, sin_k = bx.yaw_tables(yaw_steps)
        _lib.check(self.lib.r3d_engine_set_yaw_tables(handle, cos_k.ctypes.data, sin_k.ctypes.data), "set_yaw_tables")
        self._upload_db()
        if task == 'ss':
            assert map_data is not None, "semseg needs the sequence rich map {'map', 'move'}"
            m = np.ascontiguousarray(np.asarray(map_data['map']).astype(np.uint8))
            mv = np.asarray(map_data['move']).reshape(-1)
            _lib.check(self.lib.r3d_engine_set_ss_map(handle, m.ctypes.data, m.shape[0], m.shape[1], int(mv[0]),
                                                      int(mv[1])), "set_ss_map")
        self._keep = []
        self._n_scans = 0
        self._policy_set = False
        # labels/<frame>.label exists only in the semseg outputs (ss/ds:82-84); OD writes velodyne + check + label_2
        self.fetch_labels = (task == 'ss') if fetch_labels is None else bool(fetch_labels)

    # ------------------------------------------------------------------------------------------ database
    def _prepare_db(self, db):
        read = bx.read_label_line_ss if self.task == 'ss' else bx.read_label_line_od
        names, pts, offs, box_rows, cls_idx, lists, list_off, annos, strings = [], [], [0], [], [], [], [0], [], []
        for ci, cls in enumerate(self.classes):
            for name, sample in db.get(cls, []):
                pcl = np.array(sample['pcl'], dtype=np.float64, copy=True)
                if self.task == 'od':
                    pcl[:, 4] = 1                                     # od/fs:251
                anno = read(str(sample['anno'].item() if hasattr(sample['anno'], 'item') else sample['anno']))
                lists.append(len(names))
                names.append(name)
                pts.append(pcl[:, :5])
                offs.append(offs[-1] + len(pcl))
                box_rows.append(bx.object_box_record(anno))
                cls_idx.append(ci)
                annos.append(anno)
                strings.append(sample['anno'])
            list_off.append(len(lists))
        self.obj_names, self.obj_annos, self.obj_strings = names, annos, strings
        self._db_points = np.ascontiguousarray(np.concatenate(pts, axis=0))
        self._db_offsets = np.array(offs, dtype=np.int64)
        self._db_boxes = np.ascontiguousarray(np.array(box_rows, dtype=np.float64))
        self._db_cls = np.array(cls_idx, dtype=np.int32)
        self._db_list_off = np.array(list_off, dtype=np.int32)
        self._db_list = np.array(lists, dtype=np.int32)
        self.max_obj_points = int(np.diff(self._db_offsets).max())

    def _upload_db(self):
        db = _lib.ObjectDb()
        db.n_objects = len(self.obj_names)
        db.point_offsets = self._db_offsets.ctypes.data
        db.points5 = self._db_points.ctypes.data
        db.boxes = self._db_boxes.ctypes.data
        db.class_index = self._db_cls.ctypes.data
        db.class_list_offsets = self._db_list_off.ctypes.data
        db.class_list = self._db_list.ctypes.data
        _lib.check(self.lib.r3d_engine_set_objects(self.handle, C.byref(db)), "set_objects")

    # --------------------------------------------------------------------------------------------- batch
    def stage(self, scans):
        """Pack a list of ScanInput into pinned host buffers (not part of the timed e2e path's GPU work; this is the
        role of the dataset reader).  Returns an opaque staged batch for ``load``."""
        n = len(scans)
        assert 0 < n <= self.max_scans
        pt_off = np.zeros(n + 1, dtype=np.int64)
        for i, s in enumerate(scans):
            pt_off[i + 1] = pt_off[i] + len(s.xyzi)
        total = int(pt_off[-1])
        xyzi = _pinned((total, 4), np.float32)
        # labels over PCIe: semseg 2 bytes per point (they are & 0xFFFF, od/ds:65); object detection ONE BIT per point —
        # the reference collapses the labels to {Road, 1} before its loop (od/ins:353-355), "is Road" is all the path reads
        road_bits = self.task == 'od'
        labels = _pinned((total,), np.int16) if not road_bits else np.zeros(total, dtype=bool)
        box_off = np.zeros(n + 1, dtype=np.int32)
        n_events = max(int(np.asarray(s.perms).shape[0]) for s in scans)
        most = max(int(np.sum(s.counts)) for s in scans)
        if most + 1 > self.max_events:
            raise _lib.Real3DError(f"a scan asks for {most} insertions but the engine was built with max_events = "
                                   f"{self.max_events} (insertion.number_of_object / number_of_classes of the config, or "
                                   f"pass max_events)")
        nc = len(self.classes)
        counts = _pinned((n, nc), np.int32)
        counts[:] = 0
        perms = _pinned((n, n_events, nc, self.max_tries), np.int32)
        perms[:] = -1
        for i, s in enumerate(scans):
            xyzi[pt_off[i]:pt_off[i + 1]] = s.xyzi
            lab = np.asarray(s.labels)
            assert lab.size == 0 or int(lab.max()) < 65536, "semantic labels must be masked with 0xFFFF (od/ds:65)"
            if road_bits:
                labels[pt_off[i]:pt_off[i + 1]] = lab == self.road_label
            else:
                labels[pt_off[i]:pt_off[i + 1]] = lab.astype(np.uint16).view(np.int16)
            box_off[i + 1] = box_off[i] + len(s.box_dicts if s.box_dicts is not None else s.box_lines)
            counts[i] = np.asarray(s.counts, dtype=np.int32)
            p = np.asarray(s.perms, dtype=np.int32)
            perms[i, :p.shape[0], :, :p.shape[2]] = p
        # scene boxes: the annotation lines of the whole batch go through scipy's matrix <-> quaternion conversions in ONE
        # call (bit-identical to the per-line path, 18x cheaper); scans that bring box dictionaries keep the per-box path
        from_lines = bx.box_records_from_lines([line for s in scans if s.box_dicts is None for line in s.box_lines],
                                               ss=self.task == 'ss')
        boxes = _pinned((max(int(box_off[-1]), 1), 16), np.float64)[:int(box_off[-1])]
        taken = 0
        for i, s in enumerate(scans):
            k = int(box_off[i + 1] - box_off[i])
            if s.box_dicts is None:
                boxes[box_off[i]:box_off[i + 1]] = from_lines[taken:taken + k]
                taken += k
            elif k:
                boxes[box_off[i]:box_off[i + 1]] = np.array([bx.box_record(a) for a in s.box_dicts], dtype=np.float64).reshape(-1, 16)
        if road_bits:
            packed = np.packbits(labels, bitorder='little')
            labels = _pinned((max(len(packed), 1),), np.uint8)
            labels[:len(packed)] = packed
        staged = {'n': n, 'pt_off': pt_off, 'xyzi': xyzi, 'labels': labels, 'label_bits': road_bits, 'box_off': box_off, 'boxes': boxes,
                  'counts': counts, 'perms': perms, 'n_events': n_events, 'total': total}
        if self.task == 'od':
            blobs, moff, dims = [], [0], np.zeros((n, 2, 4), dtype=np.int32)
            for i, s in enumerate(scans):
                for j, key in enumerate(('Road', 'Sidewalk')):
                    md = s.maps[key]
                    m = np.ascontiguousarray(np.asarray(md['map']).astype(np.uint8))
                    blobs.append(m.reshape(-1))
                    moff.append(moff[-1] + m.size)
                    dims[i, j] = (m.shape[0], m.shape[1], int(md['min_x']), int(md['min_y']))
            maps = _pinned((moff[-1],), np.uint8)
            maps[:] = np.concatenate(blobs)
            staged.update(maps=maps, map_off=np.array(moff, dtype=np.int64), map_dims=dims)
        else:
            staged['poses'] = np.ascontiguousarray(np.stack([np.asarray(s.pose, dtype=np.float64) for s in scans]))
        return staged

    def load(self, staged):
        """Host -> device copy of a staged batch + the one-off spherical cache (A1/A2)."""
        b = _lib.Batch()
        b.n_scans = staged['n']
        b.point_offsets = staged['pt_off'].ctypes.data
        b.xyzi = staged['xyzi'].ctypes.data
        b.labels = None
        b.labels16 = None if staged.get('label_bits') else staged['labels'].ctypes.data
        b.labels1 = staged['labels'].ctypes.data if staged.get('label_bits') else None
        b.box_offsets = staged['box_off'].ctypes.data
        b.boxes = staged['boxes'].ctypes.data if staged['boxes'].size else None
        if self.task == 'od':
            b.map_offsets = staged['map_off'].ctypes.data
            b.maps = staged['maps'].ctypes.data
            b.map_dims = staged['map_dims'].ctypes.data
        else:
            b.poses = staged['poses'].ctypes.data
        b.counts = staged['counts'].ctypes.data
        b.perms = staged['perms'].ctypes.data
        b.n_events = staged['n_events']
        self._keep = [staged, b]
        self._n_scans = staged['n']
        self._in_bytes = staged['total'] * 18
        _lib.check(self.lib.r3d_engine_load_batch(self.handle, C.byref(b)), "load_batch")

    def reset(self, from_raw_points=False):
        """Re-arm the resident batch.  ``from_raw_points`` repeats the whole device path from the resident float4
        points (spherical ingest, spatial indices) instead of only resetting the flags and the scheduling state."""
        _lib.check(self.lib.r3d_engine_rearm_batch(self.handle, 1 if from_raw_points else 0), "rearm_batch")

    def run(self):
        _lib.check(self.lib.r3d_engine_run(self.handle), "run")

    def run_until(self, stop_at):
        """``run`` that returns True (still running) once at most ``stop_at`` scans are unfinished; call again with 0."""
        more = C.c_int(0)
        _lib.check(self.lib.r3d_engine_run_until(self.handle, int(stop_at), C.byref(more)), "run_until")
        return bool(more.value)

    def set_sub_batches(self, n):
        """How many contiguous sub-batches ``run`` advances concurrently on their own streams (1 = strictly serial)."""
        _lib.check(self.lib.r3d_engine_set_sub_batches(self.handle, int(n)), "set_sub_batches")

    def sync(self):
        _lib.check(self.lib.r3d_engine_sync(self.handle), "sync")

    def output_rows(self):
        a, b = C.c_int64(), C.c_int64()
        _lib.check(self.lib.r3d_engine_output_rows(self.handle, C.byref(a), C.byref(b)), "output_rows")
        return a.value, b.value

    def fetch_raw(self, buffers=None):
        """Device -> host copy of the last run's outputs into (reusable, pinned) buffers."""
        n = self._n_scans
        rows, chk = self.output_rows()
        if buffers is None or buffers['cap_points'] < rows or buffers['cap_check'] < chk:
            cap_p, cap_c = max(rows, 1), max(chk, 1)
            buffers = {'cap_points': cap_p, 'cap_check': cap_c, 'xyzi': _pinned((cap_p, 4), np.float32),
                       'labels': _pinned((cap_p,), np.int16), 'check': _pinned((cap_c, 5), np.float32)}   # labels: 16 bit over PCIe
        buffers.update(out_off=np.zeros(n + 1, dtype=np.int64), check_off=np.zeros(n + 1, dtype=np.int64),
                       n_inserted=np.zeros(n, dtype=np.int32), inserted=np.zeros((n, self.max_events, 4), dtype=np.int32),
                       inserted_box=np.zeros((n, self.max_events, 8), dtype=np.float64),
                       status=np.zeros(n, dtype=np.int32), rounds=np.zeros(1, dtype=np.int32))
        r = _lib.BatchResult()
        r.out_offsets = buffers['out_off'].ctypes.data
        r.out_xyzi = buffers['xyzi'].ctypes.data
        r.out_labels = None
        r.out_labels16 = buffers['labels'].ctypes.data if self.fetch_labels else None
        r.capacity_points = buffers['cap_points']
        r.check_offsets = buffers['check_off'].ctypes.data
        r.check_xyzil = buffers['check'].ctypes.data
        r.capacity_check = buffers['cap_check']
        r.n_inserted = buffers['n_inserted'].ctypes.data
        r.inserted = buffers['inserted'].ctypes.data
        r.inserted_box = buffers['inserted_box'].ctypes.data
        r.status = buffers['status'].ctypes.data
        r.rounds = buffers['rounds'].ctypes.data
        _lib.check(self.lib.r3d_engine_fetch(self.handle, C.byref(r)), "fetch")
        buffers['out_bytes'] = rows * (18 if self.fetch_labels else 16) + chk * 20
        return buffers

    def outputs_on_device(self):
        """The packed outputs of the last run as CUDA tensors that alias the engine's device buffers (no copy, nothing
        crosses PCIe): ``{'xyzi': float32 [total, 4], 'labels': int32 [total], 'check': float32 [total_check, 5],
        'offsets': int64 [n + 1] (host), 'check_offsets': int64 [n + 1] (host)}``; scan s owns rows
        ``offsets[s]:offsets[s + 1]``.  Valid until the engine is re-armed, loaded or run again."""
        import torch
        n = self._n_scans
        px, pl, pc = C.c_void_p(), C.c_void_p(), C.c_void_p()
        off, coff = np.zeros(n + 1, dtype=np.int64), np.zeros(n + 1, dtype=np.int64)
        _lib.check(self.lib.r3d_engine_output_device(self.handle, C.byref(px), C.byref(pl), C.byref(pc), off.ctypes.data,
                                                     coff.ctypes.data), "output_device")
        total, total_c = int(off[n]), int(coff[n])
        return {"xyzi": _cuda_tensor(px.value, (total, 4), "<f4", torch.float32),
                "labels": _cuda_tensor(pl.value, (total,), "<i4", torch.int32),
                "check": _cuda_tensor(pc.value, (total_c, 5), "<f4", torch.float32), "offsets": off, "check_offsets": coff}

    # ------------------------------------------------------------------------------- resident dataset (online)
    def set_schedule_policy(self):
        """``insertion.random`` / ``number_of_object`` / ``number_of_classes`` of the config -> the device-side draw of
        the class counts (``generate_seed`` od/ins:171-187)."""
        ins = self.config['insertion']
        rand = bool(ins.get('random', True))
        fixed = np.zeros(_lib.R3D_MAX_CLASSES, dtype=np.int32)
        if not rand:
            fixed[:len(self.classes)] = np.asarray(ins['number_of_classes'], dtype=np.int32)
        _lib.check(self.lib.r3d_engine_set_schedule_policy(self.handle, int(rand), int(ins.get('number_of_object', 0)),
                                                           fixed.ctypes.data), "set_schedule_policy")
        self._policy_set = True

    def load_resident(self, store, indices, seed, epoch):
        """Gather the scans ``indices`` (store rows, duplicates allowed) of a device-resident store
        (``online.ResidentDataset``) as the batch and draw their schedules on the device for (``seed``, ``epoch``).  Only
        the index list crosses PCIe; a scan's draws depend on (seed, epoch, store index), not on its place in the batch."""
        if not self._policy_set:
            self.set_schedule_policy()
        idx = np.ascontiguousarray(np.asarray(indices, dtype=np.int64).astype(np.int32))
        self._keep = [store, idx]
        self._n_scans = len(idx)
        mask = (1 << 64) - 1
        _lib.check(self.lib.r3d_engine_load_resident(self.handle, C.byref(store.abi), idx.ctypes.data, len(idx),
                                                     int(seed) & mask, int(epoch) & mask), "load_resident")

    def set_ss_map_device(self, map_u8, move_x, move_y):
        """Semseg: read the sequence map from a uint8 CUDA tensor [size_x, size_y] in place (kept alive by the caller)."""
        _lib.check(self.lib.r3d_engine_set_ss_map_device(self.handle, map_u8.data_ptr(), int(map_u8.shape[0]),
                                                         int(map_u8.shape[1]), int(move_x), int(move_y)), "set_ss_map_device")

    def schedule_read(self):
        """(counts int32 [n, classes], perms int32 [n, events, classes, max_tries]) of the loaded batch, on the host."""
        n, nc = self._n_scans, len(self.classes)
        counts, ne = np.zeros((n, nc), dtype=np.int32), C.c_int32()
        _lib.check(self.lib.r3d_engine_schedule_read(self.handle, counts.ctypes.data, None, C.byref(ne)), "schedule_read")
        perms = np.zeros((n, ne.value, nc, self.max_tries), dtype=np.int32)
        _lib.check(self.lib.r3d_engine_schedule_read(self.handle, counts.ctypes.data, perms.ctypes.data, C.byref(ne)),
                   "schedule_read")
        return counts, perms

    def inserted_device(self):
        """The inserted objects of the last run as CUDA tensors aliasing the engine's buffers, enqueued on the engine
        stream: ``n_inserted`` int32 [n], ``inserted`` int32 [n, max_events, 4] (object id, rotation step, class index,
        visible points) and ``boxes`` float32 [n, max_events, 7] (x, y, z_bottom, length, width, height, yaw); rows
        past ``n_inserted`` are padding.  Valid until the engine is loaded or run again."""
        import torch
        n, e = self._n_scans, self.max_events
        pn, pi, pb, p7 = C.c_void_p(), C.c_void_p(), C.c_void_p(), C.c_void_p()
        _lib.check(self.lib.r3d_engine_inserted_device(self.handle, C.byref(pn), C.byref(pi), C.byref(pb), C.byref(p7)),
                   "inserted_device")
        return {"n_inserted": _cuda_tensor(pn.value, (n,), "<i4", torch.int32),
                "inserted": _cuda_tensor(pi.value, (n, e, 4), "<i4", torch.int32),
                "boxes": _cuda_tensor(p7.value, (n, e, 7), "<f4", torch.float32)}

    def set_world_aug(self, policy):
        """World flip / rotation / scaling of the following ``load_resident`` batches (``online.WorldAug`` or any object
        with its five fields; None turns it off).  ``load`` batches are never transformed."""
        if policy is None:
            _lib.check(self.lib.r3d_engine_set_world_aug(self.handle, None), "set_world_aug")
            return
        w = _lib.WorldAug(float(policy.flip_x_prob), float(policy.flip_y_prob), float(policy.rot_max),
                          float(policy.scale_lo), float(policy.scale_hi))
        _lib.check(self.lib.r3d_engine_set_world_aug(self.handle, C.byref(w)), "set_world_aug")

    def world_device(self):
        """float32 CUDA tensor [n, 8] (fx, fy, theta, c, s, k, 0, 0) of the loaded batch, aliasing the engine's buffer;
        raises unless the batch was loaded by ``load_resident`` with a world augmentation."""
        import torch
        p = C.c_void_p()
        _lib.check(self.lib.r3d_engine_world_device(self.handle, C.byref(p)), "world_device")
        return _cuda_tensor(p.value, (self._n_scans, 8), "<f4", torch.float32)

    def set_target_classes(self, target_classes):
        """Object detection: the target classes of ``targets_device`` (class id = 1 + position in the list).  The
        dimensions of a cut object's target box are the unpadded ``l, w, h`` of its own KITTI string."""
        if self.task != 'od':
            raise _lib.Real3DError("detection targets need an object detection engine")
        target_classes = list(target_classes)
        missing = [c for c in self.classes if c not in target_classes]
        if missing:
            raise _lib.Real3DError(f"insertion classes {missing} are not in target_classes {target_classes}")
        dims = np.zeros((max(len(self.obj_strings), 1), 3), dtype=np.float32)
        for i, s in enumerate(self.obj_strings):
            items = (s.item() if hasattr(s, 'item') else str(s)).split(' ')
            dims[i] = (float(items[10]), float(items[9]), float(items[8]))
        class_target = np.array([target_classes.index(c) + 1 for c in self.classes], dtype=np.int32)
        _lib.check(self.lib.r3d_engine_set_object_targets(self.handle, dims.ctypes.data, class_target.ctypes.data),
                   "set_object_targets")
        self.target_classes = target_classes

    def targets_device(self, store, out):
        """Enqueue the detection targets of the last run (a ``load_resident`` batch of ``store``) on the engine stream
        into ``out`` = {'gt_boxes': float32 [>= n, max_targets, 7], 'gt_classes': int32 [>= n, max_targets], 'n_gt':
        int32 [>= n]} (contiguous CUDA tensors): the scan's scene boxes, then its inserted objects, then zeros."""
        if self.task != 'od':
            raise _lib.Real3DError("targets_device: detection targets need an object detection engine")
        if getattr(self, 'target_classes', None) is None:
            raise _lib.Real3DError("targets_device: call set_target_classes first")
        box7, cls = store.scene_targets(self.target_classes)
        gb, gc, ng = out['gt_boxes'], out['gt_classes'], out['n_gt']
        n, m = self._n_scans, int(gb.shape[1])
        assert gb.is_contiguous() and gc.is_contiguous() and ng.is_contiguous()
        assert gb.shape[0] >= n and gb.shape[2] == 7 and tuple(gc.shape[1:]) == (m,) and gc.shape[0] >= n and ng.shape[0] >= n
        ptr = lambda t: t.data_ptr() if t.numel() else None
        _lib.check(self.lib.r3d_engine_targets_device(self.handle, C.byref(store.abi), ptr(box7), ptr(cls), m,
                                                      gb.data_ptr(), gc.data_ptr(), ng.data_ptr()), "targets_device")

    def target_points_device(self, out, min_points, point_gt):
        """Enqueue on the engine stream, for the targets ``targets_device`` wrote into ``out`` for the last run:
        ``out['gt_points']`` (int32 [>= n, max_targets]) = output rows of the scan inside each target, and ``point_gt``
        (int32 CUDA tensor with one entry per output row at least) = index of the first target of the row's scan that
        contains the row, or -1 (inside test: include/real3d_b200.h, ``oracle.target_points``).  Targets
        with fewer than ``min_points`` points are then dropped from ``out`` in place, order kept, and ``point_gt``
        refers to the kept rows; 0 drops nothing."""
        gb, gc, ng, gp = out['gt_boxes'], out['gt_classes'], out['n_gt'], out['gt_points']
        m = int(gb.shape[1])
        assert all(t.is_contiguous() for t in (gb, gc, ng, gp, point_gt))
        assert tuple(gp.shape[1:]) == (m,) and gp.shape[0] >= self._n_scans
        _lib.check(self.lib.r3d_engine_target_points_device(self.handle, m, gb.data_ptr(), gc.data_ptr(), ng.data_ptr(),
                                                            int(min_points), gp.data_ptr(), point_gt.data_ptr()),
                   "target_points_device")

    def unpack(self, buffers, raise_on_error=True):
        """Per-scan output records in the reference's formats."""
        out = []
        ss = self.task == 'ss'
        n_ins = [int(v) for v in buffers['n_inserted'][:self._n_scans]]
        placed = [(s, j) for s in range(self._n_scans) for j in range(n_ins[s])]
        all_boxes = iter(bx.placed_box_dictionaries(                       # one scipy call for the inserted boxes of the batch
            [buffers['inserted_box'][s, j] for s, j in placed],
            [(str(c) if ss else c) for c in (self.classes[int(buffers['inserted'][s, j, 2])] for s, j in placed)], ss))
        for s in range(self._n_scans):
            st = int(buffers['status'][s])
            if st != 0 and raise_on_error:
                _lib.check(st, f"scan {s}")
            a, b = buffers['out_off'][s], buffers['out_off'][s + 1]
            ca, cb = buffers['check_off'][s], buffers['check_off'][s + 1]
            inserted, lines, boxes, visible = [], [], [], []
            for j in range(n_ins[s]):
                obj, rot, ci, nvis = (int(v) for v in buffers['inserted'][s, j])
                cls = self.classes[ci]
                box = next(all_boxes)
                inserted.append((self.obj_names[obj], rot, cls))
                boxes.append(box)
                visible.append(nvis)
                if not ss:
                    lines.append(bx.create_annotation_line(self.obj_strings[obj], box, rot * (360.0 / self.yaw_steps)))
            chk = np.array(buffers['check'][ca:cb])
            out.append(ScanResult(velodyne=np.array(buffers['xyzi'][a:b]),
                                  labels=(np.array(buffers['labels'][a:b]).view(np.uint16).astype(np.uint32) if self.fetch_labels
                                          else np.zeros(0, dtype=np.uint32)),
                                  check=chk if ss else chk[:, :4], inserted=inserted, lines=lines, boxes=boxes,
                                  visible=visible, status=st, extra={'rounds': int(buffers['rounds'][0])}))
        return out

    def augment_batch(self, scans):
        """Load, run and fetch one batch of ScanInput; returns a list of ScanResult."""
        self.load(self.stage(scans))
        self.run()
        return self.unpack(self.fetch_raw())

    def probe_places(self, scan, object_id, scene_rows9, want_points=True):
        """find_possible_places of ONE cut object against the given current scene (N' x 9 float64 working rows);
        the scan's original points / boxes / maps come from the loaded batch.  Returns (flags[K+1], boxes[K+1, 5],
        xyz [n_feasible, M, 3] or None, rotations of the feasible candidates)."""
        k1 = self.yaw_steps + 1
        rows = np.ascontiguousarray(scene_rows9, dtype=np.float64)
        flags = np.zeros(k1, dtype=np.uint8)
        boxes = np.zeros((k1, 5), dtype=np.float64)
        m = int(self._db_offsets[object_id + 1] - self._db_offsets[object_id])
        xyz = np.zeros((self.yaw_steps, m, 3), dtype=np.float64) if want_points else None
        nf = C.c_int32()
        _lib.check(self.lib.r3d_engine_probe_places(self.handle, scan, object_id, rows.ctypes.data, len(rows),
                                                    flags.ctypes.data, boxes.ctypes.data,
                                                    xyz.ctypes.data if want_points else None, self.yaw_steps,
                                                    C.byref(nf)), "probe_places")
        rots = [k for k in range(1, k1) if flags[k] == 3]
        assert len(rots) == nf.value
        return flags, boxes, (xyz[:nf.value] if want_points else None), rots

    # ------------------------------------------------------------------------------------------ profiling
    def profile(self, on=True):
        _lib.check(self.lib.r3d_engine_profile_enable(self.handle, 1 if on else 0), "profile_enable")

    def profile_read(self):
        names = C.create_string_buffer(4096)
        ms = (C.c_double * 64)()
        launches = (C.c_int64 * 64)()
        n = C.c_int()
        _lib.check(self.lib.r3d_engine_profile_read(self.handle, names, 4096, ms, launches, 64, C.byref(n)), "profile_read")
        ks = names.value.decode().split('\n')
        return {ks[i]: {'ms': ms[i], 'launches': int(launches[i])} for i in range(n.value)}

    def stats(self):
        out = np.zeros(40, dtype=np.uint64)
        _lib.check(self.lib.r3d_engine_stats_ex(self.handle, out.ctypes.data, 40), "stats")
        return {'projected_scans': int(out[0]), 'tried_objects': int(out[1]), 'masked_scans': int(out[2]),
                'patched_scans': int(out[3]), 'select_tile': int(out[4]), 'select_global': int(out[5]),
                'prefilter_survivors': int(out[6]), 'onmap_rotations': int(out[7]), 'max_steps_per_scan': int(out[8]),
                'candidate_windows': int(out[9]), 'exact_occlusion_counts': int(out[10]),
                'walker_full_reprojections': int(out[11]),
                'walker_cycles': {k: int(out[16 + i]) for i, k in enumerate(
                    ('schedule', 'update', 'setup_prefilter', 'placement', 'occlusion', 'select_insert', 'total'))},
                'walker_detail': {k: int(out[16 + 7 + i]) for i, k in enumerate(
                    ('onmap_cycles', 'level_warp_cycles', 'collide_warp_cycles', 'n_level', 'n_collide', 'apply_cycles',
                     'patch_cycles', 'closefill_cycles', 'ss_resweeps', 'ss_level_cycles'))}}

    def walk_profile(self):
        """(SM cycles each scan's walker CTA lived, cut objects it tried) for the scans of the last run."""
        n = self._n_scans
        cycles, tries = np.zeros(n, dtype=np.int64), np.zeros(n, dtype=np.int32)
        _lib.check(self.lib.r3d_engine_walk_profile(self.handle, cycles.ctypes.data, tries.ctypes.data, n), "walk_profile")
        return cycles, tries

    def surface_labels(self):
        """Semantic labels the road-level search of any class accepts (what the surface grid indexes)."""
        if self.task == 'od':
            return [int(self.config['labels']['Road'])]
        ins = self.config['insertion']
        out = set()
        for cls in self.classes:
            for v in ins['placement'][cls]:
                out.update(int(x) for x in ins['placement_labels'][v])
        return sorted(out)

    def cuda_stream(self):
        import torch
        return torch.cuda.ExternalStream(int(self.lib.r3d_engine_stream(self.handle)))

    def launch_count(self):
        return int(self.lib.r3d_launch_count())

    def debug_image(self, scan):
        out = np.zeros((self.rows, self.cols), dtype=np.float64)
        _lib.check(self.lib.r3d_engine_debug_image(self.handle, scan, out.ctypes.data), "debug_image")
        return out

    def debug_candidates(self, scan):
        k1 = self.yaw_steps + 1
        flags, level, vis = np.zeros(k1, np.uint8), np.zeros(k1, np.float64), np.zeros(k1, np.int32)
        _lib.check(self.lib.r3d_engine_debug_candidates(self.handle, scan, flags.ctypes.data, level.ctypes.data,
                                                        vis.ctypes.data), "debug_candidates")
        return flags, level, vis

    def debug_col_index(self, scan):
        """(group, off, idx, col) of the column index of scan `scan`'s original points: bucket g holds the point indices
        idx[off[g - 1]:off[g]] (off[-1] read as 0), col = every point's azimuth bin."""
        group = C.c_int32(0)
        _lib.check(self.lib.r3d_engine_debug_col_index(self.handle, scan, C.byref(group), None, None, None), "debug_col_index")
        off = np.zeros(-(-self.cols // group.value) + 1, np.int32)
        idx, col = np.zeros(self.max_points, np.int32), np.zeros(self.max_points, np.uint16)
        _lib.check(self.lib.r3d_engine_debug_col_index(self.handle, scan, C.byref(group), off.ctypes.data, idx.ctypes.data,
                                                       col.ctypes.data), "debug_col_index")
        return group.value, off, idx, col

    def close(self):
        if getattr(self, 'handle', None):
            self.lib.r3d_engine_destroy(self.handle)
            self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def scan_input_from_case(case, pose=None):
    """ScanInput from a ``synth.Case`` (used by tests, smoke and bench)."""
    return ScanInput(xyzi=np.ascontiguousarray(case.pcl5[:, :4].astype(np.float32)),
                     labels=case.pcl5[:, 4].astype(np.uint32), box_lines=list(case.box_lines),
                     counts=case.schedule.counts, perms=case.schedule.perms, maps=case.maps,
                     pose=case.pose if pose is None else pose)
