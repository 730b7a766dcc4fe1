"""Online augmentation inside a training process: the dataset stays in device memory, every epoch draws fresh
schedules on the device, and the augmented clouds and inserted boxes come back as CUDA tensors.

``ResidentDataset`` lays the scans out once in the layout of ``r3d_resident_store`` (include/real3d_b200.h): packed
float4 xyzi + 16-bit labels, the scene boxes as 16-double records, OD maps or semseg poses.  ``OnlineAugmenter`` gathers a
batch from it by index (``r3d_engine_load_resident``: the index list is the only host -> device copy), runs the engine
and hands out an ``AugmentedBatch``.  A scan's draws are keyed by (seed, epoch, store index), so they do not depend on
the batch it lands in or on the rank that owns it; they are their own random stream, not the reference's Python
``random`` / ``np.random`` stream.
"""
from __future__ import annotations

import collections
import math
import os
from dataclasses import dataclass

import numpy as np

from . import _lib
from . import boxes as bx
from .engine import Real3DEngine
from .sharding import shard_indices


def epoch_batches(n_scans, batch_size, *, rank=0, world=1, seed=0, epoch=0, shuffle=True, groups=None):
    """This rank's shard of the store (``sharding.shard_indices``) cut into batches of at most ``batch_size`` scans for
    one epoch.  ``shuffle``: the order of the scans and of the batches is a permutation drawn from (seed, epoch, rank).
    ``groups`` (one id per store scan, e.g. the semseg sequence): a batch never mixes groups."""
    assert batch_size >= 1
    idx = np.asarray(shard_indices(n_scans, rank, world), dtype=np.int64)
    rng = np.random.default_rng([int(seed) & ((1 << 64) - 1), int(epoch), int(rank)]) if shuffle else None
    if rng is not None:
        idx = rng.permutation(idx)
    keys = np.zeros(len(idx), dtype=np.int64) if groups is None else np.asarray(groups, dtype=np.int64)[idx]
    out = []
    for g in (np.unique(keys) if len(keys) else []):
        members = idx[keys == g]
        out += [members[i:i + batch_size] for i in range(0, len(members), batch_size)]
    if rng is not None:
        out = [out[i] for i in rng.permutation(len(out))]
    return out


class ResidentDataset:
    """Scans laid out in device memory (one upload when the dataset is built; ``r3d_resident_store`` layout).
    Semseg: one map per sequence on the device and a sequence id per scan."""

    def __init__(self, task, sizes, frames, seq_maps=None, sequence_ids=None, names=None):
        """``sizes``: points per scan; ``frames``: iterable of (xyzi, labels, box_lines, maps (OD) or pose (semseg)).
        ``seq_maps``: semseg {sequence id: {'map', 'move'}}; ``sequence_ids``: the sequence id of each scan."""
        torch = _lib.require_cuda()
        dev = torch.device("cuda", torch.cuda.current_device())
        self.task = task
        n = len(sizes)
        assert n > 0
        self.n_scans = n
        self.names = list(names) if names is not None else [str(i) for i in range(n)]
        self.h_point_offsets = np.zeros(n + 1, dtype=np.int64)
        self.h_point_offsets[1:] = np.cumsum(np.asarray(sizes, dtype=np.int64))
        total = int(self.h_point_offsets[-1])
        self.xyzi = torch.empty((total, 4), dtype=torch.float32, device=dev)
        self.labels = torch.empty(total, dtype=torch.int16, device=dev)          # uint16 bits
        lines, nboxes, blobs, map_off, dims, poses = [], [], [], [0], np.zeros((n, 2, 4), dtype=np.int32), []
        for i, (xyzi, labels, box_lines, extra) in enumerate(frames):
            a, b = int(self.h_point_offsets[i]), int(self.h_point_offsets[i + 1])
            assert len(xyzi) == b - a, f"scan {i}: {len(xyzi)} points, {b - a} announced"
            lab = np.asarray(labels)
            assert lab.size == 0 or int(lab.max()) < 65536, "semantic labels must be masked with 0xFFFF (od/ds:65)"
            self.xyzi[a:b].copy_(torch.from_numpy(np.ascontiguousarray(xyzi, dtype=np.float32)))
            self.labels[a:b].copy_(torch.from_numpy(lab.astype(np.uint16).view(np.int16)))
            lines += list(box_lines)
            nboxes.append(len(box_lines))
            if task == 'od':
                for j, key in enumerate(('Road', 'Sidewalk')):
                    m = np.ascontiguousarray(np.asarray(extra[key]['map']).astype(np.uint8))
                    blobs.append(torch.from_numpy(m.reshape(-1)))
                    map_off.append(map_off[-1] + m.size)
                    dims[i, j] = (m.shape[0], m.shape[1], int(extra[key]['min_x']), int(extra[key]['min_y']))
            else:
                poses.append(np.asarray(extra, dtype=np.float64).reshape(16))
        assert len(nboxes) == n, "fewer frames than sizes"
        self.h_box_offsets = np.zeros(n + 1, dtype=np.int32)
        self.h_box_offsets[1:] = np.cumsum(nboxes)
        # every annotation line through scipy's matrix <-> quaternion conversions in one call (Real3DEngine.stage does
        # the same per batch)
        recs = bx.box_records_from_lines(lines, ss=task == 'ss') if lines else np.zeros((0, 16))
        self.boxes = torch.from_numpy(np.ascontiguousarray(recs, dtype=np.float64).reshape(-1, 16)).to(dev)
        # OD: every scene box as a detection target record (bx.scene_targets_od) and the id of its name in box_names,
        # 1:1 with the box records; the class ids of a target_classes list are derived from them on the device
        self.box_names, self._scene_targets = [], {}
        if task == 'od':
            t7, names = bx.scene_targets_od(lines)
            self.box_names = sorted(set(names))
            self.h_box_name_ids = np.array([self.box_names.index(n) for n in names], dtype=np.int32)
            self.scene_box7 = torch.from_numpy(np.ascontiguousarray(t7.astype(np.float32)).reshape(-1, 7)).to(dev)
            self.box_name_ids = torch.from_numpy(self.h_box_name_ids).to(dev)
        self.point_offsets = torch.from_numpy(self.h_point_offsets).to(dev)
        self.box_offsets = torch.from_numpy(self.h_box_offsets).to(dev)
        self.max_points = int(np.diff(self.h_point_offsets).max())
        self.max_boxes = int(np.diff(self.h_box_offsets).max())
        self.maps = self.map_offsets = self.map_dims = self.poses = None
        self.seq_maps, self.sequence_ids = {}, None
        if task == 'od':
            self.maps = torch.cat(blobs).to(dev)
            self.map_offsets = torch.tensor(map_off, dtype=torch.int64, device=dev)
            self.map_dims = torch.from_numpy(dims).to(dev)
        else:
            self.poses = torch.from_numpy(np.stack(poses)).to(dev)
            self.sequence_ids = np.zeros(n, dtype=np.int64) if sequence_ids is None else np.asarray(sequence_ids, dtype=np.int64)
            assert len(self.sequence_ids) == n
            for sid, md in (seq_maps or {}).items():
                mv = np.asarray(md['move']).reshape(-1)
                m = np.ascontiguousarray(np.asarray(md['map']).astype(np.uint8))
                self.seq_maps[int(sid)] = (torch.from_numpy(m).to(dev), int(mv[0]), int(mv[1]))
            missing = set(self.sequence_ids.tolist()) - set(self.seq_maps)
            assert not missing, f"no rich map for sequences {sorted(missing)}"
        ptr = lambda t: t.data_ptr() if t is not None and t.numel() else None
        s = _lib.ResidentStore()
        s.n_scans = n
        s.xyzi, s.labels, s.point_offsets = ptr(self.xyzi), ptr(self.labels), ptr(self.point_offsets)
        s.boxes, s.box_offsets = ptr(self.boxes), ptr(self.box_offsets)
        s.maps, s.map_offsets, s.map_dims, s.poses = ptr(self.maps), ptr(self.map_offsets), ptr(self.map_dims), ptr(self.poses)
        s.h_point_offsets, s.h_box_offsets = self.h_point_offsets.ctypes.data, self.h_box_offsets.ctypes.data
        self.abi = s

    def __len__(self):
        return self.n_scans

    def scene_targets(self, target_classes):
        """(scene_box7 float32 [boxes, 7], class ids int32 [boxes]) on the device for ``target_classes``: 1-based
        position of the box's name in the list, 0 for a box that is not a target.  Mapped once per list."""
        if self.task != 'od':
            raise _lib.Real3DError("detection targets need an object detection store")
        key = tuple(target_classes)
        if key not in self._scene_targets:
            torch = _lib.require_cuda()
            lut = np.array([key.index(n) + 1 if n in key else 0 for n in self.box_names] or [0], dtype=np.int32)
            ids = torch.from_numpy(lut).to(self.box_name_ids.device)[self.box_name_ids.long()].to(torch.int32).contiguous()
            torch.cuda.current_stream().synchronize()        # the engine reads the ids back once, outside this stream
            is_target = (lut[self.h_box_name_ids] > 0).astype(np.int64)
            kept = np.cumsum(np.concatenate([[0], is_target]))[self.h_box_offsets]
            self._scene_targets[key] = (self.scene_box7, ids, int(np.diff(kept).max()))
        return self._scene_targets[key][:2]

    def max_kept_boxes(self, target_classes):
        """The most scene boxes of one scan that are ``target_classes`` targets."""
        self.scene_targets(target_classes)
        return self._scene_targets[tuple(target_classes)][2]

    @classmethod
    def from_scans(cls, task, scans, map_data=None):
        """From ``engine.ScanInput`` records (annotation lines; their schedules are not used).  Semseg: ``map_data``
        ({'map', 'move'}) is the map of the one sequence every scan belongs to."""
        assert all(s.box_dicts is None for s in scans), "the store takes annotation lines (box_lines)"
        frames = ((s.xyzi, s.labels, s.box_lines, s.maps if task == 'od' else s.pose) for s in scans)
        return cls(task, [len(s.xyzi) for s in scans], frames, seq_maps={0: map_data} if task == 'ss' else None)

    @classmethod
    def from_kitti(cls, config):
        """Every frame of KITTI's ``train.txt`` list, read as ``dataset_driver.augment_kitti`` reads it."""
        from .dataset_driver import read_kitti_frame
        from .object_detection.Real3DAug.tools.datasets import KITTI
        dataset = KITTI(config)
        files = list(dataset.velodyne_list)
        frames = ((x, l, b, m) for x, l, b, m in (read_kitti_frame(dataset, i, config['path']['maps_path'])
                                                  for i in range(len(files))))
        return cls('od', [os.path.getsize(f) // 16 for f in files], frames, names=[dataset.frame_name(f) for f in files])

    @classmethod
    def from_semantic_kitti(cls, config, sequences):
        """Every frame of the given SemanticKITTI sequences, read as ``dataset_driver.augment_semantic_kitti`` reads
        them, with one rich map per sequence (``<maps_path>/<sequence>.npz``)."""
        from .dataset_driver import read_semantic_kitti_frame
        from .semantic_segmentation.Real3DAug.tools.datasets import SemanticKITTI
        sizes, seq_ids, names, seq_maps, readers = [], [], [], {}, []
        for sid, seq in enumerate(sequences):
            dataset = SemanticKITTI(config, seq)
            files = list(dataset.velodyne_list)
            sizes += [os.path.getsize(f) // 16 for f in files]
            seq_ids += [sid] * len(files)
            names += [f'{seq}/{dataset.frame_name(f)}' for f in files]
            with np.load(f"{config['path']['maps_path']}/{seq}.npz", allow_pickle=True) as z:
                seq_maps[sid] = {'map': z['map'], 'move': z['move']}
            readers += [(dataset, i) for i in range(len(files))]
        frames = ((x, l, b, p) for x, l, p, b in (read_semantic_kitti_frame(d, i) for d, i in readers))
        ds = cls('ss', sizes, frames, seq_maps=seq_maps, sequence_ids=seq_ids, names=names)
        ds.sequences = list(sequences)
        return ds


@dataclass
class WorldAug:
    """Per-scan world augmentation after the insertion (OpenPCDet's ``random_world_flip`` / ``random_world_rotation`` /
    ``random_world_scaling``; defaults of its KITTI configs): flip along x (y -> -y) with ``flip_x_prob``, along y
    (x -> -x) with ``flip_y_prob``, rotate about z by a uniform angle in [-rot_max, rot_max], scale by a uniform factor
    in [scale_lo, scale_hi], in that order, to the points and the boxes together.  The exact arithmetic is that of
    ``r3d_world_aug`` in include/real3d_b200.h."""
    flip_x_prob: float = 0.5
    flip_y_prob: float = 0.0
    rot_max: float = math.pi / 4
    scale_lo: float = 0.95
    scale_hi: float = 1.05

    def __post_init__(self):
        vals = (self.flip_x_prob, self.flip_y_prob, self.rot_max, self.scale_lo, self.scale_hi)
        if not all(math.isfinite(float(v)) for v in vals):
            raise ValueError(f"WorldAug: non-finite value in {self}")
        if not (0.0 <= self.flip_x_prob <= 1.0 and 0.0 <= self.flip_y_prob <= 1.0):
            raise ValueError("WorldAug: flip probabilities must be in [0, 1]")
        if not 0.0 <= self.rot_max <= math.pi:
            raise ValueError("WorldAug: rot_max must be in [0, pi]")
        if not 0.0 < self.scale_lo <= self.scale_hi:
            raise ValueError("WorldAug: need 0 < scale_lo <= scale_hi")


@dataclass
class AugmentedBatch:
    """One augmented batch as CUDA tensors that alias the engine's buffers (valid until the engine that made it is
    loaded again, ``depth`` batches later).  Scan s owns rows ``offsets[s]:offsets[s + 1]`` of xyzi / labels and
    objects ``[s, :n_inserted[s]]`` of the per-object tensors (the rest is padding)."""
    xyzi: object              # float32 [total, 4]: the augmented clouds (velodyne rows)
    labels: object            # int32 [total]: semantic labels (OD: {Road, other} as the engine sees them)
    offsets: np.ndarray       # int64 [n + 1], host
    check: object             # float32 [total_check, 5]: the visible points of the inserted objects (check record)
    check_offsets: np.ndarray # int64 [n + 1], host
    n_inserted: object        # int32 [n]
    object_id: object         # int32 [n, max_events]: index into the cut-object database (engine.obj_names)
    class_index: object       # int32 [n, max_events]
    rotation: object          # int32 [n, max_events]: yaw step of the placement
    visible: object           # int32 [n, max_events]: visible points of the inserted object
    boxes: object             # float32 [n, max_events, 7]: x, y, z_bottom, length, width, height, yaw (lidar frame):
                              # the inserted objects in the engine's collision-box convention, before the world transform
    indices: np.ndarray       # int64 [n], host: the store scans of the batch
    # with target_classes: every ground-truth box of the augmented scan (scene boxes in file order, then the inserted
    # objects), OpenPCDet gt_boxes layout x, y, z_center, dx, dy, dz, heading, after the world transform
    gt_boxes: object = None   # float32 [n, max_targets, 7]; rows past n_gt are zero
    gt_classes: object = None # int32 [n, max_targets]: 1-based into target_classes, 0 = padding
    n_gt: object = None       # int32 [n]
    world: object = None      # float32 [n, 8]: with world_aug, (fx, fy, theta, c, s, k, 0, 0) of each scan


class OnlineAugmenter:
    """Real3D-Aug inside a training loop on data that stays on the GPU.  ``depth`` engines are used in turn, so that
    batch k + 1 is augmented while the consumer still works on batch k."""

    def __init__(self, task, config, db, dataset, *, batch_size, seed, yaw_steps=360, depth=2, rank=0, world=1,
                 target_classes=None, world_aug=None, **engine_kwargs):
        """``target_classes`` (object detection): the class names of ``gt_boxes`` / ``gt_classes``; every insertion
        class must be one of them.  ``world_aug``: a ``WorldAug`` applied to every batch (None: off)."""
        torch = _lib.require_cuda()
        from .dataset_driver import _objects_per_frame
        assert dataset.task == task and depth >= 1
        self.task, self.dataset, self.batch_size, self.seed = task, dataset, int(batch_size), int(seed)
        self.rank, self.world, self.depth = rank, world, depth
        kw = dict(max_scans=self.batch_size, max_points=dataset.max_points, yaw_steps=yaw_steps,
                  max_boxes=max(16, dataset.max_boxes + _objects_per_frame(config) + 1))
        if task == 'ss':                  # a starting map; set_ss_map_device switches sequences between batches
            m, mx, my = next(iter(dataset.seq_maps.values()))
            kw['map_data'] = {'map': m.cpu().numpy(), 'move': np.array([mx, my])}
        kw.update(engine_kwargs)
        self.engines = [Real3DEngine(task, config, db, **kw) for _ in range(depth)]
        self.max_events = self.engines[0].max_events
        self._streams = [e.cuda_stream() for e in self.engines]
        self._seq = [None] * depth
        self._next = 0
        self._pending = collections.deque()
        self._torch = torch
        self.world_aug = world_aug
        for e in self.engines:
            e.set_world_aug(world_aug)
        self.target_classes = None if target_classes is None else list(target_classes)
        self._targets = []
        if self.target_classes is not None:
            if task != 'od':
                raise _lib.Real3DError("detection targets need an object detection dataset")
            self.max_targets = dataset.max_kept_boxes(self.target_classes) + self.max_events - 1
            dev = dataset.xyzi.device
            for e in self.engines:             # each slot owns the buffers of the batch its engine holds
                e.set_target_classes(self.target_classes)
                self._targets.append({'gt_boxes': torch.zeros((self.batch_size, self.max_targets, 7), dtype=torch.float32, device=dev),
                                      'gt_classes': torch.zeros((self.batch_size, self.max_targets), dtype=torch.int32, device=dev),
                                      'n_gt': torch.zeros(self.batch_size, dtype=torch.int32, device=dev)})

    def _submit(self, indices, epoch):
        torch = self._torch
        slot = self._next % self.depth
        self._next += 1
        eng = self.engines[slot]
        idx = np.asarray(indices, dtype=np.int64)
        # the engine's buffers still back the batch it made last: reload only after the work the consumer has
        # queued so far (which includes every use of that batch) is done
        consumed = torch.cuda.Event()
        consumed.record(torch.cuda.current_stream())
        self._streams[slot].wait_event(consumed)
        if self.task == 'ss':
            seqs = np.unique(self.dataset.sequence_ids[idx]) if len(idx) else []
            if len(seqs) != 1:
                raise _lib.Real3DError(f"a semseg batch must come from one sequence, got {list(seqs)}")
            if self._seq[slot] != int(seqs[0]):
                m, mx, my = self.dataset.seq_maps[int(seqs[0])]
                eng.set_ss_map_device(m, mx, my)
                self._seq[slot] = int(seqs[0])
        eng.load_resident(self.dataset, idx, self.seed, epoch)
        eng.run()
        self._pending.append((slot, idx))

    def _collect(self):
        torch = self._torch
        slot, idx = self._pending.popleft()
        eng = self.engines[slot]
        out = eng.outputs_on_device()                # waits for the run: the one host synchronisation of a batch
        ins = eng.inserted_device()
        extra = {}
        if self.target_classes is not None:
            tg = self._targets[slot]
            eng.targets_device(self.dataset, tg)
            n = len(idx)
            extra.update(gt_boxes=tg['gt_boxes'][:n], gt_classes=tg['gt_classes'][:n], n_gt=tg['n_gt'][:n])
        if self.world_aug is not None:
            extra['world'] = eng.world_device()
        ready = torch.cuda.Event()
        ready.record(self._streams[slot])
        torch.cuda.current_stream().wait_event(ready)
        t = ins['inserted']
        return AugmentedBatch(xyzi=out['xyzi'], labels=out['labels'], offsets=out['offsets'], check=out['check'],
                              check_offsets=out['check_offsets'], n_inserted=ins['n_inserted'], object_id=t[..., 0],
                              rotation=t[..., 1], class_index=t[..., 2], visible=t[..., 3], boxes=ins['boxes'], indices=idx,
                              **extra)

    def augment(self, indices, epoch):
        """Augment the store scans ``indices`` (at most ``batch_size``; duplicates allowed) with the draws of
        ``epoch``.  The current torch stream is made to wait for the result."""
        assert not self._pending, "augment() called while an epoch() iteration has batches in flight"
        self._submit(indices, epoch)
        return self._collect()

    def epoch(self, epoch, shuffle=True):
        """Iterate over this rank's shard in an order shuffled per epoch; ``depth - 1`` batches are augmented ahead
        of the one handed out.  Semseg batches never mix sequences."""
        for _, batch in self.epochs([epoch], shuffle):
            yield batch

    def epochs(self, epochs, shuffle=True):
        """``epoch`` for several epochs in a row, yielding (epoch, batch): the batches of the next epoch are augmented
        ahead as well, so the device does not wait for the pipeline to refill at each epoch boundary."""
        order = [(e, b) for e in epochs
                 for b in epoch_batches(self.dataset.n_scans, self.batch_size, rank=self.rank, world=self.world,
                                        seed=self.seed, epoch=e, shuffle=shuffle, groups=self.dataset.sequence_ids)]
        ahead = self.depth - 1
        try:
            for k in range(min(ahead, len(order))):
                self._submit(order[k][1], order[k][0])
            for k in range(len(order)):
                if k + ahead < len(order):
                    self._submit(order[k + ahead][1], order[k + ahead][0])
                yield order[k][0], self._collect()
        finally:
            self._pending.clear()

    def close(self):
        for e in self.engines:
            e.close()
