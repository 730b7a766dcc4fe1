"""The script part of the reference's two ``insertion.py`` (od/ins:301-630, ss/ins:290-601) on top of the batched
CUDA engine: walk a dataset in the reference's on-disk formats, augment ``batch_size`` frames at a time and write the
files the reference writes (augmented cloud, ``check`` record, annotation / label files, ``added_objects/<frame>.txt``).

What is kept from the reference's loop: the per-frame marker file that makes concurrent runs skip frames in progress
(od/ins:335-347) and is removed when nothing could be inserted (od/ins:616-620); ``generate_seed`` drawing the class
counts from ``np.random`` (od/ins:171-187) and a uniform shuffle of each class's sample list per window (od/ins:400; seeded
from ``random``, see ``_permutation_heads``) — the
draws happen here on the host, once per frame, and are handed to the engine as tables, so a seeded ``random`` /
``np.random`` gives a reproducible run; ``setting.txt``; the run-folder numbering.
"""
from __future__ import annotations

import glob
import os
import random

import numpy as np

from .engine import MAX_NUM_TRIES, Real3DEngine, ScanInput


def load_object_db(sample_path, classes, folder_of=str):
    """Cut-object database ``{class: [(name, {'pcl', 'anno'})]}`` from ``<sample_path>/<folder>/*.npz``
    (od/ins:393, 432; ss/ins:374, 413), in sorted file-name order (the order the shuffle tables index)."""
    db = {}
    for cls in classes:
        items = []
        for path in sorted(glob.glob(f'{sample_path}/{folder_of(cls)}/*.npz')):
            with np.load(path, allow_pickle=True) as z:
                items.append((os.path.basename(path).split('.')[0], {'pcl': z['pcl'], 'anno': z['anno']}))
        if not items:
            raise FileNotFoundError(f'no cut objects for class {cls!r} under {sample_path}/{folder_of(cls)}')
        db[cls] = items
    return db


def generate_seed(config):
    """Objects to insert per class (od/ins:171-187, ss/ins:171-187)."""
    ins = config['insertion']
    if ins['random']:
        seed = np.zeros(len(ins['classes']))
        for i in np.random.randint(len(ins['classes']), size=ins['number_of_object']):
            seed[i] += 1
    else:
        seed = np.array(ins['number_of_classes'])
    return seed


def _permutation_heads(n_events, list_lens, tries):
    """One uniformly shuffled order of every class's (sorted) sample list per possible window — what ``random.shuffle``
    gives the reference at od/ins:399-402 — as an int32 table [event][class][try]; only the first ``tries`` entries of a
    shuffle can be visited before the next one.  The reference draws its shuffles where the loop needs them, so its
    stream cannot be reproduced by a table drawn up front anyway; what is kept is the SOURCE: one 64-bit draw from
    ``random`` per frame seeds the generator that shuffles (a seeded ``random`` gives a reproducible run), and the
    (events x classes) shuffles of a frame cost 0.1 ms instead of the 1 ms (6 ms for the six semseg classes) of
    ``random.shuffle`` in a Python loop."""
    rng = np.random.Generator(np.random.PCG64(random.getrandbits(64)))
    perms = np.full((n_events, len(list_lens), tries), -1, dtype=np.int32)
    for c, n in enumerate(list_lens):
        k = min(tries, n)
        if k > 0:
            perms[:, c, :k] = rng.permuted(np.tile(np.arange(n, dtype=np.int32), (n_events, 1)), axis=1)[:, :k]
    return perms


def draw_schedule(config, list_lens, tries=MAX_NUM_TRIES):
    """Pre-draw one frame's randomness: the class counts (``generate_seed``, from ``np.random`` like the reference), then
    the shuffled sample orders of every possible window (``_permutation_heads``, seeded from ``random``)."""
    counts = generate_seed(config).astype(np.int64)
    return counts, _permutation_heads(int(counts.sum()) + 1, list_lens, tries)


def read_kitti_frame(dataset, idx, maps_path):
    """One KITTI frame as the engine takes it: (xyzi, labels, scene annotation lines, {'Road', 'Sidewalk'} maps)."""
    xyzi, labels, name = dataset.read_frame(idx)
    with open(f'{dataset.data_path}/label_2/{name}.txt') as f:
        box_lines = [line for line in f if len(line.strip()) > 0]                     # od/ins:133-157
    maps = {}
    for key, sub in (('Road', 'road_maps'), ('Sidewalk', 'pedestrian_area')):        # od/ins:361-362
        with np.load(f'{maps_path}/maps/{sub}/npz/{name}.npz', allow_pickle=True) as z:
            maps[key] = {'map': z['map'], 'min_x': z['min_x'], 'min_y': z['min_y']}
    return xyzi, labels, box_lines, maps


def read_semantic_kitti_frame(dataset, idx):
    """One SemanticKITTI (or Waymo adapter) frame as the engine takes it: (xyzi, labels, lidar->world pose, scene
    annotation lines)."""
    xyzi, labels, pose, anno_path, _ = dataset.read_frame(idx)
    with open(anno_path) as f:
        box_lines = [line for line in f if len(line.strip()) > 0]
    return xyzi, labels, pose, box_lines


def _marker(out_dir, name):
    return f'{out_dir}/added_objects/{name}.txt'


def _claim(out_dir, name):
    """Frame marker (od/ins:335-347).  Returns False when another run already holds it."""
    path = _marker(out_dir, name)
    if os.path.exists(path):
        return False
    open(path, 'w').close()
    return True


def _finish(dataset, out_dir, folder, name, result, yaw_step_deg=1.0):
    """Write one frame's outputs, or drop the marker when nothing was inserted (od/ins:616-620)."""
    if not result.inserted:
        os.remove(_marker(out_dir, name))
        return False
    with open(_marker(out_dir, name), 'w') as f:
        for obj_name, rot, _ in result.inserted:
            rot = rot * yaw_step_deg
            f.write(f'{obj_name} with rotation: {int(rot) if float(rot).is_integer() else rot}\n')        # od/ins:537
    dataset.save_result(result, folder, name)
    return True


def _max_points(files, bytes_per_point=16):
    return max(os.path.getsize(f) // bytes_per_point for f in files)


def _max_boxes(anno_files, n_insert):
    """Scene boxes of the fullest frame + the boxes the insertions add (the reference has no such limit)."""
    most = 0
    for path in anno_files:
        try:
            with open(path) as f:
                most = max(most, sum(1 for line in f if line.strip()))
        except OSError:
            pass
    return max(16, most + int(n_insert) + 1)


def _objects_per_frame(config):
    ins = config['insertion']
    return int(ins['number_of_object']) if ins['random'] else int(np.sum(ins['number_of_classes']))


class FrameError(RuntimeError):
    """Frames the engine could not finish (the per-scan status the reference would have raised as an exception)."""

    def __init__(self, failures):
        self.failures = failures                       # [(frame name, status)]
        super().__init__('; '.join(f'{n}: status {st}' for n, st in failures))


def _drive(batches, engine_factory, finish, log, depth, engine_cls):
    """Reader thread -> engines -> writer thread (SURVEY 8f rows 1-2: the steps either side of the path, overlapped).

    ``batches``: iterator of (names, scans); reading files, claiming the frame markers and drawing the schedules happen
    inside it, i.e. on the READER thread, in frame order (the RNG draws stay in the reference's order).
    ``finish(name, result) -> bool`` writes one frame (writer thread).  With the CUDA engine the batches stream through
    ``ScanPipeline`` (``depth`` engines: upload, compute and download of consecutive batches overlap); any other
    ``engine_cls`` (the oracle stand-in of the CPU tests) is called batch by batch between the two threads.
    A frame whose scan ends with a non-zero status is skipped (its marker removed) and reported after every other
    frame has been written; markers of frames that were claimed but never finished are removed."""
    import queue
    import threading
    from .pipeline import ScanPipeline
    read_q, write_q = queue.Queue(maxsize=max(2, depth)), queue.Queue()
    names_of, errors, failures = {}, [], []
    counts = {'written': 0, 'skipped': 0}
    end = object()

    def reader():
        try:
            for i, (names, scans) in enumerate(batches):
                names_of[i] = names
                read_q.put((i, scans))
                if errors:
                    break
        except BaseException as exc:
            errors.append(exc)
        finally:
            read_q.put(end)

    def writer():
        while True:
            item = write_q.get()
            if item is end:
                return
            names, results = item
            try:
                for name, result in zip(names, results):
                    if result.status != 0:
                        failures.append((name, result.status))
                        finish(name, None)
                        continue
                    counts['written' if finish(name, result) else 'skipped'] += 1
                    log(f'{name}: inserted {[(n, r) for n, r, _ in result.inserted]}')
            except BaseException as exc:
                errors.append(exc)

    def read_batches():
        while True:
            item = read_q.get()
            if item is end:
                return
            yield item

    rt, wt = threading.Thread(target=reader, daemon=True), threading.Thread(target=writer, daemon=True)
    rt.start(); wt.start()
    runner = None
    try:
        if engine_cls is Real3DEngine:
            runner = engine_factory(ScanPipeline, depth)
            order = []

            def staged():
                for i, scans in read_batches():
                    order.append(i)
                    yield runner.engines[0].stage(scans)          # pinned packing, on the pipeline's producer thread
            runner.process(staged(), on_result=lambda j, eng, buf: write_q.put((names_of[order[j]], eng.unpack(buf, raise_on_error=False))))
        else:
            runner = engine_factory(None, 1)
            for i, scans in read_batches():
                write_q.put((names_of[i], runner.augment_batch(scans)))
    except BaseException as exc:
        errors.append(exc)
    finally:
        while rt.is_alive():                                       # an error upstream: let the reader run out
            try:
                read_q.get(timeout=0.05)
            except queue.Empty:
                pass
        write_q.put(end)
        rt.join(); wt.join()
        if runner is not None:
            runner.close()
    if errors:
        raise errors[0]
    return counts['written'], counts['skipped'], sorted(failures)


def augment_kitti(config, batch_size=64, yaw_steps=360, folder_number=None, engine_kwargs=None, log=print,
                  engine_cls=Real3DEngine, depth=3):
    """object_detection/Real3DAug/insertion.py ``__main__`` (od/ins:301-630) for the whole ``train.txt`` list.
    Returns (save folder, frames written, frames without an insertion)."""
    from .object_detection.Real3DAug.tools.datasets import KITTI
    dataset = KITTI(config)
    save_folder, _ = dataset.create_directories('random' if config['insertion']['random'] else 'chosen', folder_number)
    out_dir = f"{config['path']['output_path']}/{save_folder}"
    classes = config['insertion']['classes']
    db = load_object_db(config['path']['sample_path'], classes)
    list_lens = [len(db[c]) for c in classes]
    maps_path = config['path']['maps_path']
    files = list(dataset.velodyne_list)
    if not files:
        return save_folder, 0, 0
    kw = dict(max_scans=min(batch_size, len(files)), max_points=_max_points(files), yaw_steps=yaw_steps,
              max_boxes=_max_boxes([f'{dataset.data_path}/label_2/{dataset.frame_name(f)}.txt' for f in files],
                                   _objects_per_frame(config)))
    kw.update(engine_kwargs or {})
    claimed, done = set(), set()

    def batches():
        for i0 in range(0, len(files), batch_size):
            scans, names = [], []
            for idx in range(i0, min(i0 + batch_size, len(files))):
                name = dataset.frame_name(files[idx])
                if not _claim(out_dir, name):
                    log(f'{name}: already in progress')
                    continue
                claimed.add(name)
                xyzi, labels, box_lines, maps = read_kitti_frame(dataset, idx, maps_path)
                counts, perms = draw_schedule(config, list_lens)
                scans.append(ScanInput(xyzi=xyzi, labels=labels, box_lines=box_lines, counts=counts, perms=perms, maps=maps))
                names.append(name)
            if scans:
                yield names, scans

    def finish(name, result):
        done.add(name)
        if result is None:                                   # failed scan: give the frame back
            os.remove(_marker(out_dir, name))
            return False
        return _finish(dataset, out_dir, save_folder, name, result, 360.0 / yaw_steps)

    def factory(pipeline_cls, n):
        if pipeline_cls is None:
            return engine_cls('od', config, db, **kw)
        return pipeline_cls('od', config, db, depth=n, **kw)

    try:
        written, skipped, failures = _drive(batches(), factory, finish, log, depth, engine_cls)
    finally:
        for name in claimed - done:                          # claimed but never finished: do not block later runs
            if os.path.exists(_marker(out_dir, name)) and os.path.getsize(_marker(out_dir, name)) == 0:
                os.remove(_marker(out_dir, name))
    if failures:
        raise FrameError(failures)
    return save_folder, written, skipped


def augment_semantic_kitti(config, sequence, batch_size=64, yaw_steps=360, folder_number=None, reverse=False,
                           skip_scenes=0, engine_kwargs=None, log=print, dataset=None, engine_cls=Real3DEngine, depth=3):
    """semantic_segmentation/Real3DAug/insertion.py ``__main__`` (ss/ins:290-601) for one sequence (SemanticKITTI, or
    a prepared ``Waymo`` adapter through ``dataset``: only the frames of ``sequence`` are taken, the reference reloads
    the map and the save folder when the sequence changes, ss/ins:317-323).  Returns (save folder of the sequence,
    written, skipped)."""
    from .semantic_segmentation.Real3DAug.tools.datasets import SemanticKITTI
    if dataset is None:
        dataset = SemanticKITTI(config, sequence, reverse=reverse, skip_scenes=skip_scenes)
    save_folder, _ = dataset.create_directories('random' if config['insertion']['random'] else 'chosen', folder_number)
    save_folder = f'{save_folder}/{sequence}'                                                    # ss/ins:306
    out_dir = f"{config['path']['output_path']}/{save_folder}"
    classes = config['insertion']['classes']
    db = load_object_db(config['path']['bbox_path'], classes, folder_of=lambda c: config['labels'][c])
    list_lens = [len(db[c]) for c in classes]
    with np.load(f"{config['path']['maps_path']}/{sequence}.npz", allow_pickle=True) as z:      # ss/ins:312-313
        map_data = {'map': z['map'], 'move': z['move']}
    all_files = list(dataset.velodyne_list)
    # adapters that span several sequences (Waymo): one call = one sequence = one rich map / save folder
    multi = bool(getattr(dataset, 'sequence_names', None))
    indices = [i for i, f in enumerate(all_files) if not multi or f.split('/')[-3] == str(sequence)]
    files = [all_files[i] for i in indices]
    if not files:
        return save_folder, 0, 0
    if multi:
        dataset.create_subdirectories(sequence)
    per_point = 16 if files[0].endswith('.bin') else 24
    anno_dir = os.path.dirname(dataset.read_frame(indices[0])[3])
    kw = dict(max_scans=min(batch_size, len(files)), max_points=_max_points(files, per_point), yaw_steps=yaw_steps,
              map_data=map_data,
              max_boxes=_max_boxes([f'{anno_dir}/{dataset.frame_name(f)}.txt' for f in files], _objects_per_frame(config)))
    kw.update(engine_kwargs or {})
    claimed, done = set(), set()

    def batches():
        for i0 in range(0, len(files), batch_size):
            scans, names = [], []
            for k in range(i0, min(i0 + batch_size, len(files))):
                name = dataset.frame_name(files[k])
                if not _claim(out_dir, name):
                    log(f'{sequence}/{name}: already in progress')
                    continue
                claimed.add(name)
                xyzi, labels, pose, box_lines = read_semantic_kitti_frame(dataset, indices[k])
                counts, perms = draw_schedule(config, list_lens)
                scans.append(ScanInput(xyzi=xyzi, labels=labels, box_lines=box_lines, counts=counts, perms=perms, pose=pose))
                names.append(name)
            if scans:
                yield names, scans

    def finish(name, result):
        done.add(name)
        if result is None:
            os.remove(_marker(out_dir, name))
            return False
        return _finish(dataset, out_dir, save_folder, name, result, 360.0 / yaw_steps)

    def factory(pipeline_cls, n):
        if pipeline_cls is None:
            return engine_cls('ss', config, db, **kw)
        return pipeline_cls('ss', config, db, depth=n, **kw)

    try:
        written, skipped, failures = _drive(batches(), factory, finish, lambda m: log(f'{sequence}/{m}'), depth, engine_cls)
    finally:
        for name in claimed - done:
            if os.path.exists(_marker(out_dir, name)) and os.path.getsize(_marker(out_dir, name)) == 0:
                os.remove(_marker(out_dir, name))
    if failures:
        raise FrameError(failures)
    return save_folder, written, skipped
