"""CPU tier: the batching / sharding / shuffling of the online augmenter's epochs (online.epoch_batches)."""
import numpy as np

from pcl_augmentation_b200.online import epoch_batches
from pcl_augmentation_b200.sharding import shard_indices


def test_every_scan_of_the_shard_once_per_epoch():
    for world in (1, 3):
        for rank in range(world):
            batches = epoch_batches(50, 8, rank=rank, world=world, seed=7, epoch=2)
            got = np.concatenate(batches)
            assert sorted(got.tolist()) == shard_indices(50, rank, world)
            assert all(1 <= len(b) <= 8 for b in batches)


def test_shuffle_depends_on_seed_and_epoch_only():
    a = epoch_batches(40, 16, seed=3, epoch=1)
    b = epoch_batches(40, 16, seed=3, epoch=1)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    flat = lambda bs: np.concatenate(bs).tolist()
    assert flat(epoch_batches(40, 16, seed=3, epoch=2)) != flat(a)
    assert flat(epoch_batches(40, 16, seed=4, epoch=1)) != flat(a)


def test_no_shuffle_keeps_the_shard_order():
    batches = epoch_batches(10, 4, rank=1, world=2, shuffle=False)
    assert [b.tolist() for b in batches] == [[1, 3, 5, 7], [9]]


def test_batches_never_mix_groups():
    groups = np.repeat([0, 1, 2], [7, 12, 5])
    for epoch in range(4):
        batches = epoch_batches(len(groups), 4, rank=0, world=2, seed=1, epoch=epoch, groups=groups)
        assert sorted(np.concatenate(batches).tolist()) == shard_indices(len(groups), 0, 2)
        for b in batches:
            assert len(np.unique(groups[b])) == 1
