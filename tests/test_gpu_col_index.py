"""GPU tier: the column index the streaming prepass builds (col_off / col_idx, buckets of COL_GROUP adjacent image
columns) holds every original point exactly once, in the bucket of its azimuth bin, also for image widths that are not
a multiple of the group; and the slot update that reads it still gives the oracle's results at such a width."""
import numpy as np
import pytest

from pcl_augmentation_b200 import synth
from pcl_augmentation_b200.engine import scan_input_from_case
from tests.helpers import GOLDEN_SHAPE
from tests.test_gpu_engine import assert_matches_oracle, make_engine, oracle_run

pytestmark = pytest.mark.gpu


@pytest.mark.parametrize("task,seed,counts,cols", [("od", 701, [2, 1], 1440), ("od", 702, [1, 2], 1001),
                                                   ("ss", 703, [1, 1, 0, 1, 0, 1], 1953)])
def test_column_groups_hold_every_point_once(task, seed, counts, cols):
    case = synth.make_case(task, seed, shape=GOLDEN_SHAPE, counts=counts, obj_range=(4.0, 16.0))
    eng = make_engine(case, cols=cols)
    got = eng.augment_batch([scan_input_from_case(case)])[0]
    group, off, idx, col = eng.debug_col_index(0)
    eng.close()
    n0 = len(case.pcl5)
    ng = -(-cols // group)
    assert group >= 1 and len(off) == ng + 1
    assert off[ng - 1] == n0 and np.all(np.diff(off[:ng]) >= 0)
    pts = idx[:n0]
    np.testing.assert_array_equal(np.sort(pts), np.arange(n0))                  # every point exactly once
    assert col[:n0].max() < cols
    bucket = np.repeat(np.arange(ng), np.diff(np.concatenate([[0], off[:ng]])))
    np.testing.assert_array_equal(col[pts] // group, bucket)                      # in the group of its column
    ref, want = oracle_run(case, num_column=cols)
    assert_matches_oracle(case, got, ref, want)
