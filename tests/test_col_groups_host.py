"""CPU tier: the arithmetic of the column index by groups of COL_GROUP adjacent image columns (csrc/r3d_engine.cuh
col_groups, the slot update's visit in csrc/r3d_k_update_project.cuh apply_vis_mask).  For every column range [c0, c1]
of an image, the visited groups c0 // G .. c1 // G cover the range, stay inside the image's ceil(cols / G) groups and add
at most 2 (G - 1) columns."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def default_group():
    text = open(os.path.join(ROOT, "pcl_augmentation_b200", "csrc", "r3d_engine.cuh")).read()
    return int(re.search(r"#define R3D_COL_GROUP (\d+)", text).group(1))


GROUPS = sorted({1, 4, 8, 16, 32, default_group()})
WIDTHS = [1440, 2048, 1953, 1, 7, 33, 601, 1023]        # 1953: synth.SEMKITTI_SHAPE; odd widths are legal


def col_groups(cols, g):
    return (cols + g - 1) // g


@pytest.mark.parametrize("g", GROUPS)
@pytest.mark.parametrize("cols", WIDTHS)
def test_visited_groups_cover_every_column_range(cols, g):
    ng = col_groups(cols, g)
    c0, c1 = np.meshgrid(np.arange(cols), np.arange(cols), indexing="ij")
    keep = c1 >= c0
    c0, c1 = c0[keep], c1[keep]
    g0, g1 = c0 // g, c1 // g
    assert g1.max() < ng                                             # the last (partial) group exists
    first, last = g0 * g, np.minimum((g1 + 1) * g, cols) - 1         # columns the visited groups hold
    assert np.all(first <= c0) and np.all(last >= c1)
    extra = (last - first + 1) - (c1 - c0 + 1)
    assert extra.min() >= 0 and extra.max() <= 2 * (g - 1)


@pytest.mark.parametrize("g", GROUPS)
@pytest.mark.parametrize("cols", WIDTHS)
def test_group_buckets_hold_each_point_once(cols, g):
    # the CSR the prepass builds: counts per group, exclusive scan, scatter; then off[k] = END of group k's bucket
    rng = np.random.default_rng(cols * 64 + g)
    col = rng.integers(0, cols, size=5000)
    ng = col_groups(cols, g)
    off = np.cumsum(np.bincount(col // g, minlength=ng + 1))
    assert off.shape == (ng + 1,) and off[ng - 1] == len(col)
    idx = np.argsort(col // g, kind="stable")
    for c0, c1 in [(0, cols - 1), (cols // 3, cols // 2), (cols - 1, cols - 1)]:
        g0, g1 = c0 // g, c1 // g
        visited = idx[(off[g0 - 1] if g0 > 0 else 0):off[g1]]
        assert len(np.unique(visited)) == len(visited)
        want = np.flatnonzero((col >= c0) & (col <= c1))
        assert np.all(np.isin(want, visited))                        # every point of the range is visited
        assert np.all(col[visited] // g >= g0) and np.all(col[visited] // g <= g1)
