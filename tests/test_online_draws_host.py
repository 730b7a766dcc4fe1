"""CPU tier: the host restatement of the online draws (oracle/online_draws.py) that tests/test_gpu_online_draws.py
holds the device to: Philox4x32-10 against the Random123 known answers, Lemire's bounded integers exactly unbiased,
the array Fisher-Yates shuffle exactly uniform, and the vectorised reference equal to the word-by-word one."""
import itertools
import math

import numpy as np
import pytest

from oracle import online_draws as od


@pytest.mark.parametrize("ctr,key,want", [
    ((0, 0, 0, 0), (0, 0), (0x6627e8d5, 0xe169c58d, 0xbc57ac4c, 0x9b00dbd8)),
    ((0xffffffff,) * 4, (0xffffffff, 0xffffffff), (0x408f276d, 0x41c83b0e, 0xa20bc7c6, 0x6d5451fd)),
    ((0x243f6a88, 0x85a308d3, 0x13198a2e, 0x03707344), (0xa4093822, 0x299f31d0),
     (0xd16cfe09, 0x94fdcceb, 0x5001e420, 0x24126ea1)),
])
def test_philox_known_answers(ctr, key, want):
    assert tuple(int(w) for w in od.philox4x32_10(ctr, key)) == want
    # vectorised: the same counter in a batch of others gives the same words
    c0 = np.array([ctr[0], 1, 2], dtype=np.uint64)
    got = od.philox4x32_10((c0, ctr[1], ctr[2], ctr[3]), key)
    assert tuple(int(w[0]) for w in got) == want


def test_key_and_counter_words():
    assert od.key_of(2**64 - 1, 2**32 + 5) == (0xFFFFFFFF, 0xFFFFFFFF ^ 1)
    assert od.key_of(2**32, 7) == (0, 1)
    # the epoch's high word reaches the key: epochs 5 and 2^32 + 5 draw differently
    a = od.draw_counts(3, 9, 5, 16, 64)[0]
    b = od.draw_counts(3, 9, 2**32 + 5, 16, 64)[0]
    assert not np.array_equal(a, b)
    ha = od.draw_heads([3], 9, 5, 2, [50], 20)[0]
    hb = od.draw_heads([3], 9, 2**32 + 5, 2, [50], 20)[0]
    assert not np.array_equal(ha, hb)


@pytest.mark.parametrize("r", [1, 2, 3, 7, 100, 641, 5000, 65537, 129971])
def test_bounded_exactly_unbiased(r):
    """Every v in [0, r) is given by exactly floor(2^32 / r) accepted words.  The words x with floor(x r / 2^32) = v
    run from x0 = ceil(v 2^32 / r) to x1 = ceil((v + 1) 2^32 / r) - 1 and their low words step by r from
    low0 = x0 r - v 2^32 < r, so only x0 can be rejected: the count is x1 - x0 + 1 minus x0's rejection."""
    v = np.arange(r, dtype=object)
    x0 = np.array([-(-(int(a) << 32) // r) for a in v], dtype=np.uint64)
    x1 = np.array([-(-((int(a) + 1) << 32) // r) - 1 for a in v], dtype=np.uint64)
    got0, ok0 = od.bounded(x0, r)
    np.testing.assert_array_equal(got0, np.arange(r, dtype=np.uint64))
    more = x1 > x0
    got1, ok1 = od.bounded(x0[more] + np.uint64(1), r)                # the second word of each v: always accepted
    assert ok1.all() and np.array_equal(got1, np.arange(r, dtype=np.uint64)[more])
    accepted = (x1 - x0 + np.uint64(1)).astype(np.int64) - (~ok0).astype(np.int64)
    assert (accepted == (2**32) // r).all()
    assert int((~ok0).sum()) == (2**32) % r                          # the rejected words: 2^32 mod r in all
    # the words around the ends of the range
    ends = np.array([0, 1, 2**32 - 2, 2**32 - 1], dtype=np.uint64)
    vv, _ = od.bounded(ends, r)
    assert (vv < r).all() and vv[0] == 0 and vv[-1] == r - 1


@pytest.mark.parametrize("n_c", range(1, 7))
def test_fisher_yates_exactly_uniform(n_c):
    """All step sequences r_j in [j, n_c): every ordered k-subset of [0, n_c) comes out exactly once."""
    for k in range(1, n_c + 1):
        seqs = np.array(list(itertools.product(*[range(j, n_c) for j in range(k)])), dtype=np.int64)
        heads = od.fisher_yates_heads(seqs, n_c, k + 2, chunk=50)
        assert (heads[:, k:] == -1).all()
        got = sorted(map(tuple, heads[:, :k].tolist()))
        want = sorted(itertools.permutations(range(n_c), k))
        assert got == want
        assert len(got) == math.perm(n_c, k)


KEYS = [(0, 0), (77, 3), (2**64 - 1, 2**32 + 5), (2**32, 7)]


@pytest.mark.parametrize("seed,epoch", KEYS)
@pytest.mark.parametrize("n_classes", [1, 2, 3, 16])
def test_counts_vectorised_equals_scalar(seed, epoch, n_classes):
    for nobj in (0, 1, 31, 32, 127, 128, 129):
        for sidx in (0, 5, 2**31 - 1):
            a, ra = od.draw_counts(sidx, seed, epoch, n_classes, nobj)
            b, rb = od.draw_counts_scalar(sidx, seed, epoch, n_classes, nobj)
            np.testing.assert_array_equal(a, b)
            assert ra == rb and a.sum() == nobj


@pytest.mark.parametrize("seed,epoch", KEYS)
def test_heads_vectorised_equals_scalar(seed, epoch):
    idx = [4, 0, 4, 9]
    lens = [1, 0, 2, 31, 32, 33, 70]
    T, E = 32, 3
    heads, rej = od.draw_heads(idx, seed, epoch, E, lens, T)
    total = 0
    for b, i in enumerate(idx):
        for ev in range(E):
            for c, n_c in enumerate(lens):
                h, r = od.draw_head_scalar(i, seed, epoch, ev, c, n_c, T)
                np.testing.assert_array_equal(heads[b, ev, c], h)
                total += r
                k = min(T, n_c)
                assert sorted(set(h[:k].tolist())) == sorted(h[:k].tolist()) and (h[:k] < n_c).all() and (h[k:] == -1).all()
    assert rej == total
    np.testing.assert_array_equal(heads[0], heads[2])              # same store index, same draws


def test_head_rejections_are_redrawn():
    """With n_c - j = 129971 a word is rejected with probability (2^32 mod r) / 2^32 ~ 1.5e-5: 1024 steps of enough
    heads meet some, and the vectorised and word-by-word references agree on the heads that met one."""
    r, rej = od.head_steps(np.arange(256), 5, 2**32 + 5, 1, 129971, 1024)
    assert ((r >= np.arange(1024)) & (r < 129971)).all()
    hits = np.flatnonzero(rej)
    assert len(hits) >= 1                                           # this key: computed, not assumed
    heads = od.fisher_yates_heads(r[hits], 129971, 1024)
    for h, head in zip(hits[:2], heads):
        want, n_rej = od.draw_head_scalar(int(h), 5, 2**32 + 5, 0, 0, 129971, 1024)
        np.testing.assert_array_equal(head, want)
        assert n_rej == rej[h]


def test_world_draw():
    idx = np.arange(4096)
    fx, fy, theta, k = od.draw_world(idx, 31, 2**32 + 1, 0.3, 1.0, np.float32(np.pi), 0.9, 1.2)
    for a in (fx, fy, theta, k):
        assert a.dtype == np.float32
    assert set(np.unique(fx)) == {0.0, 1.0} and (fy == 1).all()
    assert (np.abs(theta) <= np.float32(np.pi)).all() and (k >= np.float32(0.9)).all() and (k <= np.float32(1.2)).all()
    fx0, fy0, t0, k0 = od.draw_world(idx[:64], 31, 2**32 + 1, 0.0, 0.0, 0.0, 1.0, 1.0)
    assert not fx0.any() and not fy0.any() and not t0.any() and (k0 == 1).all()
    # word by word: the four words of the one Philox call per scan, float32 steps with one rounding each
    f32 = np.float32
    for i in (0, 1, 4095):
        w = [int(x) for x in od.philox4x32_10((0, 0xFFFFFFFF, i, 1), od.key_of(31, 2**32 + 1))]
        u = [f32(x >> 8) * f32(2.0**-24) for x in w]
        assert fx[i] == (u[0] < f32(0.3)) and theta[i] == f32(f32(np.pi) * f32(f32(2 * u[2]) - f32(1)))
        assert k[i] == f32(f32(0.9) + f32(f32(f32(1.2) - f32(0.9)) * u[3]))
