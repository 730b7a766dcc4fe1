"""CPU tier: r3d::mean_div (csrc/r3d_common.cuh), the close / fill neighbour mean without an fp64 division, restated in
exact rational arithmetic: y = RN(1/n), q = RN(sum * y), r = RN(sum - q * n) (one fma), q' = RN(q + r * y) (one fma)
must be the correctly rounded sum / n for every n the 5 x 3 window can give (1 .. 15)."""
import math
import random
import struct
from fractions import Fraction

import pytest

N_MAX = 15


def rn(x: Fraction) -> float:
    return float(x)                     # Fraction -> float rounds to nearest, ties to even


def mean_div(s: float, n: int) -> float:
    y = rn(Fraction(1, n))
    q = rn(Fraction(s) * Fraction(y))
    r = rn(Fraction(s) - Fraction(q) * n)
    return rn(Fraction(r) * Fraction(y) + Fraction(q))


def ordered_sum(values):
    s = 0.0
    for v in values:
        s += v                          # fp64 additions in order, like the kernels' neighbour loop
    return s


def test_reciprocal_table_is_rn_of_one_over_n():
    for n in range(1, N_MAX + 1):
        assert 1.0 / n == rn(Fraction(1, n))


@pytest.mark.parametrize("n", range(1, N_MAX + 1))
def test_mean_div_matches_division_on_seeded_range_sums(n):
    # 70 000 sums per n (> 10^6 over all n): ordered fp64 sums of n ranges in (0, 500] m, half of them drawn from a
    # narrow band (neighbouring pixels of one surface), half spread over the whole range
    rng = random.Random(1000 + n)
    for i in range(70_000):
        if i & 1:
            c = rng.uniform(1e-3, 500.0)
            vals = [min(500.0, max(1e-9, c + rng.uniform(-0.5, 0.5))) for _ in range(n)]
        else:
            vals = [500.0 - rng.random() * 500.0 for _ in range(n)]
        s = ordered_sum(vals)
        assert mean_div(s, n) == s / n, (s, n)


@pytest.mark.parametrize("n", range(1, N_MAX + 1))
def test_mean_div_matches_division_on_random_mantissas(n):
    # sums with every mantissa pattern equally likely, not only the patterns that sums of ranges produce
    rng = random.Random(2000 + n)
    for _ in range(4_000):
        e = rng.randint(1013, 1036)                         # sums from ~1e-3 to ~8e3 (15 ranges of up to 500 m)
        s = struct.unpack("<d", struct.pack("<Q", (e << 52) | rng.getrandbits(52)))[0]
        assert mean_div(s, n) == s / n, (s, n)


def test_mean_div_edge_cases():
    cases = []
    for n in range(1, N_MAX + 1):
        for v in (1e-9, 0.1, 0.5, 1.0, 1.5, 3.0, 7.25, 99.99, 250.0, 499.999, 500.0):
            cases.append((ordered_sum([v] * n), n))                         # n equal values: the mean is v (or its RN)
        for k in range(-10, 13):
            cases.append((math.ldexp(1.0, k), n))                           # powers of two
            cases.append((math.ldexp(1.0, k) * n, n))                       # exact quotients
        for m in range(1, 2 * n, 2):                                        # sums next to n times a midpoint
            cases.append((rn(Fraction(n) * (1 + Fraction(m, 2 ** 53))), n))       # between two doubles of [1, 2)
        for a in (3.0, 100.0, 333.0):                                       # neighbours of an exact multiple
            s = a * n
            cases += [(math.nextafter(s, 0.0), n), (s, n), (math.nextafter(s, math.inf), n)]
    for s, n in cases:
        assert mean_div(s, n) == s / n, (s, n)
