"""The host model of tests/sparse_euclid_forms.py, without a GPU: the f64 prediction of which pairs the sparse
Euclidean call lists agrees with an exact rational N / P classification, planted records have the counts they
claim (against the oracle's k-mer counts), and the planted listed pairs really need the difference form: their exact
distance is more than 1e-9 away from the reference's, so a kernel that gave them the integer form would fail."""
import math
from fractions import Fraction

import numpy as np
import pytest

from sparse_euclid_forms import (BIG_T, NEAR_TAU_WORST, TAU, XS_I, XS_J, exact_ratio, is_listed, listed_pairs,
                                 pair_at_ratio, pair_terms, planted_record, planted_row, range_listed_count,
                                 tiles_for_rows, two_entry_ratio)
from sparse_euclid_ref import merge_matrix

TARGETS = (1 - 1e-3, 1 + 1e-3, 1.5, 3.0, 10.0)


def _terms(a, b):
    """(X, Q_a, Q_b, T_a, T_b) of two count vectors over the same indices, as Python ints"""
    a, b = [int(v) for v in a], [int(v) for v in b]
    return sum(p * q for p, q in zip(a, b)), sum(p * p for p in a), sum(q * q for q in b), sum(a), sum(b)


def _ref_error(a, b) -> float:
    """|d_ref / d - 1| of the merge-form reference over rounded frequencies against the exact distance"""
    rows = [planted_row(a, 9), planted_row(b, 9)]
    d_ref = merge_matrix(rows, [sum(a), sum(b)])[1, 0]
    x, qa, qb, ta, tb = _terms(a, b)
    nn, _ = pair_terms(x, qa, qb, ta, tb)
    r2 = Fraction(d_ref) ** 2 * (ta * tb) ** 2 / nn  # (d_ref / d)^2, exact; its f64 rounding is ~1e-16
    return abs(math.sqrt(float(r2)) - 1.0)


def test_f64_prediction_agrees_with_exact_ratio():
    """random 1- to 4-entry count rows over the same indices, scaled so that N / P spans 1e-16 .. 1e-10: away from
    TAU (1e-9 relative) the kernel's f64 test gives the exact classification"""
    rng = np.random.default_rng(13)
    seen = {False: 0, True: 0}
    for _ in range(4000):
        m = int(rng.integers(1, 5))
        big = int(10 ** rng.uniform(2, 7.5))
        a = [big] + [int(v) for v in rng.integers(0, 40, size=m - 1)]
        b = [max(0, v + int(d)) for v, d in zip(a, rng.integers(-3, 4, size=m))]
        x, qa, qb, ta, tb = _terms(a, b)
        if tb == 0:
            continue
        r = exact_ratio(x, qa, qb, ta, tb)
        if abs(r / Fraction(TAU) - 1) < Fraction(1, 10 ** 9):
            continue
        want = r != 0 and r < Fraction(TAU)
        assert is_listed(x, qa, qb, ta, tb) == want, (a, b, float(r))
        seen[want] += 1
    assert seen[True] > 200 and seen[False] > 200, seen
    # T = 0 is NaN, never listed; T_a T_b >= 2^63 is always listed, whatever N
    assert not is_listed(0, 0, 25, 0, 5)
    t0 = 3_037_000_499
    assert t0 * (t0 + 1) < BIG_T <= (t0 + 1) ** 2
    assert not is_listed(0, t0 * t0, (t0 + 1) ** 2, t0, t0 + 1)
    assert is_listed(0, (t0 + 1) ** 2, (t0 + 1) ** 2, t0 + 1, t0 + 1)


def test_pairs_at_ratio_land_where_asked():
    for r in TARGETS:
        x, y = pair_at_ratio(r * TAU)
        ratio = two_entry_ratio(x, y)
        assert abs(float(ratio) / (r * TAU) - 1) < 1e-5
        assert is_listed(*_terms([x, 1], [y, 1])) == (r < 1), (r, x, y)
    # the 1,700 / 1,800 example: one more k-mer of the same base
    assert not is_listed(*_terms([1700, 1], [1701, 1])) and is_listed(*_terms([1800, 1], [1801, 1]))


def test_near_tau_pairs_are_gram_side_with_the_largest_reference_error():
    for a, b in NEAR_TAU_WORST:
        ratio = exact_ratio(*_terms(a, b)) / Fraction(TAU)
        assert 1 < ratio < Fraction(11, 10), (a, b, float(ratio))
        assert not is_listed(*_terms(a, b))
        assert 1e-10 < _ref_error(a, b) < 0.5e-9, (a, b, _ref_error(a, b))


def test_planted_listed_pairs_need_the_difference_form():
    """pairs of [L0 + m, 1] rows (all listed) and [1800, 1] / [1801, 1]: the exact distance is more than 1e-9 from
    the reference for some of them, so routing them to the integer form would fail the 1e-9 tests"""
    rows = [[200_000 + m, 1] for m in (0, 1, 2, 7, 900, 4999)] + [[1800, 1], [1801, 1]]
    errs = []
    for i in range(len(rows)):
        for j in range(i):
            if (i >= 6) != (j >= 6):
                continue
            assert is_listed(*_terms(rows[i], rows[j]))
            errs.append(_ref_error(rows[i], rows[j]))
    assert max(errs) > 1e-9, max(errs)


@pytest.mark.parametrize("k", [9, 10, 11, 12])
def test_planted_records_have_the_claimed_counts(k):
    from oracle import oracle
    for counts in ([5, 0, 0, 0], [0, 1, 0, 0], [3, 0, 0, 7], [1, 2, 3, 4], [1800, 1], [0, 0, 200_000, 1], [0, 0, 0, 0]):
        seq = planted_record(counts, k)
        dense = oracle.kcounts(seq, k)
        idx, cnt = planted_row(counts, k)
        nz = np.flatnonzero(dense)
        assert np.array_equal(nz, idx) and np.array_equal(dense[nz], cnt), counts
        assert seq.size == sum(k + c - 1 for c in counts if c) + max(0, int(np.count_nonzero(counts)) - 1)
    # the four homopolymers lie in buckets 0, nb / 3, 2 nb / 3 and nb - 1 (bucket = index >> 12): different lanes
    idx, _ = planted_row([1, 1, 1, 1], k)
    nb = 4 ** k >> 12
    assert (idx >> 12).tolist() == [0, nb // 3, 2 * nb // 3, nb - 1]
    assert len({int(b) % 32 for b in idx >> 12}) == 4


def test_listed_pairs_matrix_and_tile_mirror():
    """listed_pairs on planted rows; the full range's tiles cover every pair of the lower triangle once, and a
    range's listed count includes the listed pairs of its tiles outside the range"""
    rows = [planted_row(c, 9) for c in ([200_000, 1], [5, 7], [200_003, 1], [0, 0, 0, 0], [200_001, 1], [5, 7])]
    listed = listed_pairs(rows, 4 ** 9)
    want = np.zeros((6, 6), dtype=bool)
    for i, j in ((2, 0), (4, 0), (4, 2)):
        want[i, j] = True
    assert np.array_equal(listed, want)  # (5, 1) is a copy (N = 0), row 3 has no k-mer
    for n in (1, 7, 8, 9, 64, 65, 130, 300):
        cover = np.zeros((n, n), dtype=int)
        for ib, jc in tiles_for_rows(n, 0, n):
            i0, j0 = ib * XS_I, jc * XS_J
            for i in range(i0, min(n, i0 + XS_I)):
                for j in range(j0, min(i + 1, j0 + XS_J)):
                    cover[i, j] += 1
        assert np.array_equal(cover, np.tril(np.ones((n, n), dtype=int))), n
    n = 200
    listed = np.tril(np.ones((n, n), dtype=bool), -1)
    assert range_listed_count(listed, 0, n) == n * (n - 1) // 2
    # rows [64, 65): tile row ib = 8 (pairs (64..71, 0..71)) and the column tiles jc = 1 below it
    want = sum(min(i, 128) - 64 for i in range(72, n)) + sum(i for i in range(64, 72))
    assert range_listed_count(listed, 64, 65) == want
    assert range_listed_count(listed, 5, 5) == 0
