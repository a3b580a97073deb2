"""Host model of which form `dvs_euclid_distances_sparse` (csrc/euclid_sparse.cu) gives each pair, and records
planted to land on either side of its threshold.

* `listed_pairs`: the pairs `k_xs_finish` puts on the list for `k_xs_pairs` (the difference form), predicted bit for
  bit from exact integers: with X = sum c_a c_b, Q_a = X_aa, P = T_b^2 Q_a + T_a^2 Q_b and N = P - 2 T_a T_b X, a pair
  is listed iff T_a T_b >= 2^63, or N != 0 and not f64(N) >= TAU * f64(P) (the kernel's u128 -> f64 conversion);
  pairs with T = 0 are NaN and never listed.
* `tiles_for_rows` / `range_listed_count`: the lower-triangle tiles a row range computes (`xs_tiles_for_rows`) and
  how many listed pairs they hold; a range call lists every listed pair of its tiles, including pairs of rows
  outside the range.
* `planted_record`: a record whose sparse row holds up to 4 entries with any counts: a run of k + c - 1 copies of
  base b gives the one k-mer b^k (index b (4^k - 1) / 3) c times, and runs are separated by an invalid byte (4).
  The four indices fall in buckets 0, nb/3, 2nb/3 and nb - 1, i.e. on different lanes of `k_xs_pairs`.
"""
from fractions import Fraction

import numpy as np
import scipy.sparse

TAU = 1e-13                      # kXsTau
XS_I, XS_J = 8, 64               # kXsI, kXsJ: rows of a tile's I block and J block
FLAG_CAP = 1 << 24               # kXsFlagCap: a call lists at most min(tile pairs, 2^24) pairs
BIG_T = 1 << 63                  # T_a T_b from here on: N no longer fits 128 bits, the pair is listed

# pairs of count rows just above TAU whose reference distance (over rounded frequencies) is furthest from the exact
# one, found by a host search over random 2- and 3-entry rows: about 1.5e-10 to 2e-10 relative, the largest
# rounding error a Gram-form pair has to stay within 1e-9 of
NEAR_TAU_WORST = [
    ([9_316_568, 17], [9_316_566, 14]),
    ([16_377_386, 56, 42], [16_377_383, 59, 45]),
    ([10_782_185, 11, 27], [10_782_186, 9, 25]),
]


def homopolymer_index(base: int, k: int) -> int:
    return base * (4 ** k - 1) // 3


def planted_record(counts, k: int) -> np.ndarray:
    """uint8 record whose k-mer row is {homopolymer_index(b, k): counts[b]} over the nonzero counts[b], b < 4"""
    assert len(counts) <= 4
    parts = []
    for b, c in enumerate(counts):
        if c:
            if parts:
                parts.append(np.array([4], dtype=np.uint8))
            parts.append(np.full(k + int(c) - 1, b, dtype=np.uint8))
    return np.concatenate(parts) if parts else np.zeros(0, dtype=np.uint8)


def planted_row(counts, k: int):
    """(ascending k-mer indices, counts) that `planted_record(counts, k)` has"""
    nz = [(homopolymer_index(b, k), int(c)) for b, c in enumerate(counts) if c]
    return (np.array([i for i, _ in nz], dtype=np.uint32), np.array([c for _, c in nz], dtype=np.uint32))


def u128_to_double(v: int) -> float:
    """xs_u128_to_double: f64(hi) * 2^64 + f64(lo), each step rounded to nearest"""
    hi, lo = v >> 64, v & ((1 << 64) - 1)
    return float(hi) * 2.0 ** 64 + float(lo) if hi else float(lo)


def pair_terms(x: int, qa: int, qb: int, ta: int, tb: int):
    """(N, P) of a pair as exact integers"""
    p = tb * tb * qa + ta * ta * qb
    return p - 2 * ta * tb * x, p


def is_listed(x: int, qa: int, qb: int, ta: int, tb: int) -> bool:
    """whether k_xs_finish hands the pair to the difference form"""
    if ta == 0 or tb == 0:
        return False
    if ta * tb >= BIG_T:
        return True
    nn, p = pair_terms(x, qa, qb, ta, tb)
    return nn != 0 and not (u128_to_double(nn) >= TAU * u128_to_double(p))


def gram_inputs(rows, dim: int):
    """(X as Python ints [n][n], T as Python ints) of sparse rows (indices, counts)"""
    n = len(rows)
    ind = np.concatenate([np.asarray(i, dtype=np.int64) for i, _ in rows]) if n else np.zeros(0, np.int64)
    val = np.concatenate([np.asarray(c, dtype=np.int64) for _, c in rows]) if n else np.zeros(0, np.int64)
    ptr = np.concatenate([[0], np.cumsum([len(i) for i, _ in rows])]).astype(np.int64)
    m = scipy.sparse.csr_matrix((val, ind, ptr), shape=(n, dim))
    x = (m @ m.T).toarray()  # exact: every X here is far below 2^63
    t = [int(np.asarray(c, dtype=np.int64).sum()) for _, c in rows]
    return x.tolist(), t


def listed_pairs(rows, dim: int) -> np.ndarray:
    """n x n bool, True at (i, j), j < i, for every pair the call over all rows lists"""
    x, t = gram_inputs(rows, dim)
    n = len(rows)
    out = np.zeros((n, n), dtype=bool)
    for i in range(n):
        xi = x[i]
        for j in range(i):
            out[i, j] = is_listed(xi[j], xi[i], x[j][j], t[i], t[j])
    return out


def exact_ratio(x: int, qa: int, qb: int, ta: int, tb: int) -> Fraction:
    nn, p = pair_terms(x, qa, qb, ta, tb)
    return Fraction(nn, p)


def tiles_for_rows(n: int, row_begin: int, row_end: int):
    """xs_tiles_for_rows: the (ib, jc) tiles of the lower triangle that hold a pair with a row in the range"""
    tiles = []
    for ib in range((n + XS_I - 1) // XS_I):
        i0, i1 = ib * XS_I, min(n, ib * XS_I + XS_I)
        i_in = i0 < row_end and i1 > row_begin
        jc = 0
        while jc * XS_J < i1:
            j0, j1 = jc * XS_J, min(i1, jc * XS_J + XS_J)
            if i_in or (j0 < row_end and j1 > row_begin):
                tiles.append((ib, jc))
            jc += 1
    return tiles


def range_listed_count(listed: np.ndarray, row_begin: int, row_end: int) -> int:
    """pairs a call for rows [row_begin, row_end) lists: the listed pairs (i, j), j < i, of its tiles (none for an
    empty range, which returns before any launch)"""
    n = listed.shape[0]
    if row_end <= row_begin:
        return 0
    cover = np.zeros((n, n), dtype=bool)
    for ib, jc in tiles_for_rows(n, row_begin, row_end):
        cover[ib * XS_I:(ib + 1) * XS_I, jc * XS_J:(jc + 1) * XS_J] = True
    return int((listed & np.tril(cover, -1)).sum())


def two_entry_ratio(x: int, y: int) -> Fraction:
    """N / P of the rows [x, 1] and [y, 1]: N = 2 (x - y)^2"""
    return exact_ratio(x * y + 1, x * x + 1, y * y + 1, x + 1, y + 1)


def pair_at_ratio(target: float, max_gap: int = 400):
    """(x, y) with rows [x, 1], [y, 1] whose N / P is within 1e-5 relative of `target`: N / P ~ (x - y)^2 /
    ((x + y) / 2)^4, so the closest y next to (gap^2 / target)^(1/4) - gap / 2 over gaps x - y = 1 .. max_gap"""
    best = None
    for gap in range(1, max_gap + 1):
        x0 = int((gap * gap / target) ** 0.25 - gap / 2)
        for x in range(x0 - 2, x0 + 3):
            dev = abs(float(two_entry_ratio(x + gap, x)) / target - 1.0)
            if best is None or dev < best[0]:
                best = (dev, x + gap, x)
    assert best[0] < 1e-5, best
    return best[1], best[2]
