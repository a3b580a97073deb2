"""Sparse Euclidean matrix (dvs_euclid_distances_sparse, csrc/euclid_sparse.cu) in both forms that can give a pair
its distance, at multi-tile shapes and row ranges:

* Gram form   - k_xs_self + k_xs_gram + k_xs_finish, exact integers: 3 launches, no pair listed;
* listed form - k_xs_finish also lists pairs with N < TAU P or T_a T_b >= 2^63, k_xs_pairs recomputes them in
                difference form and stores them into the matrix: 4 launches.

Every call asserts its launch count and that `fallback_pairs()` equals the host prediction of
tests/sparse_euclid_forms.py exactly, so a test cannot silently take the other form.  Listed pairs are planted
with homopolymer runs (`planted_record`).  Every matrix matches the sparse-row reference at 1e-9 relative (NaN
pattern equal, exact zeros exact), is bitwise symmetric with a zero diagonal, every listed entry is bitwise the
difference-form kernel's value for that pair, and every row range equals the same rows of the full matrix bitwise.
"""
import numpy as np
import pytest

from conftest import random_seqs
from sparse_euclid_forms import (BIG_T, FLAG_CAP, NEAR_TAU_WORST, TAU, listed_pairs, pair_at_ratio, planted_record,
                                 planted_row, range_listed_count, two_entry_ratio)
from sparse_euclid_ref import chunked_dense_matrix, merge_matrix

pytestmark = pytest.mark.gpu

RTOL = 1e-9
L0 = 200_000   # [L0 + m, 1] rows with m < 5,000: N / P ~ m'^2 / L0^4 < TAU / 6, every pair of them is listed
SENTINEL = -7.0


@pytest.fixture(scope="module")
def lib():
    from diverseseq_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def ctx(lib):
    return lib.Context(0)


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


# ------------------------------------------------------------------------------------------- helpers ----

def host_rows(sp):
    _, totals, _, _ = sp.stats()
    return [sp.record(r) for r in range(sp.nrec)], totals


def call(sp, listed, fn, row_begin, row_end):
    """runs one matrix call and asserts its form: launches and the exact number of listed pairs"""
    before = sp.ctx.launch_count
    out = fn()
    launches, got = sp.ctx.launch_count - before, sp.fallback_pairs()
    want = range_listed_count(listed, row_begin, row_end)
    want_launches = 0 if row_end == row_begin else 4 if want else 3
    assert (launches, got) == (want_launches, want), \
        f"rows [{row_begin}, {row_end}) of n={sp.nrec}: {launches} launches, {got} listed; expected {want_launches}, {want}"
    return out


def run(sp, listed, row_begin=0, row_end=None):
    row_end = sp.nrec if row_end is None else row_end
    return call(sp, listed, lambda: sp.euclidean(row_begin, row_end), row_begin, row_end)


def run_into(lib, ctx, sp, listed, row_begin, row_end):
    """rows [row_begin, row_end) written to a device buffer filled with SENTINEL first"""
    n = sp.nrec
    shape = (row_end - row_begin, n)
    buf = lib.DeviceBuffer(ctx, max(8, shape[0] * n * 8))
    buf.from_host(np.full(shape, SENTINEL))
    call(sp, listed, lambda: sp.euclidean_into(buf.ptr, row_begin, row_end), row_begin, row_end)
    out = buf.to_host(np.float64, shape)
    buf.close()
    return out


def assert_matches(got, exp):
    nan = np.isnan(exp)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got == 0.0, exp == 0.0)  # exact zeros are exact
    np.testing.assert_allclose(got[~nan], exp[~nan], rtol=RTOL, atol=0)


def assert_matrix_form(got):
    assert np.array_equal(got, got.T, equal_nan=True), "not bitwise symmetric"
    assert (np.diag(got) == 0.0).all(), "diagonal not exactly 0"


def assert_listed_entries(sp, got, listed):
    """every listed pair's entry is bitwise the difference-form kernel's value for that pair"""
    i, j = np.nonzero(listed)
    if i.size:
        d = sp.debug_euclid_pairs(np.stack([i, j], axis=1))
        assert np.array_equal(got[i, j], d, equal_nan=True)
        assert np.array_equal(got[j, i], d, equal_nan=True)


def gram_side_error(got, exp, listed):
    """largest relative error of the pairs the Gram form computed (finite, nonzero)"""
    il = np.tril_indices(got.shape[0], -1)
    g, e, lst = got[il], exp[il], listed[il]
    keep = ~lst & np.isfinite(e) & (e > 0)
    return float((np.abs(g[keep] - e[keep]) / e[keep]).max()) if keep.any() else 0.0


def check_full(sp, got, listed, k, merge=True, orc=None):
    rows, totals = host_rows(sp)
    if merge:
        exp = merge_matrix(rows, totals)
    else:
        exp = chunked_dense_matrix(orc, rows, totals, 4 ** k, threads=max(1, orc.hardware_threads()))
    assert_matches(got, exp)
    assert_matrix_form(got)
    assert_listed_entries(sp, got, listed)
    return exp


# ----------------------------------------------------------------------------------------- record sets ----

def mixed_records(rng, n, k):
    """random records with planted near-proportional groups, degenerate records and copies.  Family P ([L0 + m, 1]
    on the homopolymers of bases 0, 1) sits at rows 0, 7 | 8, 63 | 64, 71, 127 | 128, 200 and n - 1 (the last, often
    partial, I block): listed pairs in diagonal tiles, in jc >= 1 tiles and across the 8-, 64- and 128-row edges.
    Family Q ([1, 3, 1, L0 + m], all four lanes of k_xs_pairs; N / P ~ 13 m'^2 / L0^4, so only pairs less than
    ~3,500 apart in m are listed) at rows 4, 65, 66, 129, 250 and n - 2; row 150 is a copy of row 7 (a zero in a
    family)."""
    seqs = random_seqs(rng, n, 0, 1200, invalid_rate=0.01)
    taken = {}

    def put(pos, seq):
        if 0 <= pos < n and pos not in taken:
            taken[pos] = True
            seqs[pos] = seq

    ms = iter(rng.permutation(5000).tolist())
    for pos in (0, 7, 8, 63, 64, 71, 127, 128, 200, n - 1):
        put(pos, planted_record([L0 + next(ms), 1], k))
    if 7 in taken:
        put(150, seqs[7].copy())
    for pos in (4, 65, 66, 129, 250, n - 2):
        put(pos, planted_record([1, 3, 1, L0 + next(ms)], k))
    put(2, np.zeros(0, dtype=np.uint8))                       # empty
    put(5, np.full(300, 4, dtype=np.uint8))                   # no valid byte
    put(9, rng.integers(0, 4, size=k - 1, dtype=np.uint8))    # shorter than k
    if n > 12:
        put(12, seqs[3].copy())                               # copies of random records
        put(n - 3, seqs[1].copy())
    return seqs


def counted(lib, ctx, seqs, k):
    return lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), k)


# --------------------------------------------------------------------------------------------- tests ----

def _shape_cases():
    for k in (9, 12):
        for n in (1, 2, 7, 8, 9, 63, 64, 65, 72, 127, 129, 200, 300):
            yield pytest.param(k, n, id=f"k{k}-n{n}")
    yield pytest.param(10, 130, id="k10-n130")
    yield pytest.param(11, 77, id="k11-n77")


@pytest.mark.parametrize("k,n", list(_shape_cases()))
def test_forms_at_shapes(lib, ctx, k, n):
    seqs = mixed_records(np.random.default_rng(100 * k + n), n, k)
    sp = counted(lib, ctx, seqs, k)
    rows, _ = host_rows(sp)
    listed = listed_pairs(rows, 4 ** k)
    if n >= 2:
        assert listed[n - 1, 0]  # rows 0 and n - 1 are in the planted family P
    got = run(sp, listed)
    exp = check_full(sp, got, listed, k)
    if n >= 9:
        assert np.array_equal(sp.record(7)[0], planted_row([1, 1], k)[0]) and listed[8, 7] and listed[7, 0]
    for rb, re in ((0, 2 * n // 3), (n // 3, n)):
        assert np.array_equal(run(sp, listed, rb, re), got[rb:re], equal_nan=True), (rb, re)
    print(f"\nk={k} n={n}: {int(listed.sum())} listed pairs, Gram-side error {gram_side_error(got, exp, listed):.2e}")


def test_threshold(lib, ctx):
    """pairs at N / P = TAU * (1 - 1e-3, 1 + 1e-3, 1.5, 3, 10) and the near-TAU pairs with the largest reference
    rounding error: exactly the pairs below TAU are listed, and the Gram-side ones still meet 1e-9"""
    k = 12
    seqs, pairs = [], []
    for b, r in enumerate((1 - 1e-3, 1 + 1e-3, 1.5, 3.0, 10.0)):
        x, y = pair_at_ratio(r * TAU)
        lo = [0, 0, 0, 0]
        lo[b % 4], lo[(b + 1) % 4] = x, 1   # a different base pair per target, so targets do not mix
        hi = list(lo)
        hi[b % 4] = y
        pairs.append((len(seqs), len(seqs) + 1, r))
        seqs += [planted_record(lo, k), planted_record(hi, k)]
    for a, c in NEAR_TAU_WORST:
        pairs.append((len(seqs), len(seqs) + 1, None))
        seqs += [planted_record(a, k), planted_record(c, k)]
    rng = np.random.default_rng(41)
    seqs += random_seqs(rng, 20, 100, 2000)
    sp = counted(lib, ctx, seqs, k)
    rows, _ = host_rows(sp)
    listed = listed_pairs(rows, 4 ** k)
    for a, c, r in pairs:
        assert listed[c, a] == (r is not None and r < 1), (a, c, r)
    got = run(sp, listed)
    exp = check_full(sp, got, listed, k)
    near = [(c, a) for a, c, r in pairs if r is None or r > 1]
    rel = [abs(got[c, a] - exp[c, a]) / exp[c, a] for c, a in near]
    print(f"\nGram-side pairs just above TAU: relative errors {['%.2e' % v for v in rel]}, "
          f"largest Gram-side error {gram_side_error(got, exp, listed):.2e}")
    assert max(rel) <= RTOL


def _ranges(n):
    r = [(0, 64), (0, 8), (8, 64), (3, 61), (64, n), (60, 130), (8, n - 1), (13, n), (0, n - 1), (n - 9, n),
         (64, 128), (70, 190)]
    r += [(i, i + 1) for i in (0, 7, 8, 63, 64, n - 1)]
    r += [(5, 5), (n, n)]
    out = []
    for rb, re in r:
        re = min(re, n)
        if rb <= re and (rb, re) not in out:
            out.append((rb, re))
    return out


@pytest.mark.parametrize("n", [65, 200, 300])
def test_row_ranges_equal_full_matrix(lib, ctx, n):
    """ranges aligned and unaligned to 8 and 64, single rows at tile edges, ranges to the end and empty ranges, host
    and device output.  A matrix of other records is computed before each host-output call and the device buffer is
    filled with a sentinel, so neither stale pool memory nor a stale buffer can supply an unwritten entry."""
    k = 12
    rng = np.random.default_rng(7 * n)
    sp = counted(lib, ctx, mixed_records(rng, n, k), k)
    decoy = counted(lib, ctx, random_seqs(rng, n, 50, 400), k)
    rows, _ = host_rows(sp)
    listed = listed_pairs(rows, 4 ** k)
    full = run(sp, listed)
    check_full(sp, full, listed, k)
    for rb, re in _ranges(n):
        decoy.euclidean()
        got = run(sp, listed, rb, re)
        assert np.array_equal(got, full[rb:re], equal_nan=True), f"rows [{rb}, {re}) differ from the full matrix"
        got = run_into(lib, ctx, sp, listed, rb, re)
        assert np.array_equal(got, full[rb:re], equal_nan=True), f"device rows [{rb}, {re}) differ from the full matrix"


def test_argument_errors_and_empty_list_reset_the_counter(lib, ctx):
    k = 9
    seqs = [planted_record([L0 + m, 1], k) for m in (0, 3, 9)] + [np.full(100, 4, dtype=np.uint8)]
    sp = counted(lib, ctx, seqs, k)
    listed = listed_pairs(host_rows(sp)[0], 4 ** k)
    assert listed.sum() == 3
    plain = counted(lib, ctx, random_seqs(np.random.default_rng(3), 10, 100, 500), k)
    none = listed_pairs(host_rows(plain)[0], 4 ** k)
    assert not none.any()
    for bad in ((0, 5), (3, 2)):
        run(sp, listed)
        assert sp.fallback_pairs() == 3
        with pytest.raises(TypeError):
            sp.euclidean(*bad)
        assert sp.fallback_pairs() == 0, bad
    run(sp, listed)
    assert run(sp, listed, 2, 2).shape == (0, 4) and sp.fallback_pairs() == 0
    run(sp, listed)
    run(plain, none)  # 3 launches, 0 listed
    run(sp, listed, 0, 1)
    assert sp.fallback_pairs() == 3  # rows [0, 1): the one tile holds every pair


def two_entry_rows(xs, row_begin, row_end):
    """rows [row_begin, row_end) of the distances of the rows [x, 1] (the base-0 index below the base-1 one), in f64
    as merge_distance computes them, vectorised"""
    x = np.asarray(xs, dtype=np.float64)
    t = x + 1.0
    f0, f1 = x / t, 1.0 / t
    d0 = f0[row_begin:row_end, None] - f0[None, :]
    d1 = f1[row_begin:row_end, None] - f1[None, :]
    return np.sqrt(d0 * d0 + d1 * d1)


def test_list_overflow(lib, ctx):
    """6,000 records [L0 + m, 1] at k = 9 (1.2 Gbp): all 17,997,000 pairs are listed, more than the 2^24 a call can
    list, so the whole matrix is refused and the counter holds the overflowing count; rows [0, 64) and
    [n - 70, n) list fewer and succeed"""
    k, n = 9, 6000
    x = L0 + np.arange(n, dtype=np.int64)
    # record m = planted_record([x_m, 1], k): x_m + k - 1 bytes of base 0, an invalid byte, k bytes of base 1
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(x + 2 * k)
    flat = np.zeros(int(offsets[-1]), dtype=np.uint8)
    starts = offsets[:-1].astype(np.int64)
    sep = starts + x + k - 1
    flat[sep] = 4
    for q in range(k):
        flat[sep + 1 + q] = 1
    assert np.array_equal(flat[int(offsets[5]):int(offsets[6])], planted_record([L0 + 5, 1], k))
    ss = lib.SeqSet.upload(ctx, flat, offsets)
    sp = lib.KSparse.count(ctx, ss, k)
    ss.close()
    del flat
    _, totals, _, _ = sp.stats()
    assert np.array_equal(totals, x + 1)
    # the largest N / P of the set: the pair furthest apart at the smallest counts
    assert two_entry_ratio(int(x[-1]), int(x[0])) < TAU / 4
    listed = np.tril(np.ones((n, n), dtype=bool), -1)
    assert listed.sum() == 17_997_000 > FLAG_CAP
    with pytest.raises(ValueError, match="pairs need the difference form"):
        sp.euclidean()
    assert sp.fallback_pairs() == 17_997_000
    for rb, re in ((0, 64), (n - 70, n)):
        got = run(sp, listed, rb, re)
        assert_matches(got, two_entry_rows(x, rb, re))


def random_bases(rng, out):
    """fills `out` with random valid bases, 256 MB at a time"""
    step = 1 << 28
    for o in range(0, out.size, step):
        c = min(step, out.size - o)
        out[o:o + c] = np.frombuffer(rng.bytes(c), dtype=np.uint8) & np.uint8(3)


def test_t_product_around_2_63(lib, ctx, orc):
    """two random records of about 3 Gbp each, all bases valid: T_a T_b = 3,037,000,499 x 3,037,000,500 < 2^63
    takes the Gram form, 3,037,000,500^2 >= 2^63 is listed whatever N is.  Two calls of two records, the first
    freed before the second (each needs ~55 GB of device memory)"""
    k = 9
    t1 = 3_037_000_500
    assert (t1 - 1) * t1 < BIG_T <= t1 * t1
    la = t1 + k - 1  # bytes of a record with T = t1
    flat = np.empty(2 * la, dtype=np.uint8)
    random_bases(np.random.default_rng(263), flat)
    offsets = np.array([0, la, 2 * la], dtype=np.uint64)
    last = int(flat[la - 1])
    for t0 in (t1 - 1, t1):
        flat[la - 1] = 4 if t0 < t1 else last  # an invalid last byte takes one k-mer from record 0
        ss = lib.SeqSet.upload(ctx, flat, offsets)
        sp = lib.KSparse.count(ctx, ss, k)
        ss.close()
        _, totals, _, _ = sp.stats()
        assert totals.tolist() == [t0, t1], totals
        listed = np.zeros((2, 2), dtype=bool)
        listed[1, 0] = t0 * t1 >= BIG_T
        got = run(sp, listed)
        check_full(sp, got, listed, k, merge=False, orc=orc)
        sp.close()
