"""Euclidean distance matrix from sparse k-mer rows (dvs_euclid_distances_sparse, 9 <= k <= 12) against the
sparse-row references of tests/sparse_euclid_ref.py (the merge form is bitwise the dense oracle,
tests/test_oracle_euclid_sparse.py) at 1e-9 relative, exact zeros exact; against the dense GPU path where dense rows still fit (k = 9, 10); and the difference-form kernel that
takes the pairs the exact integer form cannot give to 1e-9 of the reference's rounded frequencies."""
import numpy as np
import pytest

from conftest import random_seqs
from sparse_euclid_ref import chunked_dense_matrix, merge_matrix

pytestmark = pytest.mark.gpu

RTOL = 1e-9


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


def oracle_matrix(orc, sp, k, merge=False):
    """merge=True: the sequential merge form (short rows); otherwise the column-sliced dense oracle"""
    _, totals, _, _ = sp.stats()
    rows = [sp.record(r) for r in range(sp.nrec)]
    if merge:
        return merge_matrix(rows, totals)
    return chunked_dense_matrix(orc, rows, totals, 4 ** k, threads=max(1, orc.hardware_threads()))


def assert_matches(got, exp):
    nan = np.isnan(exp)
    assert np.array_equal(np.isnan(got), nan)
    assert np.array_equal(got == 0.0, exp == 0.0)  # exact zeros are exact
    np.testing.assert_allclose(got[~nan], exp[~nan], rtol=RTOL, atol=0)


def assert_matrix_form(got):
    nan = np.isnan(got)
    assert np.array_equal(nan, nan.T) and np.array_equal(got[~nan], got.T[~nan])
    assert (np.diag(got) == 0.0).all()


@pytest.fixture(scope="module")
def ragged(lib, ctx):
    """ragged records with the degenerate cases: empty, no valid k-mer, homopolymer, shorter than k, repeat"""
    rng = np.random.default_rng(1212)
    seqs = random_seqs(rng, 40, 1, 60_000, invalid_rate=0.002)
    seqs[3] = np.zeros(0, dtype=np.uint8)
    seqs[5] = np.full(500, 4, dtype=np.uint8)
    seqs[7] = np.zeros(100_000, dtype=np.uint8)
    seqs[9] = rng.integers(0, 4, size=11, dtype=np.uint8)
    seqs[11] = np.tile(np.array([0, 1, 2, 3, 3, 1], dtype=np.uint8), 30_000)
    return seqs


@pytest.mark.parametrize("k", [9, 10, 11, 12])
def test_brca1_all_records(lib, ctx, orc, brca1, k):
    seqs = list(brca1.values())
    ss = lib.SeqSet.from_seqs(ctx, seqs)
    sp = lib.KSparse.count(ctx, ss, k)
    got = sp.euclidean()
    assert_matrix_form(got)
    assert_matches(got, oracle_matrix(orc, sp, k, merge=True))
    if k <= 10:  # the dense rows of the same records
        assert_matches(got, lib.KFreqs.count(ctx, ss, k).euclidean())


@pytest.mark.parametrize("k", [10, 12])
def test_ragged_degenerate_records_against_dense_and_oracle(lib, ctx, orc, ragged, k):
    ss = lib.SeqSet.from_seqs(ctx, ragged)
    sp = lib.KSparse.count(ctx, ss, k)
    got = sp.euclidean()
    assert_matrix_form(got)
    exp = oracle_matrix(orc, sp, k)
    assert_matches(got, exp)
    assert np.isnan(got[3, 0]) and np.isnan(got[5, 8]) and np.isnan(got[3, 5]) and got[3, 3] == 0.0
    if k == 10:
        assert_matches(got, lib.KFreqs.count(ctx, ss, k).euclidean())


def test_near_duplicates_copies_and_proportional_rows_k12(lib, ctx, orc):
    rng = np.random.default_rng(2038)
    base = rng.integers(0, 4, size=300_000, dtype=np.uint8)
    seqs = []
    for _ in range(24):  # a family with 0.1 % substitutions
        s = base.copy()
        hit = rng.random(s.size) < 0.001
        s[hit] = rng.integers(0, 4, size=int(hit.sum()), dtype=np.uint8)
        seqs.append(s)
    seqs += [seqs[3].copy(), seqs[7].copy(), base.copy(), base.copy()]              # exact copies: 24..27
    seqs += [np.concatenate([seqs[5], np.array([4], np.uint8), seqs[5]]),           # s || invalid || s: 28
             np.concatenate([base, np.array([9], np.uint8), base, np.array([4], np.uint8), base])]  # 3 x base: 29
    seqs += [rng.integers(0, 4, size=250_000, dtype=np.uint8) for _ in range(4)]    # unrelated rows: 30..33
    sp = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), 12)
    got = sp.euclidean()
    exp = oracle_matrix(orc, sp, 12)
    for a, b in ((3, 24), (7, 25), (26, 27), (5, 28), (26, 29), (27, 29)):
        assert exp[a, b] == 0.0 and got[a, b] == 0.0 and got[b, a] == 0.0
    near = exp[:24, :24][np.triu_indices(24, 1)]
    assert near.max() < exp[:24, 30:].min() / 5  # the family really is near-duplicate
    assert_matches(got, exp)
    assert_matrix_form(got)


def test_full_length_genomes_k12(lib, ctx, orc):
    """64 synthetic genomes of ~4 Mbp at k=12: all 2,016 pairs"""
    sp = lib.KSparse.count(ctx, lib.SeqSet.synth(ctx, 4412, 64, 8, 4_000_000), 12)
    got = sp.euclidean()
    exp = oracle_matrix(orc, sp, 12)
    assert_matches(got, exp)
    assert_matrix_form(got)
    assert not np.isnan(got).any() and (got[np.triu_indices(64, 1)] > 0).all()


@pytest.mark.parametrize("k", [9, 12])
def test_difference_form_pairs_kernel(lib, ctx, orc, ragged, k):
    sp = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, ragged), k)
    exp = oracle_matrix(orc, sp, k)
    rng = np.random.default_rng(k)
    pairs = rng.integers(0, len(ragged), size=(300, 2))
    pairs = np.concatenate([pairs, [[7, 0], [0, 7], [7, 11], [3, 5], [5, 8], [8, 3], [7, 7], [3, 3], [11, 9]]])
    got = sp.debug_euclid_pairs(pairs)
    want = exp[pairs[:, 0], pairs[:, 1]]
    assert_matches(got, want)
    # orientation does not change the bits
    assert np.array_equal(got, sp.debug_euclid_pairs(pairs[:, ::-1]), equal_nan=True)


def test_row_ranges_host_and_device_outputs(lib, ctx, brca1):
    sp = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, list(brca1.values())), 12)
    n = sp.nrec
    full = sp.euclidean()
    assert np.array_equal(sp.euclidean(5, 29), full[5:29])
    assert np.array_equal(sp.euclidean(0, 1), full[0:1]) and np.array_equal(sp.euclidean(n - 3, n), full[n - 3:])
    buf = lib.DeviceBuffer(ctx, n * n * 8)
    sp.euclidean_into(buf.ptr)
    assert np.array_equal(buf.to_host(np.float64, (n, n)), full)
    sp.euclidean_into(buf.ptr, 17, 40)
    assert np.array_equal(buf.to_host(np.float64, (23, n)), full[17:40])
    assert_matrix_form(full)


def test_ctree_k12_euclidean(lib, ctx, brca1):
    from diverseseq_b200.cluster import dvs_ctree, make_cluster_tree

    names = list(brca1)
    seqs = [brca1[x] for x in names]
    host = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), 12).euclidean()
    tree = dvs_ctree(k=12, distance_mode="euclidean", ctx=ctx)(names, seqs)
    ref = make_cluster_tree(names, host, ctx=ctx)
    assert np.array_equal(tree.children, ref.children) and np.array_equal(tree.heights, ref.heights)
    assert tree.treestring == ref.treestring and sorted(tree.get_tip_names()) == sorted(names)


def test_argument_errors(lib, ctx):
    sp = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, [np.zeros(100, dtype=np.uint8)] * 3), 9)
    with pytest.raises(TypeError):
        sp.euclidean(0, 4)
    with pytest.raises(TypeError):
        sp.euclidean(2, 1)
    with pytest.raises(TypeError):
        sp.debug_euclid_pairs([[0, 3]])
    assert sp.euclidean(1, 1).shape == (0, 3)
