"""CPU checks of the sparse-row Euclidean references (tests/sparse_euclid_ref.py): merging two ascending
(index, count) rows and summing (f_a - f_b)^2 in index order must give exactly the bits of the dense oracle's
row-difference sum (the dense sum only adds (0 - 0)^2 = +0.0 on top), NaN pairs for records without a valid k-mer
included; the column-sliced dense form must agree to 1e-12."""
import numpy as np
import pytest

from conftest import random_seqs
from sparse_euclid_ref import chunked_dense_matrix, merge_matrix


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


def sparse_rows(orc, seqs, k):
    rows, totals = [], []
    for s in seqs:
        dense = orc.kcounts(s, k)
        nz = np.flatnonzero(dense)
        rows.append((nz.astype(np.uint32), dense[nz].astype(np.uint32)))
        totals.append(int(dense.sum()))
    return rows, np.array(totals, dtype=np.uint64)


def assert_same_bits(a, b):
    assert a.shape == b.shape
    nan = np.isnan(a)
    assert np.array_equal(nan, np.isnan(b))
    assert np.array_equal(a[~nan].view(np.uint64), b[~nan].view(np.uint64))


@pytest.mark.parametrize("k", [4, 5, 6, 7, 8])
def test_sparse_oracle_is_the_dense_oracle_brca1(orc, brca1, k):
    seqs = list(brca1.values())
    rows, totals = sparse_rows(orc, seqs, k)
    dense = np.stack([orc.kfreqs_unchecked(s, k) for s in seqs])
    exp = orc.euclid_matrix(dense)
    assert_same_bits(merge_matrix(rows, totals), exp)
    got = chunked_dense_matrix(orc, rows, totals, dense.shape[1], chunk=1000)
    np.testing.assert_allclose(got, exp, rtol=1e-12, atol=0)


def test_sparse_oracle_is_the_dense_oracle_ragged_with_empty_records(orc):
    rng = np.random.default_rng(45)
    seqs = random_seqs(rng, 24, 1, 20_000, invalid_rate=0.002)
    seqs[2] = np.zeros(0, dtype=np.uint8)       # empty record
    seqs[9] = np.full(300, 5, dtype=np.uint8)   # no valid k-mer
    seqs[13] = np.zeros(5_000, dtype=np.uint8)  # homopolymer: one k-mer
    rows, totals = sparse_rows(orc, seqs, 6)
    dense = np.stack([orc.kfreqs_unchecked(s, 6) for s in seqs])
    got = merge_matrix(rows, totals)
    exp = orc.euclid_matrix(dense)
    assert_same_bits(got, exp)
    sliced = chunked_dense_matrix(orc, rows, totals, dense.shape[1], chunk=700, threads=2)
    assert np.array_equal(np.isnan(sliced), np.isnan(exp))
    np.testing.assert_allclose(sliced, exp, rtol=1e-12, atol=0)
    nan_rows = np.isnan(got).all(axis=1) | (np.isnan(got).sum(axis=1) == got.shape[0] - 1)
    assert nan_rows[[2, 9]].all() and not nan_rows[[0, 13]].any()
    assert (np.diag(got) == 0).all() and np.isnan(got[2, 9])
