"""References for the Euclidean matrix over sparse k-mer rows (record r = ascending k-mer indices with their counts and
its number of valid k-mers T_r), independent of the GPU kernels:

* `merge_matrix`: frequencies f = c / T, the two index lists merged and (f_a - f_b)^2 summed left to right in index
  order (np.cumsum is a sequential sum).  That is the dense oracle's row-difference sum without its (0 - 0)^2 = +0.0
  terms, i.e. the same bits (tests/test_oracle_euclid_sparse.py asserts it); NaN pairs for records with T = 0.
* `chunked_dense_matrix`: the dense oracle (`oracle.euclid_matrix`, multithreaded C++) on column slices of the dense
  frequency rows, the slices' squared distances added - for records whose pairs are too long for numpy merges
  (4 Mbp genomes at k=12: 3 M entries per row).  Accurate to a few ulps, not bitwise.
"""
import numpy as np


def _freqs(rows, totals):
    return [(np.asarray(i, dtype=np.int64), np.asarray(c, dtype=np.float64) / np.float64(t))
            for (i, c), t in zip(rows, np.asarray(totals, dtype=np.uint64))]


def merge_distance(a, b):
    (ia, fa), (ib, fb) = a, b
    u = np.union1d(ia, ib)
    xa = np.zeros(u.size)
    xb = np.zeros(u.size)
    xa[np.searchsorted(u, ia)] = fa
    xb[np.searchsorted(u, ib)] = fb
    x = xa - xb
    return float(np.sqrt(np.cumsum(x * x)[-1])) if u.size else 0.0


def merge_matrix(rows, totals):
    n = len(rows)
    tot = np.asarray(totals, dtype=np.uint64)
    fr = _freqs(rows, tot)
    dist = np.zeros((n, n))
    for i in range(n):
        for j in range(i):
            d = np.nan if tot[i] == 0 or tot[j] == 0 else merge_distance(fr[i], fr[j])
            dist[i, j] = dist[j, i] = d
    return dist


def chunked_dense_matrix(orc, rows, totals, dim, chunk=1 << 20, threads=1):
    n = len(rows)
    tot = np.asarray(totals, dtype=np.uint64)
    fr = _freqs(rows, tot)
    d2 = np.zeros((n, n))
    for c0 in range(0, dim, chunk):
        c1 = min(dim, c0 + chunk)
        dense = np.zeros((n, c1 - c0))
        for r, (i, f) in enumerate(fr):
            lo, hi = np.searchsorted(i, [c0, c1])
            dense[r, i[lo:hi] - c0] = f[lo:hi]
        d2 += orc.euclid_matrix(dense, threads=threads) ** 2
    d = np.sqrt(d2)
    bad = tot == 0
    d[bad, :] = np.nan
    d[:, bad] = np.nan
    np.fill_diagonal(d, 0.0)
    return d
