"""Pair-matrix hot path of the reference's ``diverse_seq/distance.py`` on the GPU.

Mirrors ``mash_sketches`` (:178-227), ``mash_distance`` (:230-291), ``mash_distances`` (:119-175),
``euclidean_distances`` (:294-332) and ``euclidean_distance`` (:335-336).  The reference wraps the
result in a cogent3 ``DistanceMatrix`` (absent here); :class:`NamedDistances` carries the same
``array`` / ``names`` / ``dists[a, b]`` surface so the callers' use is unchanged.
"""
from __future__ import annotations

from collections.abc import Sequence

import numpy as np

from . import _lib

BottomSketch = list


class NamedDistances:
    def __init__(self, matrix: np.ndarray, names: Sequence[str]):
        self.array = matrix
        self.names = list(names)
        self._index = {n: i for i, n in enumerate(self.names)}

    @classmethod
    def from_array_names(cls, matrix, names):
        return cls(np.asarray(matrix), names)

    def __getitem__(self, key):
        a, b = key
        return float(self.array[self._index[a], self._index[b]])

    def take_dists(self, names):
        idx = [self._index[n] for n in names]
        return NamedDistances(self.array[np.ix_(idx, idx)], names)


def _seqset(ctx, seq_arrays):
    return _lib.SeqSet.from_seqs(ctx, [s.get_seq() for s in seq_arrays])  # LazySeq.get_seq, src/record.rs:263


def mash_sketches(seq_arrays, k: int, sketch_size: int, num_states: int, *, mash_canonical: bool = False,
                  progress=None) -> list[BottomSketch]:
    ctx = _lib.default_context()
    sk = _lib.Sketches.sketch(ctx, _seqset(ctx, seq_arrays), k, int(sketch_size), num_states, mash_canonical)
    data, lens = sk.download()
    return [data[i, : int(lens[i])].tolist() for i in range(len(lens))]


def mash_distance(left_sketch, right_sketch, k: int, sketch_size: int) -> float:
    ctx = _lib.default_context()
    la, lb = len(left_sketch), len(right_sketch)
    stride = max(la, lb, 1)
    sk = np.zeros((2, stride), dtype=np.uint32)
    sk[0, :la] = left_sketch
    sk[1, :lb] = right_sketch
    d = _lib.Sketches.from_host(ctx, sk, np.array([la, lb], dtype=np.uint32)).distances(k, int(sketch_size))
    return float(d[0, 1])


def mash_distances(seq_arrays, k: int, sketch_size: int, num_states: int, *, mash_canonical: bool = False,
                   progress=None) -> NamedDistances:
    ctx = _lib.default_context()
    sk = _lib.Sketches.sketch(ctx, _seqset(ctx, seq_arrays), k, int(sketch_size), num_states, mash_canonical)
    dist = sk.distances(k, int(sketch_size))
    return NamedDistances.from_array_names(dist, [s.seqid for s in seq_arrays])


def counts_sparse_for_euclidean(k: int, num_states: int) -> bool:
    """Whether the Euclidean matrix is formed from sparse k-mer rows (dvs_count_kmers_sparse +
    dvs_euclid_distances_sparse) instead of dense frequency rows: for DNA at 10 <= k <= 12, where a dense row
    takes 4^k x 12 bytes and a pair 2 x 4^k flops.  At k = 9 the dense rows (3 MB) were measured ahead on
    4 Mbp genomes (13 against 18 ms for 256 of them, DESIGN.md §5.11) and stay."""
    return num_states == 4 and 10 <= k <= 12


def euclidean_distances(seq_arrays, k: int, moltype: str = "dna", *, progress=None) -> NamedDistances:
    num_states = seq_arrays[0].num_states if len(seq_arrays) and hasattr(seq_arrays[0], "num_states") else 4
    ctx = _lib.default_context()
    ss = _seqset(ctx, seq_arrays)
    if counts_sparse_for_euclidean(k, num_states):
        dist = _lib.KSparse.count(ctx, ss, k, num_states).euclidean()
    else:
        dist = _lib.KFreqs.count(ctx, ss, k, num_states).euclidean()
    return NamedDistances.from_array_names(dist, [s.seqid for s in seq_arrays])


def euclidean_distance(freq_1: np.ndarray, freq_2: np.ndarray) -> float:
    ctx = _lib.default_context()
    rows = np.stack([np.asarray(freq_1, dtype=np.float64), np.asarray(freq_2, dtype=np.float64)])
    kf = _lib.KFreqs.from_rows(ctx, rows, np.zeros(2))
    return float(kf.euclidean()[0, 1])
