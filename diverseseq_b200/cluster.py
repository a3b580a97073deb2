"""Tail of `dvs ctree` on the GPU: average-linkage cluster tree from k-mer distances.

Mirrors the tree-building part of the reference's ``diverse_seq/cluster.py``:
  :99-188   dvs_ctree.main        distances (mash | euclidean) -> make_cluster_tree
  :191-237  make_cluster_tree     sklearn AgglomerativeClustering(metric="precomputed",
                                  linkage="average").children_ -> nested tuples -> tree string
The linkage runs in csrc/cluster.cu (`dvs_linkage_average`) and returns sklearn's ``children_``
bit-for-bit, ties included.  The reference hands the string to cogent3's ``make_tree`` (absent here);
:class:`ClusterTree` keeps the same string plus the merge table.  With ``dvs_ctree`` the distance
matrix never leaves the device: the kernels of distance.py write it to device memory and the linkage
reads it there.
"""
from __future__ import annotations

from collections.abc import Sequence

import numpy as np

from . import _lib
from .distance import counts_sparse_for_euclidean


class ClusterTree:
    """The tree make_cluster_tree builds: ``treestring`` is what the reference passes to
    ``make_tree(treestring=..., underscore_unmunge=True)``; ``children`` is sklearn's ``children_``."""

    def __init__(self, names: Sequence[str], children: np.ndarray, heights: np.ndarray, counts: np.ndarray):
        self.names = list(names)
        self.children = children
        self.heights = heights
        self.counts = counts

    @property
    def nested(self):
        """nested 2-tuples of names in merge order (cluster.py:222-230)"""
        n = len(self.names)
        if n == 1:
            return self.names[0]
        node = {i: self.names[i] for i in range(n)}
        nxt = n
        for left, right in self.children:
            node[nxt] = (node.pop(int(left)), node.pop(int(right)))
            nxt += 1
        return node[nxt - 1]

    @property
    def treestring(self) -> str:
        return str(self.nested).replace("'", "")  # cluster.py:232

    def get_tip_names(self) -> list[str]:
        out, stack = [], [self.nested]
        while stack:
            t = stack.pop()
            if isinstance(t, tuple):
                stack.extend(reversed(t))
            else:
                out.append(t)
        return out

    def __str__(self) -> str:
        return self.treestring + ";"


def make_cluster_tree(seq_names: Sequence[str], pairwise_distances, *, progress=None,
                      ctx: _lib.Context | None = None) -> ClusterTree:
    """Given pairwise distances between sequences, construct a cluster tree (cluster.py:191-237).
    `pairwise_distances`: numpy n x n array, an object with ``.array`` (distance.NamedDistances), or a
    (device_ptr, n) pair for a matrix already in device memory."""
    ctx = ctx or _lib.default_context()
    if isinstance(pairwise_distances, tuple):
        dptr, n = pairwise_distances
        children, heights, counts = _lib.linkage_average(ctx, n=n, device_ptr=dptr)
    else:
        d = getattr(pairwise_distances, "array", pairwise_distances)
        children, heights, counts = _lib.linkage_average(ctx, np.asarray(d))
    if len(seq_names) != children.shape[0] + 1:
        raise ValueError("number of names does not match the distance matrix")
    return ClusterTree(seq_names, children, heights, counts)


class dvs_ctree:
    """Create a cluster tree from kmer distances (cluster.py:99-188): sequences are records of
    index-encoded bytes (`LazySeq`-like objects with ``get_seq()``, or uint8 arrays)."""

    def __init__(self, *, k: int = 12, sketch_size: int | None = 3_000, moltype: str = "dna",
                 distance_mode: str = "mash", mash_canonical_kmers: bool | None = None,
                 show_progress: bool = False, ctx: _lib.Context | None = None) -> None:
        if mash_canonical_kmers is None:
            mash_canonical_kmers = False
        if distance_mode not in ("mash", "euclidean"):
            raise ValueError(f"Unexpected distance {distance_mode!r}.")
        if moltype not in ("dna", "rna") and mash_canonical_kmers:
            raise ValueError("Canonical kmers only supported for dna/rna sequences.")
        if distance_mode == "mash" and sketch_size is None:
            raise ValueError("Expected sketch size for mash distance measure.")
        self._k, self._sketch_size, self._moltype = k, sketch_size, moltype
        self._distance_mode, self._mash_canonical = distance_mode, mash_canonical_kmers
        self._num_states = 4 if moltype in ("dna", "rna") else 20
        self._ctx = ctx

    def __call__(self, seq_names, seqs) -> ClusterTree:
        return self.main(seq_names, seqs)

    def main(self, seq_names: Sequence[str], seqs) -> ClusterTree:
        ctx = self._ctx or _lib.default_context()
        arrays = [s.get_seq() if hasattr(s, "get_seq") else s for s in seqs]
        ss = _lib.SeqSet.from_seqs(ctx, arrays)
        n = ss.nrec
        if n < 2:
            return ClusterTree(seq_names, np.zeros((0, 2), np.int32), np.zeros(0), np.zeros(0, np.uint32))
        dmat = _lib.DeviceBuffer(ctx, n * n * 8)  # the matrix never leaves the device
        if self._distance_mode == "mash":
            sk = _lib.Sketches.sketch(ctx, ss, self._k, int(self._sketch_size), self._num_states, self._mash_canonical)
            sk.distances_into(dmat.ptr, self._k, int(self._sketch_size))
        elif counts_sparse_for_euclidean(self._k, self._num_states):
            _lib.KSparse.count(ctx, ss, self._k, self._num_states).euclidean_into(dmat.ptr)
        else:
            kf = _lib.KFreqs.count(ctx, ss, self._k, self._num_states)
            kf.euclidean_into(dmat.ptr)
        tree = make_cluster_tree(seq_names, (dmat.ptr, n), ctx=ctx)
        dmat.close()
        return tree
