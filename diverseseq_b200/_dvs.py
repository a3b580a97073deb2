"""Drop-in for the hot-path surface of the reference's PyO3 module ``diverse_seq._dvs``
(/root/reference/src/lib.rs:174-189), backed by libdvs_b200.so (CUDA, sm_100a).

Same callables, keyword names, defaults, return attribute names and error types as the
reference, so its callers (diverse_seq/records.py:128,177,203,72,311,371,418;
distance.py:218,326-327; cluster.py:328,377) work unchanged:

    nmost_divergent, max_divergent, final_nmost, final_max, mash_sketch,
    get_delta_jsd_calculator, SummedRecordsResult, LazySeq,
    make_zarr_store / ZarrStoreWrapper (in-memory variant), get_seqids_from_store

There is no CPU fallback: every numeric result comes from the CUDA library and a missing
library / GPU raises.  `make_zarr_store()` gives the in-memory store the reference's tests use as
their fake backend (src/zarr_io.rs:67); `make_zarr_store(path)` opens a `.dvseqsz` directory
(diverseseq_b200/dvseqsz.py, SURVEY.md §8f-1).
"""
from __future__ import annotations

import hashlib

import numpy as np

from . import _lib
from .distance import counts_sparse_for_selection

__all__ = [
    "ZarrStoreWrapper", "SummedRecordsResult", "LazySeq", "make_zarr_store", "get_seqids_from_store",
    "nmost_divergent", "final_nmost", "max_divergent", "final_max", "mash_sketch", "get_delta_jsd_calculator",
]


# ------------------------------------------------------------------------------ storage ----
class ZarrStoreWrapper:
    """In-memory stand-in for the reference's store wrapper (src/zarr_py.rs:9-247).

    One array per UNIQUE sequence content; several seqids may share it (src/zarr_io.rs:217-235).
    """

    def __init__(self, path: str | None = None, mode: str = "r"):
        if path is not None:
            raise NotImplementedError(
                "on-disk .dvseqsz stores are read by the reference's own storage layer; "
                "this module provides the in-memory variant only (make_zarr_store())"
            )
        self._mode = mode
        self._seqid_to_key: dict[str, bytes] = {}
        self._data: dict[bytes, np.ndarray] = {}
        self._meta: dict[bytes, dict[str, str]] = {}

    def __repr__(self) -> str:
        return f"ZarrStoreWrapper(source=:memory:, n={len(self)})"

    def __contains__(self, key: str) -> bool:
        return key in self._seqid_to_key

    def __len__(self) -> int:
        return len(self._seqid_to_key)

    @property
    def source(self) -> str:
        return ":memory:"

    def write(self, seqid: str, seq, metadata: dict | None = None) -> None:
        data = np.frombuffer(bytes(seq), dtype=np.uint8) if not isinstance(seq, np.ndarray) else \
            np.ascontiguousarray(seq, dtype=np.uint8)
        if data.size == 0:  # src/zarr_io.rs:548-551
            raise ValueError(f"Failed to create add {seqid}")
        if seqid in self._seqid_to_key:  # existing seqids are skipped, src/zarr_io.rs:217-219
            return
        key = hashlib.blake2b(data.tobytes(), digest_size=8).digest()
        if key not in self._data:
            self._data[key] = data.copy()
            self._meta[key] = dict(metadata) if metadata else {"source": "unknown"}
        self._seqid_to_key[seqid] = key

    def write_log(self, unique_id: str, data: str) -> None:  # no-op upstream too (zarr_py.rs:171-178)
        return None

    def write_citations(self, data) -> None:
        return None

    def read(self, seqid: str) -> bytes:
        try:
            return self._data[self._seqid_to_key[seqid]].tobytes()
        except KeyError:
            raise RuntimeError(f"Failed to create add {seqid}") from None

    def _array(self, seqid: str) -> np.ndarray:
        try:
            return self._data[self._seqid_to_key[seqid]]
        except KeyError:
            raise RuntimeError(f"Failed to create add {seqid}") from None

    def read_metadata(self, seqid: str) -> dict:
        try:
            return dict(self._meta[self._seqid_to_key[seqid]])
        except KeyError:
            raise RuntimeError(f"Failed to read metadata for {seqid}: not found") from None

    def num_unique(self) -> int:
        return len(self._data)

    @property
    def unique_seqids(self) -> list[str]:
        """one seqid per unique sequence (upstream: arbitrary hash-map order, zarr_io.rs:376-384;
        here: first seqid written for each content, in insertion order)"""
        seen, out = set(), []
        for sid, key in self._seqid_to_key.items():
            if key not in seen:
                seen.add(key)
                out.append(sid)
        return out

    def get_seqids(self) -> list[str]:
        return list(self._seqid_to_key)

    def get_lazyseq(self, seqid: str, num_states: int) -> "LazySeq":
        return LazySeq(seqid, self, num_states)

    def get_lazyseqs(self, num_states: int) -> list["LazySeq"]:
        return [LazySeq(s, self, num_states) for s in self.get_seqids()]


def make_zarr_store(path: str | None = None, mode: str = "r"):
    """src/lib.rs:23-27: no path -> in-memory store, else the `.dvseqsz` directory store"""
    if path is None:
        return ZarrStoreWrapper(None, mode)
    from .dvseqsz import DvseqszStore
    return DvseqszStore(path, mode)


def get_seqids_from_store(path: str) -> list[str]:
    """src/lib.rs:29-34"""
    from .dvseqsz import DvseqszStore
    return DvseqszStore(path, "r").get_seqids()


# ------------------------------------------------------------------------------ results ----
class SummedRecordsResult:
    """Plain-data result, attribute- and pickle-compatible with src/records_py.rs:7-88."""

    __slots__ = ("total_jsd", "records", "mean_delta_jsd", "std_delta_jsd", "cov_delta_jsd", "size", "k",
                 "num_states")
    _FIELDS = __slots__

    def __init__(self):
        self.total_jsd = 0.0
        self.records: list[tuple[str, list[float], float]] = []
        self.mean_delta_jsd = 0.0
        self.std_delta_jsd = 0.0
        self.cov_delta_jsd = 0.0
        self.size = 0
        self.k = 0
        self.num_states = 0

    @property
    def record_names(self) -> list[str]:
        return [r[0] for r in self.records]

    def __getstate__(self) -> dict:
        return {f: getattr(self, f) for f in self._FIELDS}

    def __setstate__(self, state: dict) -> None:
        for f in self._FIELDS:
            if f not in state:
                raise KeyError(f)
            setattr(self, f, state[f])

    def __repr__(self) -> str:
        return f"SummedRecordsResult(size={self.size}, total_jsd={self.total_jsd!r}, k={self.k})"


def _make_result(names, kfreq_rows, deltas, stats, k, num_states, as_lists: bool = True) -> SummedRecordsResult:
    """as_lists=False keeps each record's frequency row a float64 ndarray (the sparse route at k >= 10, where a
    Python list of 4^k floats would take ~0.4 GB per record)"""
    r = SummedRecordsResult()
    r.records = [(names[i], kfreq_rows[i].tolist() if as_lists else kfreq_rows[i], float(deltas[i]))
                 for i in range(len(names))]
    r.total_jsd = float(stats[0])
    r.mean_delta_jsd = float(stats[1])
    r.std_delta_jsd = float(stats[2])
    r.cov_delta_jsd = float(stats[3])
    r.size = len(names)
    r.k = int(k)
    r.num_states = int(num_states)
    return r


def _stat_mode(stat: str) -> int:
    # any value other than "stdev" means cov upstream (src/lib.rs:116-120)
    return _lib.MODE_MAX_STDEV if stat == "stdev" else _lib.MODE_MAX_COV


def _read_array(store, seqid: str) -> np.ndarray:
    """sequence bytes of `seqid` from any store exposing the reference's `read(seqid)` (src/zarr_py.rs:181)"""
    fast = getattr(store, "_array", None)
    return fast(seqid) if fast is not None else np.frombuffer(bytes(store.read(seqid)), dtype=np.uint8)


def _rows_and_order(seqids):
    """distinct seqids -> row index; order[i] = row of seqids[i] (the seqid is the identity)"""
    row_of: dict[str, int] = {}
    order = np.empty(len(seqids), dtype=np.uint32)
    for i, s in enumerate(seqids):
        order[i] = row_of.setdefault(s, len(row_of))
    return list(row_of), order


def _select_from_store(store, seqids, k, num_states, mode, min_size, max_size) -> SummedRecordsResult:
    ctx = _lib.default_context()
    seqids = list(store.unique_seqids if seqids is None else seqids)
    names, order = _rows_and_order(seqids)
    if hasattr(store, "read_into"):  # on-disk .dvseqsz: threaded zstd decode into a pinned staging buffer
        from .dvseqsz import load_seqset
        seqset, _ = load_seqset(ctx, store, names)
    else:
        seqset = _lib.SeqSet.from_seqs(ctx, [_read_array(store, n) for n in names])
    if k == 0:
        raise ValueError("k cannot be 0")
    if len(seqids) < min_size:  # before any counting, like records.rs:323-325
        raise ValueError(f"The number of sequences {len(seqids)} is < n {min_size}")
    if counts_sparse_for_selection(k, num_states):  # no dense row in memory; the same selection bit for bit
        sp = _lib.KSparse.count(ctx, seqset, k, num_states, want_entropy=True)
        idx, delta, stats = sp.select(order, mode, min_size, max_size)
        return _make_result([names[r] for r in idx], sp.dense_rows(idx), delta, stats, k, num_states, as_lists=False)
    # one call: for nmost at k = 4..6 the selection rounds trail the counting (dvs_count_select); every other case runs
    # the two steps back to back inside it, with the same results and errors
    kf, idx, delta, stats = _lib.KFreqs.count_select(ctx, seqset, k, order, mode, min_size, max_size, num_states)
    rows = kf.download_rows(idx)
    return _make_result([names[r] for r in idx], rows, delta, stats, k, num_states)


def nmost_divergent(store, n: int, k: int, num_states: int = 4, seqids=None) -> SummedRecordsResult:
    """src/lib.rs:59-73 -> select_nmost_divergent (src/records.rs:311-342)."""
    return _select_from_store(store, seqids, k, num_states, _lib.MODE_NMOST, n, n)


def max_divergent(store, min_size: int, max_size: int, k: int, num_states: int = 4, seqids=None,
                  stat: str = "stdev") -> SummedRecordsResult:
    """src/lib.rs:105-137 -> select_max_divergent (src/records.rs:390-454)."""
    return _select_from_store(store, seqids, k, num_states, _stat_mode(stat), min_size, max_size)


def _select_from_results(records, mode, min_size, max_size) -> SummedRecordsResult:
    ctx = _lib.default_context()
    names_all, rows_all = [], []
    for sr in records:
        for name, kfreqs, _delta in sr.records:
            names_all.append(name)
            rows_all.append(np.asarray(kfreqs, dtype=np.float64))
    if len(names_all) < min_size:
        raise ValueError(f"The number of sequences {len(names_all)} is < n {min_size}")
    if not names_all:
        raise ValueError("records cannot be empty")
    first_row: dict[str, int] = {}
    order = np.empty(len(names_all), dtype=np.uint32)
    for i, s in enumerate(names_all):
        order[i] = first_row.setdefault(s, i)
    rows = np.stack(rows_all)
    kf = _lib.KFreqs.from_rows(ctx, rows)  # entropy recomputed as KmerSeq::new does (records.rs:353)
    idx, delta, stats = kf.select(order, mode, min_size, max_size)
    # upstream quirk kept on purpose: KmerSeq::new(seqid, kfreqs, sr.k, sr.num_states) is called with
    # k and num_states exchanged (records.rs:353 vs record.rs:157), so the merged result reports them swapped
    k_out, ns_out = records[0].num_states, records[0].k
    return _make_result([names_all[r] for r in idx], rows[idx], delta, stats, k_out, ns_out)


def final_nmost(records, n: int) -> SummedRecordsResult:
    """src/lib.rs:95-103 -> select_nmost_divergent_final (src/records.rs:363-382)."""
    return _select_from_results(list(records), _lib.MODE_NMOST, n, n)


def final_max(records, min_size: int, max_size: int, stat: str = "stdev") -> SummedRecordsResult:
    """src/lib.rs:139-160 -> select_max_divergent_final (src/records.rs:456-507)."""
    return _select_from_results(list(records), _stat_mode(stat), min_size, max_size)


# ------------------------------------------------------------------------------ sketches ----
def mash_sketch(seq_array, k: int, sketch_size: int, num_states: int = 4, mash_canonical: bool = False) -> list[int]:
    """src/distance.rs:136-182: bottom-`sketch_size` distinct k-mer hashes, ascending."""
    ctx = _lib.default_context()
    seqset = _lib.SeqSet.from_seqs(ctx, [_lib.as_u8(seq_array)])
    sk = _lib.Sketches.sketch(ctx, seqset, k, sketch_size, num_states, mash_canonical)
    data, lens = sk.download()
    return data[0, : int(lens[0])].tolist()


# ------------------------------------------------------------------------- delta-JSD app ----
class SummedRecordsWrapper:
    """src/records_py.rs:90-125 (make_summed_records, src/records.rs:509-524)."""

    def __init__(self, records, k: int, num_states: int = 4):
        self._ctx = _lib.default_context()
        self._k, self._num_states = int(k), int(num_states)
        if self._k == 0:
            raise ValueError("k cannot be 0")
        names = [r[0] for r in records]
        seqset = _lib.SeqSet.from_seqs(self._ctx, [_lib.as_u8(r[1]) for r in records])
        self._kf = _lib.KFreqs.count(self._ctx, seqset, self._k, self._num_states)
        valid = self._kf.download(counts=False, freqs=False)[3]
        members = [i for i in range(len(names)) if valid[i]]  # records without k-mers are dropped (:519-521)
        self._names = names
        self._member_names = {names[i] for i in members}
        self._summed = _lib.Summed(self._ctx, self._kf, members)

    def delta_jsd(self, seqid: str, seq) -> float:
        seqset = _lib.SeqSet.from_seqs(self._ctx, [_lib.as_u8(seq)])
        q = _lib.KFreqs.count(self._ctx, seqset, self._k, self._num_states)
        if not q.download(counts=False, freqs=False)[3][0]:
            raise ValueError(f"delta_jsd('{seqid}') failed: No valid k-mers for '{seqid}'")
        return self._summed.delta_jsd(q, 0, is_member=seqid in self._member_names)

    def delta_jsd_many(self, seqids_seqs) -> list[float]:
        """batch form of delta_jsd (one count + one scoring launch for all queries); same values and the
        same ValueError for a query without valid k-mers"""
        seqids_seqs = list(seqids_seqs)
        seqset = _lib.SeqSet.from_seqs(self._ctx, [_lib.as_u8(s) for _, s in seqids_seqs])
        q = _lib.KFreqs.count(self._ctx, seqset, self._k, self._num_states)
        member = np.array([sid in self._member_names for sid, _ in seqids_seqs], dtype=np.uint8)
        out = self._summed.delta_jsd_batch(q, member)
        for (sid, _), v in zip(seqids_seqs, out):
            if v != v:
                raise ValueError(f"delta_jsd('{sid}') failed: No valid k-mers for '{sid}'")
        return out.tolist()

    def get_result(self) -> SummedRecordsResult:
        idx, delta, stats, _low = self._summed.result()
        rows = self._kf.download_rows(idx)
        return _make_result([self._names[r] for r in idx], rows, delta, stats, self._k, self._num_states)


def get_delta_jsd_calculator(seqids_seqs, k: int, num_states: int = 4) -> SummedRecordsWrapper:
    """src/lib.rs:162-171"""
    return SummedRecordsWrapper(list(seqids_seqs), k, num_states)


# ------------------------------------------------------------------------------ LazySeq ----
class LazySeq:
    """src/record.rs:212-269"""

    def __init__(self, seqid: str, storage: ZarrStoreWrapper, num_states: int):
        self._seqid, self._storage, self._num_states = seqid, storage, int(num_states)

    @property
    def seqid(self) -> str:
        return self._seqid

    @property
    def num_states(self) -> int:
        return self._num_states

    def __repr__(self) -> str:
        return f"LazySeq(seqid={self._seqid}, num_states={self._num_states}, storage={self._storage!r})"

    def _count(self, k: int):
        if k == 0:
            raise ValueError("k cannot be 0")
        ctx = _lib.default_context()
        seqset = _lib.SeqSet.from_seqs(ctx, [_read_array(self._storage, self._seqid)])
        return _lib.KFreqs.count(ctx, seqset, k, self._num_states)

    def get_kcounts(self, k: int) -> list[int]:
        return self._count(k).download(freqs=False)[0][0].tolist()

    def get_kfreqs(self, k: int) -> list[float]:
        return self._count(k).download(counts=False)[1][0].tolist()

    def get_seq(self) -> bytes:
        return self._storage.read(self._seqid)
