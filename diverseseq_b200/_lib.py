"""ctypes binding of libdvs_b200.so (C ABI: include/dvs_b200.h).

The library is built in-tree by ``__graft_entry__.build()`` / ``make -C diverseseq_b200/csrc``.
There is no CPU fallback: a missing library or a missing CUDA device is an error.
"""
from __future__ import annotations

import ctypes as C
import pathlib
import threading

import numpy as np

_HERE = pathlib.Path(__file__).resolve().parent
LIB_PATH = _HERE / "libdvs_b200.so"

DVS_OK, DVS_ERR_VALUE, DVS_ERR_CUDA, DVS_ERR_ARG = 0, 1, 2, 3
MODE_NMOST, MODE_MAX_STDEV, MODE_MAX_COV = 0, 1, 2
PHASE_COUNT_KERNEL, PHASE_FREQ_ENTROPY, PHASE_SELECT, PHASE_SKETCH, PHASE_MASH_PAIRS, PHASE_EUCLID, PHASE_UPLOAD = range(7)
PHASE_PREP = 7
PHASE_CLUSTER = 8
PHASE_SPARSE = 9
PHASE_COUNT_LAUNCHES = 10
PHASE_EUCLID_SPARSE = 11
PHASE_EUCLID_SPARSE_ROWS = 12

_vp = C.c_void_p
_u32, _u64, _i32, _f64 = C.c_uint32, C.c_uint64, C.c_int, C.c_double

# name -> (restype, argtypes); every symbol include/dvs_b200.h declares
SIGNATURES = {
    "dvs_last_error": (C.c_char_p, []),
    "dvs_version": (C.c_char_p, []),
    "dvs_ctx_create": (_i32, [_i32, C.POINTER(_vp)]),
    "dvs_ctx_destroy": (None, [_vp]),
    "dvs_ctx_sync": (_i32, [_vp]),
    "dvs_ctx_stream": (_vp, [_vp]),
    "dvs_ctx_launch_count": (_u64, [_vp]),
    "dvs_ctx_last_upload_wire_bytes": (_u64, [_vp]),
    "dvs_ctx_enable_timing": (_i32, [_vp, _i32]),
    "dvs_ctx_phase_ms": (_f64, [_vp, _i32]),
    "dvs_device_malloc": (_i32, [_vp, _u64, C.POINTER(_vp)]),
    "dvs_device_free": (None, [_vp, _vp]),
    "dvs_device_memcpy": (_i32, [_vp, _vp, _vp, _u64]),
    "dvs_host_malloc_pinned": (_i32, [_u64, C.POINTER(_vp)]),
    "dvs_host_free_pinned": (None, [_vp]),
    "dvs_seqset_upload": (_i32, [_vp, _vp, _vp, _u32, C.POINTER(_vp)]),
    "dvs_seqset_synth": (_i32, [_vp, _u64, _u32, _u32, _u64, C.POINTER(_vp)]),
    "dvs_seqset_synth_range": (_i32, [_vp, _u64, _u32, _u32, _u32, _u64, C.POINTER(_vp)]),
    "dvs_synth_host": (_i32, [_u64, _u32, _u32, _u64, _u32, _u32, _vp, _vp]),
    "dvs_synth_lengths": (_i32, [_u64, _u32, _u64, _vp]),
    "dvs_seqset_nrec": (_u32, [_vp]),
    "dvs_seqset_total_bases": (_u64, [_vp]),
    "dvs_seqset_offsets": (_i32, [_vp, _vp]),
    "dvs_seqset_download": (_i32, [_vp, _vp, _u32, _u32, _vp]),
    "dvs_seqset_free": (None, [_vp]),
    "dvs_linkage_average": (_i32, [_vp, _vp, _u32, _vp, _vp, _vp]),
    "dvs_prep_fasta": (_i32, [_vp, _vp, _vp, _u32, C.c_char_p, C.c_char_p, _i32, _i32, C.POINTER(_vp)]),
    "dvs_count_kmers": (_i32, [_vp, _vp, _i32, _i32, C.POINTER(_vp)]),
    "dvs_kfreqs_from_rows": (_i32, [_vp, _vp, _vp, _u32, _u64, C.POINTER(_vp)]),
    "dvs_kfreqs_device_ptrs": (_i32, [_vp, C.POINTER(_vp), C.POINTER(_vp), C.POINTER(_vp)]),
    "dvs_kfreqs_from_device": (_i32, [_vp, _vp, _vp, _vp, _u32, _u64, C.POINTER(_vp)]),
    "dvs_kfreqs_take_rows": (_i32, [_vp, _vp, _vp, _u32, C.POINTER(_vp)]),
    "dvs_kfreqs_nrec": (_u32, [_vp]),
    "dvs_kfreqs_dim": (_u64, [_vp]),
    "dvs_kfreqs_download": (_i32, [_vp, _vp, _u32, _u32, _vp, _vp, _vp, _vp]),
    "dvs_kfreqs_free": (None, [_vp]),
    "dvs_count_kmers_host": (_i32, [_vp, _vp, _vp, _u32, _i32, _i32, _vp, _vp, _vp, _vp]),
    "dvs_count_kmers_sparse": (_i32, [_vp, _vp, _i32, _i32, _i32, C.POINTER(_vp)]),
    "dvs_ksparse_nrec": (_u32, [_vp]),
    "dvs_ksparse_stats": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp]),
    "dvs_ksparse_download": (_i32, [_vp, _vp, _u32, _vp, _vp, _u64, C.POINTER(_u64)]),
    "dvs_ksparse_free": (None, [_vp]),
    "dvs_euclid_distances_sparse": (_i32, [_vp, _vp, _u32, _u32, _vp]),
    "dvs_select": (_i32, [_vp, _vp, _vp, _u32, _i32, _u32, _u32, _vp, _vp, _vp, C.POINTER(_u32)]),
    "dvs_count_select": (_i32, [_vp, _vp, _i32, _i32, _vp, _u32, _i32, _u32, _u32, _u32, C.POINTER(_vp), _vp, _vp, _vp,
                                C.POINTER(_u32)]),
    "dvs_select_last_accepts": (_u32, [_vp]),
    "dvs_select_last_exact_evals": (_u32, [_vp]),
    "dvs_select_last_trail_accepts": (_u32, [_vp]),
    "dvs_select_last_trail_launches": (_u32, [_vp]),
    "dvs_select_last_trail_sms": (_u32, [_vp]),
    "dvs_summed_create": (_i32, [_vp, _vp, _vp, _u32, C.POINTER(_vp)]),
    "dvs_summed_delta_jsd": (_i32, [_vp, _vp, _vp, _u32, _i32, C.POINTER(_f64)]),
    "dvs_summed_delta_jsd_batch": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "dvs_summed_result": (_i32, [_vp, _vp, _vp, _vp, _vp, C.POINTER(_u32), C.POINTER(_u32)]),
    "dvs_summed_free": (None, [_vp]),
    "dvs_mash_sketch": (_i32, [_vp, _vp, _i32, _u64, _i32, _i32, C.POINTER(_vp)]),
    "dvs_sketches_from_host": (_i32, [_vp, _vp, _u32, _vp, _u32, C.POINTER(_vp)]),
    "dvs_sketches_nrec": (_u32, [_vp]),
    "dvs_sketches_stride": (_u32, [_vp]),
    "dvs_sketches_download": (_i32, [_vp, _vp, _vp, _vp]),
    "dvs_sketches_free": (None, [_vp]),
    "dvs_mash_distances": (_i32, [_vp, _vp, _i32, _u64, _u32, _u32, _vp, _vp, _vp]),
    "dvs_mash_sketch_host": (_i32, [_vp, _vp, _u64, _i32, _u64, _i32, _i32, _vp, _u64, C.POINTER(_u64)]),
    "dvs_euclid_distances": (_i32, [_vp, _vp, _u32, _u32, _vp]),
    "dvs_euclid_last_fallback_pairs": (_u32, [_vp]),
    "dvs_comm_create": (_i32, [_vp, _i32, _i32, _u64, C.POINTER(_vp), _vp]),
    "dvs_comm_connect": (_i32, [_vp, _vp, _vp]),
    "dvs_comm_set_host_barrier": (_i32, [_vp, _vp, _vp]),
    "dvs_comm_rank": (_i32, [_vp]),
    "dvs_comm_world": (_i32, [_vp]),
    "dvs_comm_barrier": (_i32, [_vp, _vp]),
    "dvs_comm_allgatherv": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "dvs_comm_destroy": (None, [_vp]),
    "dvs_count_kmers_sharded": (_i32, [_vp, _vp, _vp, _i32, _i32, _vp, C.POINTER(_vp)]),
    "dvs_kfreqs_allgather": (_i32, [_vp, _vp, _vp, _vp, C.POINTER(_vp)]),
    "dvs_sketches_allgather": (_i32, [_vp, _vp, _vp, _vp, _u32, C.POINTER(_vp)]),
    "dvs_mash_distances_sharded": (_i32, [_vp, _vp, _vp, _i32, _u64, _vp]),
    "dvs_euclid_distances_sharded": (_i32, [_vp, _vp, _vp, _vp]),
    "dvs_euclid_distances_sparse_sharded": (_i32, [_vp, _vp, _vp, _vp, _vp]),
    "dvs_select_sharded": (_i32, [_vp, _vp, _vp, _vp, _u32, _i32, _u32, _u32, _vp, _vp, _vp, C.POINTER(_u32)]),
    "dvs_debug_pack_host": (_i32, [_vp, _u64, _vp, _vp, _vp, _u32, C.POINTER(_u32)]),
    "dvs_debug_log2": (_i32, [_vp, _vp, _vp, _u64]),
    "dvs_debug_fast_terms": (_i32, [_vp, _vp, _vp, _vp, _vp, _vp, _u64]),
    "dvs_debug_entropy": (_i32, [_vp, _vp, _u32, _u64, _vp, _vp]),
    "dvs_debug_euclid_sparse_pairs": (_i32, [_vp, _vp, _vp, _u32, _vp]),
}

_lib = None
_lock = threading.Lock()
_shutdown = False


def _at_exit() -> None:
    """interpreter shutdown: objects finalised from here on must not call into the CUDA runtime any more
    (its own teardown may already be under way); the process exit releases everything"""
    global _shutdown
    _shutdown = True


import atexit  # noqa: E402

atexit.register(_at_exit)


def load() -> C.CDLL:
    """Load libdvs_b200.so (no GPU needed to load; needed to create a context)."""
    global _lib
    with _lock:
        if _lib is None:
            if not LIB_PATH.exists():
                raise RuntimeError(
                    f"{LIB_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                    "or `make -C diverseseq_b200/csrc`. There is no CPU fallback."
                )
            lib = C.CDLL(str(LIB_PATH))
            for name, (res, args) in SIGNATURES.items():
                fn = getattr(lib, name)  # AttributeError here == header/library mismatch
                fn.restype = res
                fn.argtypes = args
            _lib = lib
    return _lib


def last_error() -> str:
    return load().dvs_last_error().decode(errors="replace")


def check(rc: int) -> None:
    if rc == DVS_OK:
        return
    msg = last_error()
    if rc == DVS_ERR_VALUE:
        if msg == "division by zero":
            raise ZeroDivisionError(msg)
        raise ValueError(msg)  # what the reference raises for a Rust panic (src/lib.rs:36-57)
    if rc == DVS_ERR_CUDA:
        raise RuntimeError(msg)
    raise TypeError(msg) if rc == DVS_ERR_ARG else RuntimeError(msg)


def ptr(a):
    """void* of a C-contiguous numpy array (or None)."""
    if a is None:
        return None
    assert a.flags["C_CONTIGUOUS"]
    return a.ctypes.data_as(_vp)


class Context:
    """One CUDA context/stream for the hot path on one GPU (dvs_ctx)."""

    def __init__(self, device: int = 0):
        self._lib = load()
        h = _vp()
        check(self._lib.dvs_ctx_create(int(device), C.byref(h)))
        self.handle = h
        self.device = int(device)

    def close(self) -> None:
        if getattr(self, "handle", None) and not _shutdown:
            self._lib.dvs_ctx_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def sync(self) -> None:
        check(self._lib.dvs_ctx_sync(self.handle))

    def enable_timing(self, on: bool = True) -> None:
        check(self._lib.dvs_ctx_enable_timing(self.handle, int(on)))

    def phase_ms(self, phase: int) -> float:
        return float(self._lib.dvs_ctx_phase_ms(self.handle, int(phase)))

    @property
    def stream(self) -> int:
        return int(self._lib.dvs_ctx_stream(self.handle) or 0)

    @property
    def last_upload_wire_bytes(self) -> int:
        return int(self._lib.dvs_ctx_last_upload_wire_bytes(self.handle))

    @property
    def launch_count(self) -> int:
        return int(self._lib.dvs_ctx_launch_count(self.handle))


class DeviceBuffer:
    """plain device memory owned by the library (dvs_device_malloc); `.ptr` is the raw device pointer"""

    def __init__(self, ctx: Context, nbytes: int):
        self.ctx, self.nbytes = ctx, int(nbytes)
        p = _vp()
        check(ctx._lib.dvs_device_malloc(ctx.handle, self.nbytes, C.byref(p)))
        self.ptr = int(p.value)

    def to_host(self, dtype, shape) -> np.ndarray:
        out = np.empty(shape, dtype=dtype)
        assert out.nbytes <= self.nbytes
        check(self.ctx._lib.dvs_device_memcpy(self.ctx.handle, ptr(out), _vp(self.ptr), out.nbytes))
        return out

    def from_host(self, a: np.ndarray) -> None:
        a = np.ascontiguousarray(a)
        assert a.nbytes <= self.nbytes
        check(self.ctx._lib.dvs_device_memcpy(self.ctx.handle, _vp(self.ptr), ptr(a), a.nbytes))

    def close(self) -> None:
        if getattr(self, "ptr", 0) and not _shutdown and getattr(self.ctx, "handle", None):
            self.ctx._lib.dvs_device_free(self.ctx.handle, _vp(self.ptr))
        self.ptr = 0

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Pinned:
    def __init__(self, lib, p):
        self.lib, self.p = lib, p

    def __del__(self):
        try:
            if self.p and not _shutdown:
                self.lib.dvs_host_free_pinned(self.p)
        except Exception:
            pass


def pinned_array(nbytes: int) -> np.ndarray:
    """uint8 numpy array over page-locked host memory (dvs_host_malloc_pinned); freed with the array"""
    lib = load()
    p = _vp()
    check(lib.dvs_host_malloc_pinned(int(max(nbytes, 1)), C.byref(p)))
    owner = _Pinned(lib, p)
    buf = (C.c_uint8 * int(max(nbytes, 1))).from_address(p.value)
    arr = np.frombuffer(buf, dtype=np.uint8)
    _PINNED_OWNERS[id(buf)] = owner  # the ctypes buffer (kept alive by arr.base) keeps the allocation alive
    import weakref
    weakref.finalize(buf, _PINNED_OWNERS.pop, id(buf), None)
    return arr


_PINNED_OWNERS: dict = {}
_default_ctx: dict[int, Context] = {}


def default_context(device: int | None = None) -> Context:
    """Process-wide context per device; device defaults to $LOCAL_RANK or 0."""
    import os

    if device is None:
        device = int(os.environ.get("DVS_DEVICE", os.environ.get("LOCAL_RANK", "0")))
    ctx = _default_ctx.get(device)
    if ctx is None or ctx.handle is None:
        ctx = _default_ctx[device] = Context(device)
    return ctx


class _Handle:
    _free = None

    def __init__(self, ctx: Context, handle):
        self.ctx = ctx
        self.handle = handle

    def close(self) -> None:
        # a handle that outlives its context (or the interpreter) is left to the process exit
        if getattr(self, "handle", None) and not _shutdown and getattr(self.ctx, "handle", None):
            getattr(self.ctx._lib, self._free)(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


def as_u8(a) -> np.ndarray:
    if isinstance(a, (bytes, bytearray, memoryview)):
        return np.frombuffer(a, dtype=np.uint8)
    return np.ascontiguousarray(a, dtype=np.uint8)


def concat(seqs) -> tuple[np.ndarray, np.ndarray]:
    arrs = [as_u8(s) for s in seqs]
    offsets = np.zeros(len(arrs) + 1, dtype=np.uint64)
    if arrs:
        offsets[1:] = np.cumsum([a.size for a in arrs], dtype=np.uint64)
    flat = np.concatenate(arrs) if arrs and int(offsets[-1]) else np.zeros(0, dtype=np.uint8)
    return np.ascontiguousarray(flat), offsets


class SeqSet(_Handle):
    """Device-resident batch of encoded sequences (dvs_seqset)."""

    _free = "dvs_seqset_free"

    @classmethod
    def upload(cls, ctx: Context, flat: np.ndarray, offsets: np.ndarray) -> "SeqSet":
        flat = as_u8(flat)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        h = _vp()
        check(ctx._lib.dvs_seqset_upload(ctx.handle, ptr(flat) if flat.size else None, ptr(offsets),
                                         len(offsets) - 1, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_seqs(cls, ctx: Context, seqs) -> "SeqSet":
        return cls.upload(ctx, *concat(seqs))

    @classmethod
    def synth(cls, ctx: Context, seed: int, nrec: int, nfam: int, mean_len: int, first: int = 0) -> "SeqSet":
        """`nrec` synthetic records starting at record `first` of the generator keyed by `seed`"""
        h = _vp()
        check(ctx._lib.dvs_seqset_synth_range(ctx.handle, seed, first, nrec, nfam, mean_len, C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def prep_fasta(cls, ctx: Context, text, file_offsets, alphabet: str | None = None,
                   delete_chars: bytes | None = None, sep_char: int = -1, device_ptr: int | None = None) -> "SeqSet":
        """FASTA text of several files -> one encoded record per file (dvs_prep_fasta).  `text` is a
        uint8 array / bytes holding the files back to back, or None with `device_ptr` (device text)."""
        file_offsets = np.ascontiguousarray(file_offsets, dtype=np.uint64)
        h = _vp()
        if device_ptr is not None:
            tp, on_dev = _vp(device_ptr), 1
        else:
            text = as_u8(text)
            tp, on_dev = (ptr(text) if text.size else None), 0
        check(ctx._lib.dvs_prep_fasta(ctx.handle, tp, ptr(file_offsets), len(file_offsets) - 1,
                                      alphabet.encode() if alphabet is not None else None,
                                      delete_chars, sep_char, on_dev, C.byref(h)))
        return cls(ctx, h)

    @property
    def nrec(self) -> int:
        return int(self.ctx._lib.dvs_seqset_nrec(self.handle))

    @property
    def total_bases(self) -> int:
        return int(self.ctx._lib.dvs_seqset_total_bases(self.handle))

    def offsets(self) -> np.ndarray:
        out = np.zeros(self.nrec + 1, dtype=np.uint64)
        check(self.ctx._lib.dvs_seqset_offsets(self.handle, ptr(out)))
        return out

    def download(self, first: int = 0, count: int | None = None, out: np.ndarray | None = None) -> np.ndarray:
        count = self.nrec - first if count is None else count
        off = self.offsets()
        n = int(off[first + count] - off[first])
        if out is None:
            out = np.empty(max(n, 1), dtype=np.uint8)
        check(self.ctx._lib.dvs_seqset_download(self.ctx.handle, self.handle, first, count, ptr(out)))
        return out[:n]


def synth_host(seed: int, nrec: int, nfam: int, mean_len: int, first: int = 0, count: int | None = None):
    """host twin of SeqSet.synth: (flat bytes, offsets) of records [first, first+count)"""
    lib = load()
    count = nrec - first if count is None else count
    lens = np.zeros(nrec, dtype=np.uint64)
    check(lib.dvs_synth_lengths(seed, nrec, mean_len, ptr(lens)))
    total = int(lens[first:first + count].sum())
    flat = np.empty(max(total, 1), dtype=np.uint8)
    offsets = np.zeros(count + 1, dtype=np.uint64)
    check(lib.dvs_synth_host(seed, nrec, nfam, mean_len, first, count, ptr(flat), ptr(offsets)))
    return flat[:total], offsets


class KFreqs(_Handle):
    """Device-resident k-mer frequency rows + entropies (dvs_kfreqs)."""

    _free = "dvs_kfreqs_free"

    @classmethod
    def count(cls, ctx: Context, seqset: SeqSet, k: int, num_states: int = 4) -> "KFreqs":
        h = _vp()
        check(ctx._lib.dvs_count_kmers(ctx.handle, seqset.handle, int(k), int(num_states), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def count_select(cls, ctx: Context, seqset: SeqSet, k: int, order, mode: int, min_size: int, max_size: int = 0,
                     num_states: int = 4, chunks: int = 0):
        """dvs_count_select: counting with the nmost rounds trailing it; returns (KFreqs, indices, delta_jsd, stats5)"""
        order = np.ascontiguousarray(order, dtype=np.uint32)
        cap = max(int(min_size), int(max_size), 1) + 1
        if int(mode) != MODE_NMOST and int(max_size) < int(min_size):
            cap = order.size + 1
        idx = np.zeros(cap, dtype=np.uint32)
        delta = np.zeros(cap, dtype=np.float64)
        stats = np.zeros(5, dtype=np.float64)
        size = _u32(0)
        h = _vp()
        check(ctx._lib.dvs_count_select(ctx.handle, seqset.handle, int(k), int(num_states),
                                        ptr(order) if order.size else None, order.size, int(mode), int(min_size),
                                        int(max_size), int(chunks), C.byref(h), ptr(idx), ptr(delta), ptr(stats),
                                        C.byref(size)))
        n = size.value
        return cls(ctx, h), idx[:n].copy(), delta[:n].copy(), stats

    @classmethod
    def count_sharded(cls, ctx: Context, comm: "Comm", seqset: SeqSet, k: int, nrec_per_rank, num_states: int = 4) -> "KFreqs":
        """count this rank's records; the result holds the rows of ALL ranks (rank-major) on every rank"""
        npr = np.ascontiguousarray(nrec_per_rank, dtype=np.uint32)
        h = _vp()
        check(ctx._lib.dvs_count_kmers_sharded(ctx.handle, comm.handle, seqset.handle, int(k), int(num_states), ptr(npr),
                                               C.byref(h)))
        out = cls(ctx, h)
        out._comm = comm  # the rows live in the communicator's window: keep it alive
        return out

    def allgather(self, comm: "Comm", nrec_per_rank) -> "KFreqs":
        npr = np.ascontiguousarray(nrec_per_rank, dtype=np.uint32)
        h = _vp()
        check(self.ctx._lib.dvs_kfreqs_allgather(self.ctx.handle, comm.handle, self.handle, ptr(npr), C.byref(h)))
        out = KFreqs(self.ctx, h)
        out._comm = comm
        return out

    def select_sharded(self, comm: "Comm", order, mode: int, min_size: int, max_size: int = 0):
        """single-pass selection over the rows of all ranks, candidate-sharded over the GPUs (dvs_select_sharded)"""
        order = np.ascontiguousarray(order, dtype=np.uint32)
        cap = max(int(min_size), int(max_size), 1) + 1
        if int(mode) != MODE_NMOST and int(max_size) < int(min_size):
            cap = order.size + 1
        idx = np.zeros(cap, dtype=np.uint32)
        delta = np.zeros(cap, dtype=np.float64)
        stats = np.zeros(5, dtype=np.float64)
        size = _u32(0)
        check(self.ctx._lib.dvs_select_sharded(self.ctx.handle, comm.handle, self.handle, ptr(order) if order.size else None,
                                               order.size, int(mode), int(min_size), int(max_size), ptr(idx), ptr(delta),
                                               ptr(stats), C.byref(size)))
        n = size.value
        return idx[:n].copy(), delta[:n].copy(), stats

    @classmethod
    def from_rows(cls, ctx: Context, rows: np.ndarray, entropies: np.ndarray | None = None) -> "KFreqs":
        rows = np.ascontiguousarray(rows, dtype=np.float64)
        ent = None if entropies is None else np.ascontiguousarray(entropies, dtype=np.float64)
        h = _vp()
        check(ctx._lib.dvs_kfreqs_from_rows(ctx.handle, ptr(rows), ptr(ent), rows.shape[0], rows.shape[1], C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_device(cls, ctx: Context, rows_ptr: int, ent_ptr: int | None, valid_ptr: int | None, nrec: int,
                    dim: int) -> "KFreqs":
        """device-to-device copy from gathered device buffers (raw pointers on ctx's GPU); ent_ptr None
        recomputes the entropies from the rows (KmerSeq::new), valid_ptr None marks every row valid"""
        h = _vp()
        check(ctx._lib.dvs_kfreqs_from_device(ctx.handle, _vp(rows_ptr), _vp(ent_ptr) if ent_ptr else None,
                                              _vp(valid_ptr) if valid_ptr else None, nrec, dim, C.byref(h)))
        return cls(ctx, h)

    def take_rows(self, rows) -> "KFreqs":
        """device gather of the given rows into a new KFreqs (the records of a selection result)"""
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        h = _vp()
        check(self.ctx._lib.dvs_kfreqs_take_rows(self.ctx.handle, self.handle, ptr(rows) if rows.size else None,
                                                 rows.size, C.byref(h)))
        return KFreqs(self.ctx, h)

    def download_rows(self, rows) -> np.ndarray:
        """frequency rows `rows` as one [len(rows), dim] f64 array: one device gather + one copy (the
        records of a SummedRecordsResult) instead of one round trip per row"""
        rows = np.ascontiguousarray(rows, dtype=np.uint32)
        if rows.size == 0:
            return np.zeros((0, self.dim), dtype=np.float64)
        taken = self.take_rows(rows)
        out = taken.download(counts=False)[1]
        taken.close()
        return out

    def device_ptrs(self) -> tuple[int, int, int]:
        a, b, c = _vp(), _vp(), _vp()
        check(self.ctx._lib.dvs_kfreqs_device_ptrs(self.handle, C.byref(a), C.byref(b), C.byref(c)))
        return int(a.value or 0), int(b.value or 0), int(c.value or 0)

    @property
    def nrec(self) -> int:
        return int(self.ctx._lib.dvs_kfreqs_nrec(self.handle))

    @property
    def dim(self) -> int:
        return int(self.ctx._lib.dvs_kfreqs_dim(self.handle))

    def download(self, first: int = 0, count: int | None = None, counts=True, freqs=True):
        count = self.nrec - first if count is None else count
        d = self.dim
        c = np.zeros((count, d), dtype=np.uint64) if counts else None
        f = np.zeros((count, d), dtype=np.float64) if freqs else None
        e = np.zeros(count, dtype=np.float64)
        v = np.zeros(count, dtype=np.uint8)
        check(self.ctx._lib.dvs_kfreqs_download(self.ctx.handle, self.handle, first, count, ptr(c), ptr(f), ptr(e), ptr(v)))
        return c, f, e, v

    def select(self, order, mode: int, min_size: int, max_size: int = 0):
        """nmost / max selection; returns (row indices, delta_jsd, stats5)"""
        order = np.ascontiguousarray(order, dtype=np.uint32)
        cap = max(int(min_size), int(max_size), 1) + 1
        if int(mode) != MODE_NMOST and int(max_size) < int(min_size):
            cap = order.size + 1  # the set can grow without bound (dvs_b200.h, dvs_select)
        idx = np.zeros(cap, dtype=np.uint32)
        delta = np.zeros(cap, dtype=np.float64)
        stats = np.zeros(5, dtype=np.float64)
        size = _u32(0)
        check(self.ctx._lib.dvs_select(self.ctx.handle, self.handle, ptr(order) if order.size else None, order.size,
                                       int(mode), int(min_size), int(max_size), ptr(idx), ptr(delta), ptr(stats),
                                       C.byref(size)))
        n = size.value
        return idx[:n].copy(), delta[:n].copy(), stats

    def euclidean(self, row_begin: int = 0, row_end: int | None = None) -> np.ndarray:
        row_end = self.nrec if row_end is None else row_end
        out = np.zeros((row_end - row_begin, self.nrec), dtype=np.float64)
        check(self.ctx._lib.dvs_euclid_distances(self.ctx.handle, self.handle, row_begin, row_end, ptr(out)))
        return out

    def euclidean_sharded(self, comm: "Comm", device_ptr: int | None = None):
        """whole matrix over the rows of all ranks, tiles dealt over the GPUs (dvs_euclid_distances_sharded)"""
        out = None if device_ptr is not None else np.zeros((self.nrec, self.nrec), dtype=np.float64)
        check(self.ctx._lib.dvs_euclid_distances_sharded(self.ctx.handle, comm.handle, self.handle,
                                                         _vp(device_ptr) if device_ptr is not None else ptr(out)))
        return out

    def euclidean_into(self, device_ptr: int, row_begin: int = 0, row_end: int | None = None) -> None:
        """same matrix written to device memory at `device_ptr` ((row_end-row_begin) x nrec f64)"""
        row_end = self.nrec if row_end is None else row_end
        check(self.ctx._lib.dvs_euclid_distances(self.ctx.handle, self.handle, row_begin, row_end, _vp(device_ptr)))

    def fallback_pairs(self) -> int:
        """pairs that the last Euclidean call on this context took from the Gram form's list and recomputed in
        difference form (dvs_euclid_last_fallback_pairs); 0 when the difference-form tile kernel did the whole call"""
        return int(self.ctx._lib.dvs_euclid_last_fallback_pairs(self.ctx.handle))


class KSparse(_Handle):
    """Sparse (index, count) k-mer rows for 9 <= k <= 12 (dvs_ksparse)."""

    _free = "dvs_ksparse_free"

    @classmethod
    def count(cls, ctx: Context, seqset: SeqSet, k: int, num_states: int = 4, want_entropy: bool = False) -> "KSparse":
        h = _vp()
        check(ctx._lib.dvs_count_kmers_sparse(ctx.handle, seqset.handle, int(k), int(num_states), int(want_entropy),
                                              C.byref(h)))
        out = cls(ctx, h)
        out.has_entropy = bool(want_entropy)
        return out

    @property
    def nrec(self) -> int:
        return int(self.ctx._lib.dvs_ksparse_nrec(self.handle))

    def stats(self):
        """(distinct k-mers, valid k-mers, entropies or None, valid flags) per record"""
        n = self.nrec
        nnz, tot = np.zeros(n, dtype=np.uint64), np.zeros(n, dtype=np.uint64)
        ent = np.zeros(n, dtype=np.float64) if self.has_entropy else None
        valid = np.zeros(n, dtype=np.uint8)
        check(self.ctx._lib.dvs_ksparse_stats(self.ctx.handle, self.handle, ptr(nnz), ptr(tot), ptr(ent), ptr(valid)))
        return nnz, tot, ent, valid

    def record(self, rec: int):
        """(ascending k-mer indices, counts) of one record"""
        n = _u64(0)
        check(self.ctx._lib.dvs_ksparse_download(self.ctx.handle, self.handle, int(rec), None, None, 0, C.byref(n)))
        idx, cnt = np.zeros(n.value, dtype=np.uint32), np.zeros(n.value, dtype=np.uint32)
        if n.value:
            check(self.ctx._lib.dvs_ksparse_download(self.ctx.handle, self.handle, int(rec), ptr(idx), ptr(cnt), n.value,
                                                     C.byref(n)))
        return idx, cnt

    def euclidean(self, row_begin: int = 0, row_end: int | None = None) -> np.ndarray:
        """rows [row_begin, row_end) of the Euclidean distance matrix of the frequency rows (dvs_euclid_distances_sparse)"""
        row_end = self.nrec if row_end is None else row_end
        out = np.zeros((max(row_end - row_begin, 0), self.nrec), dtype=np.float64)
        check(self.ctx._lib.dvs_euclid_distances_sparse(self.ctx.handle, self.handle, row_begin, row_end, ptr(out)))
        return out

    def euclidean_into(self, device_ptr: int, row_begin: int = 0, row_end: int | None = None) -> None:
        """same matrix written to device memory at `device_ptr` ((row_end-row_begin) x nrec f64)"""
        row_end = self.nrec if row_end is None else row_end
        check(self.ctx._lib.dvs_euclid_distances_sparse(self.ctx.handle, self.handle, row_begin, row_end,
                                                        _vp(device_ptr)))

    def euclidean_sharded(self, comm: "Comm", nrec_per_rank, device_ptr: int | None = None):
        """whole matrix over the sparse rows of all ranks, each rank passing its own rows (collective,
        dvs_euclid_distances_sparse_sharded); into device memory at `device_ptr` when given (returns None)"""
        npr = np.ascontiguousarray(nrec_per_rank, dtype=np.uint32)
        assert npr.size == comm.world
        n = int(npr.sum())
        out = None if device_ptr is not None else np.zeros((n, n), dtype=np.float64)
        check(self.ctx._lib.dvs_euclid_distances_sparse_sharded(
            self.ctx.handle, comm.handle, self.handle, ptr(npr), _vp(device_ptr) if device_ptr is not None else ptr(out)))
        return out

    def fallback_pairs(self) -> int:
        """pairs that the last Euclidean call on this context listed for the difference form
        (dvs_euclid_last_fallback_pairs): 0 when the exact integer form gave every pair; after a list overflow, the
        number of pairs that overflowed the list.  After `euclidean_sharded`: the pairs this rank listed"""
        return int(self.ctx._lib.dvs_euclid_last_fallback_pairs(self.ctx.handle))

    def debug_euclid_pairs(self, pairs) -> np.ndarray:
        """difference-form distances of the given (a, b) record pairs (dvs_debug_euclid_sparse_pairs)"""
        pairs = np.ascontiguousarray(pairs, dtype=np.uint32).reshape(-1, 2)
        out = np.zeros(pairs.shape[0], dtype=np.float64)
        check(self.ctx._lib.dvs_debug_euclid_sparse_pairs(self.ctx.handle, self.handle, ptr(pairs) if pairs.size else None,
                                                          pairs.shape[0], ptr(out)))
        return out


class Comm:
    """Peer windows over NVLink (dvs_comm): one per rank; `blob` is what the ranks exchange before connect()."""

    def __init__(self, ctx: Context, rank: int, world: int, window_bytes: int):
        self.ctx, self.rank, self.world = ctx, int(rank), int(world)
        h = _vp()
        buf = C.create_string_buffer(128)
        check(ctx._lib.dvs_comm_create(ctx.handle, self.rank, self.world, int(window_bytes), C.byref(h), buf))
        self.handle = h
        self.blob = bytes(buf.raw)

    def connect(self, blobs) -> "Comm":
        blobs = list(blobs)
        assert len(blobs) == self.world and all(len(b) == 128 for b in blobs)
        check(self.ctx._lib.dvs_comm_connect(self.ctx.handle, self.handle, C.create_string_buffer(b"".join(blobs), 128 * self.world)))
        return self

    def set_host_barrier(self, fn) -> None:
        """ranks sharing one GPU: `fn()` returns once every rank has called it (dvs_comm_set_host_barrier)"""
        self._host_barrier_cb = C.CFUNCTYPE(None, _vp)(lambda _arg: fn())
        check(self.ctx._lib.dvs_comm_set_host_barrier(self.handle, C.cast(self._host_barrier_cb, _vp), None))

    def barrier(self) -> None:
        check(self.ctx._lib.dvs_comm_barrier(self.ctx.handle, self.handle))

    def allgatherv(self, src_ptr: int, nbytes, dst_ptr: int) -> None:
        """device buffers: this rank's nbytes[rank] bytes at src_ptr -> all pieces, in rank order, at dst_ptr"""
        nb = np.ascontiguousarray(nbytes, dtype=np.uint64)
        assert nb.size == self.world
        check(self.ctx._lib.dvs_comm_allgatherv(self.ctx.handle, self.handle, _vp(src_ptr) if src_ptr else None, ptr(nb),
                                                _vp(dst_ptr)))

    def close(self) -> None:
        if getattr(self, "handle", None) and not _shutdown and getattr(self.ctx, "handle", None):
            self.ctx._lib.dvs_comm_destroy(self.handle)
        self.handle = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class Summed(_Handle):
    """Device-resident SummedRecords state (dvs_summed)."""

    _free = "dvs_summed_free"

    def __init__(self, ctx: Context, kfreqs: KFreqs, members):
        members = np.ascontiguousarray(members, dtype=np.uint32)
        h = _vp()
        check(ctx._lib.dvs_summed_create(ctx.handle, kfreqs.handle, ptr(members) if members.size else None,
                                         members.size, C.byref(h)))
        super().__init__(ctx, h)
        self.kfreqs = kfreqs  # keep alive
        self.size = int(members.size)

    def delta_jsd(self, query: KFreqs, row: int = 0, is_member: bool = False) -> float:
        out = _f64(0.0)
        check(self.ctx._lib.dvs_summed_delta_jsd(self.ctx.handle, self.handle, query.handle, row, int(is_member),
                                                 C.byref(out)))
        return out.value

    def delta_jsd_batch(self, queries: KFreqs, is_member=None) -> np.ndarray:
        """delta_jsd of every row of `queries` (NaN for rows without valid k-mers)"""
        out = np.zeros(queries.nrec, dtype=np.float64)
        mem = None if is_member is None else np.ascontiguousarray(is_member, dtype=np.uint8)
        check(self.ctx._lib.dvs_summed_delta_jsd_batch(self.ctx.handle, self.handle, queries.handle, ptr(mem), ptr(out)))
        return out

    def result(self):
        idx = np.zeros(self.size, dtype=np.uint32)
        delta = np.zeros(self.size, dtype=np.float64)
        stats = np.zeros(5, dtype=np.float64)
        size, low = _u32(0), _u32(0)
        check(self.ctx._lib.dvs_summed_result(self.ctx.handle, self.handle, ptr(idx), ptr(delta), ptr(stats),
                                              C.byref(size), C.byref(low)))
        return idx[: size.value], delta[: size.value], stats, low.value


class Sketches(_Handle):
    """Device-resident MinHash sketches (dvs_sketches)."""

    _free = "dvs_sketches_free"

    @classmethod
    def sketch(cls, ctx: Context, seqset: SeqSet, k: int, sketch_size: int, num_states: int = 4,
               canonical: bool = False) -> "Sketches":
        h = _vp()
        check(ctx._lib.dvs_mash_sketch(ctx.handle, seqset.handle, int(k), int(sketch_size), int(num_states),
                                       int(bool(canonical)), C.byref(h)))
        return cls(ctx, h)

    @classmethod
    def from_host(cls, ctx: Context, sketches: np.ndarray, lens: np.ndarray) -> "Sketches":
        sk = np.ascontiguousarray(sketches, dtype=np.uint32)
        lens = np.ascontiguousarray(lens, dtype=np.uint32)
        h = _vp()
        check(ctx._lib.dvs_sketches_from_host(ctx.handle, ptr(sk), sk.shape[1], ptr(lens), sk.shape[0], C.byref(h)))
        return cls(ctx, h)

    @property
    def nrec(self) -> int:
        return int(self.ctx._lib.dvs_sketches_nrec(self.handle))

    @property
    def stride(self) -> int:
        return int(self.ctx._lib.dvs_sketches_stride(self.handle))

    def download(self):
        sk = np.zeros((self.nrec, self.stride), dtype=np.uint32)
        lens = np.zeros(self.nrec, dtype=np.uint32)
        check(self.ctx._lib.dvs_sketches_download(self.ctx.handle, self.handle, ptr(sk), ptr(lens)))
        return sk, lens

    def distances(self, k: int, sketch_size: int, row_begin: int = 0, row_end: int | None = None,
                  want_counts: bool = False):
        row_end = self.nrec if row_end is None else row_end
        shape = (row_end - row_begin, self.nrec)
        dist = np.zeros(shape, dtype=np.float64)
        inter = np.zeros(shape, dtype=np.uint32) if want_counts else None
        uni = np.zeros(shape, dtype=np.uint32) if want_counts else None
        check(self.ctx._lib.dvs_mash_distances(self.ctx.handle, self.handle, int(k), int(sketch_size), row_begin,
                                               row_end, ptr(dist), ptr(inter), ptr(uni)))
        return (dist, inter, uni) if want_counts else dist

    def allgather(self, comm: "Comm", nrec_per_rank, stride_all: int) -> "Sketches":
        npr = np.ascontiguousarray(nrec_per_rank, dtype=np.uint32)
        h = _vp()
        check(self.ctx._lib.dvs_sketches_allgather(self.ctx.handle, comm.handle, self.handle, ptr(npr), int(stride_all),
                                                   C.byref(h)))
        return Sketches(self.ctx, h)

    def distances_sharded(self, comm: "Comm", k: int, sketch_size: int, device_ptr: int | None = None):
        """whole matrix, pairs dealt over the GPUs (dvs_mash_distances_sharded)"""
        out = None if device_ptr is not None else np.zeros((self.nrec, self.nrec), dtype=np.float64)
        check(self.ctx._lib.dvs_mash_distances_sharded(self.ctx.handle, comm.handle, self.handle, int(k), int(sketch_size),
                                                       _vp(device_ptr) if device_ptr is not None else ptr(out)))
        return out

    def distances_into(self, device_ptr: int, k: int, sketch_size: int) -> None:
        """the full nrec x nrec f64 matrix written to device memory at `device_ptr`"""
        check(self.ctx._lib.dvs_mash_distances(self.ctx.handle, self.handle, int(k), int(sketch_size), 0, self.nrec,
                                               _vp(device_ptr), None, None))


def linkage_average(ctx: Context, dist=None, n: int | None = None, device_ptr: int | None = None):
    """children_ (n-1, 2), merge heights and cluster sizes of the average-linkage tree of an n x n
    distance matrix held in a numpy array or in device memory (dvs_linkage_average)"""
    if device_ptr is None:
        dist = np.ascontiguousarray(dist, dtype=np.float64)
        if dist.ndim != 2 or dist.shape[0] != dist.shape[1]:
            raise ValueError("distance matrix must be square")
        n, dp = dist.shape[0], ptr(dist)
    else:
        dp = _vp(device_ptr)
    m = max(int(n) - 1, 0)
    children = np.zeros((m, 2), dtype=np.int32)
    heights = np.zeros(m, dtype=np.float64)
    counts = np.zeros(m, dtype=np.uint32)
    check(ctx._lib.dvs_linkage_average(ctx.handle, dp, int(n), ptr(children), ptr(heights), ptr(counts)))
    return children, heights, counts


def debug_log2(ctx: Context, x: np.ndarray) -> np.ndarray:
    x = np.ascontiguousarray(x, dtype=np.float64)
    y = np.zeros_like(x)
    check(ctx._lib.dvs_debug_log2(ctx.handle, ptr(x), ptr(y), x.size))
    return y


def debug_fast_terms(ctx: Context, a: np.ndarray, b: np.ndarray):
    a = np.ascontiguousarray(a, dtype=np.float64)
    b = np.ascontiguousarray(b, dtype=np.float64)
    m, lg, sp = np.zeros_like(a), np.zeros_like(a), np.zeros(a.size, dtype=np.int32)
    check(ctx._lib.dvs_debug_fast_terms(ctx.handle, ptr(a), ptr(b), ptr(m), ptr(lg), ptr(sp), a.size))
    return m, lg, sp


def debug_entropy(ctx: Context, rows: np.ndarray):
    rows = np.ascontiguousarray(rows, dtype=np.float64)
    out = np.zeros(rows.shape[0], dtype=np.float64)
    err = np.zeros(rows.shape[0], dtype=np.uint8)
    check(ctx._lib.dvs_debug_entropy(ctx.handle, ptr(rows), rows.shape[0], rows.shape[1], ptr(out), ptr(err)))
    return out, err
