"""Multi-GPU sharding of the hot path (SURVEY.md §8e): one process (or host thread) per GPU over the
library's own peer windows (include/dvs_b200.h, dvs_comm_*): no NCCL and no torch in the product.

* counting: records are independent -> each rank counts its own shard (`count_sharded`); each chunk of
  frequency rows is pushed to every peer over the copy engines while the next chunk is being counted, so
  when counting ends every GPU holds the rows of all records.
* nmost / max: `select_sharded` = the reference's single pass (numprocs=1 semantics, src/records.rs:311-342,
  390-454) with every window of candidates scored candidate-sharded (position % world) and one 16-byte
  all-reduce(min) per round over NVLink; the state update is replayed identically on every GPU.
  `chunked_select` keeps the reference's `-np N` chunk-then-merge semantics (diverse_seq/records.py:206-251,
  a different result by design) for callers that want to reproduce numprocs > 1 outputs.
* distance matrices: sketches / rows are all-gathered, the lower triangle is dealt over the GPUs (pairs for
  mash, 128 x 128 tiles for Euclid) and every kernel stores its results straight into every peer's copy
  of the matrix.  Sparse k-mer rows (k = 9..12) are not gathered: each rank keeps its own and copies one peer's
  at a time (`sharded_euclidean_sparse`).
* nmost / max from sparse rows (k = 10..12): `select_sparse_sharded`.  Each rank keeps its own rows and scores the
  candidates it holds; only rows that enter the set (and `max`'s grow candidates) are copied to the other ranks.

The only host-side exchange is the rendezvous below (window handles and a few integers over TCP on
MASTER_ADDR:MASTER_PORT+1, or in-process for ranks that are threads of one process).
"""
from __future__ import annotations

import os
import pickle
import socket
import struct
import threading
import time

import numpy as np


def shard_bounds(n_items: int, world: int, rank: int) -> tuple[int, int]:
    """contiguous block partition [begin, end) of n_items over world ranks (sizes differ by <= 1)"""
    base, rem = divmod(n_items, world)
    begin = rank * base + min(rank, rem)
    return begin, begin + base + (1 if rank < rem else 0)


def global_order(seed: int, n_total: int) -> np.ndarray:
    """the shuffled examination order, identical on every rank (cli.py:445-446 uses default_rng(seed))"""
    return np.random.default_rng(seed).permutation(n_total).astype(np.uint32)


# ------------------------------------------------------------------------------ rendezvous ----
def _send(sock, obj) -> None:
    data = pickle.dumps(obj, protocol=pickle.HIGHEST_PROTOCOL)
    sock.sendall(struct.pack("<Q", len(data)) + data)


def _recv(sock):
    def exactly(n):
        buf = bytearray()
        while len(buf) < n:
            part = sock.recv(n - len(buf))
            if not part:
                raise ConnectionError("rendezvous peer closed the connection")
            buf += part
        return bytes(buf)

    (n,) = struct.unpack("<Q", exactly(8))
    return pickle.loads(exactly(n))


class Rendezvous:
    """all-gather of small python objects between the ranks over TCP (rank 0 listens); only used to exchange
    window handles, record counts and the like - never on the data path"""

    def __init__(self, rank: int | None = None, world: int | None = None, addr: str | None = None,
                 port: int | None = None, timeout: float = 300.0):
        self.rank = int(os.environ.get("RANK", "0")) if rank is None else int(rank)
        self.world = int(os.environ.get("WORLD_SIZE", "1")) if world is None else int(world)
        addr = addr or os.environ.get("MASTER_ADDR", "127.0.0.1")
        port = int(port if port is not None else int(os.environ.get("MASTER_PORT", "29500")) + 1)
        self.peers: list = []
        self.sock = None
        if self.world == 1:
            return
        if self.rank == 0:
            srv = socket.socket(socket.AF_INET, socket.SOCK_STREAM)
            srv.setsockopt(socket.SOL_SOCKET, socket.SO_REUSEADDR, 1)
            srv.bind((addr if addr not in ("localhost",) else "127.0.0.1", port))
            srv.listen(self.world)
            srv.settimeout(timeout)
            conns = {}
            while len(conns) < self.world - 1:
                c, _ = srv.accept()
                c.settimeout(timeout)
                conns[_recv(c)] = c
            srv.close()
            self.peers = [conns[r] for r in range(1, self.world)]
        else:
            deadline = time.time() + timeout
            while True:
                try:
                    s = socket.create_connection((addr, port), timeout=5.0)
                    break
                except OSError:
                    if time.time() > deadline:
                        raise
                    time.sleep(0.05)
            s.settimeout(timeout)
            _send(s, self.rank)
            self.sock = s

    def allgather(self, obj) -> list:
        if self.world == 1:
            return [obj]
        if self.rank == 0:
            out = [obj] + [_recv(c) for c in self.peers]
            for c in self.peers:
                _send(c, out)
            return out
        _send(self.sock, obj)
        return _recv(self.sock)

    def barrier(self) -> None:
        self.allgather(None)

    def close(self) -> None:
        for c in self.peers:
            c.close()
        if self.sock is not None:
            self.sock.close()
        self.peers, self.sock = [], None


class LocalGroup:
    """the same exchange for ranks that are THREADS of one process (tests: several ranks on one GPU, or one
    thread per GPU): `group.member(rank)` has the Rendezvous interface"""

    def __init__(self, world: int):
        self.world = world
        self._bar = threading.Barrier(world)
        self._slots = [None] * world

    def member(self, rank: int) -> "_LocalMember":
        return _LocalMember(self, rank)


class _LocalMember:
    def __init__(self, group: LocalGroup, rank: int):
        self.group, self.rank, self.world = group, rank, group.world

    def allgather(self, obj) -> list:
        g = self.group
        g._slots[self.rank] = obj
        g._bar.wait()
        out = list(g._slots)
        g._bar.wait()
        return out

    def barrier(self) -> None:
        self.group._bar.wait()

    def close(self) -> None:
        pass


def connect(ctx, rv, window_bytes: int):
    """create this rank's peer window and map everybody else's (collective over the rendezvous `rv`)"""
    from . import _lib

    comm = _lib.Comm(ctx, rv.rank, rv.world, int(window_bytes))
    comm.connect(rv.allgather(comm.blob))
    comm.rv = rv
    devices = rv.allgather((os.getpid(), ctx.device))
    if isinstance(rv, _LocalMember) and len(set(devices)) < len(devices):
        comm.set_host_barrier(rv.barrier)  # thread ranks sharing a GPU: waits are taken on the host
    return comm


def window_bytes_for(nrec_total: int, dim: int, extra: int = 0) -> int:
    """a window that holds the rows of all records (+ their scalars) and `extra` bytes of other objects"""
    return int(nrec_total * (dim * 8 + 64) + extra + (64 << 20))


def window_bytes_for_sparse(nrec_per_rank, bases_per_rank, k: int, extra: int = 0) -> int:
    """the window `sharded_euclidean_sparse` needs (the formula dvs_euclid_distances_sparse_sharded checks): the
    staged sparse rows of the largest shard - one slot per sequence byte, so known before counting; none on a single
    rank - and the n x n matrix, plus `extra` bytes of other objects"""
    def align(b):
        return (int(b) + 255) // 256 * 256
    nb = 4 ** (int(k) - 6)  # buckets per record (csrc/sparse.cu)
    max_n = max((int(x) for x in nrec_per_rank), default=0)
    max_slots = max((int(x) for x in bases_per_rank), default=0)
    n = sum(int(x) for x in nrec_per_rank)
    stage = (2 * align(max_slots * 4) + align((max_n + 1) * 8) + align(max_n * (nb + 1) * 4) + align(max_n * nb * 4)
             + align(max_n * 8))
    stage = max(stage, 256) if len(nrec_per_rank) > 1 else 0  # one rank stages nothing: no peer reads its rows
    return 64 * 1024 + stage + max(align(n * n * 8), 256) + int(extra)


def window_bytes_for_sparse_select(max_record_len: int, k: int, nrec_total: int, extra: int = 0) -> int:
    """the window `select_sparse_sharded` needs (the formula dvs_select_sparse_sharded checks): control words and the
    larger of the staging of the per-record scalars (8 bytes a record) and the outbox of one row - one slot per byte of
    the longest record of any rank, so known before counting - plus `extra` bytes of other objects.  The member-row
    cache is ordinary device memory, not window memory, so the size of the set does not enter."""
    def align(b):
        return (int(b) + 255) // 256 * 256
    nb = 4 ** (int(k) - 6)  # buckets per record (csrc/sparse.cu)
    outbox = max(2 * align(int(max_record_len) * 4) + align((nb + 1) * 4) + align(nb * 4), 256)
    return 64 * 1024 + max(align(int(nrec_total) * 8), 256, outbox) + int(extra)


# --------------------------------------------------------------------------------- counting ----
def count_sharded(ctx, comm, seqset_local, k: int, num_states: int = 4):
    """(kfreqs with the rows of ALL ranks in rank-major order, records per rank)"""
    from . import _lib

    nrec = comm.rv.allgather(int(seqset_local.nrec))
    return _lib.KFreqs.count_sharded(ctx, comm, seqset_local, k, nrec, num_states), nrec


def interleaved_order(local_orders, nrec_per_rank) -> np.ndarray:
    """a global examination order over the rank-major rows of all ranks in which consecutive positions
    come from different ranks (SURVEY.md §8e: block-cyclic by position): position world*i + r is the i-th
    record of rank r's own order; shorter ranks simply run out first"""
    world = len(nrec_per_rank)
    base = np.concatenate([[0], np.cumsum(nrec_per_rank)]).astype(np.int64)
    longest = max(len(o) for o in local_orders) if world else 0
    grid = np.full((longest, world), -1, dtype=np.int64)
    for r, o in enumerate(local_orders):
        grid[: len(o), r] = np.asarray(o, dtype=np.int64) + base[r]
    flat = grid.reshape(-1)
    return flat[flat >= 0].astype(np.uint32)


def select_sharded(ctx, comm, kf_all, order, mode: int, min_size: int, max_size: int = 0):
    """single-pass selection over all rows, candidate-sharded (identical result on every rank)"""
    return kf_all.select_sharded(comm, order, mode, min_size, max_size)


def select_sparse_sharded(ctx, comm, ks_local, order, mode: int, min_size: int, max_size: int = 0):
    """single-pass nmost / max over the sparse rows of all ranks, each rank passing its own (KSparse.count with
    want_entropy=True): identical result on every rank, bitwise KSparse.select over the union of the records.

    `order` indexes the rank-major rows of all ranks.  Any placement of the records gives the same result; the one that
    balances the work deals the shuffled seqids round-robin - rank r takes positions r, r + W, ... of the shuffled list,
    in that order - and rebuilds the global order with `interleaved_order(local orders, nrec)`, so that every window of
    candidates falls evenly on the ranks.  The window: `window_bytes_for_sparse_select`."""
    nrec = comm.rv.allgather(int(ks_local.nrec))
    return ks_local.select_sharded(comm, nrec, order, mode, min_size, max_size)


def chunked_select(ctx, comm, kf_local, local_order, mode: int, min_size: int, max_size: int):
    """The reference's multi-process selection with one chunk per GPU (-np N semantics,
    diverse_seq/records.py:206-251): select locally, gather the winners' rows, merge with final_nmost /
    final_max on every rank (src/records.rs:363-382, 456-507: entropies recomputed from the stored rows).

    Returns ((rank, local row) of every selected record, delta_jsd, stats5)."""
    from . import _lib

    idx, _delta, _stats = kf_local.select(local_order, mode, min_size, max_size)
    won = kf_local.take_rows(idx)
    counts = comm.rv.allgather(int(len(idx)))
    ids = comm.rv.allgather([(comm.rank, int(r)) for r in idx])
    gathered = won.allgather(comm, counts)
    rows_p, _e, _v = gathered.device_ptrs()
    merged = _lib.KFreqs.from_device(ctx, rows_p, None, None, gathered.nrec, gathered.dim)  # KmerSeq::new: H recomputed
    flat_ids = [x for part in ids for x in part]
    midx, mdelta, mstats = merged.select(np.arange(gathered.nrec, dtype=np.uint32), mode, min_size, max_size)
    merged.close()
    gathered.close()
    won.close()
    return [flat_ids[i] for i in midx], mdelta, mstats


# -------------------------------------------------------------------------------- distances ----
def sharded_mash_distances(ctx, comm, seqset_local, k: int, sketch_size: int, num_states: int = 4,
                           canonical: bool = False) -> np.ndarray:
    """ctree mash on N GPUs: every rank sketches its own records, the sketches are all-gathered over NVLink,
    the pairs of the lower triangle are dealt over the GPUs and each kernel stores its distances into every
    peer's copy of the matrix; returns the full matrix (rank-major record order) on every rank"""
    from . import _lib

    sk = _lib.Sketches.sketch(ctx, seqset_local, k, sketch_size, num_states, canonical)
    meta = comm.rv.allgather((int(sk.nrec), int(sk.stride)))
    allsk = sk.allgather(comm, [m[0] for m in meta], max(m[1] for m in meta))
    out = allsk.distances_sharded(comm, k, sketch_size)
    allsk.close()
    sk.close()
    return out


def sharded_euclidean_sparse(ctx, comm, ks_local, device_ptr: int | None = None):
    """ctree Euclidean at 9 <= k <= 12 on N GPUs from each rank's own sparse rows (KSparse.count of its records):
    the rows stay with their rank, a rank copies one peer's rows at a time and computes the pairs it owns, results
    are stored into every peer's matrix; returns the full matrix (rank-major record order) on every rank, or writes
    it to `device_ptr` (the window: `window_bytes_for_sparse`)"""
    nrec = comm.rv.allgather(int(ks_local.nrec))
    return ks_local.euclidean_sharded(comm, nrec, device_ptr)


def sharded_euclidean(ctx, comm, kf_local=None, kf_all=None) -> np.ndarray:
    """ctree Euclidean on N GPUs: all-gather the frequency rows (or take them from count_sharded), deal the
    128 x 128 tiles of the lower triangle over the GPUs, results stored into every peer's matrix"""
    own = kf_all is None
    if own:
        nrec = comm.rv.allgather(int(kf_local.nrec))
        kf_all = kf_local.allgather(comm, nrec)
    out = kf_all.euclidean_sharded(comm)
    if own:
        kf_all.close()
    return out
