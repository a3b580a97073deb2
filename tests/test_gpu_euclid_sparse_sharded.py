"""Sparse Euclidean matrix on several ranks (dvs_euclid_distances_sparse_sharded, csrc/euclid_sparse.cu): each rank
keeps its own k-mer rows, copies one peer's rows at a time and stores the pairs it owns into every rank's matrix.

Every rank's matrix must be bitwise the single-GPU `KSparse.count(union).euclidean()` (NaN positions included), which
is itself checked against the sparse-row reference (tests/sparse_euclid_ref.py) at 1e-9.  Each rank's
`fallback_pairs()` must equal the listed pairs (tests/sparse_euclid_forms.py) that the ownership rule gives it:
    same rank p: p;  d = (q - p) mod W < W/2: p;  d > W/2: q;
    d = W/2: r = min(p, q) if the record on r has local index < ceil(n_r / 2), else r + W/2.

The ranks are host threads of this process (a copy of test_gpu_sharded.run_ranks): one GPU each when enough are
visible, otherwise all on device 0 with the waits taken on the host.  Two real processes run
tests/sparse_sharded_worker.py over the TCP rendezvous and cudaIpc.
"""
import os
import pathlib
import subprocess
import sys
import threading
import time

import numpy as np
import pytest

from conftest import random_seqs
from sparse_euclid_forms import FLAG_CAP, listed_pairs, planted_record
from sparse_euclid_ref import merge_matrix

pytestmark = pytest.mark.gpu

ROOT = pathlib.Path(__file__).resolve().parent.parent
L0 = 200_000  # [L0 + m, 1] rows with m < 5,000: every pair of them is listed (test_gpu_euclid_sparse_forms.py)


@pytest.fixture(scope="module")
def lib():
    from diverseseq_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def ctx(lib):
    return lib.Context(0)


def device_count() -> int:
    import ctypes
    try:
        rt = ctypes.CDLL("libcudart.so")
    except OSError:
        try:
            import torch
            return torch.cuda.device_count()
        except Exception:
            return 1
    n = ctypes.c_int(0)
    return n.value if rt.cudaGetDeviceCount(ctypes.byref(n)) == 0 else 1


def run_ranks(world, fn, window_bytes=256 << 20):
    """fn(rank, ctx, comm) on `world` threads; returns the per-rank results"""
    from diverseseq_b200 import _lib, shard

    ndev = device_count()
    devices = list(range(world)) if ndev >= world else [0] * world
    old = os.environ.get("DVS_SELECT_GRID")
    os.environ["DVS_COMM_CHECK"] = "1"  # a timed-out device-side wait is reported by the call it happened in
    if ndev < world:
        os.environ["DVS_SELECT_GRID"] = str(max(8, 148 // world - 2))
    group = shard.LocalGroup(world)
    results, errors = [None] * world, []

    def worker(rank):
        try:
            ctx = _lib.Context(devices[rank])
            comm = shard.connect(ctx, group.member(rank), window_bytes)
            results[rank] = fn(rank, ctx, comm)
            ctx.sync()
            group.member(rank).barrier()
            comm.close()
        except BaseException as exc:  # noqa: BLE001
            errors.append((rank, exc))
            group._bar.abort()

    threads = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join(timeout=600)
    if old is None:
        os.environ.pop("DVS_SELECT_GRID", None)
    else:
        os.environ["DVS_SELECT_GRID"] = old
    real = [e for e in errors if not isinstance(e[1], threading.BrokenBarrierError)]
    if real or errors:
        raise (real or errors)[0][1]
    return results


# ------------------------------------------------------------------------------------------- helpers ----

def owner(gi, gj, npr):
    """rank that computes the pair of global records gi != gj under the prescribed rule"""
    base = np.concatenate([[0], np.cumsum(npr)])
    w = len(npr)
    p = int(np.searchsorted(base, gi, side="right") - 1)
    q = int(np.searchsorted(base, gj, side="right") - 1)
    if p == q:
        return p
    d = (q - p) % w
    if 2 * d < w:
        return p
    if 2 * d > w:
        return q
    r = min(p, q)
    local = (gi if p == r else gj) - int(base[r])
    return r if local < (int(npr[r]) + 1) // 2 else r + w // 2


def predicted_counts(listed, npr):
    per = [0] * len(npr)
    for i, j in zip(*np.nonzero(listed)):
        per[owner(int(i), int(j), npr)] += 1
    return per


def split(seqs, npr):
    out, o = [], 0
    for n in npr:
        out.append(seqs[o:o + n])
        o += n
    return out


def window_for(lib, shards, k):
    from diverseseq_b200 import shard
    return shard.window_bytes_for_sparse([len(s) for s in shards], [sum(len(x) for x in s) for s in shards], k,
                                         extra=1 << 20)


def sharded_matrices(lib, shards, k, window=None, calls=1):
    """each rank counts its own shard and runs the sharded call; returns [(matrix, fallback_pairs)] per rank"""
    from diverseseq_b200 import shard
    world = len(shards)

    def fn(rank, ctx, comm):
        ks = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, shards[rank]), k)
        for _ in range(calls):
            m = shard.sharded_euclidean_sparse(ctx, comm, ks)
        return m, ks.fallback_pairs()

    return run_ranks(world, fn, window or window_for(lib, shards, k))


def single(lib, ctx, seqs, k):
    """(single-GPU matrix, its listed pairs, its KSparse) over the union"""
    sp = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), k)
    full = sp.euclidean()
    count = sp.fallback_pairs()
    _, totals, _, _ = sp.stats()
    rows = [sp.record(r) for r in range(sp.nrec)]
    exp = merge_matrix(rows, totals)
    nan = np.isnan(exp)
    assert np.array_equal(np.isnan(full), nan)
    assert np.array_equal(full == 0.0, exp == 0.0)
    np.testing.assert_allclose(full[~nan], exp[~nan], rtol=1e-9, atol=0)
    listed = listed_pairs(rows, 4 ** k)
    assert count == int(listed.sum())
    return full, listed, sp


def union_records(rng, npr, k, planted):
    """random records with empty / invalid / short records on several ranks, exact copies across ranks and, when
    `planted`, the listed family [L0 + m, 1] at local rows 0, ceil(n/2) - 1, ceil(n/2) and n - 1 of every rank"""
    n = int(sum(npr))
    seqs = random_seqs(rng, n, 0, 900, invalid_rate=0.01)
    base = np.concatenate([[0], np.cumsum(npr)]).astype(int)
    ms = iter(rng.permutation(5000).tolist())
    for r, nr in enumerate(npr):
        if nr == 0:
            continue
        b = int(base[r])
        if planted:
            h = (nr + 1) // 2
            for loc in sorted({0, h - 1, h, nr - 1} & set(range(nr))):
                seqs[b + loc] = planted_record([L0 + next(ms), 1], k)
        if nr > 3:
            seqs[b + 1] = np.zeros(0, dtype=np.uint8) if r % 2 == 0 else np.full(50, 4, dtype=np.uint8)
            seqs[b + 2] = rng.integers(0, 4, size=k - 1, dtype=np.uint8)  # shorter than k: no valid k-mer
    filled = [r for r in range(len(npr)) if npr[r] > 6]
    for a, c in zip(filled, filled[1:]):  # exact copies on different ranks
        seqs[int(base[c]) + 5] = seqs[int(base[a]) + 4].copy()
    return seqs


def check_ranks(results, full, listed, npr):
    per = predicted_counts(listed, npr)
    for r, (m, fb) in enumerate(results):
        assert np.array_equal(m, full, equal_nan=True), f"rank {r}: matrix differs from the single-GPU call"
        assert fb == per[r], (r, fb, per)
    assert sum(fb for _, fb in results) == int(listed.sum())
    return per


# --------------------------------------------------------------------------------------------- tests ----

SHAPES = [
    (1, [50], 12),
    (2, [70, 133], 10),
    (2, [0, 65], 12),
    (3, [70, 9, 1], 12),
    (3, [1, 64, 72], 10),
    (4, [70, 133, 9, 0], 10),
    (4, [70, 133, 9, 0], 12),
    (4, [8, 1, 129, 63], 12),
]


@pytest.mark.parametrize("world,npr,k", SHAPES, ids=[f"w{w}-{'_'.join(map(str, n))}-k{k}" for w, n, k in SHAPES])
@pytest.mark.parametrize("planted", [False, True], ids=["plain", "planted"])
def test_matches_single_gpu(lib, ctx, world, npr, k, planted):
    """uneven shards (an empty rank, one-record ranks, sizes off the 8 / 64 grid): every rank's matrix is bitwise
    the single-GPU matrix; with the planted family, listed pairs sit inside ranks, in d < W/2 and d > W/2 blocks and
    in both halves of the W/2 block, and every rank lists exactly the pairs the rule gives it"""
    seqs = union_records(np.random.default_rng(1000 * world + sum(npr) + k), npr, k, planted)
    full, listed, sp = single(lib, ctx, seqs, k)
    if planted:
        assert listed.sum() > 0
        i, j = np.nonzero(listed)
        d = sp.debug_euclid_pairs(np.stack([i, j], axis=1))
        assert np.array_equal(full[i, j], d, equal_nan=True) and np.array_equal(full[j, i], d, equal_nan=True)
    per = check_ranks(sharded_matrices(lib, split(seqs, npr), k), full, listed, npr)
    print(f"\nW={world} npr={npr} k={k}: listed per rank {per}")


def test_every_block_kind_lists_pairs(lib, ctx):
    """W = 4 with the planted family on both halves of every rank: listed pairs in all four kinds of block, each
    counted on the rank the rule names"""
    npr, k = [20, 30, 17, 25], 12
    seqs = union_records(np.random.default_rng(5), npr, k, True)
    full, listed, _ = single(lib, ctx, seqs, k)
    base = np.concatenate([[0], np.cumsum(npr)])
    kinds = set()
    for i, j in zip(*np.nonzero(listed)):
        p = int(np.searchsorted(base, i, side="right") - 1)
        q = int(np.searchsorted(base, j, side="right") - 1)
        d = (q - p) % 4
        kinds.add("same" if p == q else "half" + str(owner(int(i), int(j), npr) >= 2) if d == 2 else "d" + str(d))
    assert {"same", "d1", "d3", "halfFalse", "halfTrue"} <= kinds, kinds
    check_ranks(sharded_matrices(lib, split(seqs, npr), k, calls=2), full, listed, npr)


def overflow_set(lib, ctx):
    """the 6,000 records [L0 + m, 1] at k = 9 of test_list_overflow: all 17,997,000 pairs are listed"""
    k, n = 9, 6000
    x = L0 + np.arange(n, dtype=np.int64)
    offsets = np.zeros(n + 1, dtype=np.uint64)
    offsets[1:] = np.cumsum(x + 2 * k)
    flat = np.zeros(int(offsets[-1]), dtype=np.uint8)
    sep = offsets[:-1].astype(np.int64) + x + k - 1
    flat[sep] = 4
    for q in range(k):
        flat[sep + 1 + q] = 1
    return k, n, flat, offsets


def shard_of(flat, offsets, first, count):
    o = offsets[first:first + count + 1]
    return flat[int(o[0]):int(o[-1])], (o - o[0]).astype(np.uint64)


def test_set_one_gpu_must_split(lib, ctx):
    """[3000, 3000] on two ranks: each lists 8,998,500 pairs (< 2^24) and the call succeeds where the single call
    overflows; the matrix equals the single-GPU row-range calls that fit the list"""
    k, n, flat, offsets = overflow_set(lib, ctx)
    ss = lib.SeqSet.upload(ctx, flat, offsets)
    sp = lib.KSparse.count(ctx, ss, k)
    ss.close()
    with pytest.raises(ValueError, match="pairs need the difference form"):
        sp.euclidean()
    assert sp.fallback_pairs() == 17_997_000 > FLAG_CAP
    ranges = [(a, min(n, a + 1000)) for a in range(0, n, 1000)]
    full = np.concatenate([sp.euclidean(a, b) for a, b in ranges])
    sp.close()
    npr = [3000, 3000]
    shards = [shard_of(flat, offsets, 0, 3000), shard_of(flat, offsets, 3000, 3000)]
    from diverseseq_b200 import shard
    window = shard.window_bytes_for_sparse(npr, [len(s[0]) for s in shards], k)

    def fn(rank, rctx, comm):
        ks = lib.KSparse.count(rctx, lib.SeqSet.upload(rctx, *shards[rank]), k)
        m = shard.sharded_euclidean_sparse(rctx, comm, ks)
        return m, ks.fallback_pairs()

    res = run_ranks(2, fn, window)
    for r, (m, fb) in enumerate(res):
        assert fb == 8_998_500, (r, fb)
        assert np.array_equal(m, full, equal_nan=True), f"rank {r}"


def test_overflow_on_one_rank_fails_every_rank(lib, ctx):
    """[6000, 0]: rank 0 lists 17,997,000 pairs, more than one rank can list; BOTH ranks raise ValueError (rank 1
    listed none), and a following call on the same communicator gives the right matrix"""
    k, n, flat, offsets = overflow_set(lib, ctx)
    small = union_records(np.random.default_rng(9), [40, 33], 12, True)
    full_small, listed_small, _ = single(lib, ctx, small, 12)
    small_shards = split(small, [40, 33])
    from diverseseq_b200 import shard
    window = shard.window_bytes_for_sparse([n, 0], [len(flat), 0], k)

    def fn(rank, rctx, comm):
        mine = (flat, offsets) if rank == 0 else (np.zeros(0, dtype=np.uint8), np.zeros(1, dtype=np.uint64))
        ks = lib.KSparse.count(rctx, lib.SeqSet.upload(rctx, *mine), k)
        t0 = time.time()
        with pytest.raises(ValueError, match="need the difference form"):
            shard.sharded_euclidean_sparse(rctx, comm, ks)
        first = (ks.fallback_pairs(), time.time() - t0)
        ks.close()
        ks2 = lib.KSparse.count(rctx, lib.SeqSet.from_seqs(rctx, small_shards[rank]), 12)
        return first, shard.sharded_euclidean_sparse(rctx, comm, ks2), ks2.fallback_pairs()

    res = run_ranks(2, fn, window)
    assert [r[0][0] for r in res] == [17_997_000, 0]
    per = predicted_counts(listed_small, [40, 33])
    for r, (_, m, fb) in enumerate(res):
        assert np.array_equal(m, full_small, equal_nan=True), f"rank {r}"
        assert fb == per[r]


@pytest.mark.parametrize("what", ["k", "nrec_per_rank"])
def test_mismatches_fail_every_rank_promptly(lib, ctx, what):
    """a different k on one rank, or a wrong nrec_per_rank on one rank: every rank raises the same TypeError at
    once, and the same communicator then runs a correct call"""
    npr = [30, 21, 17]
    seqs = union_records(np.random.default_rng(33), npr, 12, True)
    full, listed, _ = single(lib, ctx, seqs, 12)
    shards = split(seqs, npr)

    def fn(rank, rctx, comm):
        ss = lib.SeqSet.from_seqs(rctx, shards[rank])
        k = 10 if what == "k" and rank == 1 else 12
        ks = lib.KSparse.count(rctx, ss, k)
        given = list(npr)
        if what == "nrec_per_rank" and rank == 2:
            given[0] += 1
        t0 = time.time()
        try:
            ks.euclidean_sharded(comm, given)
            msg = None
        except TypeError as exc:
            msg = str(exc)
        dt = time.time() - t0
        good = lib.KSparse.count(rctx, ss, 12)
        return msg, dt, good.euclidean_sharded(comm, npr), good.fallback_pairs()

    res = run_ranks(3, fn, window_for(lib, shards, 12))
    msgs = [r[0] for r in res]
    assert msgs[0] is not None and all(m == msgs[0] for m in msgs), msgs
    assert ("counted k=10" if what == "k" else "nrec_per_rank[0] = 31") in msgs[0]
    assert max(r[1] for r in res) < 10.0, [r[1] for r in res]
    per = predicted_counts(listed, npr)
    for r, (_, _, m, fb) in enumerate(res):
        assert np.array_equal(m, full, equal_nan=True) and fb == per[r]


def test_window_too_small_fails_every_rank(lib, ctx):
    npr = [60, 21]
    seqs = union_records(np.random.default_rng(34), npr, 12, False)
    shards = split(seqs, npr)
    need = window_for(lib, shards, 12) - (1 << 20)

    def fn(rank, rctx, comm):
        ks = lib.KSparse.count(rctx, lib.SeqSet.from_seqs(rctx, shards[rank]), 12)
        with pytest.raises(TypeError, match="window_bytes_for_sparse"):
            ks.euclidean_sharded(comm, npr)
        return True

    # a window one 256-byte step below the formula's
    assert all(run_ranks(2, fn, need - 256))


def test_device_output(lib, ctx):
    npr, k = [45, 30], 12
    seqs = union_records(np.random.default_rng(35), npr, k, True)
    full, _, _ = single(lib, ctx, seqs, k)
    shards = split(seqs, npr)
    n = sum(npr)

    def fn(rank, rctx, comm):
        ks = lib.KSparse.count(rctx, lib.SeqSet.from_seqs(rctx, shards[rank]), k)
        buf = lib.DeviceBuffer(rctx, n * n * 8)
        buf.from_host(np.full((n, n), -7.0))
        assert ks.euclidean_sharded(comm, npr, buf.ptr) is None
        out = buf.to_host(np.float64, (n, n))
        buf.close()
        return out

    for m in run_ranks(2, fn, window_for(lib, shards, k)):
        assert np.array_equal(m, full, equal_nan=True)


def test_processes_over_tcp_rendezvous_and_cuda_ipc(lib):
    """two real processes (cudaIpc-mapped windows, TCP rendezvous)"""
    import socket
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    ndev = device_count()
    procs = []
    for r in range(2):
        env = dict(os.environ, RANK=str(r), WORLD_SIZE="2", MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port),
                   LOCAL_RANK=str(r if ndev >= 2 else 0))
        procs.append(subprocess.Popen([sys.executable, str(ROOT / "tests" / "sparse_sharded_worker.py")], env=env,
                                      stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "SPARSE_SHARDED_WORKER_OK" in o, o


def test_t_product_at_2_63_across_ranks(lib):
    """one record of 3,037,000,500 valid k-mers per rank: T_a T_b >= 2^63, so the cross pair is listed and given by
    the difference form"""
    if device_count() < 2:
        pytest.skip("needs two GPUs: two ranks of a ~3 Gbp record on one GPU would need an estimated 150 GB "
                    "(not measured)")
    from diverseseq_b200 import shard
    k = 9
    t1 = 3_037_000_500
    la = t1 + k - 1
    flat = np.empty(2 * la, dtype=np.uint8)
    rng = np.random.default_rng(263)
    step = 1 << 28
    for o in range(0, flat.size, step):
        c = min(step, flat.size - o)
        flat[o:o + c] = np.frombuffer(rng.bytes(c), dtype=np.uint8) & np.uint8(3)
    shards = [(flat[:la], np.array([0, la], dtype=np.uint64)), (flat[la:], np.array([0, la], dtype=np.uint64))]

    def fn(rank, rctx, comm):
        ks = lib.KSparse.count(rctx, lib.SeqSet.upload(rctx, *shards[rank]), k)
        return shard.sharded_euclidean_sparse(rctx, comm, ks), ks.fallback_pairs()

    res = run_ranks(2, fn, shard.window_bytes_for_sparse([1, 1], [la, la], k))
    assert [r[1] for r in res] == [1, 0]  # (d = W/2: rank 0's record has local index 0 < ceil(1/2))
    m0 = res[0][0]
    assert np.array_equal(res[1][0], m0) and m0[0, 1] == m0[1, 0] and m0[0, 0] == 0.0
    # the reference: the single-GPU call over both records (each call frees its rows first)
    ctx0 = lib.Context(0)
    sp = lib.KSparse.count(ctx0, lib.SeqSet.upload(ctx0, flat, np.array([0, la, 2 * la], dtype=np.uint64)), k)
    assert np.array_equal(sp.euclidean(), m0)
    assert sp.fallback_pairs() == 1


def test_single_rank_window_holds_no_staged_rows(lib, ctx):
    """one rank stages nothing: the window of the formula (control words + matrix) is enough"""
    from diverseseq_b200 import shard
    seqs = union_records(np.random.default_rng(36), [90], 12, True)
    full, listed, _ = single(lib, ctx, seqs, 12)
    window = shard.window_bytes_for_sparse([90], [sum(len(x) for x in seqs)], 12)
    assert window == 64 * 1024 + (90 * 90 * 8 + 255) // 256 * 256
    res = sharded_matrices(lib, [seqs], 12, window=window)
    check_ranks(res, full, listed, [90])
