"""nmost / max from sparse k-mer rows on several ranks, each rank keeping its own rows (dvs_select_sparse_sharded,
csrc/select.cu, DESIGN.md §5.13).

Every rank's result - selected rows, delta_jsd, statistics, accepts and exact evaluations - must be bitwise the
single-GPU `KSparse.count(union).select(order)`, which tests/test_gpu_select_sparse.py checks against the dense path
and the oracle.  A rank copies in only rows that enter the set (owner-computes), which `rows_fetched()` shows.

The ranks are host threads of this process (a copy of test_gpu_euclid_sparse_sharded.run_ranks): one GPU each when
enough are visible, otherwise all on device 0 with the waits taken on the host.  Two real processes run
tests/select_sparse_sharded_worker.py over the TCP rendezvous and cudaIpc.
"""
import os
import pathlib
import subprocess
import sys
import threading

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = pathlib.Path(__file__).resolve().parent.parent
MODES = [("nmost", 10, 10), ("stdev", 5, 12), ("cov", 5, 12)]


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

def mode_id(lib, mode):
    return {"nmost": lib.MODE_NMOST, "stdev": lib.MODE_MAX_STDEV, "cov": lib.MODE_MAX_COV}[mode]


def split(seqs, npr):
    out, o = [], 0
    for n in npr:
        out.append(seqs[o:o + n])
        o += n
    return out


def window_for(seqs, k):
    from diverseseq_b200 import shard
    return shard.window_bytes_for_sparse_select(max((len(s) for s in seqs), default=0), k, len(seqs), extra=1 << 20)


def counters(ctx):
    lib, h = ctx._lib, ctx.handle
    return int(lib.dvs_select_last_accepts(h)), int(lib.dvs_select_last_exact_evals(h))


def single(lib, ctx, seqs, k, calls):
    """[(idx, delta, stats, accepts, exact_evals)] of KSparse.select over the union for each (order, mode, lo, hi)"""
    sp = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), k, want_entropy=True)
    out = []
    for order, mode, lo, hi in calls:
        res = sp.select(order, mode_id(lib, mode), lo, hi)
        out.append(res + counters(ctx))
    sp.close()
    return out


def sharded(lib, seqs, npr, k, calls, window=None):
    """per rank: [(idx, delta, stats, accepts, exact_evals, rows_fetched)] of select_sparse_sharded for each call"""
    from diverseseq_b200 import shard
    shards = split(seqs, npr)

    def fn(rank, rctx, comm):
        ks = lib.KSparse.count(rctx, lib.SeqSet.from_seqs(rctx, shards[rank]), k, want_entropy=True)
        out = []
        for order, mode, lo, hi in calls:
            res = shard.select_sparse_sharded(rctx, comm, ks, order, mode_id(lib, mode), lo, hi)
            out.append(res + counters(rctx) + (ks.rows_fetched()[0],))
        return out

    return run_ranks(len(npr), fn, window or window_for(seqs, k))


def assert_same(a, b):
    assert a[0].tolist() == b[0].tolist()
    assert np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))  # bitwise, NaN and -0.0 included
    assert np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))
    assert a[3:5] == b[3:5]  # accepts, exact evaluations


def check_all(lib, ctx, seqs, npr, k, calls, window=None):
    """every rank bitwise the single-GPU call; returns the per-rank results"""
    exp = single(lib, ctx, seqs, k, calls)
    res = sharded(lib, seqs, npr, k, calls, window)
    for rank_res in res:
        for (order, mode, lo, hi), got, e in zip(calls, rank_res, exp):
            assert_same(got, e)
            fetched = got[5]
            if len(npr) == 1:
                assert fetched == 0
            elif mode == "nmost":
                assert fetched <= lo + got[3]  # the initial set and the accepted candidates, nothing else
            else:
                assert fetched <= lo + got[3] + len(order)
    return res, exp


def orders(npr, seed):
    """a random global order and the interleaved one built from per-rank random orders"""
    from diverseseq_b200 import shard
    rng = np.random.default_rng(seed)
    n = sum(npr)
    local = [rng.permutation(x).astype(np.uint32) for x in npr]
    return [rng.permutation(n).astype(np.uint32), shard.interleaved_order(local, npr)]


@pytest.fixture(scope="module")
def brca1_seqs(brca1):
    return list(brca1.values())


# --------------------------------------------------------------------------------------------- tests ----

SHAPES = [([30, 25], 10), ([20, 0, 35], 11), ([5, 17, 9, 24], 12), ([41, 14], 12)]


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact_only"])
@pytest.mark.parametrize("npr,k", SHAPES, ids=[f"w{len(p)}_k{k}" for p, k in SHAPES])
def test_bit_identical_to_single_gpu(lib, ctx, brca1_seqs, monkeypatch, npr, k, exact):
    """uneven shards (one rank without records), every mode, a random and an interleaved order"""
    monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "1" if exact else "0")
    calls = [(o, mode, lo, hi) for o in orders(npr, 7 + k) for mode, lo, hi in MODES]
    res, _ = check_all(lib, ctx, brca1_seqs, npr, k, calls)
    assert any(r[5] > 0 for rank_res in res for r in rank_res)


def test_one_rank_fetches_nothing(lib, ctx, brca1_seqs):
    calls = [(o, mode, lo, hi) for o in orders([55], 3)[:1] for mode, lo, hi in MODES]
    check_all(lib, ctx, brca1_seqs, [55], 10, calls)


def near_tie_set(rng):
    """(as in test_gpu_select_sparse.py) exact copies and proportional rows: leave-one-out values tie or nearly tie,
    so the bounded-error kernels cannot decide and hand over"""
    base = [rng.integers(0, 4, size=int(rng.integers(2000, 4000)), dtype=np.uint8) for _ in range(10)]
    seqs = []
    for i, b in enumerate(base):
        seqs += [b, b.copy(), np.concatenate([b, b])] if i % 2 == 0 else [b]
    return [seqs[i] for i in rng.permutation(len(seqs))]


def test_exact_fallback_is_exercised(lib, ctx, monkeypatch):
    monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "0")
    seqs = near_tie_set(np.random.default_rng(7))
    order = np.arange(len(seqs), dtype=np.uint32)
    calls = [(order, "nmost", 6, 6), (order, "stdev", 4, 10), (order, "cov", 4, 10)]
    res, exp = check_all(lib, ctx, seqs, [6, 5, 9], 10, calls)
    for i in range(len(calls)):
        assert exp[i][4] > 0
        assert len({rank_res[i][4] for rank_res in res}) == 1


def edge_set(rng):
    """(as in test_gpu_select_sparse.py) records without a valid k-mer, shorter than k, with invalid runs,
    homopolymers and rows whose entries all fall in one bucket, among ordinary ones"""
    seqs = [rng.integers(0, 4, size=int(rng.integers(3000, 9000)), dtype=np.uint8) for _ in range(24)]
    seqs[3] = np.full(500, 4, dtype=np.uint8)
    seqs[5] = rng.integers(0, 4, size=7, dtype=np.uint8)
    seqs[8][100:2000] = 4
    seqs[8][2500:2510] = 5
    seqs[11] = np.zeros(200_000, dtype=np.uint8)
    seqs[13] = np.full(50_000, 3, dtype=np.uint8)
    seqs[16] = np.concatenate([np.zeros(60, dtype=np.uint8), rng.integers(0, 4, size=4, dtype=np.uint8)])
    seqs[19] = np.zeros(0, dtype=np.uint8)
    seqs[21] = np.tile(np.array([0, 1], dtype=np.uint8), 3000)
    return seqs


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact_only"])
def test_edge_records(lib, ctx, monkeypatch, exact):
    monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "1" if exact else "0")
    seqs = edge_set(np.random.default_rng(11))
    calls = [(np.random.default_rng(seed).permutation(24).astype(np.uint32), mode, lo, hi)
             for seed in (0, 1) for mode, lo, hi in [("nmost", 6, 6), ("stdev", 4, 12), ("cov", 3, 9)]]
    res, _ = check_all(lib, ctx, seqs, [4, 12, 8], 10, calls)
    for r in res[0]:
        assert not set(r[0].tolist()) & {3, 5, 19}


def test_winners_on_one_rank(lib, ctx, brca1_seqs):
    """every record the selection keeps lives on rank 0: rank 1 holds none of them and has to fetch each one"""
    order = np.random.default_rng(21).permutation(55).astype(np.uint32)
    calls = [(order, "nmost", 8, 8), (order, "stdev", 5, 12)]
    winners = set()
    for r in single(lib, ctx, brca1_seqs, 10, calls):
        winners |= set(r[0].tolist())
    perm = sorted(winners) + [i for i in range(55) if i not in winners]
    new_id = np.empty(55, dtype=np.uint32)
    new_id[perm] = np.arange(55, dtype=np.uint32)
    seqs = [brca1_seqs[p] for p in perm]
    calls = [(new_id[order], mode, lo, hi) for _, mode, lo, hi in calls]
    npr = [len(winners) + 2, 55 - len(winners) - 2]
    res, exp = check_all(lib, ctx, seqs, npr, 10, calls)
    for i, e in enumerate(exp):
        assert max(e[0].tolist()) < npr[0]
        assert res[1][i][5] >= len(set(e[0].tolist()))  # every winner came over


def errors_of(lib, npr, fn, window):
    """per rank (exception type, message) of fn(rank, ctx, comm)"""
    def wrap(rank, rctx, comm):
        try:
            fn(rank, rctx, comm)
        except (ValueError, TypeError, RuntimeError) as exc:
            return type(exc), str(exc)
        return None
    return run_ranks(len(npr), wrap, window)


def test_errors_agree_on_every_rank(lib, ctx, brca1_seqs):
    from diverseseq_b200 import shard
    seqs = edge_set(np.random.default_rng(11))
    npr = [10, 14]
    shards = split(seqs, npr)
    sp = lib.KSparse.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), 10, want_entropy=True)
    bad_first = np.array([3, 5] + [i for i in range(24) if i not in (3, 5)], dtype=np.uint32)
    one_valid = np.array([3, 0] + [i for i in range(24) if i not in (3, 0)], dtype=np.uint32)
    cases = [(np.arange(24, dtype=np.uint32), 25), (bad_first, 2), (one_valid, 2)]
    expected = []
    for order, n in cases:
        with pytest.raises(ValueError) as e:
            sp.select(order, lib.MODE_NMOST, n)
        expected.append(str(e.value))
    assert expected == ["The number of sequences 24 is < n 25", "records cannot be empty", "must have > 1 KmerSeq"]
    window = window_for(seqs, 10)

    for (order, n), text in zip(cases, expected):
        def fn(rank, rctx, comm, order=order, n=n):
            ks = lib.KSparse.count(rctx, lib.SeqSet.from_seqs(rctx, shards[rank]), 10, want_entropy=True)
            shard.select_sparse_sharded(rctx, comm, ks, order, lib.MODE_NMOST, n)
        assert errors_of(lib, npr, fn, window) == [(ValueError, text)] * 2

    def arg_case(kind):
        def fn(rank, rctx, comm):
            k = 11 if kind == "k" and rank == 1 else 10
            ks = lib.KSparse.count(rctx, lib.SeqSet.from_seqs(rctx, shards[rank]), k,
                                   want_entropy=not (kind == "entropy" and rank == 1))
            nrec = [10, 15] if kind == "npr" and rank == 0 else npr
            ks.select_sharded(comm, nrec, np.arange(24, dtype=np.uint32), lib.MODE_NMOST, 4)
        return fn

    for kind, needle in [("entropy", "without entropies"), ("k", "counted k=11"), ("npr", "nrec_per_rank[1] = 15")]:
        errs = errors_of(lib, npr, arg_case(kind), window)
        assert errs[0] == errs[1] and errs[0][0] is TypeError and needle in errs[0][1], errs

    # a window too small for the call: the message gives both sizes
    need = shard.window_bytes_for_sparse_select(max(len(s) for s in seqs), 10, 24)
    small = 64 * 1024 + (1 << 20)
    assert need > small + 256
    errs = errors_of(lib, npr, arg_case("none"), small)
    assert errs[0] == errs[1] and errs[0][0] is TypeError
    assert f"window of {need} bytes, the window has {small}" in errs[0][1]


def test_matches_oracle_brca1_k10(lib, brca1):
    from oracle import oracle as orc
    seqs = list(brca1.values())
    flat, off = lib.concat(seqs)
    order = np.random.default_rng(55).permutation(55).astype(np.uint32)
    calls = [(order, mode, lo, hi) for mode, lo, hi in MODES]
    res = sharded(lib, seqs, [28, 27], 10, calls)
    for (order, mode, lo, hi), got in zip(calls, res[1]):
        exp = orc.select_seqs(flat, off, order, 10, mode, lo, hi)
        assert got[0].tolist() == exp.ids.tolist() and np.array_equal(got[1], exp.delta_jsd)
        assert got[2][0] == exp.total_jsd and got[2][2] == exp.std_delta_jsd


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
        procs.append(subprocess.Popen([sys.executable, str(ROOT / "tests" / "select_sparse_sharded_worker.py")],
                                      env=env, stdout=subprocess.PIPE, stderr=subprocess.STDOUT, text=True))
    outs = [p.communicate(timeout=600)[0] for p in procs]
    for p, o in zip(procs, outs):
        assert p.returncode == 0, o
        assert "SELECT_SPARSE_SHARDED_WORKER_OK" in o, o
