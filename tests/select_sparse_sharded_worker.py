"""One rank of the multi-process sparse selection test (launched by tests/test_gpu_select_sparse_sharded.py, or by hand
under torchrun: RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT from the environment).  Every rank counts
its own records, runs dvs_select_sparse_sharded for nmost and max stdev and checks the result bitwise against the
single-GPU call over the union; it prints SELECT_SPARSE_SHARDED_WORKER_OK."""
import os
import pathlib
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from diverseseq_b200 import _lib, shard  # noqa: E402


def main():
    rv = shard.Rendezvous()
    rank, world = rv.rank, rv.world
    ctx = _lib.Context(int(os.environ.get("LOCAL_RANK", "0")))
    npr = [37 + 11 * r for r in range(world)]
    total, first = sum(npr), sum(npr[:rank])
    mine = _lib.synth_host(2028, total, 5, 3_000, first, npr[rank])
    flat, off = _lib.synth_host(2028, total, 5, 3_000)
    longest = rv.allgather(int(np.diff(mine[1]).max()))
    comm = shard.connect(ctx, rv, shard.window_bytes_for_sparse_select(max(longest), 12, total))
    ks = _lib.KSparse.count(ctx, _lib.SeqSet.upload(ctx, *mine), 12, want_entropy=True)
    ref = _lib.KSparse.count(ctx, _lib.SeqSet.upload(ctx, flat, off), 12, want_entropy=True)
    order = shard.global_order(5, total)
    for mode, lo, hi in ((_lib.MODE_NMOST, 8, 8), (_lib.MODE_MAX_STDEV, 4, 10)):
        got = shard.select_sparse_sharded(ctx, comm, ks, order, mode, lo, hi)
        exp = ref.select(order, mode, lo, hi)
        assert got[0].tolist() == exp[0].tolist(), "selection differs from the single-GPU call"
        assert np.array_equal(got[1].view(np.uint64), exp[1].view(np.uint64))
        assert np.array_equal(got[2].view(np.uint64), exp[2].view(np.uint64))
    ctx.sync()
    rv.barrier()
    comm.close()
    rv.close()
    print(f"SELECT_SPARSE_SHARDED_WORKER_OK rank {rank}/{world}", flush=True)


if __name__ == "__main__":
    main()
