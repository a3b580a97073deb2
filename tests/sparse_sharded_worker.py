"""One rank of the multi-process sparse Euclidean test (launched by tests/test_gpu_euclid_sparse_sharded.py, or by
hand under torchrun: RANK / WORLD_SIZE / LOCAL_RANK / MASTER_ADDR / MASTER_PORT from the environment).  Every rank
counts its own records, runs dvs_euclid_distances_sparse_sharded and checks its matrix bitwise against the
single-GPU call over the union; it prints SPARSE_SHARDED_WORKER_OK."""
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
    npr = [75 + 58 * r for r in range(world)]  # not multiples of 8 or 64
    total, first = sum(npr), sum(npr[:rank])
    mine = _lib.synth_host(2027, total, 5, 20_000, first, npr[rank])
    flat, off = _lib.synth_host(2027, total, 5, 20_000)
    bases = rv.allgather(int(mine[1][-1]))
    comm = shard.connect(ctx, rv, shard.window_bytes_for_sparse(npr, bases, 12))
    ks = _lib.KSparse.count(ctx, _lib.SeqSet.upload(ctx, *mine), 12)
    got = shard.sharded_euclidean_sparse(ctx, comm, ks)
    exp = _lib.KSparse.count(ctx, _lib.SeqSet.upload(ctx, flat, off), 12).euclidean()
    assert np.array_equal(got, exp, equal_nan=True), "matrix differs from the single-GPU call"
    ctx.sync()
    rv.barrier()
    comm.close()
    rv.close()
    print(f"SPARSE_SHARDED_WORKER_OK rank {rank}/{world}", flush=True)


if __name__ == "__main__":
    main()
