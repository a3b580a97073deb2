#!/usr/bin/env python3
"""Sparse Euclidean matrix on W GPUs (dvs_euclid_distances_sparse_sharded), one thread rank per GPU; prints one
JSON line and writes it to --out (default profiles/r4_bench_euclid_sparse_sharded.json).

    python tools/bench_euclid_sparse_sharded.py [--workloads a,b,c] [--worlds 1,2,4,8] [--reps 3] [--out FILE]

  a  1,000 synthetic genomes of ~4 Mbp at k=12 (single-GPU reference: 954 ms, profiles/r3_bench_euclid_sparse.json)
  b  10,000 records of ~1.5 kbp at k=12 (single-GPU reference: 5,199 ms)
  c  10,500 genomes of ~4 Mbp at k=12 on 8 GPUs only (the rows, ~340 GB, do not fit fewer): time, memory and 20
     sampled pairs against the sparse-row reference (tests/sparse_euclid_ref.py)

Each rank generates its own records (SeqSet.synth of its range) and counts them; a W that the machine has no GPUs
for is reported as not measured.  Per W: `call_ms` = host clock around the call on every rank (all ranks enter
together, the call ends with a device synchronise), median of --reps after one warm-up; per rank the
DVS_PHASE_EUCLID_SPARSE time (its blocks, copies included), the peer row copies (DVS_PHASE_EUCLID_SPARSE_ROWS) and
the peak device memory during the calls (the high-water mark of the device's default memory pool, which holds the
library's buffers and the rank's own rows, plus the peer window); `bitwise_equal_w1` compares the SHA-256 of every
rank's matrix with W = 1's."""
import argparse
import ctypes
import hashlib
import json
import pathlib
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
sys.path.insert(0, str(ROOT / "tests"))
from diverseseq_b200 import _lib, shard  # noqa: E402

SEED, K = 20261020, 12
CU_MEMPOOL_ATTR_USED_MEM_HIGH = 8


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm",
                        "--format=csv,noheader,nounits"], capture_output=True, text=True, check=True).stdout
    rows = [line.split(", ") for line in q.strip().splitlines()]
    return [{"index": int(r[0]), "gpu": r[1], "power_limit_w": float(r[2]), "sm_clock_max_mhz": float(r[3])}
            for r in rows]


class PoolHigh:
    """high-water mark of a device's default memory pool (driver API)"""

    def __init__(self):
        self.cu = ctypes.CDLL("libcuda.so.1")
        assert self.cu.cuInit(0) == 0

    def _pool(self, device):
        dev, pool = ctypes.c_int(0), ctypes.c_void_p()
        assert self.cu.cuDeviceGet(ctypes.byref(dev), device) == 0
        assert self.cu.cuDeviceGetDefaultMemPool(ctypes.byref(pool), dev) == 0
        return pool

    def reset(self, device):
        v = ctypes.c_uint64(0)
        assert self.cu.cuMemPoolSetAttribute(self._pool(device), CU_MEMPOOL_ATTR_USED_MEM_HIGH, ctypes.byref(v)) == 0

    def get(self, device):
        v = ctypes.c_uint64(0)
        assert self.cu.cuMemPoolGetAttribute(self._pool(device), CU_MEMPOOL_ATTR_USED_MEM_HIGH, ctypes.byref(v)) == 0
        return int(v.value)


def run_world(world, nrec, mean_len, reps, pools, sample=None):
    """one thread rank per GPU; returns the per-rank results"""
    group = shard.LocalGroup(world)
    npr = [shard.shard_bounds(nrec, world, r)[1] - shard.shard_bounds(nrec, world, r)[0] for r in range(world)]
    bases = [None] * world
    out, errors = [None] * world, []

    def worker(rank):
        try:
            rv = group.member(rank)
            ctx = _lib.Context(rank)
            first = shard.shard_bounds(nrec, world, rank)[0]
            ss = _lib.SeqSet.synth(ctx, SEED, npr[rank], max(1, nrec // 16), mean_len, first)
            bases[rank] = ss.total_bases
            rv.barrier()
            window = shard.window_bytes_for_sparse(npr, bases, K)
            comm = shard.connect(ctx, rv, window)
            ks = _lib.KSparse.count(ctx, ss, K)
            ss.close()
            pools.reset(rank)  # (the high-water mark restarts at what is in use now: this rank's rows)
            ctx.enable_timing(True)
            buf = _lib.DeviceBuffer(ctx, nrec * nrec * 8)
            walls, phases, rows = [], [], []
            for it in range(reps + 1):
                rv.barrier()
                t0 = time.perf_counter()
                ks.euclidean_sharded(comm, npr, buf.ptr)
                dt = (time.perf_counter() - t0) * 1e3
                if it:
                    walls.append(dt)
                    phases.append(ctx.phase_ms(_lib.PHASE_EUCLID_SPARSE))
                    rows.append(ctx.phase_ms(_lib.PHASE_EUCLID_SPARSE_ROWS))
            res = {"rank": rank, "nrec": npr[rank], "bases": bases[rank], "call_runs_ms": walls,
                   "euclid_sparse_phase_ms": statistics.median(phases), "row_copy_ms": statistics.median(rows),
                   "fallback_pairs": ks.fallback_pairs(), "window_bytes": window,
                   "peak_device_bytes": pools.get(rank) + window}
            if sample is None:
                m = buf.to_host(np.float64, (nrec, nrec))
                res["sha256"] = hashlib.sha256(m.tobytes()).hexdigest()
                del m
            else:  # (c): the sampled pairs' entries and this rank's rows of them
                m = buf.to_host(np.float64, (nrec, nrec)) if rank == 0 else None
                lo = shard.shard_bounds(nrec, world, rank)[0]
                need = sorted({g for pr in sample for g in pr if lo <= g < lo + npr[rank]})
                _, tot, _, _ = ks.stats()
                res["rows"] = {g: (ks.record(g - lo), int(tot[g - lo])) for g in need}
                if m is not None:
                    res["entries"] = [float(m[a, b]) for a, b in sample]
                    res["sha256"] = hashlib.sha256(m.tobytes()).hexdigest()
                del m
            buf.close()
            ks.close()
            ctx.sync()
            rv.barrier()
            comm.close()
            out[rank] = res
        except BaseException as exc:  # noqa: BLE001
            errors.append((rank, exc))
            group._bar.abort()

    threads = [threading.Thread(target=worker, args=(r,)) for r in range(world)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    real = [e for e in errors if not isinstance(e[1], threading.BrokenBarrierError)]
    if real or errors:
        raise (real or errors)[0][1]
    return out


def summarise(world, ranks, ref_hash):
    per_rep = [max(r["call_runs_ms"][i] for r in ranks) for i in range(len(ranks[0]["call_runs_ms"]))]
    res = {"world": world, "call_ms": statistics.median(per_rep), "call_runs_ms": per_rep,
           "ranks": [{k: v for k, v in r.items() if k not in ("rows", "entries")} for r in ranks]}
    if ref_hash is not None:
        res["bitwise_equal_w1"] = all(r["sha256"] == ref_hash for r in ranks)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="a,b,c")
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r4_bench_euclid_sparse_sharded.json"))
    a = ap.parse_args()
    info = gpu_info()
    ngpu = len(info)
    pools = PoolHigh()
    worlds = [int(w) for w in a.worlds.split(",")]
    res = {"gpus": info, "k": K, "reps": a.reps, "results": [], "not_measured": []}
    specs = {"a": (1000, 4_000_000), "b": (10_000, 1_500)}
    for wl in a.workloads.split(","):
        if wl in specs:
            nrec, mean_len = specs[wl]
            entry = {"workload": wl, "nrec": nrec, "mean_len": mean_len, "worlds": []}
            ref = None
            for w in worlds:
                if w > ngpu:
                    res["not_measured"].append(f"({wl}) at W={w}: {ngpu} GPU(s) visible")
                    continue
                ranks = run_world(w, nrec, mean_len, a.reps, pools)
                if w == 1:
                    ref = ranks[0]["sha256"]
                entry["worlds"].append(summarise(w, ranks, ref))
            res["results"].append(entry)
        elif wl == "c":
            if ngpu < 8:
                res["not_measured"].append(f"(c) 10,500 x 4 Mbp on 8 GPUs: {ngpu} GPU(s) visible")
                continue
            from sparse_euclid_ref import merge_distance
            nrec = 10_500
            rng = np.random.default_rng(7)
            sample = [tuple(sorted(rng.choice(nrec, 2, replace=False).tolist())) for _ in range(20)]
            ranks = run_world(8, nrec, 4_000_000, 1, pools, sample=sample)
            rows = {g: v for r in ranks for g, v in r["rows"].items()}
            errs = []
            for (x, y), got in zip(sample, ranks[0]["entries"]):
                (ia, ca), ta = rows[x]
                (ib, cb), tb = rows[y]
                ref = merge_distance((ia, ca / ta), (ib, cb / tb))
                errs.append(abs(got - ref) / ref if ref else abs(got))
            entry = summarise(8, ranks, None)
            entry.update({"workload": "c", "nrec": nrec, "mean_len": 4_000_000, "sampled_pairs": sample,
                          "sampled_max_rel_err": max(errs), "sampled_match_1e-9": max(errs) <= 1e-9})
            res["results"].append(entry)
    line = json.dumps(res)
    print(line)
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
