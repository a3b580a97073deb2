#!/usr/bin/env python3
"""Euclidean distance matrix from sparse k-mer rows (dvs_euclid_distances_sparse) on one GPU; prints one JSON line.

    python tools/bench_euclid_sparse.py [--workloads a,b,c] [--reps 5] [--out FILE]

  a  1,000 synthetic genomes of ~4 Mbp (SeqSet.synth) at k=12
  b  10,000 synthetic records of ~1.5 kbp at k=12 (16S-sized tree-building input)
  c  dense (dvs_count_kmers + dvs_euclid_distances) against sparse on 256 x 4 Mbp at k = 9, 10, 11, 12, the largest
     set whose dense k=12 rows (51 GB) still fit; the two matrices are compared at 1e-9 relative in the same run

Times are CUDA events of the library's phases (dvs_ctx_phase_ms), median of --reps runs after one warm-up run.
`products` = pairs x mean distinct k-mers per record; the kernel's own work is counted from the tile shape
(DESIGN.md §5.11): every J entry is visited once per 8-row I block, a visit is 2 LDS.128 + 8 IMAD.WIDE.U32 and
reads 8 bytes of the sparse rows.  The CPU line is the dense oracle (one thread, the reference's norm over 4^k-entry
frequency rows) on the pairs of the first --cpu-records records, extrapolated in proportion to the pairs."""
import argparse
import json
import pathlib
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from diverseseq_b200 import _lib  # noqa: E402

I_ROWS = 8  # kXsI in csrc/euclid_sparse.cu


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1]), "sm_clock_max_mhz": float(q[2])}


def kernel_visits(nnz):
    """J-entry visits of k_xs_gram over the whole lower triangle: I block ib meets every row j <= its last row"""
    cum = np.cumsum(nnz.astype(np.float64))
    n = nnz.size
    last = np.minimum(np.arange(0, n, I_ROWS) + I_ROWS - 1, n - 1)
    return float(cum[last].sum())


def bounds(visits, info, sms):
    rate = sms * info["sm_clock_max_mhz"] * 1e6  # SM-clocks per second at the highest SM clock
    # IMAD.WIDE.U32 writes a register pair: 32 per SM and clock (half the 64-lane IMAD rate); shared memory
    # delivers 128 B per SM and clock, a visit reads 32 B -> both pipes allow 4 visits per SM and clock
    return {"int_pipe_s": 8 * visits / (32 * rate), "lds_s": 32 * visits / (128 * rate), "l2_bytes": 8 * visits}


def median_ms(fn, phase_ids, ctx, reps):
    fn()  # warm-up
    runs = []
    for _ in range(reps):
        fn()
        runs.append(sum(ctx.phase_ms(p) for p in phase_ids))
    return statistics.median(runs), runs


def sparse_workload(ctx, info, sms, name, nrec, mean_len, k, reps, cpu_records):
    ss = _lib.SeqSet.synth(ctx, 20261020, nrec, max(1, nrec // 16), mean_len)
    holder = {}

    def count():
        holder["sp"] = _lib.KSparse.count(ctx, ss, k)

    count_ms, _ = median_ms(count, [_lib.PHASE_SPARSE], ctx, reps)
    sp = holder["sp"]
    nnz, tot, _, _ = sp.stats()
    out = _lib.DeviceBuffer(ctx, nrec * nrec * 8)
    dist_ms, runs = median_ms(lambda: sp.euclidean_into(out.ptr), [_lib.PHASE_EUCLID_SPARSE], ctx, reps)
    pairs = nrec * (nrec - 1) / 2
    products = pairs * float(nnz.mean())
    visits = kernel_visits(nnz)
    b = bounds(visits, info, sms)
    res = {"workload": name, "nrec": nrec, "mean_len": mean_len, "k": k, "bases": ss.total_bases,
           "mean_distinct_kmers": float(nnz.mean()), "count_ms": count_ms, "distance_ms": dist_ms,
           "distance_runs_ms": runs, "fallback_pairs": int(ctx._lib.dvs_euclid_last_fallback_pairs(ctx.handle)),
           "pairs": pairs, "products": products, "products_per_s": products / (dist_ms / 1e3),
           "pairs_per_s": pairs / (dist_ms / 1e3), "kernel_visits": visits,
           "int_pipe_bound_ms": b["int_pipe_s"] * 1e3, "lds_bound_ms": b["lds_s"] * 1e3,
           "share_of_int_pipe_bound": b["int_pipe_s"] * 1e3 / dist_ms,
           "row_bytes_read_per_s": b["l2_bytes"] / (dist_ms / 1e3)}
    if cpu_records:  # the reference's arithmetic: norm of the difference of two dense 4^k frequency rows
        from oracle import oracle as orc
        m = min(cpu_records, nrec)
        dense = np.zeros((m, 4 ** k))
        for r in range(m):
            idx, cnt = sp.record(r)
            dense[r, idx] = cnt / float(tot[r])
        t0 = time.perf_counter()
        orc.euclid_matrix(dense, threads=1)
        dt = time.perf_counter() - t0
        sub = m * (m - 1) / 2
        res["cpu_oracle"] = {"form": "dense rows (oracle.euclid_matrix)", "records": m, "pairs_timed": sub,
                             "seconds_timed": dt, "threads": 1, "extrapolated_seconds_all_pairs": dt * pairs / sub}
    out.close()
    return res


def dense_vs_sparse(ctx, reps):
    nrec, mean_len = 256, 4_000_000
    ss = _lib.SeqSet.synth(ctx, 20261021, nrec, 16, mean_len)
    rows = []
    for k in (9, 10, 11, 12):
        h = {}

        def dcount():
            h.pop("kf", None)
            h["kf"] = _lib.KFreqs.count(ctx, ss, k)

        dcount_ms, _ = median_ms(dcount, [_lib.PHASE_COUNT_KERNEL, _lib.PHASE_FREQ_ENTROPY], ctx, reps)
        dense_out = _lib.DeviceBuffer(ctx, nrec * nrec * 8)
        ddist_ms, _ = median_ms(lambda: h["kf"].euclidean_into(dense_out.ptr), [_lib.PHASE_EUCLID], ctx, reps)
        dense = dense_out.to_host(np.float64, (nrec, nrec))
        h.pop("kf").close()

        def scount():
            h.pop("sp", None)
            h["sp"] = _lib.KSparse.count(ctx, ss, k)

        scount_ms, _ = median_ms(scount, [_lib.PHASE_SPARSE], ctx, reps)
        sdist_ms, _ = median_ms(lambda: h["sp"].euclidean_into(dense_out.ptr), [_lib.PHASE_EUCLID_SPARSE], ctx, reps)
        sparse = dense_out.to_host(np.float64, (nrec, nrec))
        nnz = h["sp"].stats()[0]
        h.pop("sp").close()
        dense_out.close()
        off = ~np.eye(nrec, dtype=bool)
        rel = float(np.max(np.abs(sparse[off] - dense[off]) / dense[off]))
        rows.append({"k": k, "dense_count_ms": dcount_ms, "dense_distance_ms": ddist_ms, "sparse_count_ms": scount_ms,
                     "sparse_distance_ms": sdist_ms, "dense_total_ms": dcount_ms + ddist_ms,
                     "sparse_total_ms": scount_ms + sdist_ms, "mean_distinct_kmers": float(nnz.mean()),
                     "max_rel_diff": rel, "match_1e-9": bool(rel <= 1e-9)})
    return {"workload": "c", "nrec": nrec, "mean_len": mean_len, "rows": rows}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="a,b,c")
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--cpu-records", type=int, default=6, help="records whose pairs the CPU oracle times (0: none)")
    ap.add_argument("--out", default=None, help="also write the JSON line to this file")
    a = ap.parse_args()
    info = gpu_info()
    ctx = _lib.Context(0)
    ctx.enable_timing(True)
    import torch
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    res = dict(info, sms=sms, reps=a.reps, results=[])
    wl = a.workloads.split(",")
    if "a" in wl:
        res["results"].append(sparse_workload(ctx, info, sms, "a", 1000, 4_000_000, 12, a.reps, a.cpu_records))
    if "b" in wl:
        res["results"].append(sparse_workload(ctx, info, sms, "b", 10_000, 1_500, 12, a.reps, a.cpu_records))
    if "c" in wl:
        res["results"].append(dense_vs_sparse(ctx, a.reps))
    line = json.dumps(res)
    print(line)
    if a.out:
        pathlib.Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        pathlib.Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
