#!/usr/bin/env python3
"""nmost / max from sparse k-mer rows kept by W ranks (dvs_select_sparse_sharded); prints one JSON line and writes it
to --out (default profiles/r6_bench_select_sparse_sharded.json).

    python tools/bench_select_sparse_sharded.py [--workloads a,b,c] [--worlds 1,2,4,8] [--reps 3] [--out FILE]

  a  1,000 synthetic records of ~1.5 kbp at k = 10: nmost n = 100 and max stdev 5..100
  b  1,000 synthetic genomes of ~4 Mbp at k = 12: nmost n = 100
  c  10,500 synthetic genomes of ~4 Mbp at k = 12, nmost n = 100, on 8 GPUs only: the sparse rows of this set do not
     fit one GPU

Rank r holds the contiguous block shard.shard_bounds(n, W, r) of the records (SeqSet.synth with `first`) and counts it
itself; the examination order is one random permutation of all records, the same for every W, so every W makes the
same selection.  The ranks are threads of this process with one GPU each; a W larger than the visible GPUs is reported
as "not measured".  Per W: a host clock around the call on every rank, started after a barrier and stopped after a
device synchronise (the largest rank's time; median and spread of --reps runs after a warm-up, one run at k = 12),
accepts, exact evaluations, and the rows and bytes each rank copied in from its peers.  The card's name and power limit
are read in the same run."""
import argparse
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
from diverseseq_b200 import _lib, shard  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1]), "sm_clock_max_mhz": float(q[2])}


def device_count():
    import torch
    return torch.cuda.device_count()


def run_world(W, nrec, mean_len, seed, k, order, selections, reps):
    """one rank per GPU (threads); returns {selection name: result}"""
    group = shard.LocalGroup(W)
    npr = [b - a for a, b in (shard.shard_bounds(nrec, W, r) for r in range(W))]
    # a synthetic record is at most 1.25x the mean length (syn_max_len, csrc/synth.cu); the window is sized for twice it
    window = shard.window_bytes_for_sparse_select(2 * mean_len, k, nrec, extra=1 << 20)
    per_rank = [None] * W
    errors = []

    def worker(r):
        try:
            ctx = _lib.Context(r)
            rv = group.member(r)
            comm = shard.connect(ctx, rv, window)
            first = shard.shard_bounds(nrec, W, r)[0]
            ks = _lib.KSparse.count(ctx, _lib.SeqSet.synth(ctx, seed, npr[r], 40, mean_len, first), k,
                                    want_entropy=True)
            ctx.sync()
            out = {}
            warm = order[:min(200, nrec)]
            ks.select_sharded(comm, npr, warm, _lib.MODE_NMOST, 10, 10)
            for name, mode, lo, hi in selections:
                runs = []
                for _ in range(reps):
                    rv.barrier()
                    t0 = time.perf_counter()
                    res = ks.select_sharded(comm, npr, order, mode, lo, hi)
                    ctx.sync()
                    runs.append(time.perf_counter() - t0)
                rows, nbytes = ks.rows_fetched()
                out[name] = {"runs_s": runs, "size": int(res[0].size), "sel": res[0].tolist(),
                             "accepts": int(ctx._lib.dvs_select_last_accepts(ctx.handle)),
                             "exact_evals": int(ctx._lib.dvs_select_last_exact_evals(ctx.handle)),
                             "rows_fetched": rows, "bytes_fetched": nbytes}
            per_rank[r] = out
            ks.close()
            rv.barrier()
            comm.close()
        except BaseException as exc:  # noqa: BLE001
            errors.append(exc)
            group._bar.abort()

    threads = [threading.Thread(target=worker, args=(r,)) for r in range(W)]
    for t in threads:
        t.start()
    for t in threads:
        t.join()
    if errors:
        raise errors[0]
    result = {}
    for name, *_ in selections:
        rs = [p[name] for p in per_rank]
        assert all(x["sel"] == rs[0]["sel"] for x in rs), "ranks disagree"
        times = [max(x["runs_s"][i] for x in rs) for i in range(reps)]
        result[name] = {"median_s": round(statistics.median(times), 4), "min_s": round(min(times), 4),
                        "max_s": round(max(times), 4), "runs": reps, "size": rs[0]["size"],
                        "accepts": rs[0]["accepts"], "exact_evals": rs[0]["exact_evals"],
                        "rows_fetched": [x["rows_fetched"] for x in rs],
                        "bytes_fetched": [x["bytes_fetched"] for x in rs], "selection": rs[0]["sel"]}
    return result


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="a,b,c")
    ap.add_argument("--worlds", default="1,2,4,8")
    ap.add_argument("--reps", type=int, default=3, help="timed runs of workload a (k = 12: one)")
    ap.add_argument("--out", default=str(ROOT / "profiles" / "r6_bench_select_sparse_sharded.json"))
    args = ap.parse_args()
    ndev = device_count()
    out = {"bench": "select_sparse_sharded", **gpu_info(), "visible_gpus": ndev,
           "timing": "host clock around synchronised calls, largest rank"}

    def save():
        pathlib.Path(args.out).write_text(json.dumps(out) + "\n")

    nmost100 = ("nmost_n100", _lib.MODE_NMOST, 100, 100)
    stdev = ("max_stdev_5_100", _lib.MODE_MAX_STDEV, 5, 100)
    specs = {"a": ("a_1000x1.5kbp_k10", 1000, 1500, 1010, 10, [nmost100, stdev], args.reps, None),
             "b": ("b_1000x4Mbp_k12", 1000, 4_000_000, 4242, 12, [nmost100], 1, None),
             "c": ("c_10500x4Mbp_k12", 10_500, 4_000_000, 4343, 12, [nmost100], 1, [8])}
    for w in args.workloads.split(","):
        key, nrec, mean_len, seed, k, sels, reps, only = specs[w]
        order = np.random.default_rng(seed).permutation(nrec).astype(np.uint32)
        out[key] = {}
        ref = None
        for W in (int(x) for x in args.worlds.split(",")):
            if only and W not in only:
                continue
            if W > ndev:
                out[key][f"W{W}"] = "not measured"
                save()
                continue
            res = run_world(W, nrec, mean_len, seed, k, order, sels, reps)
            if ref is None:
                ref = {n: r["selection"] for n, r in res.items()}
            for n, r in res.items():
                r["same_selection_as_first_W"] = r.pop("selection") == ref[n]
            out[key][f"W{W}"] = res
            save()
    line = json.dumps(out)
    print(line)
    save()


if __name__ == "__main__":
    main()
