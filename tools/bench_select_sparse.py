#!/usr/bin/env python3
"""nmost / max from sparse k-mer rows (dvs_count_kmers_sparse + dvs_select_sparse) on one GPU; prints one JSON line.

    python tools/bench_select_sparse.py [--workloads a,b,c] [--reps 3] [--out FILE]

  a  1,000 synthetic genomes of ~4 Mbp (SeqSet.synth) at k = 12, nmost n = 100
  b  10,000 synthetic records of ~1.5 kbp at k = 12 (gene-sized input), nmost n = 100 and max stdev 5..100
  c  the same 1,000 x 1.5 kbp records at k = 10 through the dense route (dvs_count_kmers + dvs_select) and the sparse
     one, nmost n = 100 and max stdev 5..100; the selections are compared bit for bit in the same run (the evidence
     for the lower k of distance.counts_sparse_for_selection)

Counting and selection times are a host clock around calls that end in a device synchronise: median and the spread
(min, max) of --reps runs after a warm-up.  At k = 12 (a, b) one selection takes minutes, so the warm-up there is an
nmost n = 10 over the first 200 positions of the same rows (it loads every kernel of the timed call) and the timed
runs are --reps-k12 (default 1); the JSON is rewritten after every selection, so a run cut short keeps what it
measured.  `exact_evals` counts the exact re-evaluations the bounded-error kernels handed over.  `peak_mem_gb`: device-wide memory in use, sampled every 10 ms during the runs, above what was in
use before the workload (so it includes the rows and the selection state).  The card's name and power limit are read in
the same run."""
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
from diverseseq_b200 import _lib  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader,nounits",
                        "-i", "0"], capture_output=True, text=True, check=True).stdout.strip().split(", ")
    return {"gpu": q[0], "power_limit_w": float(q[1]), "sm_clock_max_mhz": float(q[2])}


class MemPeak:
    """device-wide used memory, sampled from a thread (torch.cuda.mem_get_info) while the block runs"""

    def __init__(self):
        import torch
        self._get = lambda: torch.cuda.mem_get_info(0)
        free, total = self._get()
        self.base, self.total, self.peak, self._stop = total - free, total, total - free, False

    def __enter__(self):
        def run():
            while not self._stop:
                free, _ = self._get()
                self.peak = max(self.peak, self.total - free)
                time.sleep(0.01)
        self._t = threading.Thread(target=run, daemon=True)
        self._t.start()
        return self

    def __exit__(self, *exc):
        self._stop = True
        self._t.join()

    def gb(self):
        return round((self.peak - self.base) / 1e9, 3)


def timed(fn, reps, warm=None):
    (warm or fn)()
    runs = []
    for _ in range(reps):
        t0 = time.perf_counter()
        out = fn()
        runs.append((time.perf_counter() - t0) * 1e3)
    return out, {"median_ms": round(statistics.median(runs), 3), "min_ms": round(min(runs), 3),
                 "max_ms": round(max(runs), 3), "runs": len(runs)}


def select_stats(ctx, fn, reps, warm=None):
    out, t = timed(fn, reps, warm)
    t["accepts"] = int(ctx._lib.dvs_select_last_accepts(ctx.handle))
    t["exact_evals"] = int(ctx._lib.dvs_select_last_exact_evals(ctx.handle))
    t["size"] = int(out[0].size)
    return out, t


def counted(ctx, fn):
    out = fn()
    ctx.sync()
    return out


def sparse_case(ctx, ss, k, order, selections, reps, small_warm, save):
    res = {}
    with MemPeak() as mp:
        sp, res["count"] = timed(lambda: counted(ctx, lambda: _lib.KSparse.count(ctx, ss, k, want_entropy=True)), reps)
        res["sparse_rows_gb"] = round(8 * float(sp.stats()[0].sum()) / 1e9, 3)
        warm = (lambda: sp.select(order[:200], _lib.MODE_NMOST, 10, 10)) if small_warm else None
        for name, mode, lo, hi in selections:
            _, res[name] = select_stats(ctx, lambda: sp.select(order, mode, lo, hi), reps, warm)
            res["peak_mem_gb"] = mp.gb()
            save(res)
    return res, sp


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--workloads", default="a,b,c")
    ap.add_argument("--reps", type=int, default=3, help="timed runs of workload c")
    ap.add_argument("--reps-k12", type=int, default=1, help="timed runs of workloads a and b")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    ctx = _lib.Context(0)
    out = {"bench": "select_sparse", **gpu_info(), "reps": args.reps, "reps_k12": args.reps_k12,
           "timing": "host clock around synchronised calls"}

    def saver(key):
        def save(res):
            out[key] = res
            if args.out:
                pathlib.Path(args.out).write_text(json.dumps(out) + "\n")
        return save
    nmost100 = ("nmost_n100", _lib.MODE_NMOST, 100, 100)
    stdev = ("max_stdev_5_100", _lib.MODE_MAX_STDEV, 5, 100)
    for w in args.workloads.split(","):
        if w == "a":
            nrec = 1000
            ss = _lib.SeqSet.synth(ctx, 4242, nrec, 40, 4_000_000)
            order = np.random.default_rng(1).permutation(nrec).astype(np.uint32)
            res, sp = sparse_case(ctx, ss, 12, order, [nmost100], args.reps_k12, True, saver("a_1000x4Mbp_k12"))
            del sp, ss
        elif w == "b":
            nrec = 10_000
            ss = _lib.SeqSet.upload(ctx, *_lib.synth_host(1515, nrec, 200, 1500))
            order = np.random.default_rng(2).permutation(nrec).astype(np.uint32)
            res, sp = sparse_case(ctx, ss, 12, order, [nmost100, stdev], args.reps_k12, True, saver("b_10000x1.5kbp_k12"))
            del sp, ss
        elif w == "c":
            nrec = 1000
            ss = _lib.SeqSet.upload(ctx, *_lib.synth_host(1010, nrec, 40, 1500))
            order = np.random.default_rng(3).permutation(nrec).astype(np.uint32)
            res_s, sp = sparse_case(ctx, ss, 10, order, [nmost100, stdev], args.reps, False, lambda res: None)
            res_d = {}
            with MemPeak() as mp:
                kf, res_d["count"] = timed(lambda: counted(ctx, lambda: _lib.KFreqs.count(ctx, ss, 10)), args.reps)
                same = True
                for name, mode, lo, hi in (nmost100, stdev):
                    d, res_d[name] = select_stats(ctx, lambda: kf.select(order, mode, lo, hi), args.reps)
                    s = sp.select(order, mode, lo, hi)
                    same &= d[0].tolist() == s[0].tolist() and np.array_equal(d[1], s[1]) and \
                        np.array_equal(d[2], s[2])
            res_d["peak_mem_gb"] = mp.gb()
            out["c_1000x1.5kbp_k10"] = {"sparse": res_s, "dense": res_d, "bit_identical": bool(same)}
            del sp, kf, ss
    line = json.dumps(out)
    print(line)
    if args.out:
        pathlib.Path(args.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
