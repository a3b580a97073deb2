#!/usr/bin/env python3
"""Counting-kernel A/B timings on the bench workload (10,500 synthetic genomes, k=6 by default):

    python tools/bench_count.py [--k 6] [--nrec 10500] [--variants default,super]

A variant is a comma-free name from VARIANTS below (a set of environment switches read by dvs_count_kmers on every
call).  Every variant's count rows are compared with the default kernel's on a sample of records."""
import argparse
import os
import pathlib
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
from diverseseq_b200 import _lib  # noqa: E402

VARIANTS = {
    "default": {},                                   # (k+2)-mers / 16-bit halves, 1024 threads x 3 KB-steps in flight
    "super": {"DVS_COUNT_S3": "0"},                   # (k+1)-mer kernel of round 1
}
KEYS = sorted({k for v in VARIANTS.values() for k in v})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--k", type=int, default=6)
    ap.add_argument("--nrec", type=int, default=10500)
    ap.add_argument("--mean-len", type=int, default=4_000_000)
    ap.add_argument("--variants", default="default,super")
    ap.add_argument("--reps", type=int, default=5)
    a = ap.parse_args()
    ctx = _lib.Context(0)
    ctx.enable_timing(True)
    ss = _lib.SeqSet.synth(ctx, 20261017, a.nrec, 64, a.mean_len)
    bases = ss.total_bases
    sample = np.unique(np.linspace(0, a.nrec - 1, 40).astype(int))
    ref = None
    for name in a.variants.split(","):
        for kk in KEYS:
            os.environ.pop(kk, None)
        os.environ.update(VARIANTS[name])
        ms = []
        for _ in range(a.reps):
            kf = _lib.KFreqs.count(ctx, ss, a.k)
            ms.append(ctx.phase_ms(_lib.PHASE_COUNT_KERNEL))
        rows = np.stack([kf.download(int(r), 1, freqs=False)[0][0] for r in sample])
        if ref is None:
            ref = rows
        same = bool(np.array_equal(rows, ref))
        best = min(ms)
        print(f"{name:10s} k={a.k} count kernel best {best:8.3f} ms  median {np.median(ms):8.3f} ms  "
              f"{bases / best / 1e6:8.1f} Gbp/s  ({bases * 1.008 / best / 1e6 / 6550.1:.3f} of 6550 GB/s)  rows==default: {same}",
              flush=True)
        del kf


if __name__ == "__main__":
    main()
