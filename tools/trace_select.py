#!/usr/bin/env python3
"""Per-round phase timeline of the persistent selection kernels (CTA 0, %globaltimer) and the select
wall time of each form on the benchmark set (nmost n=100, k=6, 10.5k genomes):

    python tools/trace_select.py [--mean-len 4000000] [--out gpurun_out/sel_trace.txt]

DVS_SELECT_PERSIST: 0 = host-driven rounds, 1 = global-state persistent kernel, 2 = SM-replicated."""
from __future__ import annotations

import argparse
import os
import pathlib
import sys

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))
SEED = 20261017


def main() -> int:
    ap = argparse.ArgumentParser()
    ap.add_argument("--nrec", type=int, default=10500)
    ap.add_argument("--mean-len", type=int, default=4_000_000)
    ap.add_argument("--k", type=int, default=6)
    ap.add_argument("--n", type=int, default=100)
    ap.add_argument("--out", default="gpurun_out/sel_trace.txt")
    a = ap.parse_args()
    from diverseseq_b200 import _lib

    ctx = _lib.Context(0)
    ctx.enable_timing(True)
    ss = _lib.SeqSet.synth(ctx, SEED, a.nrec, 64, a.mean_len)
    kf = _lib.KFreqs.count(ctx, ss, a.k)
    order = np.random.default_rng(SEED).permutation(a.nrec).astype(np.uint32)
    ref = None
    for mode in ("0", "1", "2"):
        os.environ["DVS_SELECT_PERSIST"] = mode
        os.environ.pop("DVS_SELECT_TRACE", None)
        ms = []
        for _ in range(4):
            idx, delta, stats = kf.select(order, _lib.MODE_NMOST, a.n)
            ms.append(ctx.phase_ms(_lib.PHASE_SELECT))
        acc = int(ctx._lib.dvs_select_last_accepts(ctx.handle))
        key = (idx.tolist(), delta.tolist(), stats.tolist())
        ref = ref or key
        print(f"persist={mode}: select ms {['%.3f' % m for m in ms]} accepts {acc} exact_evals "
              f"{int(ctx._lib.dvs_select_last_exact_evals(ctx.handle))} same_result {key == ref}", flush=True)
        if mode == "0":
            continue
        out = pathlib.Path(f"{a.out}.{mode}")
        out.parent.mkdir(parents=True, exist_ok=True)
        out.unlink(missing_ok=True)
        os.environ["DVS_SELECT_TRACE"] = str(out)
        kf.select(order, _lib.MODE_NMOST, a.n)
        os.environ.pop("DVS_SELECT_TRACE", None)
        rows = np.loadtxt(out, comments="#", ndmin=2)
        if rows.size:
            r = rows[1:, 1:]
            r = r[(r < 1e6).all(axis=1)]
            print(f"  {out.read_text().splitlines()[0]}", flush=True)
            print(f"  rounds traced {len(r)}: mean ns {np.round(r.mean(axis=0), 0).tolist()} "
                  f"median {np.median(r, axis=0).tolist()} sum/round = {r.sum(axis=1).mean():.0f}", flush=True)
            acc = r[r[:, 3] > 0] if r.shape[1] > 4 else r
            print(f"  accepting rounds {len(acc)}: median {np.median(acc, axis=0).tolist()} sum = {acc.sum(axis=1).mean():.0f}",
                  flush=True)
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
