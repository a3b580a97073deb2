#!/usr/bin/env python3
"""bench.py — the hot path's headline measurement (BASELINE.json configs[1]).

Workload: "prep + nmost -n 100 k=6, 10.5k synthetic microbial genomes (~4 Mbp each), 1 B200".
One step = k-mer counting (k=6) of every genome into 4^k frequency rows + Shannon entropies,
followed by the order-preserving nmost (n=100) selection over the shuffled record order.
Metric = whole-step throughput in Gbp/s (bases consumed / step time).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--dump-outputs DIR]

N>1 is launched by torchrun (one rank per GPU); each rank counts its own 10.5k-genome shard (weak
scaling) and pushes its frequency rows to every peer over NVLink while it is still counting; the nmost
selection is then ONE single pass over all N x 10.5k records (numprocs=1 semantics) with every window of
candidates scored candidate-sharded and a 16-byte all-reduce(min) per round through the library's peer
windows (no NCCL in the data path; torch.distributed only carries the timing reductions).  --multi chunked
runs the reference's -np semantics instead (select per GPU, final_nmost merge of the winners).
`value` times the step with inputs already in HBM; `e2e` times the same step through
the public host-buffer API (pinned host -> device copy + result read-back inside the timed region).
`--impl reference` times the CPU restatement of the reference (oracle/) on the host cores.
`--dump-outputs DIR` writes what the last timed step returned to its caller as DIR/<name>.npy (see
dump_outputs); the inputs depend on the arguments alone, so two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import pathlib
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = pathlib.Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))
# kernels of different ranks wait for each other: keep every stream on its own hardware queue (before CUDA starts)
os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")

SEED = 20261017
METRIC = "prep_nmost_throughput"
UNIT = "Gbp/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--nrec", type=int, default=10500)
    ap.add_argument("--mean-len", type=int, default=4_000_000)
    ap.add_argument("--nfam", type=int, default=64)
    ap.add_argument("--k", type=int, default=6)
    ap.add_argument("--n", type=int, default=100)
    ap.add_argument("--multi", default="sharded", choices=["sharded", "chunked"],
                    help="N>1 selection: 'sharded' = ONE single-pass selection over all records, candidate-sharded "
                         "with a per-round all-reduce(min) over NVLink; 'chunked' = the reference's -np N semantics "
                         "(select per GPU, merge with final_nmost)")
    ap.add_argument("--overlap", default="on", choices=["on", "off"],
                    help="N=1: dvs_count_select (the nmost rounds trail the counting on SMs of their own) instead of the "
                         "two calls back to back (profiles/r2_overlap_ab.txt)")
    ap.add_argument("--chunks", type=int, default=0, help="counting launches of dvs_count_select (0 = library default)")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-ctree", action="store_true", help="skip the ctree pairs/s side measurements (N=1 only)")
    ap.add_argument("--cpu-seconds", type=float, default=12.0, help="target wall time of one CPU sample")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the results of the last timed step as DIR/<name>.npy (float64, < 64 MB in all)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs is not None and a.impl != "b200":
        ap.error("--dump-outputs needs --impl b200")
    return a


def workload_config(a, world):
    return {
        "workload": f"prep+nmost: count k={a.k} + entropy + nmost n={a.n} over {a.nrec} synthetic genomes "
                    f"(~{a.mean_len / 1e6:g} Mbp each, {a.nfam} Markov families, invalid runs 1e-4) per GPU "
                    "[BASELINE.json configs[1]]",
        "nrec_per_gpu": a.nrec, "mean_len": a.mean_len, "k": a.k, "n": a.n, "seed": SEED,
        "parallelism": ("1 GPU" if world == 1 else
                        f"records sharded x{world}; nmost per GPU then final_nmost merge of the {world}x{a.n} winners "
                        "(reference -np semantics, records.py:206-251)" if a.multi == "chunked" else
                        f"records sharded x{world} (rows pushed to all peers during counting); ONE single-pass nmost "
                        f"over all {world}x{a.nrec} records, candidate-sharded, all-reduce(min) per round over NVLink"),
        "l2": "inputs (~42 GB/GPU) are far larger than the 126 MB L2, no flush needed",
        "overlap": ("dvs_count_select: records counted in the selection's examination order on a second stream in 6 "
                    "launches; the nmost rounds trail the published rows on 36 SMs of their own, the counting keeps the "
                    "other 112" if world == 1 and a.overlap == "on" else "none (count, then select)"),
    }


# ------------------------------------------------- timing plumbing (torch.distributed only) ----
def max_over_ranks(value: float, device=None) -> float:
    """timing rule: a multi-GPU duration is the max over ranks"""
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()):
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def sum_over_ranks(value: float, device=None) -> float:
    import torch
    import torch.distributed as dist

    if not (dist.is_available() and dist.is_initialized()):
        return float(value)
    t = torch.tensor([float(value)], dtype=torch.float64, device=device if device is not None else "cpu")
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    return float(t.item())


# --------------------------------------------------------------------------- clocks ----
class ClockSampler:
    """SM clock + clock-event reasons DURING the timed region.  The timed region of the default run is
    tens of milliseconds, far below nvidia-smi's practical sampling period, so NVML is polled in-process
    from a thread (ctypes calls into libdvs release the GIL); `nvidia-smi -lms` is the fallback when the
    NVML binding is unavailable.  CUDA_VISIBLE_DEVICES remapping is resolved through the PCI bus id."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int, pci_bus_id: str | None = None):
        self.index = index
        self.pci = pci_bus_id
        self.proc = None
        self.lines = []
        self.nvml = None
        self.samples = []  # (sm_mhz, power_w, reasons_mask)
        self._stop = threading.Event()

    def start(self):
        try:
            import pynvml
            pynvml.nvmlInit()
            try:
                h = pynvml.nvmlDeviceGetHandleByPciBusId(self.pci.encode())
            except Exception:
                h = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml, self.h = pynvml, h
            self.thread = threading.Thread(target=self._poll, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "50", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _poll(self):
        nv, h = self.nvml, self.h
        reasons = getattr(nv, "nvmlDeviceGetCurrentClocksEventReasons", None) or nv.nvmlDeviceGetCurrentClocksThrottleReasons
        while not self._stop.is_set():
            try:
                self.samples.append((float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)),
                                     nv.nvmlDeviceGetPowerUsage(h) / 1000.0, int(reasons(h))))
            except Exception:
                pass
            time.sleep(0.002)

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    @staticmethod
    def _summary(sm, mx, pw, reasons, how):
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"], "how": how}
        # "under load": samples in the upper half of the observed power range
        thr = (max(pw) + min(pw)) / 2
        load = [s for s, p in zip(sm, pw) if p >= thr] or sm
        return {"sm_mhz": float(np.median(load)), "sm_max_mhz": float(mx), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons), "how": how}

    def stop(self):
        if self.nvml is not None:
            self._stop.set()
            self.thread.join(timeout=2)
            nv = self.nvml
            names = {"hw_slowdown": "nvmlClocksThrottleReasonHwSlowdown",
                     "hw_thermal_slowdown": "nvmlClocksThrottleReasonHwThermalSlowdown",
                     "sw_thermal_slowdown": "nvmlClocksThrottleReasonSwThermalSlowdown",
                     "sw_power_cap": "nvmlClocksThrottleReasonSwPowerCap"}
            seen = set()
            for _, _, mask in self.samples:
                for name, attr in names.items():
                    if mask & int(getattr(nv, attr, 0)):
                        seen.add(name)
            out = self._summary([s[0] for s in self.samples], self.sm_max, [s[1] for s in self.samples], seen,
                                "NVML polled in-process every ~2 ms during the timed region")
            try:
                nv.nvmlShutdown()
            except Exception:
                pass
            return out
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvml and nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2])); pw.append(float(f[3]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return self._summary(sm, max(mx) if mx else None, pw, reasons, "nvidia-smi -lms 50")


# ------------------------------------------------------------------- CPU (oracle) leg ----
def cpu_sample_run(flat, offsets, k, n, threads):
    """the reference's path on the host: count+freq+entropy over all host threads, then the (serial)
    nmost selection — returns seconds"""
    from oracle import oracle as orc

    nrec = len(offsets) - 1
    t0 = time.perf_counter()
    _, freqs, ent, valid = orc.count_batch(flat, offsets, k, threads=threads, want_counts=False)
    t1 = time.perf_counter()
    order = np.random.default_rng(SEED).permutation(nrec)
    nn = min(n, max(2, nrec // 2))
    orc.select_rows(freqs, ent, order, "nmost", nn, valid=valid)
    t2 = time.perf_counter()
    return t2 - t0, t1 - t0, t2 - t1, nn


def make_cpu_sample(a, want_records, seqset=None):
    """first `want_records` genomes of the synthetic set as host arrays"""
    from diverseseq_b200 import _lib

    if seqset is not None:
        off = seqset.offsets()
        flat = seqset.download(0, want_records)
        return flat, (off[: want_records + 1] - off[0]).astype(np.uint64)
    return _lib.synth_host(SEED, a.nrec, a.nfam, a.mean_len, 0, want_records)


def cpu_baseline(a, seqset=None, target_s=12.0):
    from oracle import oracle as orc

    threads = max(1, orc.hardware_threads())
    probe_n = min(a.nrec, max(2, threads))
    flat, off = make_cpu_sample(a, probe_n, seqset)
    dt, *_ = cpu_sample_run(flat, off, a.k, a.n, threads)
    rate = float(off[-1]) / max(dt, 1e-6)  # bases/s on the probe
    avail = 8e9
    try:
        for ln in open("/proc/meminfo"):
            if ln.startswith("MemAvailable"):
                avail = float(ln.split()[1]) * 1024
    except OSError:
        pass
    want_bases = min(rate * target_s, 0.25 * avail)
    want = int(min(a.nrec, max(probe_n, want_bases / a.mean_len)))
    flat, off = make_cpu_sample(a, want, seqset)
    dt, t_count, t_sel, nn = cpu_sample_run(flat, off, a.k, a.n, threads)
    bases = float(off[-1])
    return {"value": bases / dt / 1e9, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"first {want} of {a.nrec} genomes ({bases / 1e9:.2f} Gbp): count+entropy on {threads} threads "
                      f"{t_count:.2f}s + serial nmost n={nn} {t_sel:.2f}s",
            "seconds": dt}


def run_reference(a):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    seqset = None
    try:
        from diverseseq_b200 import _lib
        ctx = _lib.Context(int(os.environ.get("LOCAL_RANK", "0")))
        seqset = _lib.SeqSet.synth(ctx, SEED, a.nrec, a.nfam, a.mean_len)  # generator only; timing is CPU-only
    except Exception:
        seqset = None
    vals = []
    base = None
    for i in range(a.warmup + a.steps):
        base = cpu_baseline(a, seqset, target_s=a.cpu_seconds if i >= a.warmup else a.cpu_seconds / 4)
        if i >= a.warmup:
            vals.append(base)
    dt = float(np.mean([v["seconds"] for v in vals]))
    v = float(np.mean([v["value"] for v in vals]))
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8 counts / f64 entropy", "data": "synthetic",
            "config": workload_config(a, 1),
            "cpu_baseline": {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")} | {"value": v},
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0}
    emit(line)
    return 0



# ------------------------------------------------------------- side metrics (configs[2..4], k=12) ----
FP64_PEAK_TFLOPS = 40.0   # B200 nominal FP64 (vector = tensor); MEASURED_PEAKS.json carries no FP64 figure
INT32_PEAK_TOPS = 148 * 128 * 1.965e9 / 1e12  # 128 INT32 lanes per SM and clock (nominal issue rate)


def side_metrics(a, ctx, comm, rank, world, device, barrier, hbm_peak):
    import torch

    from diverseseq_b200 import _lib, shard

    def wall(fn):
        barrier()
        t0 = time.perf_counter()
        out = fn()
        ctx.sync()
        barrier()
        return max_over_ranks(time.perf_counter() - t0, device), out

    out = {"scaling": "strong: one record set split over the ranks", "n_gpus": world}
    # ---- configs[3]: mash k=16 s=3000 on 1,000 genomes ----
    n_m = 1000
    b, e = shard.shard_bounds(n_m, world, rank)
    ss = _lib.SeqSet.synth(ctx, SEED, e - b, a.nfam, a.mean_len, first=b)
    _lib.Sketches.sketch(ctx, ss, 16, 3000, 4, True).close()
    sk_wall, sk = wall(lambda: _lib.Sketches.sketch(ctx, ss, 16, 3000, 4, True))
    sk_ms = max_over_ranks(ctx.phase_ms(_lib.PHASE_SKETCH), device)
    mash_bases = sum_over_ranks(ss.total_bases, device)
    npm = n_m * (n_m - 1) // 2
    dmat = _lib.DeviceBuffer(ctx, n_m * n_m * 8)
    if world > 1:
        meta = comm.rv.allgather((int(sk.nrec), int(sk.stride)))
        allsk = sk.allgather(comm, [m[0] for m in meta], max(m[1] for m in meta))
        allsk.distances_sharded(comm, 16, 3000, dmat.ptr)
        pairs_wall, _ = wall(lambda: allsk.distances_sharded(comm, 16, 3000, dmat.ptr))
        allsk.close()
    else:
        sk.distances_into(dmat.ptr, 16, 3000)
        pairs_wall, _ = wall(lambda: sk.distances_into(dmat.ptr, 16, 3000))
    pairs_ms = max_over_ranks(ctx.phase_ms(_lib.PHASE_MASH_PAIRS), device)
    int_ops = (6 * 16 + 8) * mash_bases  # SURVEY 8d: ~(6k+8) integer ops per window
    out["mash_k16_s3000_1k_genomes"] = {
        "sketch_ms": sk_ms, "sketch_gbp_per_s": mash_bases / sk_ms / 1e6, "pairs": npm, "pairs_kernel_ms": pairs_ms,
        "pairs_per_s": npm / pairs_ms * 1e3, "pairs_per_s_wall": npm / pairs_wall,
        "roofline_sketch": {"bound": "int32-alu", "achieved": int_ops / sk_ms / 1e9, "peak": INT32_PEAK_TOPS * world,
                            "unit": "Tint-op/s", "frac": int_ops / sk_ms / 1e9 / (INT32_PEAK_TOPS * world),
                            "note": "(6k+8) integer ops per window (SURVEY 8d) vs 128 INT32 lanes/SM/clk nominal"},
        "roofline_pairs": {"bound": "latency (L2-resident sketches)", "achieved": npm * 8 * 3000 / pairs_ms / 1e6,
                           "unit": "GB/s nominal (8 s bytes per pair)", "peak": None, "frac": None}}
    sk.close(); dmat.close(); ss.close()

    # ---- configs[4] / configs[2]: 10.5k genomes at k=8 (rows depend on nrec x 4^8 only: 400 kbp genomes) ----
    n_e = a.nrec
    b, e = shard.shard_bounds(n_e, world, rank)
    ss = _lib.SeqSet.synth(ctx, SEED, e - b, a.nfam, 400_000, first=b)
    if world > 1:
        kf8, _ = shard.count_sharded(ctx, comm, ss, 8)
    else:
        kf8 = _lib.KFreqs.count(ctx, ss, 8)
    npe = n_e * (n_e - 1) // 2
    dmat = _lib.DeviceBuffer(ctx, n_e * n_e * 8)
    if world > 1:
        eu_wall, _ = wall(lambda: kf8.euclidean_sharded(comm, dmat.ptr))
    else:
        eu_wall, _ = wall(lambda: kf8.euclidean_into(dmat.ptr))
    eu_ms = max_over_ranks(ctx.phase_ms(_lib.PHASE_EUCLID), device)
    tf = 2.0 * 65536 * npe / eu_ms / 1e9
    entry = {"pairs": npe, "kernel_ms": eu_ms, "pairs_per_s": npe / eu_ms * 1e3, "pairs_per_s_wall": npe / eu_wall,
             "roofline": {"bound": "fp64", "achieved": tf, "peak": FP64_PEAK_TFLOPS * world, "unit": "TFLOP/s",
                          "frac": tf / (FP64_PEAK_TFLOPS * world),
                          "note": "useful flops 2 D per pair (the difference form issues 3 D); nominal FP64 peak"}}
    if rank == 0:
        t0 = time.perf_counter()
        children, _, _ = _lib.linkage_average(ctx, n=n_e, device_ptr=dmat.ptr)
        entry["average_linkage"] = {"device_ms": ctx.phase_ms(_lib.PHASE_CLUSTER), "wall_ms": (time.perf_counter() - t0) * 1e3,
                                    "merges": int(children.shape[0]), "note": "replicas only: rank 0 builds the tree"}
    out[f"euclid_k8_{n_e}_genomes"] = entry
    dmat.close()
    order8 = shard.global_order(SEED, n_e)
    sweeps = {}
    for name, mode, lo, hi in (("stdev_5_10", _lib.MODE_MAX_STDEV, 5, 10), ("stdev_10_100", _lib.MODE_MAX_STDEV, 10, 100),
                               ("cov_10_100", _lib.MODE_MAX_COV, 10, 100), ("nmost_100", _lib.MODE_NMOST, 100, 100)):
        sel = (lambda m=mode, l=lo, h=hi: kf8.select_sharded(comm, order8, m, l, h)) if world > 1 else \
              (lambda m=mode, l=lo, h=hi: kf8.select(order8, m, l, h))
        sel()
        w, (idx, _d, st) = wall(sel)
        sweeps[name] = {"wall_s": w, "device_ms": max_over_ranks(ctx.phase_ms(_lib.PHASE_SELECT), device),
                        "size": int(idx.size), "total_jsd": float(st[0]), "head": idx[:4].tolist(),
                        "scan_bytes_per_pass": n_e * 65536 * 8}
    out[f"max_k8_{n_e}_genomes"] = sweeps
    kf8.close(); ss.close()

    # ---- north star: k=12 counting, records sharded, no collective ----
    # sparse rows (distinct k-mers + counts, 8 bytes each: the only form that holds 10.5k genomes) ...
    n12 = 512
    ss = _lib.SeqSet.synth(ctx, SEED + 12 + rank, n12, a.nfam, a.mean_len)
    _lib.KSparse.count(ctx, ss, 12).close()
    w12, sp = wall(lambda: _lib.KSparse.count(ctx, ss, 12))
    ms12 = max_over_ranks(ctx.phase_ms(_lib.PHASE_SPARSE), device)
    nnz, tot, _e, _v = sp.stats()
    b12 = sum_over_ranks(ss.total_bases, device)
    nnz_all = sum_over_ranks(float(nnz.sum()), device)
    sparse_bytes = b12 + 8.0 * nnz_all  # SURVEY 8d: L + 8 D_r per record
    out["count_k12_sparse"] = {"genomes": n12 * world, "gbp": b12 / 1e9, "kernel_ms": ms12, "gbp_per_s": b12 / ms12 / 1e6,
                               "gbp_per_s_wall": b12 / w12 / 1e9, "distinct_per_valid_kmer": nnz_all / max(sum_over_ranks(float(tot.sum()), device), 1.0),
                               "roofline": {"bound": "hbm", "achieved": sparse_bytes / ms12 / 1e6, "peak": hbm_peak * world,
                                            "unit": "GB/s", "frac": sparse_bytes / ms12 / 1e6 / (hbm_peak * world),
                                            "note": "sparse rows: L + 8 D_r bytes per record (~8 B/bp); three radix passes "
                                                    "through shared memory (csrc/sparse.cu)"}}
    sp.close(); ss.close()
    # ... and the dense u32 rows of round 1 (global RED.ADD into an L2-resident 64 MB row), for comparison
    n12 = 64
    ss = _lib.SeqSet.synth(ctx, SEED + 12 + rank, n12, a.nfam, a.mean_len)
    _lib.KFreqs.count(ctx, ss, 12).close()
    w12, kf12 = wall(lambda: _lib.KFreqs.count(ctx, ss, 12))
    ms12 = max_over_ranks(ctx.phase_ms(_lib.PHASE_COUNT_KERNEL), device)
    b12 = sum_over_ranks(ss.total_bases, device)
    dense_bytes = b12 + n12 * world * 4 * 4 ** 12
    out["count_k12_dense"] = {"genomes": n12 * world, "gbp": b12 / 1e9, "kernel_ms": ms12, "gbp_per_s": b12 / ms12 / 1e6,
                              "roofline": {"bound": "hbm", "achieved": dense_bytes / ms12 / 1e6, "peak": hbm_peak * world,
                                           "unit": "GB/s", "frac": dense_bytes / ms12 / 1e6 / (hbm_peak * world),
                                           "note": "dense u32 rows: L + 4*4^k bytes per record (17.8 B/bp)"}}
    kf12.close(); ss.close()
    return out


# ------------------------------------------------------------------------ --dump-outputs ----
DUMP_ROWS = 512              # frequency rows in the seeded sample ...
DUMP_FREQ_BYTES = 16 << 20   # ... and their size at most (columns are sampled too when rows are wider)


def dump_outputs(out_dir, kf, idx, delta, stats):
    """What one step hands its caller, as float64 .npy files: the selection (`selected_indices` in Vec order,
    `delta_jsd`, `selection_stats` = total_jsd, mean, std and cov of delta_jsd, summed entropies) and, of the
    frequency rows it leaves on the device, every record's `entropies` and `valid` flag plus `freqs_sample`,
    the rows `freqs_sample_rows` x columns `freqs_sample_cols` drawn with a fixed seed."""
    out = pathlib.Path(out_dir)
    out.mkdir(parents=True, exist_ok=True)
    nrec, dim = kf.nrec, kf.dim
    rng = np.random.default_rng(SEED)
    rows = np.sort(rng.choice(nrec, size=min(nrec, DUMP_ROWS), replace=False))
    ncols = min(dim, DUMP_FREQ_BYTES // (8 * max(rows.size, 1)))
    cols = np.arange(dim) if ncols == dim else np.sort(rng.choice(dim, size=ncols, replace=False))
    sample = np.empty((rows.size, cols.size), dtype=np.float64)
    for i, r in enumerate(rows):
        sample[i] = kf.download(int(r), 1, counts=False)[1][0, cols]
    _, _, ent, valid = kf.download(counts=False, freqs=False)
    arrays = {"selected_indices": idx, "delta_jsd": delta, "selection_stats": stats, "entropies": ent, "valid": valid,
              "freqs_sample": sample, "freqs_sample_rows": rows, "freqs_sample_cols": cols}
    for name, arr in arrays.items():
        np.save(out / f"{name}.npy", np.asarray(arr, dtype=np.float64))


# ------------------------------------------------------------------------ B200 leg ----
_REAL_STDOUT = None


def claim_stdout():
    """stdout carries exactly ONE JSON line: everything else any library prints to fd 1 (NCCL's version
    banner, torchrun notices) is sent to stderr; emit() writes the line to the real stdout."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.fdopen(os.dup(1), "w")
        os.dup2(2, 1)


def emit(line: dict) -> None:
    out = _REAL_STDOUT or sys.stdout
    out.write(json.dumps(line) + "\n")
    out.flush()


def main():
    a = parse_args()
    claim_stdout()
    if a.impl == "reference":
        return run_reference(a)

    import torch
    import torch.distributed as dist

    from diverseseq_b200 import _lib, shard

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=device)  # timing reductions / barriers only
    ctx = _lib.Context(local)
    ctx.enable_timing(True)
    stream = torch.cuda.ExternalStream(ctx.stream, device=device)
    comm = None
    if world > 1:
        # the library's own peer windows: rows of all ranks at k (headline) and, for the side metrics, the
        # 10.5k x 4^8 rows + the n x n matrix of the ctree configs
        rv = shard.Rendezvous()
        need = max(shard.window_bytes_for(a.nrec * world, 4 ** a.k),
                   0 if a.no_ctree else shard.window_bytes_for(a.nrec, 4 ** 8, a.nrec * a.nrec * 8))
        comm = shard.connect(ctx, rv, need)

    # ---- synthetic inputs, resident in HBM (rank r holds records of seed SEED+r) ----
    seqset = _lib.SeqSet.synth(ctx, SEED + rank, a.nrec, a.nfam, a.mean_len)
    bases = seqset.total_bases
    total_bases = sum_over_ranks(bases, device)
    order = shard.global_order(SEED, a.nrec)
    local_order = shard.global_order(SEED + rank, a.nrec)
    if world > 1:  # position-interleaved global order over the rank-major rows of all ranks
        order = shard.interleaved_order([shard.global_order(SEED + r, a.nrec) for r in range(world)], [a.nrec] * world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(device)

    phase = {}
    kept = []  # the frequency rows of a step run with keep=True (--dump-outputs: the last timed step)

    def release(kf, keep):
        if keep:
            kept.append(kf)
        else:
            kf.close()

    def step(ss, keep=False):
        t0 = time.perf_counter()
        if world > 1 and a.multi == "sharded":
            kf, _ = shard.count_sharded(ctx, comm, ss, a.k)
            t1 = time.perf_counter()
            idx, delta, stats = shard.select_sharded(ctx, comm, kf, order, _lib.MODE_NMOST, a.n)
            release(kf, keep)
        else:
            if world == 1 and a.overlap == "on":
                # counting with the nmost rounds trailing it (dvs_count_select): one call, two streams
                kf, idx, delta, stats = _lib.KFreqs.count_select(ctx, ss, a.k, order, _lib.MODE_NMOST, a.n, a.n,
                                                                 chunks=a.chunks)
                t1 = time.perf_counter()
                release(kf, keep)
                phase["trail_accepts"] = int(ctx._lib.dvs_select_last_trail_accepts(ctx.handle))
                phase["count_ms"] = ctx.phase_ms(_lib.PHASE_COUNT_LAUNCHES)  # the counting launches alone, summed
                phase["count_region_ms"] = ctx.phase_ms(_lib.PHASE_COUNT_KERNEL)  # first launch .. last entropy launch
                phase["freq_entropy_ms"] = 0.0  # (inside the chunk loop)
                phase["select_ms"] = ctx.phase_ms(_lib.PHASE_SELECT)
                phase["host_wall_ms"] = {"count_select_call": (t1 - t0) * 1e3}
                return idx, delta, stats
            kf = _lib.KFreqs.count(ctx, ss, a.k)
            t1 = time.perf_counter()
            if world > 1:
                idx, delta, stats = shard.chunked_select(ctx, comm, kf, local_order, _lib.MODE_NMOST, a.n, a.n)
                idx = np.array([r * a.nrec + i for r, i in idx], dtype=np.uint32)
            else:
                idx, delta, stats = kf.select(order, _lib.MODE_NMOST, a.n)
            release(kf, keep)
        t3 = time.perf_counter()
        phase["count_ms"] = ctx.phase_ms(_lib.PHASE_COUNT_KERNEL)
        phase["freq_entropy_ms"] = ctx.phase_ms(_lib.PHASE_FREQ_ENTROPY)
        phase["select_ms"] = ctx.phase_ms(_lib.PHASE_SELECT)
        phase["host_wall_ms"] = {"count_call": (t1 - t0) * 1e3, "select_call": (t3 - t1) * 1e3}
        return idx, delta, stats

    def timed(fn, steps):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        out = None
        for _ in range(steps):
            out = fn()
        e1.record(stream)
        barrier()
        return max_over_ranks(e0.elapsed_time(e1), device) / steps, out

    for _ in range(a.warmup):
        step(seqset)
    try:
        pr = torch.cuda.get_device_properties(local)
        pci = f"{pr.pci_domain_id:08x}:{pr.pci_bus_id:02x}:{pr.pci_device_id:02x}.0"
    except Exception:
        pci = None
    sampler = ClockSampler(local, pci)
    if rank == 0:
        sampler.start()
    launches0 = ctx.launch_count
    count_ms, fe_ms, sel_ms = [], [], []

    def step_resident():
        r = step(seqset, keep=a.dump_outputs is not None and len(count_ms) == a.steps - 1)
        count_ms.append(phase["count_ms"]); fe_ms.append(phase["freq_entropy_ms"]); sel_ms.append(phase["select_ms"])
        return r

    ms_step, (idx, delta, stats) = timed(step_resident, a.steps)
    launches = ctx.launch_count - launches0  # kernels of libdvs_b200.so launched inside the timed region (all K steps)
    accepts = int(ctx._lib.dvs_select_last_accepts(ctx.handle))
    if kept:  # before any further step: the peer window of the sharded path holds the rows of one step only
        if rank == 0:
            dump_outputs(a.dump_outputs, kept[0], idx, delta, stats)
        kept.pop().close()
    # NVML sometimes answers only once or twice inside a 70 ms timed region: keep the load on with further identical
    # (untimed) steps until the sampler has a usable number of readings; every rank runs the same number of steps
    in_region = len(sampler.samples) if rank == 0 else 0
    extra_steps = 0
    while max_over_ranks(1.0 if (rank == 0 and len(sampler.samples) < 12 and extra_steps < 60) else 0.0, device) > 0.0:
        step(seqset)
        extra_steps += 1
    clocks = sampler.stop() if rank == 0 else None
    if clocks is not None and extra_steps:
        clocks["how"] += f"; {in_region} readings fell inside the timed region, the rest during {extra_steps} further identical steps right after it"
    value = total_bases / (ms_step * 1e-3) / 1e9

    overlapped = world == 1 and a.overlap == "on"
    alone_ms = None
    if overlapped:  # the same kernel without the selection beside it (explains the in-step figure; not the headline)
        _lib.KFreqs.count(ctx, seqset, a.k).close()
        al = []
        for _ in range(3):
            kfa = _lib.KFreqs.count(ctx, seqset, a.k)
            ctx.sync()
            al.append(ctx.phase_ms(_lib.PHASE_COUNT_KERNEL))
            kfa.close()
        alone_ms = float(np.median(al))

    # ---- roofline of the dominant kernel (k_count), timed live by CUDA events on its stream ----
    kc_ms = float(np.mean(count_ms))
    dim = 4 ** a.k
    algo_bytes = bases + a.nrec * (8 * dim + 8)  # SURVEY §8d: L + 8*4^k + 8 per record
    peaks = {}
    try:
        peaks = json.loads((ROOT / "MEASURED_PEAKS.json").read_text())
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    achieved = algo_bytes / (kc_ms * 1e-3) / 1e9
    traffic = None  # dram__bytes_read.sum + dram__bytes_write.sum of one launch, from the committed ncu capture
    try:
        tr = json.loads((ROOT / "profiles" / "r2_k_count_traffic.json").read_text())
        wl = tr["workload"]
        if (wl["nrec"], wl["mean_len"], wl["k"]) == (a.nrec, a.mean_len, a.k):
            traffic = tr["traffic_bytes_per_launch"]
    except Exception:
        pass
    roofline = {"bound": "hbm", "kernel": "k_count", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "peak_source": "MEASURED_PEAKS.json hbm_gbs (burst copy)" if peaks else "fallback 6650 GB/s",
                "kernel_ms": kc_ms, "algorithmic_bytes_per_launch": algo_bytes}
    if overlapped:
        roofline["note"] = ("in-step: sum of the 6 counting launches of a step; from the third launch on the selection "
                            "kernel owns 36 of the 148 SMs, so the counting runs on 112; `alone` = the same kernel as one "
                            "launch on the whole GPU, timed in the same run after the timed region; `step_frac` = "
                            "algorithmic bytes / ms_per_step / peak")
        roofline["step_frac"] = algo_bytes / (ms_step * 1e-3) / 1e9 / peak
        roofline["alone"] = {"kernel_ms": alone_ms, "achieved": algo_bytes / (alone_ms * 1e-3) / 1e9,
                             "frac": algo_bytes / (alone_ms * 1e-3) / 1e9 / peak}

    # ---- end to end through the host-buffer API: pinned host -> device copy inside the timed region ----
    e2e = None
    if not a.no_e2e:
        # stage 1 (collective decision): can every local rank pin its whole input?  Refuse (e2e.value =
        # null with the reason) rather than risk the host OOM killer when the box cannot hold N x 42 GB.
        why, pinned = None, None
        try:
            lws = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
            avail = None
            for ln in open("/proc/meminfo"):
                if ln.startswith("MemAvailable"):
                    avail = float(ln.split()[1]) * 1024
            if avail is not None and bases * lws * 1.25 > avail:
                raise MemoryError(f"host MemAvailable {avail / 1e9:.0f} GB < {lws} ranks x {bases / 1e9:.0f} GB pinned input")
            pinned = torch.empty(int(bases) + 64, dtype=torch.uint8, pin_memory=True)
        except Exception as exc:
            why = f"{type(exc).__name__}: {exc}"
        all_ok = sum_over_ranks(0.0 if why is None else 1.0, device) == 0.0
        if not all_ok:
            e2e = {"value": None, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0,
                   "error": why or "another rank could not pin its input"}
            pinned = None
        else:
            host = pinned.numpy()
            seqset.download(0, a.nrec, out=host)
            offsets = seqset.offsets()
            del seqset
            seqset = None

            def step_e2e():
                ss = _lib.SeqSet.upload(ctx, host[: int(bases)], offsets)
                r = step(ss)
                ss.close()
                return r

            step_e2e()
            ms_e2e, (idx2, _d2, _s2) = timed(step_e2e, a.steps)
            assert idx2.tolist() == idx.tolist(), "e2e selection differs from the resident-input run"
            d2h = idx.nbytes + delta.nbytes + 5 * 8 + 4
            e2e = {"value": total_bases / (ms_e2e * 1e-3) / 1e9, "unit": UNIT,
                   "h2d_bytes_per_step": int(bases + offsets.nbytes + order.nbytes), "d2h_bytes_per_step": int(d2h),
                   "ms_per_step": ms_e2e, "upload_ms": ctx.phase_ms(_lib.PHASE_UPLOAD),
                   "h2d_wire_bytes_per_step": ctx.last_upload_wire_bytes,
                   "note": "pinned host buffer (1 byte/base, the reference layout) -> dvs_seqset_upload (host threads "
                           "pack 2 bits/base, PCIe, device unpack to the same bytes) -> count -> nmost -> read back "
                           "indices/deltas; h2d_bytes_per_step counts the host bytes handed to the API"}

    base = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        if seqset is None:
            seqset = _lib.SeqSet.synth(ctx, SEED, a.nrec, a.nfam, a.mean_len)
        base = cpu_baseline(a, seqset, a.cpu_seconds)
        base = {k: base[k] for k in ("value", "unit", "cores", "kind", "sample")}

    # BASELINE.json's other configs as side metrics, outside the timed step, at every N (strong scaling: the SAME
    # record sets split over the ranks): configs[2] `max` sweeps at k=8 (candidate-sharded), configs[3] mash k=16
    # s=3000 on 1,000 genomes (pairs dealt over the GPUs), configs[4] Euclidean k=8 on 10.5k genomes (tiles dealt
    # over the GPUs), the north star's k=12 counting, each with the roofline that bounds it
    ctree = None
    if not a.no_ctree:
        try:
            del seqset
            seqset = None
            ctree = side_metrics(a, ctx, comm, rank, world, device, barrier, peak)
        except Exception as exc:
            ctree = {"error": f"{type(exc).__name__}: {exc}"}

    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
                "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8 bases -> u32 counts -> f64 frequencies/entropy/JSD", "data": "synthetic",
                "config": workload_config(a, world), "roofline": roofline, "cpu_baseline": base, "e2e": e2e,
                "gpu_launches": int(launches), "clocks": clocks,
                "extra": {"gpu_launches_per_step": int(launches) // max(a.steps, 1),
                          "count_kernel_gbp_per_s": bases / (kc_ms * 1e-3) / 1e9, "count_kernel_ms": kc_ms,
                          "freq_entropy_ms": float(np.mean(fe_ms)), "nmost_wall_s": float(np.mean(sel_ms)) * 1e-3,
                          "nmost_accepts": accepts, "total_gbp": total_bases / 1e9,
                          "selected_head": idx[:8].tolist(), "total_jsd": float(stats[0]),
                          "host_wall_ms_last_step": phase.get("host_wall_ms"),
                          "count_region_ms": phase.get("count_region_ms"), "trail_accepts": phase.get("trail_accepts"),
                          "ctree": ctree}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    raise SystemExit(main())
