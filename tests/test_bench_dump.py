"""bench.py --dump-outputs: a small run writes what its last timed step returned (the nmost selection, every
entropy and validity flag, a seeded sample of the frequency rows) as float64 .npy files, equal to the oracle's."""
import json
import pathlib
import subprocess
import sys

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = pathlib.Path(__file__).resolve().parent.parent
NAMES = {"selected_indices", "delta_jsd", "selection_stats", "entropies", "valid", "freqs_sample",
         "freqs_sample_rows", "freqs_sample_cols"}


@pytest.mark.timeout(300)  # a fresh process: torch and the CUDA context start again
def test_bench_dump_outputs_equal_the_oracle(tmp_path):
    import bench
    from diverseseq_b200 import _lib
    from oracle import oracle as orc

    nrec, nfam, mean_len, k, n = 128, 64, 30_000, 6, 16  # the set still changes after it first fills
    out = tmp_path / "dump"
    cmd = [sys.executable, str(ROOT / "bench.py"), "--steps", "2", "--warmup", "1", "--nrec", str(nrec),
           "--nfam", str(nfam), "--mean-len", str(mean_len), "--k", str(k), "--n", str(n),
           "--no-e2e", "--no-cpu-baseline", "--no-ctree", "--dump-outputs", str(out)]
    r = subprocess.run(cmd, capture_output=True, text=True, timeout=280)
    assert r.returncode == 0, r.stderr[-4000:]
    line = json.loads(r.stdout.strip().splitlines()[-1])
    assert line["steps"] == 2 and line["config"]["nrec_per_gpu"] == nrec

    paths = list(out.glob("*.npy"))
    assert {p.stem for p in paths} == NAMES
    assert sum(p.stat().st_size for p in paths) <= 64 << 20
    got = {p.stem: np.load(p) for p in paths}
    assert all(a.dtype == np.float64 for a in got.values())

    flat, off = _lib.synth_host(bench.SEED, nrec, nfam, mean_len)
    _, freqs, ent, valid = orc.count_batch(flat, off, k, want_counts=False)
    order = np.random.default_rng(bench.SEED).permutation(nrec)
    exp = orc.select_rows(freqs, ent, order, "nmost", n, valid=valid)
    assert got["selected_indices"].tolist() == exp.ids.tolist()
    assert np.array_equal(got["delta_jsd"], exp.delta_jsd)
    assert got["selection_stats"][0] == exp.total_jsd
    assert np.array_equal(got["entropies"], ent) and np.array_equal(got["valid"], valid)
    rows, cols = got["freqs_sample_rows"].astype(np.int64), got["freqs_sample_cols"].astype(np.int64)
    assert rows.size == nrec and cols.size == 4 ** k  # small enough to be dumped whole
    assert np.array_equal(got["freqs_sample"], freqs[np.ix_(rows, cols)])
