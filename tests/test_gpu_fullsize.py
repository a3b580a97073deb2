"""Full-size parity (BASELINE.json configs[1]: 10,500 synthetic genomes x ~4 Mbp, k=6, nmost n=100).

The oracle cannot run on the GPU box in seconds at this size, so it was run once on the CPU
(tests/golden/make_fullsize_golden.py, no GPU involved) and its results are committed as
tests/golden/fullsize_k6_n100.npz: per-record k-mer totals, an order-sensitive 64-bit checksum of every
record's count row, every record's entropy (bit pattern), and the nmost selection (ids in Vec order,
delta_jsd bit patterns, total_jsd, summed entropies).  The device generator is the bit-exact twin of the
host generator (test_synth_device_equals_host), so the CUDA path must reproduce all of it exactly."""
import pathlib

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEED, NREC, NFAM, MEAN_LEN, K, N = 20261017, 10500, 64, 4_000_000, 6, 100
GOLDEN = pathlib.Path(__file__).resolve().parent / "golden" / "fullsize_k6_n100.npz"
MIX = np.uint64(0x9E3779B97F4A7C15)


@pytest.fixture(scope="module")
def full():
    from diverseseq_b200 import _lib

    ctx = _lib.Context(0)
    try:
        ss = _lib.SeqSet.synth(ctx, SEED, NREC, NFAM, MEAN_LEN)  # 42 GB in HBM
    except Exception as exc:  # a smaller GPU than the B200 this is sized for
        pytest.skip(f"cannot hold the full-size set on this device: {exc}")
    kf = _lib.KFreqs.count(ctx, ss, K)
    return _lib, ctx, ss, kf, np.load(GOLDEN)


def test_fullsize_counts_and_entropies_equal_the_oracle(full):
    lib, ctx, ss, kf, g = full
    assert ss.total_bases == 42_046_293_768
    ent = np.zeros(NREC)
    valid = np.zeros(NREC, dtype=np.uint8)
    totals = np.zeros(NREC, dtype=np.uint64)
    sums = np.zeros(NREC, dtype=np.uint64)
    w = np.arange(4 ** K, dtype=np.uint64) * MIX + np.uint64(1)
    step = 1500
    for first in range(0, NREC, step):  # rows in slices: 1500 x 4096 x u64 = 49 MB at a time
        cnt = min(step, NREC - first)
        c, _, e, v = kf.download(first, cnt, freqs=False)
        ent[first:first + cnt], valid[first:first + cnt] = e, v
        totals[first:first + cnt] = c.sum(axis=1, dtype=np.uint64)
        with np.errstate(over="ignore"):
            sums[first:first + cnt] = (c * w).sum(axis=1, dtype=np.uint64)
    assert np.array_equal(valid, g["valid"]) and valid.all()
    assert np.array_equal(totals, g["totals"])                 # every record's number of valid 6-mers
    assert np.array_equal(sums, g["count_checksums"])          # every record's count row (order-sensitive checksum)
    assert np.array_equal(ent.view(np.uint64), g["entropy_bits"])  # every entropy, bit for bit
    off = ss.offsets()
    lens = np.diff(off).astype(np.int64)
    missing = lens - (K - 1) - totals.astype(np.int64)         # windows lost to invalid bytes
    assert (missing >= 0).all() and 0 < missing.sum() < 1e-2 * lens.sum()


def test_fullsize_nmost_equals_the_oracle_in_every_round_form(full, monkeypatch):
    lib, ctx, ss, kf, g = full
    order = np.random.default_rng(SEED).permutation(NREC).astype(np.uint32)
    for persist in ("2", "1", "0"):  # SM-replicated rounds, cooperative grid.sync rounds, host-driven rounds
        monkeypatch.setenv("DVS_SELECT_PERSIST", persist)
        idx, delta, stats = kf.select(order, lib.MODE_NMOST, N)
        assert idx.tolist() == g["ids"].tolist()                                  # same set, same Vec order
        assert np.array_equal(delta.view(np.uint64), g["delta_jsd_bits"])         # bitwise
        assert stats[0] == float(g["total_jsd"]) and stats[4] == float(g["summed_entropies"])
        assert int(ctx._lib.dvs_select_last_accepts(ctx.handle)) == 350
        assert int(ctx._lib.dvs_select_last_exact_evals(ctx.handle)) == 0
