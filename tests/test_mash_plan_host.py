"""The host model of tests/mash_plan.py, without a GPU: `window_hashes` is the reference's hash_kmer on every valid
window, its bottom-s distinct set is the oracle's sketch for the inputs that drive the retry passes, and `plan`
reports for each of those inputs the branch of `dvs_mash_sketch` that tests/test_gpu_mash_paths.py names it for."""
import numpy as np
import pytest

from mash_plan import (ALL, KSORT_REC_MAX, bottom_s, overflow_record, plan_seqs, random_record, widen_record,
                       window_hashes)


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("k", [1, 5, 12, 15, 16])
def test_window_hashes_equal_hash_kmer(orc, k, canonical):
    rng = np.random.default_rng(100 + k)
    seq = rng.integers(0, 4, size=3000, dtype=np.uint8)
    seq[rng.random(seq.size) < 0.01] = 4
    # palindromic k-mers (k-mer == its reverse complement; only for even k): ties keep the k-mer
    for at in range(100, 2900, 300):
        if k % 2 == 0:
            half = rng.integers(0, 4, size=k // 2, dtype=np.uint8)
            seq[at:at + k] = np.concatenate([half, (half[::-1] + 2) % 4])
    got = window_hashes(seq, k, canonical)
    starts = [i for i in range(seq.size - k + 1) if (seq[i:i + k] < 4).all()]
    exp = np.array([orc.hash_kmer(seq[i:i + k], canonical) for i in starts], dtype=np.uint32)
    assert np.array_equal(got, exp)
    if k % 2 == 0:
        pal = seq[100:100 + k]
        assert np.array_equal(orc.reverse_complement(pal), pal)
    assert window_hashes(seq[:k - 1], k, canonical).size == 0


RETRY_INPUTS = {
    "widen": lambda: (widen_record(1, 12, 64, False), False),
    "widen_canonical": lambda: (widen_record(5, 12, 64, True), True),
    "overflow_global": lambda: (overflow_record(2, 12, 64, False), False),
    "overflow_record": lambda: (overflow_record(3, 12, 64, True, n_repeat=100_000), True),
}


@pytest.mark.parametrize("name", sorted(RETRY_INPUTS))
def test_bottom_s_equals_oracle_sketch(orc, name):
    seq, canonical = RETRY_INPUTS[name]()
    exp = orc.mash_sketch(seq, 12, 64, canonical=canonical)
    assert np.array_equal(bottom_s(window_hashes(seq, 12, canonical), 64), exp)


def test_plan_widen_ends_in_global_sort():
    for name in ("widen", "widen_canonical"):
        seq, canonical = RETRY_INPUTS[name]()
        passes = plan_seqs([seq], 12, 64, canonical)
        assert passes[0].counts == [0] and passes[0].widened == [0]
        assert passes[-1].thresh == [ALL] and passes[-1].sort == "global" and passes[-1].counts[0] > KSORT_REC_MAX
        assert sum(1 for p in passes if p.widened) >= 3
        assert np.unique(window_hashes(seq, 12, canonical)).size < 64


def test_plan_overflow_redo_both_sort_paths():
    seq, canonical = RETRY_INPUTS["overflow_global"]()
    p = plan_seqs([seq], 12, 64, canonical)
    assert [q.overflow for q in p] == [True, False] and p[0].thresh == [3_436_021] and p[0].cap == [2304]
    assert p[1].sort == "global" and p[1].counts[0] > KSORT_REC_MAX and not p[1].widened
    seq, canonical = RETRY_INPUTS["overflow_record"]()
    p = plan_seqs([seq], 12, 64, canonical)
    assert [q.overflow for q in p] == [True, False] and p[1].sort == "record" and p[1].counts[0] > p[0].cap[0]


def test_plan_mixed_call_shrinks_the_active_set():
    rng = np.random.default_rng(9)
    seqs = [random_record(rng, 50_000), RETRY_INPUTS["widen"]()[0], random_record(rng, 3000),
            RETRY_INPUTS["overflow_record"]()[0][:300_000], np.zeros(0, np.uint8), random_record(rng, 700_000)]
    p = plan_seqs(seqs, 12, 64, False)
    assert p[0].active == [0, 1, 2, 3, 5] and p[0].overflow
    assert p[1].sort == "record" and p[1].widened == [1]
    assert p[-1].active == [1] and p[-1].sort == "global"


def test_plan_large_sketch_sizes_reach_global_steps():
    rng = np.random.default_rng(4)
    p = plan_seqs([random_record(rng, n) for n in (1_000_000, 900_000, 1_100_000)], 12, 20_000, False)
    assert len(p) == 1 and p[0].sort == "global" and p[0].npad >= 1 << 17
    p = plan_seqs([random_record(rng, n) for n in (100_000, 90_000, 110_000)], 12, 4_000_000_000, False)
    assert len(p) == 1 and p[0].sort == "global" and p[0].thresh == [ALL] * 3 and p[0].npad >= 1 << 17
