"""GPU parity tests: the CUDA path (through the C ABI) against the CPU oracle.

Bar (BASELINE.json north_star): k-mer counts, sketches, mash intersections and selected
sets/orders bit-exact; entropies / JSD / distances within 1e-9 relative.  The CUDA path
replays the reference's f64 operation order (DESIGN.md §exactness), so most f64 results
are asserted bit-identical, which is stronger than the stated tolerance.
"""
import numpy as np
import pytest

from conftest import random_seqs

pytestmark = pytest.mark.gpu

RTOL = 1e-9  # stated tolerance for floating point results


@pytest.fixture(scope="module")
def lib():
    from diverseseq_b200 import _lib
    return _lib


@pytest.fixture(scope="module")
def ctx(lib):
    return lib.Context(0)


@pytest.fixture(scope="module")
def orc():
    from oracle import oracle
    return oracle


# ------------------------------------------------------------------ log2 / entropy ----

def test_log2_device_bit_identical_to_libm(lib, ctx, orc):
    xs, ys = orc.log2_samples(20261017, 2_000_000)
    got = lib.debug_log2(ctx, xs)
    same = (got.view(np.uint64) == ys.view(np.uint64)) | (np.isnan(got) & np.isnan(ys))
    assert same.all(), f"first mismatch at x={xs[~same][0]!r}"


def test_fast_terms_division_and_table_log2_are_bit_exact(lib, ctx, orc):
    """building blocks of the SM-replicated selection rounds: the reciprocal + fused-remainder division
    must equal IEEE division and the table path of the log2 restatement must equal libm wherever it
    applies; everything else must be flagged"""
    rng = np.random.default_rng(2026)
    n = 1_500_000
    b = rng.integers(1, 4100, n).astype(np.float64)
    a = np.empty(n)
    third = n // 3
    a[:third] = rng.integers(0, 200_000, third) / rng.integers(1, 5_000_000, third)      # frequency-like
    a[third:2 * third] = np.ldexp(rng.random(third) + 1.0, rng.integers(-200, 12, third))  # any mantissa / exponent
    a[2 * third:] = b[2 * third:] * (1.0 + (rng.random(n - 2 * third) - 0.5) * 0.12)        # quotients around 1
    a[::97] = 0.0
    a[1::1013] *= -1.0
    m, lg, sp = lib.debug_fast_terms(ctx, a, b)
    ref_m = a / b
    nz = a != 0
    assert np.array_equal(m[nz].view(np.uint64), ref_m[nz].view(np.uint64)) and (m[~nz] == 0).all()
    near1 = (ref_m >= float.fromhex("0x1.ea4afp-1")) & (ref_m < float.fromhex("0x1.0b559p+0"))
    expect_sp = near1 | ~(ref_m > 0) | (ref_m < 2.2250738585072014e-308)
    assert np.array_equal(sp != 0, expect_sp)
    ok = ~expect_sp
    assert ok.sum() > n // 2
    ref_l = lib.debug_log2(ctx, ref_m[ok])  # = libm bit for bit (test_log2_device_bit_identical_to_libm)
    assert np.array_equal(lg[ok].view(np.uint64), ref_l.view(np.uint64))
    xs, ys = orc.log2_samples(7, 200_000)
    m2, lg2, sp2 = lib.debug_fast_terms(ctx, xs, np.ones_like(xs))
    good = sp2 == 0
    assert good.sum() > 50_000 and np.array_equal(lg2[good].view(np.uint64), ys[good].view(np.uint64))


@pytest.mark.parametrize("dim", [1, 2, 4, 5, 63, 64, 511, 512, 513, 1024, 4096, 5000])
def test_entropy_device_matches_reference_order(lib, ctx, orc, dim):
    rng = np.random.default_rng(dim)
    rows = rng.random((7, dim))
    rows[rng.random((7, dim)) < 0.3] = 0.0
    rows[:, 0] += 1e-3
    rows /= rows.sum(axis=1, keepdims=True)
    got, err = lib.debug_entropy(ctx, rows)
    for r in range(7):
        try:
            exp = orc.entropy(rows[r])
            assert err[r] == 0
            assert got[r] == exp  # bitwise
        except ValueError:
            assert err[r] == 1


def test_entropy_panic_cases(lib, ctx):
    rows = np.array([[0.0, 0.0, 0.0, 0.0], [0.9, 0.9, 0.0, 0.0], [1.9, 0.0, 0.0, 0.0], [0.25, 0.25, 0.25, 0.25]])
    got, err = lib.debug_entropy(ctx, rows)  # record.rs:284-292
    assert err.tolist() == [1, 1, 1, 0] and got[3] == 2.0


# ------------------------------------------------------------------------ counting ----

def _check_counts(lib, ctx, orc, seqs, k, ns=4):
    flat, off = lib.concat(seqs)
    kf = lib.KFreqs.count(ctx, lib.SeqSet.upload(ctx, flat, off), k, ns)
    c, f, e, v = kf.download()
    oc, of, oe, ov = orc.count_batch(flat, off, k, ns)
    assert np.array_equal(c, oc)
    assert np.array_equal(v, ov)
    ok = ov.astype(bool)
    assert np.array_equal(f[ok], of[ok]) and np.array_equal(e[ok], oe[ok])  # bit-identical
    assert np.isnan(f[~ok]).all()  # LazySeq.get_kfreqs yields 0/0 (record.rs:256-261)
    return c


def test_count_reference_kat(lib, ctx, orc):
    seq = np.array([2, 5, 1, 5, 0, 0, 2, 1, 0, 0, 3, 0, 0, 3, 1, 0, 2, 1, 1, 5, 1], dtype=np.uint8)
    c = _check_counts(lib, ctx, orc, [seq], 2)  # record.rs:306-314
    assert c[0].tolist() == [3, 0, 2, 2, 2, 1, 0, 0, 0, 2, 0, 0, 1, 1, 0, 0]


@pytest.mark.parametrize("k", [1, 2, 3, 5, 6, 7, 8, 9, 10])
def test_count_brca1(lib, ctx, orc, brca1, k):
    _check_counts(lib, ctx, orc, list(brca1.values()), k)


@pytest.mark.parametrize("k", [1, 2, 4, 6, 8, 11])
def test_count_ragged_with_invalid_and_edges(lib, ctx, orc, k):
    rng = np.random.default_rng(100 + k)
    seqs = random_seqs(rng, 40, 1, 3000, invalid_rate=0.02)
    seqs += [np.zeros(0, dtype=np.uint8), np.array([4, 4, 4], dtype=np.uint8), np.array([1], dtype=np.uint8),
             np.full(k - 1, 2, dtype=np.uint8), np.full(k, 3, dtype=np.uint8), np.full(5000, 0, dtype=np.uint8),
             rng.integers(4, 255, size=700, dtype=np.uint8)]
    rng.shuffle(seqs)
    _check_counts(lib, ctx, orc, seqs, k)


def test_count_long_records_split_across_ctas(lib, ctx, orc):
    rng = np.random.default_rng(5)
    seqs = [rng.integers(0, 4, size=n, dtype=np.uint8) for n in (3_000_001, 1_234_567, 17)]
    seqs[0][rng.integers(0, 3_000_001, size=300)] = 4
    _check_counts(lib, ctx, orc, seqs, 6)
    _check_counts(lib, ctx, orc, seqs, 8)


@pytest.mark.parametrize("k", [4, 5, 6])
def test_count_s3_16bit_overflow_retry(lib, ctx, orc, k, monkeypatch):
    """(k+2)-mers at every third position with 16-bit packed counters: homopolymers / period-3 repeats
    push one half past 65,535, which must be detected and the item recounted exactly"""
    monkeypatch.setenv("DVS_COUNT_S3", "1")
    rng = np.random.default_rng(40 + k)
    poly = np.zeros(400_000, dtype=np.uint8)                       # one (k+2)-mer 133k times
    rep3 = np.tile(np.array([0, 1, 2], dtype=np.uint8), 150_000)  # period 3: the same (k+2)-mer at every p
    mixed = rng.integers(0, 4, size=500_000, dtype=np.uint8)
    mixed[100_000:330_000] = 3                                     # overflow inside an otherwise random record
    mixed[rng.integers(0, 500_000, size=50)] = 4
    edge = np.full(3 * 65_536 + 7, 2, dtype=np.uint8)              # just at / over the limit
    seqs = [poly, rep3, mixed, edge, rng.integers(0, 4, size=70_000, dtype=np.uint8)]
    _check_counts(lib, ctx, orc, seqs, k)


@pytest.mark.parametrize("k", [4, 6])
def test_count_s3_phase_and_record_end_cases(lib, ctx, orc, k, monkeypatch):
    """record lengths / starts in every residue mod 3 and mod 16, ends on block boundaries, invalid bytes
    next to triplet boundaries"""
    monkeypatch.setenv("DVS_COUNT_S3", "1")
    rng = np.random.default_rng(50 + k)
    seqs = []
    for n in list(range(0, 70)) + [95, 96, 97, 111, 112, 113, 127, 128, 129, 511, 512, 513, 1023, 1024, 1025, 8191,
                                   8192, 8193, 16384, 16385, 16386, 65535, 65536, 65537]:
        s = rng.integers(0, 4, size=n, dtype=np.uint8)
        if n > 40:
            s[rng.integers(0, n, size=max(1, n // 200))] = 4
        seqs.append(s)
    _check_counts(lib, ctx, orc, seqs, k)
    # the same records in another order shift every start by a different amount
    rng.shuffle(seqs)
    _check_counts(lib, ctx, orc, seqs, k)
    clean = [rng.integers(0, 4, size=n, dtype=np.uint8) for n in (48, 49, 50, 160, 161, 162, 4096, 4097, 4098)]
    _check_counts(lib, ctx, orc, clean, k)


@pytest.mark.parametrize("k", [5, 6])
def test_count_s3_kernel_general_records(lib, ctx, orc, k, monkeypatch):
    """DVS_COUNT_S3=1: the opt-in (k+2)-mer / 16-bit kernel on ragged records with invalid bytes"""
    monkeypatch.setenv("DVS_COUNT_S3", "1")
    rng = np.random.default_rng(60 + k)
    seqs = [rng.integers(0, 5, size=int(n), dtype=np.uint8) for n in rng.integers(0, 30_000, size=20)]
    seqs.append(rng.integers(0, 4, size=1_500_000, dtype=np.uint8))
    _check_counts(lib, ctx, orc, seqs, k)


def test_count_k12_global_atomic_path(lib, ctx, orc, brca1):
    """north-star headline k: 4^12 bins per record, global RED.ADD path"""
    seqs = [brca1["Human"], brca1["Dugong"], np.zeros(5, np.uint8)]
    _check_counts(lib, ctx, orc, seqs, 12)


@pytest.mark.parametrize("ns,k", [(5, 3), (20, 2), (2, 7), (3, 1)])
def test_count_other_num_states(lib, ctx, orc, ns, k):
    rng = np.random.default_rng(ns * 31 + k)
    seqs = [rng.integers(0, ns + 2, size=int(n), dtype=np.uint8) for n in rng.integers(0, 2000, size=12)]
    _check_counts(lib, ctx, orc, seqs, k, ns)


def test_count_errors(lib, ctx):
    s = lib.SeqSet.from_seqs(ctx, [np.array([0, 1, 2, 3], dtype=np.uint8)])
    with pytest.raises(ValueError, match="k cannot be 0"):
        lib.KFreqs.count(ctx, s, 0)
    with pytest.raises(TypeError):
        lib.KFreqs.count(ctx, s, 17)


def test_synth_device_equals_host(lib, ctx):
    dev = lib.SeqSet.synth(ctx, 20261017, 64, 5, 40_000)
    flat, off = lib.synth_host(20261017, 64, 5, 40_000)
    assert np.array_equal(dev.offsets(), off)
    assert np.array_equal(dev.download(), flat)
    part, poff = lib.synth_host(20261017, 64, 5, 40_000, first=10, count=7)
    assert np.array_equal(part, flat[int(off[10]):int(off[17])])
    assert (flat == 4).sum() > 0 and (flat > 4).sum() == 0


# ----------------------------------------------------------------------- selection ----

def _check_select(lib, ctx, orc, seqs, k, order, mode, lo, hi=0):
    flat, off = lib.concat(seqs)
    kf = lib.KFreqs.count(ctx, lib.SeqSet.upload(ctx, flat, off), k)
    _, of, oe, ov = orc.count_batch(flat, off, k)
    omode = {lib.MODE_NMOST: "nmost", lib.MODE_MAX_STDEV: "stdev", lib.MODE_MAX_COV: "cov"}[mode]
    exp = orc.select_rows(of, oe, order, omode, lo, hi, valid=ov)
    idx, delta, stats = kf.select(order, mode, lo, hi)
    assert idx.tolist() == exp.ids.tolist()  # same set AND same Vec order
    assert np.array_equal(delta, exp.delta_jsd)  # bitwise
    assert stats[0] == exp.total_jsd and stats[4] == exp.summed_entropies
    np.testing.assert_allclose(stats[1:4], [exp.mean_delta_jsd, exp.std_delta_jsd, exp.cov_delta_jsd], rtol=RTOL)
    assert stats[1] == exp.mean_delta_jsd and stats[2] == exp.std_delta_jsd
    return exp


@pytest.mark.parametrize("k,n", [(6, 10), (1, 3), (3, 5), (8, 4)])
def test_nmost_brca1(lib, ctx, orc, brca1, k, n):  # BASELINE config 1: brca1 -> nmost -n 10 -k 6
    seqs = list(brca1.values())
    for seed in (1, 2, 3):
        order = np.random.default_rng(seed).permutation(len(seqs)).astype(np.uint32)
        exp = _check_select(lib, ctx, orc, seqs, k, order, lib.MODE_NMOST, n)
        assert exp.size == n


@pytest.mark.parametrize("mode", ["stdev", "cov"])
@pytest.mark.parametrize("k", [2, 5])
def test_max_brca1(lib, ctx, orc, brca1, mode, k):
    seqs = list(brca1.values())
    m = lib.MODE_MAX_STDEV if mode == "stdev" else lib.MODE_MAX_COV
    for seed, lo, hi in ((1, 3, 12), (2, 5, 5), (3, 2, 100)):
        order = np.random.default_rng(seed).permutation(len(seqs)).astype(np.uint32)
        exp = _check_select(lib, ctx, orc, seqs, k, order, m, lo, hi)
        assert lo <= exp.size <= min(hi, len(seqs))


def test_select_random_families_with_invalid_records(lib, ctx, orc):
    rng = np.random.default_rng(77)
    seqs = random_seqs(rng, 150, 200, 1500, invalid_rate=0.01)
    for i in (0, 3, 50, 149):
        seqs[i] = np.full(30, 4, dtype=np.uint8)  # no valid k-mers -> skipped silently
    order = rng.permutation(150).astype(np.uint32)
    exp = _check_select(lib, ctx, orc, seqs, 4, order, lib.MODE_NMOST, 12)
    assert exp.size == 11 and len(exp.trace) > 5  # one of the first 12 is invalid -> smaller set
    _check_select(lib, ctx, orc, seqs, 4, order, lib.MODE_MAX_STDEV, 6, 20)
    _check_select(lib, ctx, orc, seqs, 4, order[:77], lib.MODE_MAX_COV, 6, 20)


def test_select_duplicates_and_subset_order(lib, ctx, orc):
    rng = np.random.default_rng(9)
    base = random_seqs(rng, 30, 300, 800, invalid_rate=0.0)
    seqs = base + [b.copy() for b in base[:10]]  # identical sequences under different ids -> exact ties
    order = rng.permutation(len(seqs)).astype(np.uint32)
    _check_select(lib, ctx, orc, seqs, 3, order, lib.MODE_NMOST, 7)
    dup_order = np.concatenate([order, order[:15]]).astype(np.uint32)  # same seqid listed twice
    _check_select(lib, ctx, orc, seqs, 3, dup_order, lib.MODE_NMOST, 7)


def test_select_reference_tiny_goldens(lib, ctx, orc):
    z = [[0, 0, 1, 1], [1, 1, 1, 3], [0, 0, 0, 2, 2, 2], [1, 1, 1, 1, 3], [1, 2]]  # records.rs:696-702
    seqs = [np.array(s, dtype=np.uint8) for s in z]
    import itertools
    for perm in itertools.permutations(range(5)):
        _check_select(lib, ctx, orc, seqs, 1, np.array(perm, dtype=np.uint32), lib.MODE_NMOST, 3)
    for perm in list(itertools.permutations(range(5)))[::7]:
        _check_select(lib, ctx, orc, seqs, 1, np.array(perm, dtype=np.uint32), lib.MODE_MAX_STDEV, 3, 4)
        _check_select(lib, ctx, orc, seqs, 1, np.array(perm, dtype=np.uint32), lib.MODE_MAX_COV, 3, 4)


def test_select_fast_path_equals_exact_only(lib, ctx, orc, monkeypatch):
    """the bounded-error fast path must take exactly the decisions of the exact-only loop"""
    flat, off = lib.synth_host(99, 1500, 12, 6000)
    kf = lib.KFreqs.count(ctx, lib.SeqSet.upload(ctx, flat, off), 5)
    order = np.random.default_rng(3).permutation(1500).astype(np.uint32)
    for mode, lo, hi in ((lib.MODE_NMOST, 40, 40), (lib.MODE_MAX_STDEV, 10, 30), (lib.MODE_MAX_COV, 10, 60)):
        monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "1")
        i0, d0, s0 = kf.select(order, mode, lo, hi)
        assert ctx._lib.dvs_select_last_exact_evals(ctx.handle) == 0
        monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "0")
        # host-driven fast rounds, the global-state persistent kernel, the SM-replicated persistent
        # kernel (default)
        for persist in ("0", "1", "2"):
            monkeypatch.setenv("DVS_SELECT_PERSIST", persist)
            i1, d1, s1 = kf.select(order, mode, lo, hi)
            assert i0.tolist() == i1.tolist() and np.array_equal(d0, d1) and np.array_equal(s0, s1)
            assert ctx._lib.dvs_select_last_exact_evals(ctx.handle) <= 5  # decisions are far from ties here
    monkeypatch.delenv("DVS_SELECT_PERSIST")
    # max modes: batched grow attempts (default) against one host-driven attempt per candidate
    for mode, lo, hi in ((lib.MODE_MAX_STDEV, 10, 30), (lib.MODE_MAX_COV, 10, 60), (lib.MODE_MAX_STDEV, 3, 1500)):
        monkeypatch.setenv("DVS_SELECT_GROW_BATCH", "0")
        i0, d0, s0 = kf.select(order, mode, lo, hi)
        monkeypatch.delenv("DVS_SELECT_GROW_BATCH")
        i1, d1, s1 = kf.select(order, mode, lo, hi)
        assert i0.tolist() == i1.tolist() and np.array_equal(d0, d1) and np.array_equal(s0, s1)
    _, of, oe, ov = orc.count_batch(flat, off, 5)
    exp = orc.select_rows(of, oe, order, "nmost", 40, valid=ov)
    i1, d1, s1 = kf.select(order, lib.MODE_NMOST, 40)
    assert i1.tolist() == exp.ids.tolist() and np.array_equal(d1, exp.delta_jsd)


@pytest.mark.parametrize("n", [3, 30, 160])
def test_select_sm_replicated_rounds_k6(lib, ctx, orc, monkeypatch, n):
    """k=6 (4096-element vectors): the SM-replicated kernel splits one candidate over 4 / 2 / 1 CTAs and
    loops member tasks when n + 1 exceeds the grid; decisions must equal the oracle's and the other forms'"""
    flat, off = lib.synth_host(4242 + n, 1300, 9, 20_000)
    kf = lib.KFreqs.count(ctx, lib.SeqSet.upload(ctx, flat, off), 6)
    _, of, oe, ov = orc.count_batch(flat, off, 6)
    order = np.random.default_rng(n).permutation(1300).astype(np.uint32)
    exp = orc.select_rows(of, oe, order, "nmost", n, valid=ov)
    res = {}
    for persist in ("2", "1", "0"):
        monkeypatch.setenv("DVS_SELECT_PERSIST", persist)
        idx, delta, stats = kf.select(order, lib.MODE_NMOST, n)
        res[persist] = (idx.tolist(), delta.tolist(), stats.tolist(), int(ctx._lib.dvs_select_last_accepts(ctx.handle)))
        assert idx.tolist() == exp.ids.tolist() and np.array_equal(delta, exp.delta_jsd)
        assert stats[0] == exp.total_jsd and stats[4] == exp.summed_entropies
    assert res["2"] == res["1"] == res["0"]
    assert res["2"][3] > 5  # the rounds actually accepted candidates
    monkeypatch.setenv("DVS_SELECT_PERSIST", "2")
    m_idx, m_delta, m_stats = kf.select(order, lib.MODE_MAX_COV, 10, 40)
    mexp = orc.select_rows(of, oe, order, "cov", 10, 40, valid=ov)
    assert m_idx.tolist() == mexp.ids.tolist() and np.array_equal(m_delta, mexp.delta_jsd)


def test_select_large_sets_match_oracle(lib, ctx, orc):
    """bigger selections (n well above one warp / one CTA of members) and a long max growth phase"""
    flat, off = lib.synth_host(123, 2500, 20, 3000)
    kf = lib.KFreqs.count(ctx, lib.SeqSet.upload(ctx, flat, off), 4)
    _, of, oe, ov = orc.count_batch(flat, off, 4)
    order = np.random.default_rng(5).permutation(2500).astype(np.uint32)
    for mode, omode, lo, hi in ((lib.MODE_NMOST, "nmost", 700, 700), (lib.MODE_MAX_COV, "cov", 50, 400),
                                (lib.MODE_MAX_STDEV, "stdev", 20, 2500)):
        exp = orc.select_rows(of, oe, order, omode, lo, hi, valid=ov)
        idx, delta, stats = kf.select(order, mode, lo, hi)
        assert idx.tolist() == exp.ids.tolist() and np.array_equal(delta, exp.delta_jsd)
        assert stats[0] == exp.total_jsd and stats[2] == exp.std_delta_jsd


def test_select_errors(lib, ctx):
    seqs = [np.array(s, dtype=np.uint8) for s in ([0, 0, 1, 1], [1, 1, 1, 3], [4, 4], [4])]
    kf = lib.KFreqs.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), 1)
    with pytest.raises(ValueError, match="The number of sequences 4 is < n 20"):  # records.rs:323-325
        kf.select(np.arange(4, dtype=np.uint32), lib.MODE_NMOST, 20)
    with pytest.raises(ValueError, match="must have > 1 KmerSeq"):  # records.rs:227-230
        kf.select(np.array([0, 2, 3, 1], dtype=np.uint32), lib.MODE_NMOST, 3)
    with pytest.raises(ValueError, match="records cannot be empty"):  # records.rs:28-30
        kf.select(np.array([2, 3, 0, 1], dtype=np.uint32), lib.MODE_NMOST, 2)


# ----------------------------------------------------------------- the _dvs surface ----

def _store(dvs, named):
    st = dvs.make_zarr_store()
    for name, arr in named.items():
        st.write(name, arr.tobytes())
    return st


def test_dvs_summed_goldens(orc):  # records.rs:602-621, 676-685 through the drop-in module
    from diverseseq_b200 import _dvs as dvs
    recs = [("seq1", bytes([0, 1, 2, 3])), ("seq2", bytes([0, 1, 2, 2, 3])), ("seq3", bytes([3, 0, 0]))]
    calc = dvs.get_delta_jsd_calculator(recs, k=1, num_states=4)
    r = calc.get_result()
    assert r.size == 3 and r.total_jsd == 0.31174344844038515
    assert [x[2] for x in r.records] == [-0.09602255461972087, -0.013445832597674734, 0.2931216853661194]
    assert r.mean_delta_jsd == 0.061217766049574594 and r.std_delta_jsd == 0.20503487410866827
    assert r.cov_delta_jsd == r.std_delta_jsd / r.mean_delta_jsd
    assert r.records[0][1] == [0.25, 0.25, 0.25, 0.25] and r.record_names == ["seq1", "seq2", "seq3"]
    assert calc.delta_jsd("seq1", bytes([0, 1, 2, 3])) == 0.0  # records.rs:641-645
    better = calc.delta_jsd("seq4", bytes([0, 1, 2, 1]))
    assert better > r.total_jsd and better == orc.Summed([list(b) for _, b in recs], 1).delta_jsd([0, 1, 2, 1])
    with pytest.raises(ValueError, match=r"delta_jsd\('bad'\) failed: No valid k-mers for 'bad'"):
        calc.delta_jsd("bad", bytes([4, 4, 4]))  # records_py.rs:113-118, tests/test_records.py:285-291
    many = calc.delta_jsd_many([("seq4", bytes([0, 1, 2, 1])), ("seq1", bytes([0, 1, 2, 3])), ("q", bytes([3, 3, 1]))])
    assert many[0] == better and many[1] == 0.0 and many[2] == calc.delta_jsd("q", bytes([3, 3, 1]))
    with pytest.raises(ValueError, match="No valid k-mers for 'bad'"):
        calc.delta_jsd_many([("seq4", bytes([0, 1, 2, 1])), ("bad", bytes([4]))])


def test_dvs_nmost_max_pickle_and_errors(brca1, orc):
    import pickle
    from diverseseq_b200 import _dvs as dvs
    st = _store(dvs, {"a": np.array([2, 2, 2, 2], np.uint8), "b": np.array([2, 2, 2, 2], np.uint8),
                      "c": np.array([0, 0, 0, 0], np.uint8), "d": np.array([2, 1, 3, 0], np.uint8)})
    assert st.num_unique() == 3 and len(st) == 4 and "a" in st
    got = dvs.nmost_divergent(st, n=3, k=1)  # tests/test_records.py:73-79
    assert got.size == 3 and set(got.record_names) == set(st.unique_seqids)
    assert pickle.loads(pickle.dumps(got)).size == 3  # :88-98
    assert dvs.max_divergent(st, min_size=2, max_size=2, k=1).size == 2  # :59-63
    with pytest.raises(ValueError):
        dvs.nmost_divergent(st, n=30, k=1)  # :82-85
    with pytest.raises(ValueError):
        dvs.max_divergent(st, min_size=30, max_size=2, k=1)  # :66-70
    # brca1 through the store path == oracle streaming path
    bst = _store(dvs, brca1)
    names = list(brca1)
    order = np.random.default_rng(4).permutation(len(names))
    seqids = [names[i] for i in order]
    got = dvs.nmost_divergent(bst, n=10, k=6, seqids=seqids)
    flat, off = orc.concat(list(brca1.values()))
    exp = orc.select_seqs(flat, off, order, 6, "nmost", 10, want_freqs=True)
    assert got.record_names == [names[i] for i in exp.ids]
    assert [r[2] for r in got.records] == exp.delta_jsd.tolist() and got.total_jsd == exp.total_jsd
    assert np.array_equal(np.array([r[1] for r in got.records]), exp.kfreqs)
    assert (got.k, got.num_states) == (6, 4)
    # merge of per-chunk results (final_nmost), incl. the upstream k/num_states swap (records.rs:353)
    r1 = dvs.nmost_divergent(bst, n=5, k=3, seqids=seqids[:25])
    r2 = dvs.nmost_divergent(bst, n=5, k=3, seqids=seqids[25:])
    merged = dvs.final_nmost([r1, r2], 5)
    rows = np.array([r[1] for r in r1.records + r2.records])
    exp = orc.select_rows(rows, None, np.arange(10), "nmost", 5, recompute_entropy=True)
    all_names = r1.record_names + r2.record_names
    assert merged.record_names == [all_names[i] for i in exp.ids]
    assert [r[2] for r in merged.records] == exp.delta_jsd.tolist()
    assert (merged.k, merged.num_states) == (4, 3)
    fm = dvs.final_max([r1, r2], 3, 8, stat="cov")
    exp = orc.select_rows(rows, None, np.arange(10), "cov", 3, 8, recompute_entropy=True)
    assert fm.record_names == [all_names[i] for i in exp.ids]
    with pytest.raises(ValueError):
        dvs.final_nmost([r1, r2], 50)


def test_dvs_lazyseq(brca1, orc):
    from diverseseq_b200 import _dvs as dvs
    st = _store(dvs, {"Human": brca1["Human"], "junk": np.array([4, 4, 5], np.uint8)})
    lz = st.get_lazyseq("Human", 4)
    assert lz.get_seq() == brca1["Human"].tobytes() and lz.seqid == "Human" and lz.num_states == 4
    assert lz.get_kcounts(3) == orc.kcounts(brca1["Human"], 3).tolist()
    assert lz.get_kfreqs(3) == orc.kfreqs_unchecked(brca1["Human"], 3).tolist()
    assert all(np.isnan(st.get_lazyseq("junk", 4).get_kfreqs(2)))


# ---------------------------------------------------------------------------- mash ----

def _check_sketches(lib, ctx, orc, seqs, k, s, canonical, ns=4):
    flat, off = lib.concat(seqs)
    sk = lib.Sketches.sketch(ctx, lib.SeqSet.upload(ctx, flat, off), k, s, ns, canonical)
    data, lens = sk.download()
    for i, q in enumerate(seqs):
        exp = orc.mash_sketch(q, k, s, ns, canonical)
        assert lens[i] == len(exp), (i, lens[i], len(exp))
        assert np.array_equal(data[i, : lens[i]], exp)
    return sk, data, lens


@pytest.mark.parametrize("canonical", [False, True])
@pytest.mark.parametrize("k,s", [(16, 400), (12, 3000), (5, 50), (1, 10), (16, 4_000_000_000)])
def test_sketch_brca1(lib, ctx, orc, brca1, k, s, canonical):  # tests/test_ctree.py:9-27 uses 400 and 4e9
    _check_sketches(lib, ctx, orc, list(brca1.values())[:12], k, s, canonical)


def test_sketch_edges_and_generic_paths(lib, ctx, orc):
    rng = np.random.default_rng(3)
    seqs = random_seqs(rng, 10, 1, 4000, invalid_rate=0.02)
    seqs += [np.zeros(0, np.uint8), np.array([4, 4], np.uint8), np.full(9000, 1, np.uint8),
             np.tile(np.array([0, 1, 2, 3], np.uint8), 3000)]  # repetitive: few distinct hashes
    _check_sketches(lib, ctx, orc, seqs, 8, 64, True)
    _check_sketches(lib, ctx, orc, seqs, 21, 100, True)     # k > 16 -> generic kernel
    _check_sketches(lib, ctx, orc, seqs, 21, 100, False)
    seqs5 = [rng.integers(0, 7, size=int(n), dtype=np.uint8) for n in (0, 5, 1000, 3000)]
    _check_sketches(lib, ctx, orc, seqs5, 4, 32, False, ns=5)  # num_states != 4 -> generic kernel


def test_sketch_long_record(lib, ctx, orc):
    rng = np.random.default_rng(8)
    seq = rng.integers(0, 4, size=1_500_000, dtype=np.uint8)
    seq[rng.integers(0, seq.size, size=100)] = 4
    _check_sketches(lib, ctx, orc, [seq, seq[:700_000]], 16, 3000, True)


def test_mash_distances(lib, ctx, orc, brca1):
    names = ["Human", "Chimpanzee", "Manatee", "Dugong", "Rhesus"] + list(brca1)[:20]
    seqs = [brca1[n] for n in names]
    for k, s, canonical in ((16, 400, True), (12, 3000, False), (4, 40, False)):
        sk, data, lens = _check_sketches(lib, ctx, orc, seqs, k, s, canonical)
        dist, inter, uni = sk.distances(k, s, want_counts=True)
        od, oi, ou = orc.mash_matrix(data, lens, k, s)
        assert np.array_equal(inter, oi) and np.array_equal(uni, ou)  # integer work: bit-exact
        np.testing.assert_allclose(dist, od, rtol=RTOL, atol=0)
        assert (np.diag(dist) == 0).all() and np.array_equal(dist, dist.T)
        part = sk.distances(k, s, 7, 13)  # row shard == the same rows of the full matrix
        assert np.array_equal(part, dist[7:13])
    from diverseseq_b200 import _dvs as dvs, distance
    assert dvs.mash_sketch(brca1["Human"].tobytes(), 16, 400, 4, True) == \
        orc.mash_sketch(brca1["Human"], 16, 400, canonical=True).tolist()
    d = distance.mash_distance(orc.mash_sketch(brca1["Human"], 16, 400, canonical=True).tolist(),
                               orc.mash_sketch(brca1["Chimpanzee"], 16, 400, canonical=True).tolist(), 16, 400)
    assert abs(d - 0.009634417489203647) <= RTOL * d


def test_mash_distance_empty_sketches(lib, ctx):
    sk = lib.Sketches.from_host(ctx, np.zeros((2, 4), np.uint32), np.array([0, 0], np.uint32))
    with pytest.raises(ZeroDivisionError):
        sk.distances(4, 10)


# ----------------------------------------------------------------------- euclidean ----

@pytest.mark.parametrize("k", [1, 5, 8])
def test_euclidean(lib, ctx, orc, brca1, k):
    seqs = list(brca1.values())
    flat, off = lib.concat(seqs)
    kf = lib.KFreqs.count(ctx, lib.SeqSet.upload(ctx, flat, off), k)
    _, of, _, _ = orc.count_batch(flat, off, k)
    exp = orc.euclid_matrix(of)
    got = kf.euclidean()
    np.testing.assert_allclose(got, exp, rtol=RTOL, atol=0)
    assert (np.diag(got) == 0).all() and np.array_equal(got, got.T)
    assert np.array_equal(kf.euclidean(10, 31), got[10:31])
    assert np.array_equal(kf.euclidean(0, 1), got[0:1])


def test_dvs_on_disk_store_matches_in_memory(tmp_path, brca1, orc):
    """`.dvseqsz` directory store (threaded zstd decode -> pinned staging -> GPU) == in-memory store"""
    from diverseseq_b200 import _dvs as dvs, dvseqsz, _lib
    path = tmp_path / "brca1.dvseqsz"
    disk = dvs.make_zarr_store(str(path), mode="w")
    mem = dvs.make_zarr_store()
    for name, arr in brca1.items():
        disk.write(name, arr.tobytes(), {"source": f"brca1-dataset:{name}"})
        mem.write(name, arr.tobytes())
    names = list(brca1)
    order = np.random.default_rng(8).permutation(len(names))
    seqids = [names[i] for i in order]
    ro = dvs.make_zarr_store(str(path))
    a = dvs.nmost_divergent(ro, n=10, k=6, seqids=seqids)
    b = dvs.nmost_divergent(mem, n=10, k=6, seqids=seqids)
    assert a.record_names == b.record_names and a.records == b.records and a.total_jsd == b.total_jsd
    m = dvs.max_divergent(ro, min_size=5, max_size=12, k=3, seqids=seqids, stat="cov")
    flat, off = orc.concat(list(brca1.values()))
    exp = orc.select_seqs(flat, off, order, 3, "cov", 5, 12)
    assert m.record_names == [names[i] for i in exp.ids] and [r[2] for r in m.records] == exp.delta_jsd.tolist()
    ctx = _lib.default_context()
    ss, offsets = dvseqsz.load_seqset(ctx, ro, names, threads=4)
    assert np.array_equal(ss.download(), flat) and np.array_equal(offsets, off)
    assert ro.get_lazyseq("Human", 4).get_kcounts(2) == orc.kcounts(brca1["Human"], 2).tolist()


def test_packed_upload_reconstructs_bytes_exactly(lib, ctx, monkeypatch):
    """2-bit packed PCIe path (csrc/upload.cu): the device must end up with the caller's bytes, incl.
    arbitrary bytes >= 4 (exceptions), a block with too many of them (raw fallback) and a ragged tail"""
    rng = np.random.default_rng(12)
    monkeypatch.setenv("DVS_UPLOAD_PACKED", "1")
    n = (256 << 20) + (256 << 20) + 1_234_567  # three blocks, the last one short and odd sized
    flat = rng.integers(0, 4, size=n, dtype=np.uint8)
    bad = rng.integers(0, n, size=200_000)
    flat[bad] = rng.integers(4, 256, size=bad.size, dtype=np.uint8)          # sparse exceptions everywhere
    flat[(256 << 20) + 1000:(256 << 20) + 9_000_000] = 78                      # block 1: > 1/64 invalid -> raw
    offsets = np.array([0, 5, 5, 1_000_003, (256 << 20) + 7, n], dtype=np.uint64)
    ss = lib.SeqSet.upload(ctx, flat, offsets)
    got = ss.download()
    assert got.size == n and np.array_equal(got, flat)
    small = rng.integers(0, 6, size=1001, dtype=np.uint8)
    s2 = lib.SeqSet.upload(ctx, small, np.array([0, 1001], dtype=np.uint64))
    assert np.array_equal(s2.download(), small)
    monkeypatch.setenv("DVS_UPLOAD_PACKED", "0")
    s3 = lib.SeqSet.upload(ctx, small, np.array([0, 1001], dtype=np.uint64))
    assert np.array_equal(s3.download(), small)
