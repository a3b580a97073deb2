"""nmost / max from sparse k-mer rows held on the device (dvs_select_sparse, 10 <= k <= 12).

The selection runs the host-driven rounds of dvs_select with every row element staged from the sparse rows, so the
selected rows, their order, delta_jsd and the statistics must be the dense path's bit for bit - with the bounded-error
kernels and with DVS_SELECT_EXACT_ONLY=1 - and the oracle's where the oracle's dense rows fit the host."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

MODES = [("nmost", 5, 5), ("nmost", 10, 10), ("stdev", 5, 12), ("cov", 5, 12)]


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


def mode_id(lib, mode):
    return {"nmost": lib.MODE_NMOST, "stdev": lib.MODE_MAX_STDEV, "cov": lib.MODE_MAX_COV}[mode]


def exact_evals(ctx):
    return int(ctx._lib.dvs_select_last_exact_evals(ctx.handle))


def both(lib, ctx, kf, sp, order, mode, lo, hi, monkeypatch, exact):
    """(dense, sparse) results of one selection, with or without the bounded-error kernels"""
    monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "1" if exact else "0")
    m = mode_id(lib, mode)
    return kf.select(order, m, lo, hi), sp.select(order, m, lo, hi)


def assert_same(a, b):
    assert a[0].tolist() == b[0].tolist()
    assert np.array_equal(a[1].view(np.uint64), b[1].view(np.uint64))  # bitwise, NaN and -0.0 included
    assert np.array_equal(a[2].view(np.uint64), b[2].view(np.uint64))


@pytest.fixture(scope="module")
def brca1_rows(lib, ctx, brca1):
    """brca1 (55 records) counted dense and sparse at k = 10, 11, 12 (dense k = 12 rows: 11 GB)"""
    flat, off = lib.concat(list(brca1.values()))
    ss = lib.SeqSet.upload(ctx, flat, off)
    order = np.random.default_rng(55).permutation(len(brca1)).astype(np.uint32)
    cache = {}

    def get(k):
        if k not in cache:
            cache.clear()  # one k at a time on the device
            cache[k] = (lib.KFreqs.count(ctx, ss, k), lib.KSparse.count(ctx, ss, k, want_entropy=True))
        return cache[k]
    return get, order, flat, off


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact_only"])
@pytest.mark.parametrize("mode,lo,hi", MODES)
@pytest.mark.parametrize("k", [10, 11, 12])
def test_brca1_bit_identical_to_dense(lib, ctx, brca1_rows, monkeypatch, k, mode, lo, hi, exact):
    get, order, _, _ = brca1_rows
    kf, sp = get(k)
    d, s = both(lib, ctx, kf, sp, order, mode, lo, hi, monkeypatch, exact)
    assert_same(d, s)
    assert lo <= s[0].size <= hi


def test_brca1_k10_matches_oracle(lib, ctx, orc, brca1_rows):
    get, order, flat, off = brca1_rows
    _, sp = get(10)
    for mode, lo, hi in MODES:
        exp = orc.select_seqs(flat, off, order, 10, mode, lo, hi)
        idx, delta, stats = sp.select(order, mode_id(lib, mode), lo, hi)
        assert idx.tolist() == exp.ids.tolist() and np.array_equal(delta, exp.delta_jsd)
        assert stats[0] == exp.total_jsd and stats[1] == exp.mean_delta_jsd and stats[2] == exp.std_delta_jsd


def test_k12_matches_oracle(lib, ctx, orc, brca1):
    """16 records at k = 12 (the oracle's dense rows: 134 MB each on the host)"""
    names = sorted(brca1)[:16]
    flat, off = lib.concat([brca1[n] for n in names])
    sp = lib.KSparse.count(ctx, lib.SeqSet.upload(ctx, flat, off), 12, want_entropy=True)
    order = np.random.default_rng(16).permutation(16).astype(np.uint32)
    for mode, lo, hi in (("nmost", 5, 5), ("stdev", 4, 8)):
        exp = orc.select_seqs(flat, off, order, 12, mode, lo, hi)
        idx, delta, stats = sp.select(order, mode_id(lib, mode), lo, hi)
        assert idx.tolist() == exp.ids.tolist() and np.array_equal(delta, exp.delta_jsd)
        assert stats[0] == exp.total_jsd and stats[2] == exp.std_delta_jsd


def near_tie_set(rng):
    """exact copies and proportional rows (a record and its doubling count nearly the same k-mers in proportion):
    leave-one-out values tie or nearly tie, so the bounded-error kernels cannot decide and hand over"""
    base = [rng.integers(0, 4, size=int(rng.integers(2000, 4000)), dtype=np.uint8) for _ in range(10)]
    seqs = []
    for i, b in enumerate(base):
        seqs += [b, b.copy(), np.concatenate([b, b])] if i % 2 == 0 else [b]
    return [seqs[i] for i in rng.permutation(len(seqs))]


@pytest.mark.parametrize("mode,lo,hi", [("nmost", 6, 6), ("stdev", 4, 10), ("cov", 4, 10)])
def test_exact_fallback_is_exercised(lib, ctx, monkeypatch, mode, lo, hi):
    seqs = near_tie_set(np.random.default_rng(7))
    flat, off = lib.concat(seqs)
    ss = lib.SeqSet.upload(ctx, flat, off)
    kf, sp = lib.KFreqs.count(ctx, ss, 10), lib.KSparse.count(ctx, ss, 10, want_entropy=True)
    order = np.arange(len(seqs), dtype=np.uint32)
    d_fast, s_fast = both(lib, ctx, kf, sp, order, mode, lo, hi, monkeypatch, exact=False)
    evals = exact_evals(ctx)
    d_ex, s_ex = both(lib, ctx, kf, sp, order, mode, lo, hi, monkeypatch, exact=True)
    assert evals > 0
    assert_same(s_fast, s_ex)
    assert_same(s_fast, d_fast)
    assert_same(s_ex, d_ex)


def edge_set(rng):
    """records without a valid k-mer, shorter than k, with invalid runs, homopolymers (one entry, huge count) and
    rows whose entries all fall in one bucket, among ordinary ones"""
    seqs = [rng.integers(0, 4, size=int(rng.integers(3000, 9000)), dtype=np.uint8) for _ in range(24)]
    seqs[3] = np.full(500, 4, dtype=np.uint8)                                   # no valid k-mer
    seqs[5] = rng.integers(0, 4, size=7, dtype=np.uint8)                        # shorter than k
    seqs[8][100:2000] = 4                                                       # a long invalid run
    seqs[8][2500:2510] = 5
    seqs[11] = np.zeros(200_000, dtype=np.uint8)                               # homopolymer: index 0 only
    seqs[13] = np.full(50_000, 3, dtype=np.uint8)                              # homopolymer: the last index
    seqs[16] = np.concatenate([np.zeros(60, dtype=np.uint8), rng.integers(0, 4, size=4, dtype=np.uint8)])  # bucket 0
    seqs[19] = np.zeros(0, dtype=np.uint8)                                      # empty
    seqs[21] = np.tile(np.array([0, 1], dtype=np.uint8), 3000)                  # two k-mers
    return seqs


@pytest.mark.parametrize("exact", [False, True], ids=["fast", "exact_only"])
@pytest.mark.parametrize("mode,lo,hi", [("nmost", 6, 6), ("stdev", 4, 12), ("cov", 3, 9)])
def test_edge_records(lib, ctx, monkeypatch, mode, lo, hi, exact):
    seqs = edge_set(np.random.default_rng(11))
    flat, off = lib.concat(seqs)
    ss = lib.SeqSet.upload(ctx, flat, off)
    kf, sp = lib.KFreqs.count(ctx, ss, 10), lib.KSparse.count(ctx, ss, 10, want_entropy=True)
    for seed in (0, 1):
        order = np.random.default_rng(seed).permutation(len(seqs)).astype(np.uint32)
        d, s = both(lib, ctx, kf, sp, order, mode, lo, hi, monkeypatch, exact)
        assert_same(d, s)
        assert not set(s[0].tolist()) & {3, 5, 19}  # records without valid k-mers are skipped silently


def test_error_texts(lib, ctx, brca1):
    flat, off = lib.concat(list(brca1.values())[:8])
    ss = lib.SeqSet.upload(ctx, flat, off)
    kf, sp = lib.KFreqs.count(ctx, ss, 10), lib.KSparse.count(ctx, ss, 10, want_entropy=True)
    order = np.arange(8, dtype=np.uint32)
    with pytest.raises(ValueError) as dense_err:
        kf.select(order, lib.MODE_NMOST, 9)
    with pytest.raises(ValueError) as sparse_err:
        sp.select(order, lib.MODE_NMOST, 9)
    assert str(sparse_err.value) == str(dense_err.value) == "The number of sequences 8 is < n 9"
    no_ent = lib.KSparse.count(ctx, ss, 10)
    with pytest.raises(TypeError, match="counted without entropies"):
        no_ent.select(order, lib.MODE_NMOST, 4)


def gene_store(lib, nrec, seed):
    from diverseseq_b200 import _dvs
    flat, off = lib.synth_host(seed, nrec, 40, 1500)
    store = _dvs.make_zarr_store()
    names = [f"g{i:05d}" for i in range(nrec)]
    for i, nm in enumerate(names):
        store.write(nm, flat[int(off[i]):int(off[i + 1])].tobytes())
    return store, names, flat, off


def test_thousand_genes_at_k12(lib, ctx, monkeypatch):
    """1,000 records of ~1.5 kbp at k = 12: dense rows would take 201 GB, the sparse ones 12 MB"""
    from diverseseq_b200 import _dvs
    store, names, flat, off = gene_store(lib, 1000, 1500)
    with pytest.raises((RuntimeError, TypeError, ValueError)):
        lib.KFreqs.count(ctx, lib.SeqSet.upload(ctx, flat, off), 12)
    monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "0")
    fast = _dvs.nmost_divergent(store, 8, 12, seqids=names)
    monkeypatch.setenv("DVS_SELECT_EXACT_ONLY", "1")
    exact = _dvs.nmost_divergent(store, 8, 12, seqids=names)
    assert fast.record_names == exact.record_names and fast.total_jsd == exact.total_jsd
    assert [r[2] for r in fast.records] == [r[2] for r in exact.records]
    sp = lib.KSparse.count(ctx, lib.SeqSet.upload(ctx, flat, off), 12, want_entropy=True)
    rows = sp.dense_rows([names.index(n) for n in fast.record_names])
    for i, (_, row, _) in enumerate(fast.records):
        assert isinstance(row, np.ndarray) and row.dtype == np.float64 and row.size == 4 ** 12
        assert np.array_equal(row, rows[i])
        assert abs(row.sum() - 1.0) < 1e-9


def test_public_surface_k12_matches_dense_route(lib, ctx, brca1, monkeypatch):
    """_dvs.nmost_divergent / max_divergent and records.select_nmost --include at k = 12 from an in-memory store:
    the sparse route against the dense one (forced through the predicate)"""
    from diverseseq_b200 import _dvs, records
    store = _dvs.make_zarr_store()
    for nm, s in brca1.items():
        store.write(nm, s.tobytes())
    seqids = records.shuffled_seqids(store.get_seqids(), 3)
    calls = [
        lambda: _dvs.nmost_divergent(store, 4, 12, seqids=seqids),
        lambda: _dvs.max_divergent(store, 3, 6, 12, seqids=seqids, stat="cov"),
        lambda: records.select_nmost(store, 3, 12, seed=3, include=["Human"]),
    ]
    sparse = [c() for c in calls]
    monkeypatch.setattr(_dvs, "counts_sparse_for_selection", lambda k, ns: False)
    dense = [c() for c in calls]
    for a, b in zip(sparse, dense):
        assert a.record_names == b.record_names and a.size == b.size
        assert [r[2] for r in a.records] == [r[2] for r in b.records]
        assert (a.total_jsd, a.mean_delta_jsd, a.std_delta_jsd, a.cov_delta_jsd) == \
            (b.total_jsd, b.mean_delta_jsd, b.std_delta_jsd, b.cov_delta_jsd)
        for ra, rb in zip(a.records, b.records):
            assert isinstance(ra[1], np.ndarray) and isinstance(rb[1], list)
            assert np.array_equal(ra[1], np.asarray(rb[1]))
