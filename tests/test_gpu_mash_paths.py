"""MinHash sketches and the mash matrix on every path of csrc/mash.cu against the CPU oracle.

Sketches are compared bit for bit (lengths and contents) with `oracle.mash_sketch_batch`:
* every filter kernel (`k_mash_filter16<CANON>`, `k_mash_filter` at k < 16 and at k = 16 through
  DVS_MASH_FILTER16=0, `k_mash_filter_generic` at k > 16 and at num_states = 5) with the per-record sort and with the
  global bitonic network (DVS_MASH_GLOBAL_SORT=1), on a ragged set with records starting at every residue mod 16,
  lengths around k and the 16-byte blocks, invalid bytes on block edges and records spanning the 256 KiB work items;
* the retry passes, driven by the input alone: a repeat that widens its threshold until it is all ones, a repeated
  low-hash k-mer that overflows the candidate buffer, both mixed with ordinary records in one call, and sketch
  sizes whose key buffer takes several global bitonic steps.  Each case first shows through tests/mash_plan.py that
  its input really takes the branch it is named for;
* ctree's default (k = 12, s = 3000) on synthetic genomes of 2-4 Mbp, also through `distance.mash_distances` and
  `dvs_ctree`.
The matrix (`k_mash_pairs`) is checked on host-built sketches over many blocks and row ranges, and the sharded
matrix on three ranks whose sketch strides differ."""
import numpy as np
import pytest

from mash_plan import (ALL, CHUNK, KSORT_REC_MAX, bottom_s, first_thresh_cap, overflow_record, plan_seqs,
                       random_record, widen_record, window_hashes)
from test_gpu_sharded import make_shards, run_ranks

pytestmark = pytest.mark.gpu

RTOL = 1e-9


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


def _threads(orc):
    return max(1, orc.hardware_threads())


def check_sketches(lib, ctx, orc, flat, off, k, s, canonical, ns=4, expected=None):
    """sketch on the GPU, compare with the oracle bit for bit; returns (Sketches, data, lens)"""
    sk = lib.Sketches.sketch(ctx, lib.SeqSet.upload(ctx, flat, off), k, s, ns, canonical)
    data, lens = sk.download()
    o_sk, o_lens = expected if expected is not None else \
        orc.mash_sketch_batch(flat, off, k, s, ns, canonical, threads=_threads(orc))
    assert data.shape == o_sk.shape
    bad = np.flatnonzero(lens != o_lens)
    assert bad.size == 0, f"lengths differ at records {bad[:10].tolist()}: {lens[bad[:10]]} vs {o_lens[bad[:10]]}"
    used = np.arange(data.shape[1])[None, :] < lens[:, None]
    diff = np.flatnonzero((data != o_sk) & used) // max(data.shape[1], 1)
    assert diff.size == 0, f"sketch contents differ at records {np.unique(diff)[:10].tolist()}"
    return sk, data, lens


def _split(flat, off):
    return [flat[int(off[i]):int(off[i + 1])] for i in range(len(off) - 1)]


# --------------------------------------------------------------------- kernel forms x sort paths ----

def ragged_set(k: int, ns: int, seed: int):
    """(flat, offsets): lengths k-1, k, k+1 and around the 16-byte blocks, starts at every residue mod 16, two
    records longer than a work item, invalid bytes inside records and on 16-byte block edges"""
    rng = np.random.default_rng(seed)
    lens = [max(k - 1, 0), k, k + 1, 15, 16, 17, 31, 32, 33, 0, 2 * CHUNK + 75_000 + 3]
    lens += [17] * 16  # each start one byte further mod 16
    lens += [CHUNK + 44_000 + 1, 5000, 2, 1, 64, 2 * k + 1]
    seqs = []
    for n in lens:
        q = rng.integers(0, ns, size=n, dtype=np.uint8)
        q[rng.random(n) < 0.005] = ns + rng.integers(0, 3)
        seqs.append(q)
    flat, off = np.concatenate(seqs), np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    starts = off[:-1][np.diff(off) > 0]
    assert set((starts % 16).tolist()) == set(range(16))
    edges = np.flatnonzero(np.isin(np.arange(flat.size) % 16, (0, 15)))
    flat[rng.choice(edges, size=edges.size // 150, replace=False)] = ns + 1
    return flat, off


# (id, k, num_states, canonical, env)
FORMS = [
    ("filter16", 16, 4, False, {}),
    ("filter16-canonical", 16, 4, True, {}),
    ("filter-k16", 16, 4, False, {"DVS_MASH_FILTER16": "0"}),
    ("filter-k16-canonical", 16, 4, True, {"DVS_MASH_FILTER16": "0"}),
    ("filter-k1", 1, 4, True, {}),
    ("filter-k5", 5, 4, False, {}),
    ("filter-k8", 8, 4, True, {}),
    ("filter-k12", 12, 4, False, {}),
    ("filter-k12-canonical", 12, 4, True, {}),
    ("filter-k15", 15, 4, True, {}),
    ("generic-k17", 17, 4, True, {}),
    ("generic-k21", 21, 4, False, {}),
    ("generic-k32", 32, 4, True, {}),
    ("generic-k40", 40, 4, False, {}),
    ("generic-ns5-canonical", 6, 5, True, {}),
]


@pytest.mark.parametrize("name,k,ns,canonical,env", FORMS, ids=[f[0] for f in FORMS])
def test_filter_kernels_both_sort_paths(lib, ctx, orc, monkeypatch, name, k, ns, canonical, env):
    """every filter kernel with the per-record sort and with the global bitonic network gives the oracle's
    sketches; s = 64 leaves the long records a threshold below all ones, the short ones none"""
    flat, off = ragged_set(k, ns, 7 + k)
    s = 64
    assert first_thresh_cap(int(np.diff(off).max()) - k + 1, s)[0] < ALL
    for key, val in env.items():
        monkeypatch.setenv(key, val)
    exp = orc.mash_sketch_batch(flat, off, k, s, ns, canonical, threads=_threads(orc))
    monkeypatch.delenv("DVS_MASH_GLOBAL_SORT", raising=False)
    _, d1, l1 = check_sketches(lib, ctx, orc, flat, off, k, s, canonical, ns, expected=exp)
    monkeypatch.setenv("DVS_MASH_GLOBAL_SORT", "1")
    _, d2, l2 = check_sketches(lib, ctx, orc, flat, off, k, s, canonical, ns, expected=exp)
    assert np.array_equal(l1, l2)
    if ns == 4 and k <= 16:  # without the switch, the first sorted pass takes the per-record sort
        passes = plan_seqs(_split(flat, off), k, s, canonical)
        assert [p.sort for p in passes if not p.overflow][0] == "record"


# ------------------------------------------------------------------------------- retry passes ----

@pytest.mark.parametrize("canonical", [False, True])
def test_widen_passes_end_in_global_sort(lib, ctx, orc, canonical):
    """a period-40 repeat whose hashes all exceed the first threshold: pass 1 finds no candidate, the threshold is
    widened x8 pass after pass (without canonical k-mers one pass also overflows its buffer on the way) and the
    last pass, at an all-ones threshold, sorts 300k candidates in the global network"""
    seq = widen_record(1 if not canonical else 5, 12, 64, canonical)
    passes = plan_seqs([seq], 12, 64, canonical)
    assert passes[0].counts == [0] and passes[0].sort == "record" and passes[0].widened == [0]
    assert sum(1 for p in passes if p.widened) >= 3
    assert passes[-1].thresh == [ALL] and passes[-1].sort == "global" and passes[-1].counts[0] > KSORT_REC_MAX
    flat, off = lib.concat([seq])
    _, _, lens = check_sketches(lib, ctx, orc, flat, off, 12, 64, canonical)
    assert 0 < lens[0] < 64


@pytest.mark.parametrize("n_repeat,sort", [(600_000, "global"), (100_000, "record")])
def test_overflow_redo(lib, ctx, orc, n_repeat, sort):
    """random bytes + a period-12 repeat with a k-mer below the record's s-th smallest hash: that k-mer occurs
    n_repeat / 12 times, beyond the first cap, so pass 1 overflows and is redone with a bigger buffer; at 600 kbp
    the redo has > 32,768 candidates and the global network drops ~50,000 copies of one key"""
    canonical = sort == "record"
    seq = overflow_record(2 if sort == "global" else 3, 12, 64, canonical, n_repeat=n_repeat)
    passes = plan_seqs([seq], 12, 64, canonical)
    assert [p.overflow for p in passes] == [True, False] and passes[1].sort == sort
    assert passes[0].counts[0] > passes[0].cap[0] and not passes[1].widened
    if sort == "global":
        assert passes[1].counts[0] > KSORT_REC_MAX
    # the repeated k-mer sits in the first half of the sketch, so copies of it that were not dropped would show
    rep = np.unique(window_hashes(seq[-n_repeat:], 12, canonical))
    at = np.flatnonzero(np.isin(bottom_s(window_hashes(seq, 12, canonical), 64), rep))
    assert at.size >= 1 and at[0] <= 32
    flat, off = lib.concat([seq])
    check_sketches(lib, ctx, orc, flat, off, 12, 64, canonical)


def test_mixed_call_slots_after_the_active_set_shrinks(lib, ctx, orc):
    """ordinary records (done in the first sorted pass) with an overflowing and a widening record in one call:
    the redo after the overflow holds every record, then only the widening one is left (slot 0 of later passes
    is record 1) and ends in the global network"""
    rng = np.random.default_rng(9)
    seqs = [random_record(rng, 50_000), widen_record(1, 12, 64, False), random_record(rng, 3000),
            overflow_record(3, 12, 64, True, n_repeat=100_000)[:300_000], np.zeros(0, np.uint8),
            random_record(rng, 700_000)]
    passes = plan_seqs(seqs, 12, 64, False)
    assert passes[0].active == [0, 1, 2, 3, 5] and passes[0].overflow
    assert passes[1].sort == "record" and passes[1].widened == [1]
    assert passes[-1].active == [1] and passes[-1].sort == "global"
    check_sketches(lib, ctx, orc, *lib.concat(seqs), 12, 64, False)


@pytest.mark.parametrize("s,lengths", [(20_000, (1_000_000, 900_003, 1_100_005)),
                                       (4_000_000_000, (100_000, 90_001, 110_007))])
def test_large_sketch_size_global_network(lib, ctx, orc, s, lengths):
    """sketch sizes whose candidates exceed the per-record sort: the padded key buffer holds >= 2^17 keys, so
    the global network runs several k_bitonic_global steps; s = 4e9 is upstream's "all" """
    rng = np.random.default_rng(s % 1000)
    seqs = [random_record(rng, n) for n in lengths]
    for q in seqs:
        q[rng.integers(0, q.size, size=50)] = 4
    passes = plan_seqs(seqs, 12, s, False)
    assert len(passes) == 1 and passes[0].sort == "global" and passes[0].npad >= 1 << 17
    check_sketches(lib, ctx, orc, *lib.concat(seqs), 12, s, False)


# ------------------------------------------------------------------- ctree defaults at genome length ----

class _Rec:
    def __init__(self, name, seq):
        self.seqid, self._seq = name, seq

    def get_seq(self):
        return self._seq


@pytest.mark.parametrize("canonical", [False, True])
def test_ctree_default_k12_s3000_genomes(lib, ctx, orc, canonical):
    """k = 12, s = 3000 (dvs_ctree's defaults) on 16 synthetic genomes of 2.25-3.75 Mbp: `k_mash_filter` at
    genome length; the matrix through Sketches.distances, distance.mash_distances and dvs_ctree is the same"""
    from diverseseq_b200 import cluster, distance
    flat, off = lib.synth_host(20261022, 16, 4, 3_000_000)
    assert int(np.diff(off).min()) >= 2_000_000
    assert first_thresh_cap(int(np.diff(off).min()) - 11, 3000)[0] < ALL
    sk, data, lens = check_sketches(lib, ctx, orc, flat, off, 12, 3000, canonical)
    assert (lens == 3000).all()
    dist, inter, uni = sk.distances(12, 3000, want_counts=True)
    od, oi, ou = orc.mash_matrix(data, lens, 12, 3000)
    assert np.array_equal(inter, oi) and np.array_equal(uni, ou)
    np.testing.assert_allclose(dist, od, rtol=RTOL, atol=0)
    assert (dist[~np.eye(16, dtype=bool)] > 0).all()
    recs = [_Rec(f"g{i}", q) for i, q in enumerate(_split(flat, off))]
    nd = distance.mash_distances(recs, 12, 3000, 4, mash_canonical=canonical)
    assert np.array_equal(nd.array, dist) and nd.names == [r.seqid for r in recs]
    tree = cluster.dvs_ctree(mash_canonical_kmers=canonical, ctx=ctx)([r.seqid for r in recs], recs)
    children, heights, _ = lib.linkage_average(ctx, dist)
    assert np.array_equal(tree.children, children) and np.array_equal(tree.heights, heights)


# ------------------------------------------------------------------------------------- matrix ----

def host_sketches(n: int, stride: int, seed: int):
    """ascending distinct rows of lengths 0..stride: overlaps drawn from a shared pool, copies of the row before,
    rows disjoint from every other row, random rows over all of u32 (0 and 2^32 - 1 included); one empty row"""
    rng = np.random.default_rng(seed)
    pool = np.unique(rng.integers(0, 1 << 32, size=3 * stride, dtype=np.uint64))
    data = np.zeros((n, stride), dtype=np.uint32)
    lens = np.zeros(n, dtype=np.uint32)
    span = (1 << 32) // n
    for i in range(n):
        kind = i % 6
        m = int(rng.integers(1, stride + 1)) if kind != 3 else stride
        if kind in (0, 3):
            row = np.sort(rng.choice(pool, size=min(m, pool.size), replace=False))
        elif kind == 1:
            row = data[i - 1, :lens[i - 1]].copy()
        elif kind == 2:  # values only row i can hold
            row = np.unique(rng.integers(i * span, (i + 1) * span, size=m, dtype=np.uint64))
        elif kind == 4:
            row = np.unique(np.concatenate([[0], rng.integers(1, (1 << 32) - 1, size=max(m - 2, 0), dtype=np.uint64),
                                            [(1 << 32) - 1]]))[:m]
        else:  # a prefix of an earlier row, then pool values
            src = data[i // 2, :lens[i // 2]]
            row = np.unique(np.concatenate([src[:len(src) // 2], rng.choice(pool, size=m)]))[:m]
        data[i, :len(row)] = row
        lens[i] = len(row)
    lens[n // 3] = 0
    data[n // 3] = 0
    inner = np.arange(stride - 1)[None, :] < lens[:, None].astype(np.int64) - 1
    assert (np.diff(data.astype(np.int64), axis=1)[inner] > 0).all()
    return data, lens


def _ulps(a, b):
    return int(np.abs(a.view(np.int64) - b.view(np.int64)).max())


@pytest.fixture(scope="module")
def matrix_set(lib, ctx, orc):
    data, lens = host_sketches(1037, 157, 31)
    sk = lib.Sketches.from_host(ctx, data, lens)
    return sk, data, lens


@pytest.mark.parametrize("s_kind", ["below", "equal", "above", "all"])
def test_mash_matrix_many_blocks(lib, ctx, orc, matrix_set, s_kind):
    """1,037 rows (1.07 M pairs over 8,400 blocks of 128): counts exact, distances within 1e-9, symmetric with a
    zero diagonal; the empty row is at distance 1 from every other row; sketch_size below, equal to and above the
    row lengths"""
    sk, data, lens = matrix_set
    n, stride = data.shape
    s = {"below": stride // 3, "equal": stride, "above": 2 * stride + 5, "all": 4_000_000_000}[s_kind]
    dist, inter, uni = sk.distances(12, s, want_counts=True)
    od, oi, ou = orc.mash_matrix(data, lens, 12, s, threads=_threads(orc))
    assert np.array_equal(inter, oi) and np.array_equal(uni, ou)
    np.testing.assert_allclose(dist, od, rtol=RTOL, atol=0)
    print(f"sketch_size {s}: largest gap to the oracle {_ulps(dist, od)} ulp")
    assert np.array_equal(dist, dist.T) and (np.diag(dist) == 0).all()
    e = n // 3
    assert (np.delete(dist[e], e) == 1.0).all()
    assert ((dist == 0.0) & ~np.eye(n, dtype=bool)).any() and ((dist == 1.0) & (inter == 0)).sum() > n
    assert np.array_equal(sk.distances(12, s), dist)  # without the counts


def test_mash_matrix_row_ranges_and_device_output(lib, ctx, orc, matrix_set):
    """row ranges (full, single rows, the last row, ranges starting and ending inside a block of 128 threads,
    empty) equal the rows of the full matrix; distances_into a DeviceBuffer equals distances"""
    sk, data, lens = matrix_set
    n = data.shape[0]
    full, fi, fu = sk.distances(12, 100, want_counts=True)
    for a, b in [(0, n), (0, 1), (n // 3, n // 3 + 1), (517, 518), (n - 1, n), (37, 613), (1, n - 1), (5, 5)]:
        d, i, u = sk.distances(12, 100, a, b, want_counts=True)
        assert d.shape == (b - a, n)
        assert np.array_equal(d, full[a:b]) and np.array_equal(i, fi[a:b]) and np.array_equal(u, fu[a:b]), (a, b)
    buf = lib.DeviceBuffer(ctx, n * n * 8)
    sk.distances_into(buf.ptr, 12, 100)
    assert np.array_equal(buf.to_host(np.float64, (n, n)), full)
    buf.close()


def test_mash_matrix_two_empty_sketches_raise(lib, ctx, matrix_set):
    """two empty sketches among non-empty ones: union 0, ZeroDivisionError as in the reference, also for a row
    range holding one of them"""
    _, data, lens = matrix_set
    lens = lens.copy()
    lens[700] = 0
    sk = lib.Sketches.from_host(ctx, data, lens)
    with pytest.raises(ZeroDivisionError):
        sk.distances(12, 100)
    with pytest.raises(ZeroDivisionError):
        sk.distances(12, 100, 690, 710)


# ------------------------------------------------------------------------------------ sharded ----

@pytest.mark.parametrize("layout", ["full-empty-short", "short-full-empty"])
def test_sharded_mash_unequal_strides(lib, ctx, orc, layout):
    """three ranks: one with records longer than s, one with none (stride 1) and one whose records are all
    shorter than s (a smaller stride, widened by the all-gather); every rank's matrix equals the single-GPU one
    bit for bit"""
    from diverseseq_b200 import shard
    s = 300
    full, _, _ = make_shards(lib, 808, [23], 4, 9000)
    short, _, _ = make_shards(lib, 809, [17], 3, 200)
    assert int(np.diff(short[0][1]).max()) - 12 + 1 < s
    empty = (np.zeros(0, np.uint8), np.zeros(1, np.uint64))
    shards = {"full-empty-short": [full[0], empty, short[0]], "short-full-empty": [short[0], full[0], empty]}[layout]
    flat, off = lib.concat([q for f, o in shards for q in _split(f, o)])
    sk, data, lens = check_sketches(lib, ctx, orc, flat, off, 12, s, True)
    single = sk.distances(12, s)
    np.testing.assert_allclose(single, orc.mash_matrix(data, lens, 12, s)[0], rtol=RTOL, atol=0)
    strides = []

    def fn(rank, rctx, comm):
        strides.append((rank, lib.Sketches.sketch(rctx, lib.SeqSet.upload(rctx, *shards[rank]), 12, s, 4,
                                                  True).stride))
        return shard.sharded_mash_distances(rctx, comm, lib.SeqSet.upload(rctx, *shards[rank]), 12, s, 4, True)

    for m in run_ranks(3, fn):
        assert np.array_equal(m, single)
    st = dict(strides)
    assert len(set(st.values())) == 3 and max(st.values()) == s
