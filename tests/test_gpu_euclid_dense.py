"""Dense Euclidean distance matrix (dvs_euclid_distances / dvs_euclid_distances_sharded, csrc/euclid.cu) in each
of the forms that can produce a pair's distance, against a plain long-double reference:

* tiles      - the difference-form tile kernel k_euclid_tiles does the whole call (DVS_EUCLID_GRAM=0, odd row
               length): 1 launch, no listed pair;
* gram       - k_eg_norms + k_eg_gram (FP64 tensor cores, K in slices of 2,048 columns) + k_eg_finish: 3 launches,
               no listed pair;
* gram_list  - the same, and pairs with d^2 < 5e-4 (|a|^2 + |b|^2) recomputed in difference form by k_eg_pairs:
               4 launches, listed pairs > 0;
* overflow   - more than an eighth of the pairs listed, so the tile kernel redoes the call: 4 launches, none listed.

Every call asserts the signature of the form it is built to take, so a test cannot silently take another path.
Every matrix matches the reference at 1e-9 relative (NaN pattern equal, exact zeros exact), is bitwise symmetric
with a zero diagonal, and every row range equals the same rows of the full matrix bitwise (DESIGN.md §5.5).
"""
import functools
import math

import numpy as np
import pytest

from test_gpu_sharded import make_shards, run_ranks

RTOL = 1e-9
TAU = 5e-4        # kEgTau: the Gram form is used for a pair only when d^2 >= TAU (|a|^2 + |b|^2)
TILE = 128        # kEuT = kEgT
SLICE = 2048      # kEgSlice
SIGNATURE = {"tiles": (1, False), "gram": (3, False), "gram_list": (4, True), "overflow": (4, False)}

# form case -> (form, row length, DVS_EUCLID_GRAM=0)
CASES = {
    "tiles-env": ("tiles", 64, True),
    "tiles-odd": ("tiles", 63, False),
    "gram": ("gram", 64, False),
    "gram_list": ("gram_list", 64, False),
    "overflow": ("overflow", 64, False),
}


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


# ------------------------------------------------------------------------------------------ reference ----

def reference(rows) -> np.ndarray:
    """d(i, j) = sqrt(sum (a - b)^2) of f64 rows, evaluated in long double (64-bit significand): NaN for the pairs
    of a row holding a NaN, exactly 0 on the diagonal"""
    assert np.finfo(np.longdouble).nmant >= 63
    x = np.asarray(rows, dtype=np.longdouble)
    n = x.shape[0]
    out = np.zeros((n, n))
    for i in range(1, n):
        d = x[:i] - x[i]
        out[i, :i] = np.sqrt((d * d).sum(axis=1))
    iu = np.triu_indices(n, 1)
    out[iu] = out.T[iu]
    return out


def oracle_reference(orc, rows) -> np.ndarray:
    """for row lengths of 65,536 and more: the oracle adds the non-negative terms (a - b)^2 in sequence in f64, so
    its d^2 is within about (dim + 2) u d^2 of the exact value (1.2e-10 relative at dim = 2^20), far inside 1e-9"""
    return orc.euclid_matrix(np.ascontiguousarray(rows, dtype=np.float64), threads=max(1, orc.hardware_threads()))


def gram_ratio(rows, ref):
    """d^2 / (|a|^2 + |b|^2) of every pair i > j, the quantity the Gram form's threshold tests"""
    nrm = np.einsum("ij,ij->i", rows, rows)
    il = np.tril_indices(rows.shape[0], -1)
    return ref[il] ** 2 / (nrm[il[0]] + nrm[il[1]]), il


def assert_matrix(got, ref):
    np.testing.assert_allclose(got, ref, rtol=RTOL, atol=0, equal_nan=True)
    assert np.array_equal(got, got.T, equal_nan=True), "not bitwise symmetric"
    assert (np.diag(got) == 0).all(), "diagonal not exactly 0"


# ----------------------------------------------------------------------------------------------- rows ----

def far_rows(rng, n, dim):
    """rows whose pairs all have d^2 >= 2 TAU (|a|^2 + |b|^2), so the Gram form lists none of them; two columns
    are too few for random rows, so there the rows are distinct points of the integer grid [0, 16)^2
    (d^2 >= 1 and |a|^2 + |b|^2 <= 900)"""
    if dim == 2:
        assert n <= 256
        pts = rng.choice(256, size=n, replace=False)
        return np.stack([pts // 16, pts % 16], axis=1).astype(np.float64)
    return rng.random((n, dim))


def near_rows(rng, n, dim):
    """every pair a near-duplicate (d^2 ~ 1e-8 |a|^2) and two exact copies: every pair goes on the list"""
    base = rng.random(dim) + 0.5
    rows = base * (1.0 + 1e-4 * rng.standard_normal((n, dim)))
    if n >= 6:
        rows[5] = rows[2]
    if n > TILE + 3:
        rows[TILE + 3] = rows[1]
    return rows


def plant_near_pairs(rng, rows):
    """a near-duplicate pair inside every 128-row block, so that every row range lists at least one pair, and an
    exact copy of row 0 in the last row (a listed pair across blocks)"""
    rows = rows.copy()
    n = rows.shape[0]
    for b0 in range(0, n - 1, TILE):
        rows[b0 + 1] = rows[b0] * (1.0 + 1e-6 * rng.standard_normal(rows.shape[1]))
    if n >= 4:
        rows[n - 1] = rows[0]
    return rows


def rows_for(form, rng, n, dim):
    if form == "gram":
        return far_rows(rng, n, dim)
    if form == "overflow":
        return near_rows(rng, n, dim)
    return plant_near_pairs(rng, far_rows(rng, n, dim))


def check_rows_suit(form, rows, ref):
    """the rows really are what the form needs (far pairs for the Gram form, all pairs near for an overflow)"""
    if rows.shape[0] < 2 or form == "tiles":
        return
    ratio, _ = gram_ratio(rows, ref)
    if form == "gram":
        assert ratio.min() >= 2 * TAU
    elif form == "overflow":
        assert ratio.max() < TAU / 2
    else:
        assert ((ratio < TAU / 2) | (ratio >= 2 * TAU)).all() and (ratio < TAU / 2).any()


def set_form_env(monkeypatch, env_off):
    if env_off:
        monkeypatch.setenv("DVS_EUCLID_GRAM", "0")
    else:
        monkeypatch.delenv("DVS_EUCLID_GRAM", raising=False)


def signature(kf, fn):
    """(result, launches, listed pairs) of one Euclidean call"""
    before = kf.ctx.launch_count
    out = fn()
    return out, kf.ctx.launch_count - before, kf.fallback_pairs()


def run(kf, form, row_begin=0, row_end=None):
    """rows [row_begin, row_end) of the matrix; asserts that `form` computed them"""
    row_end = kf.nrec if row_end is None else row_end
    out, launches, listed = signature(kf, lambda: kf.euclidean(row_begin, row_end))
    if row_end == row_begin:
        assert launches == 0 and out.shape == (0, kf.nrec)
        return out
    want_launches, want_listed = SIGNATURE[form]
    assert (launches, listed > 0) == (want_launches, want_listed), \
        f"rows [{row_begin}, {row_end}) of n={kf.nrec}: {launches} launches, {listed} listed pairs; expected {form}"
    return out


# ---------------------------------------------------------------------------------------------- tests ----

def test_reference_agrees_with_oracle(orc):
    """the long-double reference and the oracle's f64 difference form agree to 1e-13 (NaN pattern included) on
    random rows, near-duplicate rows (d^2 ~ 1e-8 |a|^2), exact copies and a NaN row"""
    rng = np.random.default_rng(11)
    rand = rng.random((40, 37))
    near = near_rows(rng, 30, 50)
    near[7] = np.nan
    for rows in (rand, near):
        ref = reference(rows)
        np.testing.assert_allclose(ref, orc.euclid_matrix(rows), rtol=1e-13, atol=0, equal_nan=True)
        assert (np.diag(ref) == 0).all() and np.array_equal(ref, ref.T, equal_nan=True)
    assert reference(near)[2, 5] == 0.0 and np.isnan(reference(near)[7]).sum() == 29


def _shape_cases():
    for name in CASES:
        for n in (1, 2, 127, 128, 129, 257, 300, 680):
            form = CASES[name][0]
            # one row has no pair to list; the list holds at least 1,024 pairs before it can overflow
            if (form == "gram_list" and n < 2) or (form == "overflow" and n < 127):
                continue
            yield pytest.param(name, n, id=f"{name}-n{n}")


@pytest.mark.gpu
@pytest.mark.parametrize("case,n", list(_shape_cases()))
def test_forms_at_shapes(lib, ctx, monkeypatch, case, n):
    """1 to 6 tile rows, tile-aligned and not: the whole matrix, an aligned-begin range and a range to the end"""
    form, dim, env_off = CASES[case]
    set_form_env(monkeypatch, env_off)
    rows = rows_for(form, np.random.default_rng(1000 + n), n, dim)
    ref = reference(rows)
    check_rows_suit(form, rows, ref)
    kf = lib.KFreqs.from_rows(ctx, rows)
    got = run(kf, form)
    assert_matrix(got, ref)
    for rb, re in ((0, 2 * n // 3), (n // 3, n)):
        assert np.array_equal(run(kf, form, rb, re), got[rb:re], equal_nan=True), (rb, re)


def _dim_cases():
    for dim in (1, 2, 3, 15, 16, 17, 1024, 2047, 2048, 2049, 4097):
        yield pytest.param("tiles", dim, dim % 2 == 0, id=f"tiles-dim{dim}")
    # the Gram form needs an even row length (16-byte rows); around 2,048 these put 1, 2 or 3 slices in K
    for form in ("gram", "gram_list", "overflow"):
        for dim in (2, 16, 1024, 2046, 2048, 2050, 4096, 4098):
            yield pytest.param(form, dim, False, id=f"{form}-dim{dim}")


@pytest.mark.gpu
@pytest.mark.parametrize("form,dim,env_off", list(_dim_cases()))
def test_forms_at_row_lengths(lib, ctx, monkeypatch, form, dim, env_off):
    """row lengths around the 16-column slabs, the 2-column vector loads and the 2,048-column Gram slices; an odd
    length alone sends the call to the tile kernel"""
    set_form_env(monkeypatch, env_off)
    n = 160
    rows = rows_for(form, np.random.default_rng(dim), n, dim)
    ref = reference(rows)
    check_rows_suit(form, rows, ref)
    kf = lib.KFreqs.from_rows(ctx, rows)
    got = run(kf, form)
    assert_matrix(got, ref)
    assert np.array_equal(run(kf, form, 0, 150), got[:150], equal_nan=True)


def _ranges(n):
    return [(0, 200), (0, 129), (128, n), (128, 200), (37, n - 50), (127, 128), (128, 129), (129, 130), (n - 1, n),
            (200, n), (150, 150), (n, n)]


@pytest.mark.gpu
@pytest.mark.parametrize("n", [300, 680])
@pytest.mark.parametrize("case", list(CASES))
def test_row_ranges_equal_full_matrix(lib, ctx, monkeypatch, case, n):
    """the row-sharding hook: aligned begin with unaligned end (the tile kernel skips an upper tile whose transpose
    stops at row_end), unaligned begin, single rows either side of a tile edge, row_end == n, empty ranges; host
    and device output.  A matrix of different rows is computed just before every range call, so that a stale
    pool block cannot supply entries that the call failed to write."""
    form, dim, env_off = CASES[case]
    set_form_env(monkeypatch, env_off)
    rng = np.random.default_rng(n + len(case))
    rows = rows_for(form, rng, n, dim)
    ref = reference(rows)
    check_rows_suit(form, rows, ref)
    kf = lib.KFreqs.from_rows(ctx, rows)
    decoy = lib.KFreqs.from_rows(ctx, rng.random((n, dim)) + 3.0)
    full = run(kf, form)
    assert_matrix(full, ref)
    for rb, re in _ranges(n):
        decoy.euclidean()
        got = run(kf, form, rb, re)
        assert np.array_equal(got, full[rb:re], equal_nan=True), f"rows [{rb}, {re}) differ from the full matrix"
    for rb, re in ((0, 200), (37, n - 50)):
        decoy.euclidean()
        buf = lib.DeviceBuffer(ctx, (re - rb) * n * 8)
        _, launches, listed = signature(kf, lambda: kf.euclidean_into(buf.ptr, rb, re))
        assert (launches, listed > 0) == SIGNATURE[form]
        assert np.array_equal(buf.to_host(np.float64, (re - rb, n)), full[rb:re], equal_nan=True)
        buf.close()


@pytest.mark.gpu
@pytest.mark.parametrize("env_off", [False, True], ids=["gram_list", "tiles"])
def test_counted_set_with_invalid_records(lib, ctx, monkeypatch, env_off):
    """records without a valid k-mer (empty, shorter than k, all invalid bytes) have NaN rows and NaN pairs; those
    pairs go on the Gram form's list"""
    set_form_env(monkeypatch, env_off)
    rng = np.random.default_rng(77)
    base = rng.integers(0, 4, size=3000, dtype=np.uint8)
    seqs = []
    for i in range(150):
        s = base[: int(rng.integers(1500, 3000))].copy()
        hit = rng.random(s.size) < rng.choice([0.001, 0.05, 0.5])
        s[hit] = rng.integers(0, 4, size=int(hit.sum()), dtype=np.uint8)
        seqs.append(s)
    bad = [3, 64, 140]
    seqs[3] = np.zeros(0, dtype=np.uint8)
    seqs[64] = np.array([0, 1, 2], dtype=np.uint8)
    seqs[140] = np.full(500, 7, dtype=np.uint8)
    seqs[20] = seqs[10].copy()
    kf = lib.KFreqs.count(ctx, lib.SeqSet.from_seqs(ctx, seqs), 4)
    _, rows, _, valid = kf.download(counts=False)
    assert np.isnan(rows[bad]).all() and not valid[bad].any() and not np.isnan(np.delete(rows, bad, 0)).any()
    ref = reference(rows)
    got = run(kf, "tiles" if env_off else "gram_list")
    assert_matrix(got, ref)
    assert np.isnan(got[bad][:, [0, 1, 149]]).all() and got[10, 20] == 0.0
    if not env_off:
        assert kf.fallback_pairs() >= 3 * 147 + 3


@pytest.mark.gpu
def test_nan_rows_alone_overflow_the_list(lib, ctx, monkeypatch):
    """far rows apart from 70 NaN rows: their 18,515 NaN pairs are more than an eighth of the pairs, so the
    call overflows the list and the tile kernel computes it"""
    set_form_env(monkeypatch, False)
    rng = np.random.default_rng(5)
    n = 300
    rows = far_rows(rng, n, 64)
    bad = rng.choice(n, size=70, replace=False)
    rows[bad] = np.nan
    ref = reference(rows)
    ratio, _ = gram_ratio(rows, ref)
    assert np.nanmin(ratio) >= 2 * TAU and np.isnan(ratio).sum() == 70 * 230 + 70 * 69 // 2
    kf = lib.KFreqs.from_rows(ctx, rows)
    got = run(kf, "overflow")
    assert_matrix(got, ref)
    assert np.array_equal(run(kf, "overflow", 0, 200), got[:200], equal_nan=True)


def threshold_rows(rng, n, dim):
    """integer counts of about 4 M per row, divided by their total: a common base plus +-a on m random columns,
    sized so that row i lies at d^2 / (|a|^2 + |b|^2) ~ 1e-7 ... 1e-2 (log-spaced) from the rows before it"""
    base = rng.poisson(4_000_000 / dim, size=dim).astype(np.float64)
    nb2 = float(base @ base)
    rows = np.empty((n, dim))
    for i, target in enumerate(np.logspace(-7, -2, n)):
        need = 2.0 * target * nb2  # sum of squared count changes
        a = max(1.0, math.ceil(math.sqrt(need / (dim / 4))))
        m = max(1, int(round(need / (a * a))))
        cols = rng.choice(dim, size=m, replace=False)
        c = base.copy()
        c[cols] += a * rng.choice([-1.0, 1.0], size=m)
        np.maximum(c, 0.0, out=c)
        rows[i] = c / c.sum()
    return rows


@pytest.mark.gpu
@pytest.mark.parametrize("dim", [65_536, 262_144, 1_048_576])
def test_gram_threshold(lib, ctx, orc, monkeypatch, dim):
    """pairs either side of the Gram threshold, at 32, 128 and 512 slices: exactly the pairs below TAU are listed
    (up to a 1e-6 band around it) and the Gram-form distances are within 1e-9 relative"""
    set_form_env(monkeypatch, False)
    rows = threshold_rows(np.random.default_rng(dim), 64, dim)
    ref = oracle_reference(orc, rows)
    ratio, il = gram_ratio(rows, ref)
    assert ((ratio >= TAU / 2) & (ratio < TAU)).sum() >= 50 and ((ratio >= TAU) & (ratio <= 2 * TAU)).sum() >= 50
    assert ratio.min() < 1e-6 and ratio.max() > 5e-3
    kf = lib.KFreqs.from_rows(ctx, rows)
    got = run(kf, "gram_list")
    assert (ratio < TAU * (1 - 1e-6)).sum() <= kf.fallback_pairs() <= (ratio < TAU * (1 + 1e-6)).sum()
    gram = ratio >= TAU * (1 + 1e-6)
    rel = np.abs(got[il][gram] - ref[il][gram]) / ref[il][gram]
    print(f"\ndim {dim} ({dim // SLICE} slices): {gram.sum()} Gram-form pairs, largest relative error {rel.max():.3e}")
    assert rel.max() <= 1e-9
    assert_matrix(got, ref)


@pytest.mark.gpu
def test_argument_errors(lib, ctx):
    kf = lib.KFreqs.from_rows(ctx, np.random.default_rng(0).random((5, 8)))
    out = np.zeros((8, 5))
    for rb, re in ((0, 6), (3, 2), (6, 6)):
        assert kf.ctx._lib.dvs_euclid_distances(ctx.handle, kf.handle, rb, re, lib.ptr(out)) == lib.DVS_ERR_ARG, (rb, re)


# -------------------------------------------------------------------------------------------- sharded ----

SHARD_NPR = {2: [290, 310], 3: [190, 200, 210]}  # the same 600 records in both splits


@functools.lru_cache(maxsize=None)
def _counted_600():
    from diverseseq_b200 import _lib
    from oracle import oracle
    shards = {w: make_shards(_lib, 606, npr, 6, 6000) for w, npr in SHARD_NPR.items()}
    _, flat, off = shards[2]
    _, of, _, ov = oracle.count_batch(flat, off, 5, want_counts=False)
    assert ov.all() and np.array_equal(shards[3][1], flat)
    return shards, flat, off, of, reference(of)


def _sharded(lib, world, fn_rows):
    """each rank's (matrix, launches, listed pairs) of dvs_euclid_distances_sharded"""
    def fn(rank, ctx, comm):
        kf = fn_rows(rank, ctx, comm)
        return signature(kf, lambda: kf.euclidean_sharded(comm))
    return run_ranks(world, fn)


@pytest.mark.gpu
@pytest.mark.parametrize("env_off", [False, True], ids=["default", "tiles"])
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_equals_reference_and_single_gpu(lib, monkeypatch, world, env_off):
    """600 records, 15 lower-triangle tiles dealt over 2 or 3 GPUs: every rank's matrix matches the reference and
    is bitwise the single-GPU matrix of the same form"""
    from diverseseq_b200 import shard
    set_form_env(monkeypatch, env_off)
    shards, flat, off, _, ref = _counted_600()
    ctx0 = lib.Context(0)
    kf0 = lib.KFreqs.count(ctx0, lib.SeqSet.upload(ctx0, flat, off), 5)
    single, launches, listed = signature(kf0, kf0.euclidean)
    if env_off:
        assert (launches, listed) == (1, 0)
    else:
        assert (launches, listed > 0) in ((3, False), (4, True)), (launches, listed)
    assert_matrix(single, ref)

    def rows(rank, ctx, comm):
        return shard.count_sharded(ctx, comm, lib.SeqSet.upload(ctx, *shards[world][0][rank]), 5)[0]

    for rank, (m, launches, listed) in enumerate(_sharded(lib, world, rows)):
        if env_off:
            assert (launches, listed) == (1, 0), rank
        else:
            assert (launches, listed > 0) in ((3, False), (4, True)), (rank, launches, listed)
        assert np.array_equal(m, single), f"rank {rank} differs from the single-GPU matrix"


def predicted_rank_forms(n, world, near):
    """the form of each rank's share when the rows `near` are near-duplicates of each other and every other pair is
    far: tiles t = rank, rank + world, ... of the lower triangle; a list of more than max(tiles * 2048, 1024) pairs
    overflows"""
    nt = (n + TILE - 1) // TILE
    tiles = [(ti, tj) for ti in range(nt) for tj in range(ti + 1)]
    forms = []
    for rank in range(world):
        mine = tiles[rank::world]
        listed = 0
        for ti, tj in mine:
            a = int(near[ti * TILE:(ti + 1) * TILE].sum())
            b = int(near[tj * TILE:(tj + 1) * TILE].sum())
            listed += a * (a - 1) // 2 if ti == tj else a * b
        cap = max(len(mine) * TILE * TILE // 8, 1024)
        forms.append("overflow" if listed > cap else "gram_list" if listed else "gram")
    return forms


@pytest.mark.gpu
@pytest.mark.parametrize("world", [2, 3])
def test_sharded_list_overflows_on_one_rank_only(lib, monkeypatch, world):
    """rows 0-255 near-duplicates of each other: the rank holding tile (1, 0) overflows its list and runs the tile
    kernel over its own tiles, the others finish in the Gram form with their lists; the matrix is still whole"""
    set_form_env(monkeypatch, False)
    rng = np.random.default_rng(600 + world)
    n, dim = 600, 64
    rows = far_rows(rng, n, dim)
    rows[:256] = near_rows(rng, 256, dim)
    near = np.zeros(n, dtype=bool)
    near[:256] = True
    ref = reference(rows)
    ratio, il = gram_ratio(rows, ref)
    both = near[il[0]] & near[il[1]]
    assert ratio[both].max() < TAU / 2 and ratio[~both].min() >= 2 * TAU
    forms = predicted_rank_forms(n, world, near)
    assert "overflow" in forms and "gram_list" in forms, forms

    def from_rows(rank, ctx, comm):
        return lib.KFreqs.from_rows(ctx, rows)

    for rank, (m, launches, listed) in enumerate(_sharded(lib, world, from_rows)):
        assert (launches, listed > 0) == SIGNATURE[forms[rank]], (rank, forms[rank], launches, listed)
        assert_matrix(m, ref)
