"""Host model of the decisions `dvs_mash_sketch` (csrc/mash.cu) takes for each pass over the records, and the
reference hash of every k-mer window, so that a test can show its input really reaches the branch it names.

* `window_hashes`: hash_kmer (distance.rs:65-87) of every fully valid window of one record, in window order, for
  num_states = 4 and k <= 16, vectorised over numpy uint32: pack the k-mer (first base most significant), take
  min(k-mer, reverse complement) for canonical k-mers, k murmur rounds of one base each, then fmix.  A byte >= 4
  ends a run, as in get_kmer_hashes (distance.rs:101-134).
* `plan`: replays the host loop of `dvs_mash_sketch` pass by pass with the same formulas.  Per record:
  target = 2 min(s, nk) + 512, thresh = (target << 32) / nk (all ones when nk <= target),
  cap = min(2 target + 1024, nk).  Per pass: a record whose candidate count exceeds its cap gets
  cap = min(max(2 count, 2 cap), nk) and the whole pass is redone; otherwise every record is sorted in shared memory
  when no count exceeds KSORT_REC_MAX, else by the global bitonic network over the padded key buffer; a record with
  fewer than min(s, stride) distinct candidates under a threshold below all ones gets thresh = 8 thresh + 7 and
  cap = 8 cap (nk once the threshold is all ones) and is redone in the next pass, alone with the others like it.
"""
from dataclasses import dataclass, field

import numpy as np

ALL = 0xFFFFFFFF
KSORT_REC_MAX = 32768  # kSortRecMax: most candidates a record may have for the per-record sort
KSORT_TILE = 2048      # kSortTile: the global key buffer is padded to a power of two >= this
CHUNK = 256 << 10      # bytes of one work item of the filter kernels

_U = np.uint32


def _rotl(x, r):
    return (x << _U(r)) | (x >> _U(32 - r))


def _round(h, b):
    t = _rotl(b * _U(0xCC9E2D51), 15) * _U(0x1B873593)
    return _rotl(h ^ t, 13) * _U(5) + _U(0xE6546B64)


def _fmix(h):
    h = h ^ (h >> _U(16))
    h = h * _U(0x85EBCA6B)
    h = h ^ (h >> _U(13))
    h = h * _U(0xC2B2AE35)
    return h ^ (h >> _U(16))


def window_hashes(seq, k: int, canonical: bool) -> np.ndarray:
    """uint32 hash of every window of k bytes < 4, in window order (duplicates kept)"""
    assert 1 <= k <= 16
    seq = np.asarray(seq, dtype=np.uint8)
    nk = seq.size - k + 1
    if nk <= 0:
        return np.zeros(0, dtype=np.uint32)
    bad = np.concatenate([[0], np.cumsum(seq >= 4)])
    ok = (bad[k:] - bad[:nk]) == 0
    b = np.where(seq < 4, seq, 0).astype(np.uint32)
    v = np.zeros(nk, dtype=np.uint32)
    for j in range(k):
        v = (v << _U(2)) | b[j:j + nk]
    if canonical:
        rc = np.zeros(nk, dtype=np.uint32)
        for j in range(k):
            rc = (rc << _U(2)) | (b[k - 1 - j:k - 1 - j + nk] ^ _U(2))
        v = np.minimum(v, rc)  # lexicographic order of the bases == integer order of the packed k-mer
    v = v[ok]
    h = np.full(v.size, 0x9747B28C ^ k, dtype=np.uint32)
    for i in range(k - 1, -1, -1):
        h = _round(h, (v >> _U(2 * i)) & _U(3))
    return _fmix(h)


def bottom_s(hashes, s: int) -> np.ndarray:
    """the sketch: the s smallest distinct hashes, ascending"""
    return np.unique(np.asarray(hashes, dtype=np.uint32))[:s]


@dataclass
class Pass:
    active: list            # record indices of this pass, in slot order
    thresh: list            # per active record
    cap: list               # per active record (before this pass's overflow rule)
    counts: list            # candidates (hashes <= thresh) per active record
    overflow: bool          # some count > cap: the pass is redone with bigger buffers
    sort: str | None        # "record" (k_mash_sort_record), "global" (bitonic network) or None after an overflow
    npad: int               # keys in the padded buffer of the global network
    widened: list = field(default_factory=list)  # records redone in the next pass with a wider threshold


def first_thresh_cap(nk: int, s: int):
    target = 2 * min(s, nk) + 512
    if nk <= target:
        return ALL, min(nk, ALL)
    return min((target << 32) // nk, ALL), min(2 * target + 1024, nk)


def plan(nk_and_hashes, s: int, global_sort: bool = False) -> list:
    """the passes `dvs_mash_sketch` makes over records given as (nk, window hashes); nk counts every window
    (len - k + 1, valid or not); `global_sort` is DVS_MASH_GLOBAL_SORT=1"""
    nk = [int(n) for n, _ in nk_and_hashes]
    hashes = [np.asarray(h, dtype=np.uint32) for _, h in nk_and_hashes]
    uniq = [np.unique(h) for h in hashes]
    stride = max(1, min(s, max(nk, default=0)))
    want = min(s, stride)
    thresh, cap = [ALL] * len(nk), [0] * len(nk)
    act = []
    for r, n in enumerate(nk):
        if n == 0 or s == 0:
            continue
        thresh[r], cap[r] = first_thresh_cap(n, s)
        act.append(r)
    passes = []
    while act:
        counts = [int(np.count_nonzero(hashes[r] <= thresh[r])) for r in act]
        total_cap = sum(cap[r] for r in act)
        npad = KSORT_TILE
        while npad < total_cap:
            npad <<= 1
        p = Pass(list(act), [thresh[r] for r in act], [cap[r] for r in act], counts, False, None, npad)
        passes.append(p)
        for r, c in zip(act, counts):
            if c > cap[r]:
                p.overflow = True
                cap[r] = min(max(2 * c, 2 * cap[r]), nk[r])
        if p.overflow:
            continue
        p.sort = "record" if max(counts) <= KSORT_REC_MAX and not global_sort else "global"
        again = []
        for r in act:
            nd = int(np.searchsorted(uniq[r], thresh[r], side="right"))
            if nd < want and thresh[r] != ALL:
                thresh[r] = min(thresh[r] * 8 + 7, ALL)
                cap[r] = min(cap[r] * 8, nk[r])
                if thresh[r] == ALL:
                    cap[r] = min(nk[r], ALL)
                again.append(r)
        p.widened = again
        act = again
    return passes


def plan_seqs(seqs, k: int, s: int, canonical: bool, global_sort: bool = False) -> list:
    return plan([(max(len(q) - k + 1, 0), window_hashes(q, k, canonical)) for q in seqs], s, global_sort)


# ---- inputs that drive the retry passes ---------------------------------------------------------------------

def random_record(rng, n: int) -> np.ndarray:
    return rng.integers(0, 4, size=n, dtype=np.uint8)


def repeat_record(pattern, n: int) -> np.ndarray:
    return np.resize(np.asarray(pattern, dtype=np.uint8), n)


def find_pattern(rng, period: int, k: int, canonical: bool, ok, tries: int = 200_000) -> np.ndarray:
    """a random period-`period` pattern whose distinct window hashes h (of the tiled pattern) satisfy ok(h)"""
    for _ in range(tries):
        pat = rng.integers(0, 4, size=period, dtype=np.uint8)
        h = np.unique(window_hashes(repeat_record(pat, period + k - 1), k, canonical))
        if ok(h):
            return pat
    raise AssertionError("no pattern found")


def widen_record(seed: int, k: int, s: int, canonical: bool, n: int = 300_000, period: int = 40) -> np.ndarray:
    """a period-`period` repeat (fewer than s distinct k-mers) of n bytes whose hashes all exceed the first
    threshold: every pass finds fewer than s distinct candidates and widens, until the threshold is all ones"""
    t0, _ = first_thresh_cap(n - k + 1, s)
    pat = find_pattern(np.random.default_rng(seed), period, k, canonical, lambda h: h.min() > t0 and h.size < s)
    return repeat_record(pat, n)


def overflow_record(seed: int, k: int, s: int, canonical: bool, n_random: int = 200_000, n_repeat: int = 600_000,
                    period: int = 12) -> np.ndarray:
    """random bytes followed by a period-`period` repeat one of whose k-mers hashes below the (s/2)-th smallest hash
    of the random part (so below the first threshold, and in the first half of the sketch, where copies of it that
    were not dropped would show): that k-mer occurs about n_repeat / period times, more than the record's first
    cap"""
    rng = np.random.default_rng(seed)
    head = random_record(rng, n_random)
    bound = int(bottom_s(window_hashes(head, k, canonical), s)[s // 2])
    pat = find_pattern(rng, period, k, canonical, lambda h: int(h[0]) < bound)
    return np.concatenate([head, repeat_record(pat, n_repeat)])
