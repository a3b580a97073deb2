// SummedRecords on the device: JSD / delta-JSD state and the order-preserving nmost / max
// selection loops.  Replaces /root/reference/src/records.rs:10-524.
//
// Exactness: every entropy the reference evaluates is evaluated here in the reference's own
// sequential order (entropy.cuh), and every elementwise update of summed_kfreqs /
// summed_entropies uses the same operations in the same order (explicit __d*_rn, no FMA), so
// the state is bitwise the reference's and every `>` / `<` decision is the reference's.
//
// Parallel shape: the reference streams candidates one at a time (records.rs:331-340).  Here a
// WINDOW of candidates following the cursor is scored concurrently (one CTA per candidate)
// against the current state; the FIRST position whose predicate `delta_jsd > total_jsd + EPS`
// holds is the one the reference would accept next (everything before it was rejected against
// the same state; everything after it is stale and is re-scored after the update).  A min-index
// reduction (atomicMin) finds it; the state update then runs as three small kernels.
#include <limits.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <limits>
#include <optional>
#include <type_traits>

#include <cooperative_groups.h>

#include "comm.cuh"
#include "common.cuh"
#include "entropy.cuh"
#include "fused.cuh"
#include "sparse.cuh"

namespace cg = cooperative_groups;

namespace dvs {

constexpr unsigned kNone = 0xFFFFFFFFu;

struct SelScal {
    double E;          // summed_entropies
    double total_jsd;
    double mean, stdv, cov;  // mean/std/cov of member delta_jsd
    double panic_total;      // offending total for a state-level entropy panic
    unsigned n;              // size
    unsigned lowest;         // lowest_index
    unsigned first_true;     // scan result: first position whose predicate holds
    unsigned first_panic;    // scan result: first position whose evaluation panics
    unsigned panic;          // 0 none; 1 = entropy sum check failed while updating the state
    unsigned ticket;         // last-block-done counter
    // ---- bounded-error fast path (see "fast path" below) ----
    double total_bound;      // |total_jsd - exact total_jsd| <= total_bound (0 when exact)
    unsigned first_unsure;   // scan result: first position the fast scan could not decide
    unsigned state_unsure;   // fast update could not certify lowest_index / the sum checks
    unsigned exact;          // 1 when total_jsd / mdelta / lowest come from the exact kernel
    unsigned pad0_;
    double std_bound;        // fast path: |stdv - reference std_delta_jsd| <= std_bound  (0 when exact)
    double cov_bound;        // fast path: same for cov (infinite when the mean is too close to 0)
    // ---- device-driven rounds (k_sel_persist / k_sel_persist_sm_t) ----
    unsigned cursor;         // next position to examine
    unsigned window;         // candidates scored per round
    unsigned window_max;
    unsigned num;            // number of positions
    unsigned halt;           // 1: the host must resolve an undecided candidate / state exactly
    unsigned accepts;        // candidates that replaced the lowest record so far
    unsigned which;          // which copy of the double-buffered S / member list is current
    unsigned limit;          // trailing rounds: positions below it had been published when the kernel returned
};

struct SelState {
    // S and the member list are double buffered: the fused fast replace+update kernel reads one copy
    // and writes the other, so it needs no grid-wide barrier between "update S" and "use S"
    DevBuf<double> Sbuf[2];          // summed_kfreqs [dim]
    DevBuf<unsigned> membuf[2];      // row indices in Vec order [cap]
    int which = 0;
    DevBuf<double> mdelta;     // delta_jsd per member [cap]
    DevBuf<double> mbound;     // fast path: error bound of each member's value [cap]
    DevBuf<SelScal> sc;
    unsigned cap = 0;
    double* S() { return Sbuf[which].p; }
    unsigned* members() { return membuf[which].p; }
    double* S_other() { return Sbuf[which ^ 1].p; }
    unsigned* members_other() { return membuf[which ^ 1].p; }
    void flip() { which ^= 1; }
    int alloc(uint64_t dim, unsigned capacity) {
        cap = capacity;
        for (int b = 0; b < 2; ++b) {
            DVS_TRY(Sbuf[b].alloc(dim));
            DVS_TRY(membuf[b].alloc(capacity));
        }
        DVS_TRY(mdelta.alloc(capacity));
        DVS_TRY(mbound.alloc(capacity));
        DVS_TRY(sc.alloc(1));
        return DVS_OK;
    }
};

// ------------------------------------------------------------------------------ row sources ----
// Where a kernel gets element i of a record's frequency row.  A kernel binds the rows it reads to the slots of a
// view (v.row(slot, record, dim)) and hands the view to the entropy helper as its staging hook.
//   DenseRows   the [nrec][dim] rows of a dvs_kfreqs: a bound row is F + record * dim; nothing is staged.
//   SparseRows  the bucket-major (index, count) rows of a dvs_ksparse (sparse.cuh).  A bucket holds the entries of
//               4,096 consecutive bins: one pass of the bounded-error kernels (8 x kFastThreads elements) and
//               kEntStageTiles tiles of the exact ones.  Before a pass, the CTA stages the bucket's counts of every
//               bound row in shared memory (16 KB per row, 0 where the row has no entry), and element i is then
//               div_exact(count, total): the division k_freq_entropy forms the dense row with.  Every element, and
//               with it every sum, error bound and decision, is therefore the dense path's bit for bit.
// The selection state S stays dense either way (4^k f64): the clamps and the reference's sums run over all elements.
struct DenseRows {
    static constexpr bool kSparse = false;
    const double* __restrict__ F;
    struct View {
        const double* __restrict__ F;
        __device__ __forceinline__ const double* row(int, unsigned r, uint64_t dim) const { return F + (size_t)r * dim; }
        // a candidate row of another dvs_kfreqs (dvs_summed_delta_jsd)
        __device__ __forceinline__ const double* cand_row(const double* C, int, unsigned r, uint64_t dim) const {
            return C + (size_t)r * dim;
        }
        __device__ __forceinline__ void operator()(uint64_t) const {}
    };
    __device__ __forceinline__ View view(uint32_t*) const { return View{F}; }
};

static_assert(kEntTile * kEntStageTiles == (int)kSpLowBins, "a tile group of the exact kernels must be one bucket");
constexpr int kStageSlots = 3;  // rows one kernel reads at most (the fused replace + update: lowest, candidate, member)
constexpr size_t kStageBytes = (size_t)kSpLowBins * sizeof(uint32_t);

struct SpRow {
    const uint32_t* s;  // staged counts of the current bucket
    FastDiv dv;         // the record's number of valid k-mers
    __device__ __forceinline__ double operator[](uint64_t i) const {
        return div_exact((double)s[i & (kSpLowBins - 1u)], dv);
    }
};

struct SparseRowsData {
    const uint32_t *idx, *cnt, *bucket_ptr, *bucket_nnz;
    const uint64_t *offsets, *totals;
    uint32_t nb;
    // first slot and entries of bucket b of record r
    __device__ __forceinline__ uint64_t bucket_at(unsigned r, uint32_t b) const {
        return offsets[r] + bucket_ptr[(size_t)r * (nb + 1) + b];
    }
    __device__ __forceinline__ uint32_t bucket_len(unsigned r, uint32_t b) const { return bucket_nnz[(size_t)r * nb + b]; }
    // the arrays that hold record r, and r's row in them: these
    __device__ __forceinline__ const SparseRowsData& part(unsigned&) const { return *this; }
};

// dvs_select_sparse_sharded: the rows a rank reads are its own (`local`) or peer rows copied into its member-row
// cache (`cache`, one row per slot); where[r] tells which for global row r.  Totals are indexed by global row.
constexpr uint32_t kCachedRow = 0x80000000u;  // where[r]: cache slot (low bits) instead of a local row
constexpr uint32_t kAbsentRow = 0xFFFFFFFFu;  // where[r]: neither (never read)
struct ShardRowsData {
    SparseRowsData local, cache;
    const uint32_t* where;
    const uint64_t* totals;
    __device__ __forceinline__ SparseRowsData part(unsigned& r) const {
        const uint32_t w = where[r];
        r = w & ~kCachedRow;
        return (w & kCachedRow) ? cache : local;
    }
};

template <class D>
struct SparseRowsT : D {
    static constexpr bool kSparse = true;
    struct View {
        D src;
        uint32_t* smem;  // kStageSlots x 4,096 counts
        unsigned rows[kStageSlots];
        int nbound;
        __device__ __forceinline__ SpRow row(int slot, unsigned r, uint64_t) {
            rows[slot] = r;
            nbound = max(nbound, slot + 1);
            return SpRow{smem + (size_t)slot * kSpLowBins, make_fast_div((double)src.totals[r])};
        }
        __device__ __forceinline__ SpRow cand_row(const double*, int slot, unsigned r, uint64_t dim) { return row(slot, r, dim); }
        // every thread of the CTA: stage the bucket that starts at element `base` of every bound row
        __device__ void operator()(uint64_t base) const {
            const uint32_t b = (uint32_t)(base >> kSpLowBits);
            __syncthreads();  // the previous bucket has been read
            uint4* z = reinterpret_cast<uint4*>(smem);
            for (unsigned i = threadIdx.x; i < (unsigned)nbound * (kSpLowBins / 4); i += blockDim.x) z[i] = make_uint4(0, 0, 0, 0);
            __syncthreads();
#pragma unroll
            for (int q = 0; q < kStageSlots; ++q) {
                if (q < nbound) {
                    unsigned r = rows[q];
                    const auto& p = src.part(r);
                    const uint64_t at = p.bucket_at(r, b);
                    const uint32_t n = p.bucket_len(r, b);
                    uint32_t* d = smem + (size_t)q * kSpLowBins;
                    for (uint32_t e = threadIdx.x; e < n; e += blockDim.x) d[p.idx[at + e] & (kSpLowBins - 1u)] = p.cnt[at + e];
                }
            }
            __syncthreads();
        }
    };
    __device__ __forceinline__ View view(uint32_t* smem) const { return View{*this, smem, {0u, 0u, 0u}, 0}; }
};
struct SparseRows : SparseRowsT<SparseRowsData> {};
struct ShardRows : SparseRowsT<ShardRowsData> {};

// the staging hook a kernel hands to the entropy helpers: the view itself, or nothing for dense rows
__device__ __forceinline__ NoStage stager(const DenseRows::View&) { return NoStage{}; }
__device__ __forceinline__ const SparseRows::View& stager(const SparseRows::View& v) { return v; }
__device__ __forceinline__ const ShardRows::View& stager(const ShardRows::View& v) { return v; }

// the staging area of the bounded-error kernels: their dynamic shared memory (the exact kernels place it after
// their tiles); dense rows have none
template <class Src>
__device__ __forceinline__ uint32_t* stage_smem() { return nullptr; }
template <>
__device__ __forceinline__ uint32_t* stage_smem<SparseRows>() {
    extern __shared__ __align__(16) uint32_t sel_stage_smem[];
    return sel_stage_smem;
}
template <>
__device__ __forceinline__ uint32_t* stage_smem<ShardRows>() {
    extern __shared__ __align__(16) uint32_t sel_stage_smem[];
    return sel_stage_smem;
}
template <class Src>
__device__ __forceinline__ uint32_t* exact_stage_smem(double* ent_smem) {
    return Src::kSparse ? reinterpret_cast<uint32_t*>(ent_smem + kEntSmemBytes / sizeof(double)) : nullptr;
}
// dynamic shared memory of a kernel that binds `slots` rows (on top of what the dense form uses)
template <class Src>
constexpr size_t stage_bytes(int slots) { return Src::kSparse ? (size_t)slots * kStageBytes : 0; }

__device__ __forceinline__ void sum_scalars(const double* __restrict__ H, const unsigned* __restrict__ members, unsigned n,
                                            int extra_row, unsigned* __restrict__ members_out, SelScal* sc) {
    double e = 0.0;
    for (unsigned j = 0; j < n; ++j) e = __dadd_rn(e, H[members[j]]);
    if (extra_row >= 0) e = __dadd_rn(e, H[extra_row]);
    unsigned nn = n;
    if (members_out != members)
        for (unsigned j = 0; j < n; ++j) members_out[j] = members[j];
    if (extra_row >= 0) members_out[nn++] = (unsigned)extra_row;
    sc->E = e;
    sc->n = nn;
    sc->panic = 0;
    sc->panic_total = 0.0;
    sc->ticket = 0;
    sc->first_true = kNone;
    sc->first_panic = kNone;
    sc->first_unsure = kNone;
    sc->state_unsure = 0;
    sc->total_bound = 0.0;
    sc->exact = 0;
}

// S[i] = ((0 + f_m0[i]) + f_m1[i]) + ... (+ f_extra[i]);  E likewise  (records.rs:36-42, :129-133)
// Sparse rows: one CTA per bucket zeroes its 4,096 elements of S and adds the members' entries one member after
// another, in member order.  An absent entry would add +0.0, which leaves every sum (all >= +0) as it is, so per
// element these are the same additions in the same order.
template <class Src>
__global__ void k_sel_sum(const Src src, const double* __restrict__ H, uint64_t dim,
                          const unsigned* __restrict__ members, unsigned n, int extra_row, double* __restrict__ S,
                          unsigned* __restrict__ members_out, SelScal* sc) {
    if constexpr (Src::kSparse) {
        const uint32_t b = blockIdx.x;
        double* Sb = S + ((uint64_t)b << kSpLowBits);
        for (unsigned i = threadIdx.x; i < kSpLowBins; i += blockDim.x) Sb[i] = 0.0;
        const unsigned nn = n + (extra_row >= 0 ? 1u : 0u);
        for (unsigned j = 0; j < nn; ++j) {
            __syncthreads();  // member j - 1 is in
            const unsigned r = j < n ? members[j] : (unsigned)extra_row;
            unsigned pr = r;
            const auto& d = src.part(pr);
            const uint64_t at = d.bucket_at(pr, b);
            const uint32_t m = d.bucket_len(pr, b);
            const FastDiv dv = make_fast_div((double)src.totals[r]);
            for (uint32_t e = threadIdx.x; e < m; e += blockDim.x) {
                double* p = Sb + (d.idx[at + e] & (kSpLowBins - 1u));
                *p = __dadd_rn(*p, div_exact((double)d.cnt[at + e], dv));
            }
        }
        if (b == 0 && threadIdx.x == 0) sum_scalars(H, members, n, extra_row, members_out, sc);
    } else {
        const double* F = src.F;
        uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i < dim) {
            double s = 0.0;
            for (unsigned j = 0; j < n; ++j) s = __dadd_rn(s, F[(size_t)members[j] * dim + i]);
            if (extra_row >= 0) s = __dadd_rn(s, F[(size_t)extra_row * dim + i]);
            S[i] = s;
        }
        if (i == 0) sum_scalars(H, members, n, extra_row, members_out, sc);
    }
}

// replace_lowest (records.rs:94-135): drop_lowest + push on summed_kfreqs, elementwise; the LAST
// CTA to finish then updates the scalars and the member Vec: E -= H_low; E += H_c;
// Vec::remove(lowest); push(c).  Sparse rows: one CTA per bucket, over every element of S (the clamp too).
template <class Src>
__global__ void k_sel_replace_vec(const Src src, const double* __restrict__ H, uint64_t dim,
                                  unsigned* __restrict__ members, uint8_t* __restrict__ is_member, SelScal* sc,
                                  unsigned cand_row, double* __restrict__ S) {
    __shared__ unsigned s_last;
    const unsigned low = sc->lowest;
    const unsigned low_row = members[low];
    if constexpr (Src::kSparse) {
        auto v = src.view(stage_smem<Src>());
        const SpRow fl = v.row(0, low_row, dim), fc = v.row(1, cand_row, dim);
        const uint64_t base = (uint64_t)blockIdx.x << kSpLowBits;
        v(base);
        for (unsigned q = threadIdx.x; q < kSpLowBins; q += blockDim.x) {
            double s = __dsub_rn(S[base + q], fl[q]);
            if (s <= kEps) s = 0.0;
            S[base + q] = __dadd_rn(s, fc[q]);
        }
    } else {
        const double* F = src.F;
        const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
        if (i < dim) {
            double s = __dsub_rn(S[i], F[(size_t)low_row * dim + i]);
            if (s <= kEps) s = 0.0;
            S[i] = __dadd_rn(s, F[(size_t)cand_row * dim + i]);
        }
    }
    __syncthreads();  // every read of members[]/lowest by this CTA is done
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(&sc->ticket, 1u) == gridDim.x - 1) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {  // block-uniform
        const unsigned n = sc->n;
        // Vec::remove(low) + push(cand): every thread moves a strided share, reads before writes
        unsigned keep[8];
        const unsigned per = (n + blockDim.x - 1) / blockDim.x;
        if (per <= 8) {
            for (unsigned q = 0; q < per; ++q) {
                const unsigned j = threadIdx.x + q * blockDim.x;
                keep[q] = (j >= low && j + 1 < n) ? members[j + 1] : 0u;
            }
            __syncthreads();
            for (unsigned q = 0; q < per; ++q) {
                const unsigned j = threadIdx.x + q * blockDim.x;
                if (j >= low && j + 1 < n) members[j] = keep[q];
            }
        } else if (threadIdx.x == 0) {
            for (unsigned j = low; j + 1 < n; ++j) members[j] = members[j + 1];
        }
        if (threadIdx.x == 0) {
            double e = __dsub_rn(sc->E, H[low_row]);
            sc->E = __dadd_rn(e, H[cand_row]);
            members[n - 1] = cand_row;
            if (is_member) {
                is_member[low_row] = 0;
                is_member[cand_row] = 1;
            }
            sc->ticket = 0;
        }
    }
}

// total_jsd and get_lowest_record_index in one launch (records.rs:136-146, 220-252): CTA j < n
// evaluates member j's leave-one-out entropy, CTA n evaluates H(S/n); none of these entropies
// depends on another, only the final scalar arithmetic does, so the last CTA to finish forms
// total_jsd = H(S/n) - E/n, delta_j = total_jsd - (H(m_j) - (E - H_j)/(n-1)), the strict-<
// argmin and the mean/std/cov statistics (:153-172) in the reference's order.
template <class Src>
__global__ void __launch_bounds__(kEntThreads)
k_sel_update(const Src src, const double* __restrict__ H, uint64_t dim, const double* __restrict__ S,
             const unsigned* __restrict__ members, double* __restrict__ mdelta, SelScal* sc) {
    extern __shared__ __align__(16) double ent_smem[];
    __shared__ unsigned s_last;
    const unsigned j = blockIdx.x, n = sc->n;
    const double nd = (double)n;
    if (j == n) {
        EntropyResult h = block_entropy_exact(dim, [&](uint64_t i) { return __ddiv_rn(S[i], nd); }, ent_smem);
        if (threadIdx.x == 0) {
            sc->total_jsd = __dsub_rn(h.e, __ddiv_rn(sc->E, nd));
            if (entropy_total_bad(h.t, dim) && atomicCAS(&sc->panic, 0u, 1u) == 0u) sc->panic_total = h.t;
        }
    } else {
        const unsigned row = members[j];
        const double div = __dsub_rn(nd, 1.0);
        auto v = src.view(exact_stage_smem<Src>(ent_smem));
        const auto f = v.row(0, row, dim);
        EntropyResult h = block_entropy_exact(
            dim,
            [&](uint64_t i) {
                double m = __ddiv_rn(__dsub_rn(S[i], f[i]), div);
                return (m <= kEps) ? 0.0 : m;  // updated_mean_freqs clamp, records.rs:281-284
            },
            ent_smem, stager(v));
        if (threadIdx.x == 0) {
            const double mean_entropy = __ddiv_rn(__dsub_rn(sc->E, H[row]), div);
            mdelta[j] = __dsub_rn(h.e, mean_entropy);  // jsd without record j; delta formed below
            // the reference panics at the first member whose sum check fails; any failure is fatal
            if (entropy_total_bad(h.t, dim) && atomicCAS(&sc->panic, 0u, 1u) == 0u) sc->panic_total = h.t;
        }
    }
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(&sc->ticket, 1u) == n) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {  // block-uniform: the last CTA finishes get_lowest_record_index + the statistics
        __threadfence();
        // the sums below are sequential (reference order); stage the n values in shared memory first so
        // the single summing thread does not pay one L2 round trip per member
        constexpr unsigned kStage = (unsigned)(kEntSmemBytes / sizeof(double));
        const bool staged = n <= kStage;
        if (staged) {
            for (unsigned t = threadIdx.x; t < n; t += blockDim.x) ent_smem[t] = __ldcg(&mdelta[t]);
            __syncthreads();
        }
        if (threadIdx.x == 0) {
            volatile double* mdv = mdelta;
            const double total_jsd = __ldcg(&sc->total_jsd);
            double mn = 1e6;
            unsigned low = 0;
            double sum = 0.0;
            for (unsigned t = 0; t < n; ++t) {
                const double d = __dsub_rn(total_jsd, staged ? ent_smem[t] : mdv[t]);
                if (staged) ent_smem[t] = d; else mdv[t] = d;
                if (d < mn) {
                    mn = d;
                    low = t;
                }
                sum = __dadd_rn(sum, d);
            }
            const double mean = __ddiv_rn(sum, nd);
            double ss = 0.0;
            for (unsigned t = 0; t < n; ++t) {
                const double d = __dsub_rn(staged ? ent_smem[t] : mdv[t], mean);
                ss = __dadd_rn(ss, __dmul_rn(d, d));
            }
            const double sd = __dsqrt_rn(__ddiv_rn(ss, __dsub_rn(nd, 1.0)));
            sc->lowest = low;
            sc->mean = mean;
            sc->stdv = sd;
            sc->cov = __ddiv_rn(sd, mean);
            sc->ticket = 0;
            sc->first_true = kNone;
            sc->first_panic = kNone;
            sc->first_unsure = kNone;
            sc->total_bound = 0.0;
            sc->std_bound = 0.0;
            sc->cov_bound = 0.0;
            sc->state_unsure = 0;
            sc->exact = 1;
        }
        if (staged) {
            __syncthreads();
            for (unsigned t = threadIdx.x; t < n; t += blockDim.x) mdelta[t] = ent_smem[t];
        }
    }
}

// increases_jsd for a window of candidates (records.rs:70-92); one CTA per position.  Sparse rows: the candidates
// are rows of the same source (candF unused).
template <class Src>
__global__ void __launch_bounds__(kEntThreads)
k_sel_scan(const Src src, const double* __restrict__ H, uint64_t dim, const double* __restrict__ S,
           const unsigned* __restrict__ members, SelScal* sc, const double* __restrict__ candF,
           const double* __restrict__ candH, const uint8_t* __restrict__ cand_valid,
           const uint8_t* __restrict__ is_member, const unsigned* __restrict__ order, unsigned pos0,
           double* __restrict__ delta_out) {
    extern __shared__ __align__(16) double ent_smem[];
    const unsigned pos = pos0 + blockIdx.x;
    const unsigned row = order ? order[pos] : pos;
    if (cand_valid && !cand_valid[row]) return;     // Err("No valid k-mers") -> skipped
    if (is_member && is_member[row]) return;        // seqid already in the set -> false
    const unsigned n = sc->n;
    const double nd = (double)n;
    const unsigned low_row = members[sc->lowest];
    auto v = src.view(exact_stage_smem<Src>(ent_smem));
    const auto fl = v.row(0, low_row, dim);
    const auto fc = v.cand_row(candF, 1, row, dim);
    EntropyResult h = block_entropy_exact(
        dim, [&](uint64_t i) { return __ddiv_rn(__dadd_rn(__dsub_rn(S[i], fl[i]), fc[i]), nd); }, ent_smem, stager(v));
    if (threadIdx.x == 0) {
        const double mean_entropy = __ddiv_rn(__dadd_rn(__dsub_rn(sc->E, H[low_row]), candH[row]), nd);
        const double d = __dsub_rn(h.e, mean_entropy);
        if (delta_out) delta_out[blockIdx.x] = d;
        if (entropy_total_bad(h.t, dim)) atomicMin(&sc->first_panic, pos);
        if (d > __dadd_rn(sc->total_jsd, kEps)) atomicMin(&sc->first_true, pos);
    }
}

#include "select_shard.cuh"
#include "select_fast.cuh"
#include "select_grow.cuh"
#include "select_sm.cuh"

static_assert(8 * kFastThreads == (int)kSpLowBins, "a pass of the bounded-error kernels must be one bucket");

constexpr auto k_sel_persist_sm_full = k_sel_persist_sm_t<kFastThreads, 1, kSmMaxN, kSmChunk>;

// test hook: the two building blocks of block_entropy_ilp on arbitrary operands
__global__ void k_debug_fast_terms(const double* a, const double* b, double* m_out, double* l_out, int* sp_out, uint64_t n) {
    __shared__ double2 ltab[64];
    dvs_log2_stage_table(ltab);
    __syncthreads();
    const uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    const double m = div_exact(a[i], make_fast_div(b[i]));
    int sp = 0;
    const double l = dvs_log2_main(m, ltab, sp);
    m_out[i] = m;
    l_out[i] = l;
    sp_out[i] = sp;
}

__global__ void k_sel_set_dev(SelScal* sc, unsigned cursor, unsigned window, unsigned window_max, unsigned num,
                              unsigned accepts, unsigned which) {
    sc->cursor = cursor;
    sc->window = window;
    sc->window_max = window_max;
    sc->num = num;
    sc->accepts = accepts;
    sc->which = which;
    sc->halt = 0;
}

__global__ void k_set_members(uint8_t* is_member, const unsigned* members, unsigned n, uint8_t v) {
    unsigned i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) is_member[members[i]] = v;
}

static int panic_error(const SelScal& h) {
    if (h.panic == 2u) {
        set_error("dvs_select_sharded: a peer GPU did not answer an exchange within 20 s (a rank is missing or died)");
        return DVS_ERR_CUDA;
    }
    set_error("cannot calculate entropy as frequency vector total %.17g!=1.0", h.panic_total);
    return DVS_ERR_VALUE;
}

// The record set of dvs_select_sparse_sharded on one rank (DESIGN.md §5.13).  The per-record scalars of ALL
// records are gathered once per call and indexed by global (rank-major) row, as the kernels and read_flags expect.
// The rows are this rank's own (`local`) plus a cache of peer rows: the members of the set and the candidate being
// decided, copied in from their owner's window outbox.  `owned` (valid and held here) is the validity mask the
// candidate scans and the grow filter see, so each rank scores exactly the candidates whose rows it holds.
struct SparseShard {
    dvs_comm* comm = nullptr;
    const dvs_ksparse* local = nullptr;
    uint32_t nrec = 0, nb = 0;
    int k = 0;
    uint64_t dim = 0;
    std::vector<uint32_t> rank_base;  // [world + 1]: global row of each rank's first record
    std::vector<uint64_t> lens;       // slots of every record's region (its byte length)
    DevBuf<uint8_t> valid, err, owned;
    DevBuf<double> err_total, entropy;
    DevBuf<uint64_t> totals;
    // member-row cache: slot s holds one peer row in entries [s * slot_len, (s + 1) * slot_len) and bucket tables
    uint64_t slot_len = 0;
    mutable DevBuf<uint32_t> c_idx, c_cnt, c_bp, c_nnz;  // (allocated by the call once it knows the set's size)
    mutable DevBuf<uint64_t> c_off;
    DevBuf<uint32_t> where;
    uint64_t outbox = 0;  // heap offset of this rank's outbox in its window
    // host bookkeeping, identical on every rank (each step is taken on all ranks with the same arguments)
    mutable std::vector<uint32_t> h_where;
    mutable std::vector<unsigned> refs;  // references to each row: members (a row may repeat) + the candidate
    mutable std::vector<unsigned> free_slots;
    mutable uint32_t fetched = 0;
    mutable uint64_t fetched_bytes = 0;
    unsigned owner_of(unsigned row) const {
        return (unsigned)(std::upper_bound(rank_base.begin(), rank_base.end(), row) - rank_base.begin()) - 1u;
    }
};

// byte layout of one row in an outbox
struct ShardRowLayout {
    uint64_t cnt, bp, nnz, bytes;
};
static uint64_t ss_align(uint64_t b) { return (b + 255) & ~255ull; }
static ShardRowLayout shard_row_layout(uint64_t slot_len, uint32_t nb) {
    ShardRowLayout L;
    L.cnt = ss_align(slot_len * 4);
    L.bp = 2 * L.cnt;
    L.nnz = L.bp + ss_align((nb + 1ull) * 4);
    L.bytes = std::max<uint64_t>(L.nnz + ss_align((uint64_t)nb * 4), 256);
    return L;
}
// window bytes dvs_select_sparse_sharded needs (shard.window_bytes_for_sparse_select): control words + the larger
// of the staging of the per-record scalars (8 bytes a record at most) and the outbox of one row
static uint64_t shard_window_need(uint64_t nrec_total, uint64_t slot_len, uint32_t nb) {
    return kCommCtrlBytes + std::max(std::max<uint64_t>(ss_align(nrec_total * 8), 256), shard_row_layout(slot_len, nb).bytes);
}

// the device row source of a record set, and the candidate rows k_sel_scan reads besides it
inline DenseRows row_source(const dvs_kfreqs* f) { return DenseRows{f->freqs.p}; }
inline SparseRows row_source(const dvs_ksparse* sp) {
    return SparseRows{{{sp->idx.p, sp->cnt.p, sp->bucket_ptr.p, sp->bucket_nnz.p, sp->offsets.p, sp->totals.p, sp->nb}}};
}
inline ShardRows row_source(const SparseShard* s) {
    const dvs_ksparse* l = s->local;
    ShardRows r;
    r.local = SparseRowsData{l->idx.p, l->cnt.p, l->bucket_ptr.p, l->bucket_nnz.p, l->offsets.p, l->totals.p, s->nb};
    r.cache = SparseRowsData{s->c_idx.p, s->c_cnt.p, s->c_bp.p, s->c_nnz.p, s->c_off.p, nullptr, s->nb};
    r.where = s->where.p;
    r.totals = s->totals.p;
    return r;
}
inline const double* cand_rows(const dvs_kfreqs* q) { return q->freqs.p; }
inline const double* cand_rows(const dvs_ksparse*) { return nullptr; }
inline const double* cand_rows(const SparseShard*) { return nullptr; }
// the validity mask of the candidates this GPU scores
inline const uint8_t* cand_valid(const dvs_kfreqs* q) { return q->valid.p; }
inline const uint8_t* cand_valid(const dvs_ksparse* q) { return q->valid.p; }
inline const uint8_t* cand_valid(const SparseShard* q) { return q->owned.p; }

// The launches of the host-driven rounds over one record set: RS is dvs_kfreqs (dense rows) or dvs_ksparse.
template <class RS>
struct Selector {
    using Src = decltype(row_source((const RS*)nullptr));
    dvs_ctx* ctx;
    const RS* f;
    uint64_t dim;
    cudaStream_t st;
    SelScal* h_sc;  // pinned

    Src rows() const { return row_source(f); }
    int read(SelState& s) {
        DVS_CUDA_TRY(cudaMemcpyAsync(h_sc, s.sc.p, sizeof(SelScal), cudaMemcpyDeviceToHost, st));
        DVS_CUDA_TRY(cudaStreamSynchronize(st));
        return DVS_OK;
    }
    // elementwise kernels (k_sel_sum, k_sel_replace_vec): 256 threads per 256 elements, or per bucket of a sparse row
    unsigned vec_grid() const {
        if constexpr (Src::kSparse) return f->nb;
        else return (unsigned)((dim + 255) / 256);
    }
    int reset_scan(SelState& s) {
        static_assert(offsetof(SelScal, first_panic) == offsetof(SelScal, first_true) + sizeof(unsigned), "layout");
        DVS_CUDA_TRY(cudaMemsetAsync((char*)s.sc.p + offsetof(SelScal, first_true), 0xFF, 2 * sizeof(unsigned), st));
        DVS_CUDA_TRY(cudaMemsetAsync((char*)s.sc.p + offsetof(SelScal, first_unsure), 0xFF, sizeof(unsigned), st));
        return DVS_OK;
    }
    int update_fast(SelState& s, unsigned n) {
        k_sel_update_fast<<<n + 1, kFastThreads, stage_bytes<Src>(1), st>>>(rows(), f->entropy.p, dim, s.S(), s.members(),
                                                                          s.mdelta.p, s.mbound.p, s.sc.p);
        DVS_LAUNCHED(ctx);
        return DVS_OK;
    }
    int replace_fast(SelState& s, unsigned n, unsigned cand_row, uint8_t* is_member) {
        k_sel_replace_update_fast<<<n + 1, kFastThreads, stage_bytes<Src>(3), st>>>(
            rows(), f->entropy.p, dim, s.S(), s.S_other(), s.members(), s.members_other(), is_member, s.mdelta.p,
            s.mbound.p, s.sc.p, cand_row);
        DVS_LAUNCHED(ctx);
        s.flip();
        return DVS_OK;
    }
    // (first_true / first_unsure are re-armed by every update kernel and stay armed after an empty
    // window; the caller resets them explicitly after an exact single-candidate scan)
    int scan_fast(SelState& s, const uint8_t* is_member, const unsigned* d_order, unsigned pos0, unsigned count) {
        k_sel_scan_fast<<<count, kFastThreads, stage_bytes<Src>(2), st>>>(rows(), f->entropy.p, dim, s.S(), s.members(),
                                                                        s.sc.p, cand_valid(f), is_member, d_order, pos0);
        DVS_LAUNCHED(ctx);
        return DVS_OK;
    }
    // one candidate row of another kfreqs object, no order / validity / membership filters
    int scan_raw(SelState& s, const double* candF, const double* candH, unsigned row, double* delta_out) {
        DVS_TRY(reset_scan(s));
        k_sel_scan<<<1, kEntThreads, kEntSmemBytes, st>>>(rows(), f->entropy.p, dim, s.S(), s.members(), s.sc.p, candF,
                                                           candH, nullptr, nullptr, nullptr, row, delta_out);
        DVS_LAUNCHED(ctx);
        return DVS_OK;
    }

    // SummedRecords::new over `members` (+ optional pushed row): sums, then total_jsd + member deltas
    int sum(SelState& s, const unsigned* d_members, unsigned n, int extra_row) {
        k_sel_sum<<<vec_grid(), 256, 0, st>>>(rows(), f->entropy.p, dim, d_members, n, extra_row, s.S(), s.members(),
                                              s.sc.p);
        DVS_LAUNCHED(ctx);
        return DVS_OK;
    }
    int build(SelState& s, const unsigned* d_members, unsigned n, int extra_row) {
        DVS_TRY(sum(s, d_members, n, extra_row));
        return update(s, n + (extra_row >= 0 ? 1u : 0u));
    }
    // fast SummedRecords::new (+ optional pushed row): exact sums, bounded-error total / deltas / stats
    int build_fast(SelState& s, const unsigned* d_members, unsigned n, int extra_row) {
        DVS_TRY(sum(s, d_members, n, extra_row));
        return update_fast(s, n + (extra_row >= 0 ? 1u : 0u));
    }
    int update(SelState& s, unsigned n) {
        k_sel_update<<<n + 1, kEntThreads, kEntSmemBytes + stage_bytes<Src>(1), st>>>(rows(), f->entropy.p, dim, s.S(),
                                                                                     s.members(), s.mdelta.p, s.sc.p);
        DVS_LAUNCHED(ctx);
        return DVS_OK;
    }
    int replace(SelState& s, unsigned n, unsigned cand_row, uint8_t* is_member) {
        k_sel_replace_vec<<<vec_grid(), 256, stage_bytes<Src>(2), st>>>(rows(), f->entropy.p, dim, s.members(), is_member,
                                                                        s.sc.p, cand_row, s.S());
        DVS_LAUNCHED(ctx);
        return update(s, n);
    }
    int scan(SelState& s, const RS* q, const uint8_t* is_member, const unsigned* d_order, unsigned pos0,
             unsigned count, double* delta_out) {
        DVS_TRY(reset_scan(s));  // re-arm the min-index reduction
        k_sel_scan<<<count, kEntThreads, kEntSmemBytes + stage_bytes<Src>(2), st>>>(
            rows(), f->entropy.p, dim, s.S(), s.members(), s.sc.p, cand_rows(q), q->entropy.p, cand_valid(q), is_member,
            d_order, pos0, delta_out);
        DVS_LAUNCHED(ctx);
        return DVS_OK;
    }
};

// The sparse forms stage up to 48 KB of rows on top of their own shared memory
static int sparse_smem_setup() {
    auto allow = [](auto kernel, size_t bytes) {
        return cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
    };
    cudaError_t e = cudaSuccess;
    for (cudaError_t x : {allow(k_sel_scan_fast<SparseRows>, 2 * kStageBytes), allow(k_sel_update_fast<SparseRows>, kStageBytes),
                          allow(k_sel_replace_update_fast<SparseRows>, 3 * kStageBytes),
                          allow(k_grow_eval<SparseRows>, 2 * kStageBytes), allow(k_sel_replace_vec<SparseRows>, 2 * kStageBytes),
                          allow(k_sel_update<SparseRows>, kEntSmemBytes + kStageBytes),
                          allow(k_sel_scan<SparseRows>, kEntSmemBytes + 2 * kStageBytes),
                          allow(k_sel_scan_fast<ShardRows>, 2 * kStageBytes), allow(k_sel_update_fast<ShardRows>, kStageBytes),
                          allow(k_sel_replace_update_fast<ShardRows>, 3 * kStageBytes),
                          allow(k_grow_eval<ShardRows>, 2 * kStageBytes), allow(k_sel_replace_vec<ShardRows>, 2 * kStageBytes),
                          allow(k_sel_update<ShardRows>, kEntSmemBytes + kStageBytes),
                          allow(k_sel_scan<ShardRows>, kEntSmemBytes + 2 * kStageBytes)})
        if (x != cudaSuccess && e == cudaSuccess) e = x;
    if (e != cudaSuccess) {
        set_error("dvs_select_sparse: shared memory for the staged rows: %s", cudaGetErrorString(e));
        return DVS_ERR_CUDA;
    }
    return DVS_OK;
}

// One selection call: its arguments, the state and buffers on the device, and where the loop stands.  Each step
// of the loop in select_core is a function of its own below.  RS: the record set (dvs_kfreqs or dvs_ksparse).
template <class RS>
struct SelRun {
    using Src = typename Selector<RS>::Src;
    dvs_ctx* ctx;
    dvs_comm* comm;
    const RS* f;
    const uint32_t* order;
    uint32_t num;
    int mode;
    uint32_t min_size, max_size;
    uint32_t* sel_idx;
    double* sel_delta;
    double* stats5;
    uint32_t* size_out;
    const TrailArgs* trail;
    cudaStream_t st = nullptr;
    uint64_t dim = 0;
    unsigned world = 1, rank = 0;
    ShardArgs shard;
    bool grow_mode = false;  // max / max_cov: the set grows to max_size before candidates replace its lowest record
    bool use_fast = true;    // bounded-error kernels, exact evaluation only where they cannot decide
    // trailing (dvs_count_select): the rows are still being produced on another stream; positions below
    // `trail_limit` have been published
    unsigned trail_limit = 0;
    std::vector<uint8_t> valid, err;  // validity / panic flags of the records
    std::vector<double> err_total;
    Selector<RS> sel;
    SelState A, B;
    SelState* cur = &A;
    SelState* alt = &B;
    unsigned cap = 0, n = 0;
    DevBuf<uint8_t> is_member;
    DevBuf<unsigned> d_order, d_init;
    std::optional<PhaseTimer> pt;
    unsigned cursor = 0, accepts = 0, exact_evals = 0;
    unsigned window = 64, window_max = 64;  // adaptive: grows while windows come back empty, shrinks after a hit
    // persistent rounds
    bool use_persist = false, sm_ok = false;
    unsigned persist_grid = 0, sm_grid = 0;
    DevBuf<SlicePart> d_slparts;  // k_sel_persist: partial sums of sliced vectors and their arrival tickets
    DevBuf<unsigned> d_slticks;
    DevBuf<SmPart> d_spart, d_upart, d_dpart;
    // batched grow attempts (see k_grow_eval)
    bool use_grow_batch = false;
    unsigned grow_window_max = 64, grow_window = 16;
    SelState fresh;  // clone(): the members re-summed in order (S, E), refreshed whenever the set changes
    DevBuf<FastSum> d_gparts;
    DevBuf<double> d_gmd, d_gmb;
    DevBuf<SelScal> d_gscratch;
    DevBuf<unsigned> d_ginteresting;
    bool fresh_valid = false;
    unsigned fresh_n = 0;
    const SelState* fresh_of = nullptr;
    int fresh_which = -1;
    bool single_candidate = false;  // the grow filter has already isolated the candidate at `cursor`
    // while the set grows at almost every candidate (e.g. cov right after the start) the filter skips
    // nothing: after two such windows in a row it is bypassed for 1, 2, 4, 8 candidates
    unsigned filter_streak = 0, filter_bypass = 0;
};

// trailing: wait until every record has been counted
template <class RS>
static int wait_counted(SelRun<RS>& r) {
    if (r.trail_limit >= r.num) return DVS_OK;
    DVS_CUDA_TRY(cudaStreamWaitEvent(r.st, r.trail->count_done, 0));
    r.trail_limit = r.num;
    return DVS_OK;
}

// ---- dvs_select_sparse_sharded: rows stay with their owner (DESIGN.md §5.13) ------------------------------------
// Every rank runs the same host loop over the same replicated state; these steps are taken on all ranks with the same
// arguments, so the barriers and all-reduces below line up.
template <class RS>
constexpr bool kByOwner = std::is_same_v<RS, SparseShard>;
constexpr const char* kShardName = "dvs_select_sparse_sharded";

// device memory of the peer-row cache (cap + 1 slots) and of the gathered per-record scalars
template <class RS>
static uint64_t shard_bytes(const SelRun<RS>& r) {
    if constexpr (kByOwner<RS>) {
        const SparseShard& s = *r.f;
        return (r.cap + 1ull) * (s.slot_len * 2 * sizeof(uint32_t) + (2ull * s.nb + 1) * sizeof(uint32_t) + sizeof(uint64_t)) +
               (uint64_t)s.nrec * (3 * sizeof(uint8_t) + 3 * sizeof(double) + sizeof(uint32_t));
    } else {
        return 0;
    }
}

// every rank returns the worst status of any rank (a CUDA failure before a bad argument before a value error); a
// rank whose own status is the worst keeps its own message
static int agree_status(dvs_ctx* ctx, dvs_comm* c, int rc) {
    enum : uint32_t { kCuda = 0, kArg = 1, kValue = 2, kOk = 3 };
    const uint32_t mine = rc == DVS_OK ? kOk : rc == DVS_ERR_VALUE ? kValue : rc == DVS_ERR_ARG ? kArg : kCuda;
    uint32_t* h = reinterpret_cast<uint32_t*>(reinterpret_cast<char*>(ctx->pinned) + sizeof(SelScal) + 16);
    DevBuf<uint32_t> d;
    DVS_TRY(d.alloc(1));
    *h = mine;
    DVS_CUDA_TRY(cudaMemcpyAsync(d.p, h, sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    DVS_TRY(comm_barrier(ctx, c));
    DVS_TRY(comm_min_u32(ctx, c, d.p, d.p));
    DVS_CUDA_TRY(cudaMemcpyAsync(h, d.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    const uint32_t all = *h;
    DVS_TRY(comm_check_error(ctx, c, kShardName));
    if (all == kOk) return DVS_OK;
    if (all != mine)
        set_error("%s: the call failed on another rank (%s)", kShardName,
                  all == kValue ? "value error" : all == kArg ? "bad argument" : "CUDA error");
    return all == kValue ? DVS_ERR_VALUE : all == kArg ? DVS_ERR_ARG : DVS_ERR_CUDA;
}

// the scan results of this rank's candidates -> the first interesting positions over all ranks
template <class RS>
static int agree_scan(SelRun<RS>& r) {
    if constexpr (kByOwner<RS>) {
        char* sc = reinterpret_cast<char*>(r.cur->sc.p);
        for (size_t off : {offsetof(SelScal, first_true), offsetof(SelScal, first_panic), offsetof(SelScal, first_unsure)}) {
            uint32_t* w = reinterpret_cast<uint32_t*>(sc + off);
            DVS_TRY(comm_min_u32(r.ctx, r.comm, w, w));
        }
    }
    return DVS_OK;
}

// A row enters the state (a member of the initial set, a replacing candidate, a grow attempt).  Its owner copies it
// into its window outbox; every other rank pulls it into a free cache slot (fetch and replicate).  The first barrier
// means every rank has pulled the previous row, so the outbox may be overwritten; the second, that this row is in it.
// A cache slot is written only by its own rank, on its stream, so every kernel that read the slot's previous row has
// finished before the copy starts.
template <class RS>
static int take_row(SelRun<RS>& r, unsigned row) {
    if constexpr (kByOwner<RS>) {
        const SparseShard& s = *r.f;
        if (s.refs[row]++ > 0) return DVS_OK;  // already here (a row that repeats in the set)
        dvs_comm* c = s.comm;
        const unsigned owner = s.owner_of(row), me = (unsigned)c->rank;
        const uint64_t len = s.lens[row];
        const uint32_t nb = s.nb;
        const ShardRowLayout L = shard_row_layout(s.slot_len, nb);
        cudaStream_t st = r.st;
        DVS_TRY(comm_barrier(r.ctx, c));
        if (owner == me) {
            const dvs_ksparse* l = s.local;
            const uint32_t lr = row - s.rank_base[me];
            const uint64_t at = l->h_offsets[lr];
            uint8_t* ob = c->window + s.outbox;
            if (len) {
                DVS_CUDA_TRY(cudaMemcpyAsync(ob, l->idx.p + at, len * 4, cudaMemcpyDeviceToDevice, st));
                DVS_CUDA_TRY(cudaMemcpyAsync(ob + L.cnt, l->cnt.p + at, len * 4, cudaMemcpyDeviceToDevice, st));
            }
            DVS_CUDA_TRY(cudaMemcpyAsync(ob + L.bp, l->bucket_ptr.p + (size_t)lr * (nb + 1), (nb + 1ull) * 4,
                                         cudaMemcpyDeviceToDevice, st));
            DVS_CUDA_TRY(cudaMemcpyAsync(ob + L.nnz, l->bucket_nnz.p + (size_t)lr * nb, nb * 4ull, cudaMemcpyDeviceToDevice, st));
        }
        DVS_TRY(comm_barrier(r.ctx, c));
        if (owner != me) {
            if (s.free_slots.empty()) {
                set_error("%s: no free slot in the row cache for record %u", kShardName, row);
                return DVS_ERR_CUDA;
            }
            const unsigned slot = s.free_slots.back();
            s.free_slots.pop_back();
            const uint8_t* ob = c->peer[owner] + s.outbox;
            if (len) {
                DVS_CUDA_TRY(cudaMemcpyAsync(s.c_idx.p + slot * s.slot_len, ob, len * 4, cudaMemcpyDeviceToDevice, st));
                DVS_CUDA_TRY(cudaMemcpyAsync(s.c_cnt.p + slot * s.slot_len, ob + L.cnt, len * 4, cudaMemcpyDeviceToDevice, st));
            }
            DVS_CUDA_TRY(cudaMemcpyAsync(s.c_bp.p + (size_t)slot * (nb + 1), ob + L.bp, (nb + 1ull) * 4,
                                         cudaMemcpyDeviceToDevice, st));
            DVS_CUDA_TRY(cudaMemcpyAsync(s.c_nnz.p + (size_t)slot * nb, ob + L.nnz, nb * 4ull, cudaMemcpyDeviceToDevice, st));
            s.h_where[row] = kCachedRow | slot;
            DVS_CUDA_TRY(cudaMemcpyAsync(s.where.p + row, &s.h_where[row], sizeof(uint32_t), cudaMemcpyHostToDevice, st));
            ++s.fetched;
            s.fetched_bytes += len * 8 + (2ull * nb + 1) * 4;
        }
    }
    return DVS_OK;
}

// a row leaves the state (the replaced lowest member, a discarded grow candidate): its slot is free once nothing
// refers to it.  (where[] on the device keeps the old slot: a row that is neither member nor candidate is never read.)
template <class RS>
static void drop_row(SelRun<RS>& r, unsigned row) {
    if constexpr (kByOwner<RS>) {
        const SparseShard& s = *r.f;
        if (--s.refs[row] > 0) return;
        const uint32_t w = s.h_where[row];
        if (w != kAbsentRow && (w & kCachedRow)) {
            s.free_slots.push_back(w & ~kCachedRow);
            s.h_where[row] = kAbsentRow;
        }
    }
}

// the row of member `j` of the current state
template <class RS>
static int member_row(SelRun<RS>& r, unsigned j, unsigned& row) {
    unsigned* h = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(r.ctx->pinned) + sizeof(SelScal) + 16);
    DVS_CUDA_TRY(cudaMemcpyAsync(h, r.cur->members() + j, sizeof(unsigned), cudaMemcpyDeviceToHost, r.st));
    DVS_CUDA_TRY(cudaStreamSynchronize(r.st));
    row = *h;
    return DVS_OK;
}

// reads the validity / panic flags of the records.  Every record in `order` goes through KmerSeq::new ->
// entropy(), where a failing sum check panics: checked here for the positions below `upto`.
template <class RS>
static int read_flags(SelRun<RS>& r, unsigned upto) {
    const RS* f = r.f;
    if (f->nrec) {
        DVS_CUDA_TRY(cudaMemcpyAsync(r.valid.data(), f->valid.p, f->nrec, cudaMemcpyDeviceToHost, r.st));
        DVS_CUDA_TRY(cudaMemcpyAsync(r.err.data(), f->err.p, f->nrec, cudaMemcpyDeviceToHost, r.st));
        DVS_CUDA_TRY(cudaMemcpyAsync(r.err_total.data(), f->err_total.p, f->nrec * sizeof(double),
                                     cudaMemcpyDeviceToHost, r.st));
        DVS_CUDA_TRY(cudaStreamSynchronize(r.st));
    }
    for (uint32_t i = 0; i < upto; ++i)
        if (r.valid[r.order[i]] && r.err[r.order[i]]) {
            set_error("cannot calculate entropy as frequency vector total %.17g!=1.0", r.err_total[r.order[i]]);
            return DVS_ERR_VALUE;
        }
    return DVS_OK;
}

// Sparse rows: the selection state is dense (S double buffered, 4^k f64 each), and `max` keeps two more copies for
// the grown set and clone().  Fail with the sizes when they do not fit instead of on an allocation.  Memory that the
// stream-ordered pool holds but does not use counts as free.
template <class RS>
static int sparse_state_fits(SelRun<RS>& r) {
    const bool grow = r.grow_mode;
    const uint64_t per = 2 * (r.dim * sizeof(double) + (uint64_t)r.cap * (sizeof(unsigned) + 2 * sizeof(double)));
    const uint64_t need = per * (grow ? 3u : 1u) + (uint64_t)r.f->nrec + (uint64_t)r.num * sizeof(unsigned) +
                          (grow ? (uint64_t)r.grow_window_max * r.cap * (sizeof(FastSum) + 2 * sizeof(double)) : 0u) +
                          shard_bytes(r);
    size_t free_b = 0, total_b = 0;
    DVS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    uint64_t avail = free_b;
    cudaMemPool_t pool;
    if (cudaDeviceGetDefaultMemPool(&pool, r.ctx->device) == cudaSuccess) {
        uint64_t reserved = 0, used = 0;
        if (cudaMemPoolGetAttribute(pool, cudaMemPoolAttrReservedMemCurrent, &reserved) == cudaSuccess &&
            cudaMemPoolGetAttribute(pool, cudaMemPoolAttrUsedMemCurrent, &used) == cudaSuccess && reserved > used)
            avail += reserved - used;
    }
    (void)cudaGetLastError();
    if (need + (64ull << 20) > avail) {
        set_error("dvs_select_sparse: the selection state at k=%d needs %.1f MB of device memory (%s%s), %.1f MB are free",
                  r.f->k, need / 1e6, grow ? "max: three double-buffered 4^k f64 sums" : "a double-buffered 4^k f64 sum",
                  shard_bytes(r) ? ", the peer-row cache and every record's scalars" : "", avail / 1e6);
        return DVS_ERR_CUDA;
    }
    return DVS_OK;
}

// after the argument checks: the memory check and the cache on every rank (all fail together), then the rows of the
// initial set
static int shard_prepare(SelRun<SparseShard>& r, const std::vector<unsigned>& init) {
    const SparseShard& s = *r.f;
    const unsigned slots = r.cap + 1;
    int rc = sparse_state_fits(r);
    if (rc == DVS_OK) rc = s.c_idx.alloc((size_t)slots * s.slot_len);
    if (rc == DVS_OK) rc = s.c_cnt.alloc((size_t)slots * s.slot_len);
    if (rc == DVS_OK) rc = s.c_bp.alloc((size_t)slots * (s.nb + 1));
    if (rc == DVS_OK) rc = s.c_nnz.alloc((size_t)slots * s.nb);
    if (rc == DVS_OK) rc = s.c_off.alloc(slots);
    if (rc == DVS_OK) {
        std::vector<uint64_t> off(slots);
        for (unsigned q = 0; q < slots; ++q) off[q] = (uint64_t)q * s.slot_len;
        if (cudaMemcpyAsync(s.c_off.p, off.data(), slots * sizeof(uint64_t), cudaMemcpyHostToDevice, r.st) != cudaSuccess ||
            cudaStreamSynchronize(r.st) != cudaSuccess) {
            set_error("%s: setting up the row cache failed", kShardName);
            rc = DVS_ERR_CUDA;
        }
    }
    s.free_slots.clear();
    for (unsigned q = slots; q-- > 0;) s.free_slots.push_back(q);
    DVS_TRY(agree_status(r.ctx, r.comm, rc));
    for (unsigned row : init) DVS_TRY(take_row(r, row));
    return DVS_OK;
}

// argument checks, the panic check over the published positions, the initial set and its state, the buffers,
// and the round forms this call can use
template <class RS>
static int select_setup(SelRun<RS>& r) {
    dvs_ctx* ctx = r.ctx;
    const RS* f = r.f;
    const uint32_t* order = r.order;
    const uint32_t num = r.num;
    if (!ctx || !f || (!order && num) || !r.size_out) {
        set_error("dvs_select: NULL argument");
        return DVS_ERR_ARG;
    }
    if (r.mode < DVS_MODE_NMOST || r.mode > DVS_MODE_MAX_COV) {
        set_error("dvs_select: bad mode %d", r.mode);
        return DVS_ERR_ARG;
    }
    ctx->last_accepts = 0;
    ctx->last_trail_accepts = 0;
    ctx->last_trail_launches = 0;
    ctx->last_trail_sms = 0xFFFFFFFFu;
    if (num < r.min_size) {  // records.rs:323-325, :404-410
        set_error("The number of sequences %u is < n %u", num, r.min_size);
        return DVS_ERR_VALUE;
    }
    if (r.mode == DVS_MODE_NMOST) r.max_size = r.min_size;
    if (!(num > r.max_size)) r.max_size = num;  // records.rs:412-416
    for (uint32_t i = 0; i < num; ++i)
        if (order[i] >= f->nrec) {
            set_error("dvs_select: order[%u]=%u out of range (nrec=%u)", i, order[i], f->nrec);
            return DVS_ERR_ARG;
        }
    DVS_CUDA_TRY(dvs::enter(ctx));
    r.st = ctx->stream;
    r.dim = f->dim;
    dvs_comm* comm = r.comm;
    r.world = comm ? (unsigned)comm->world : 1u;
    r.rank = comm ? (unsigned)comm->rank : 0u;
    memset(&r.shard, 0, sizeof r.shard);
    r.shard.rank = (int)r.rank;
    r.shard.world = (int)r.world;
    for (unsigned q = 0; q < r.world && comm; ++q) r.shard.xbase[q] = comm->peer[q];
    if (r.world > 1) DVS_TRY(comm_barrier(ctx, comm));  // every rank is here: exchange slots of earlier calls are dead
    // trailing: start once the first chunk (>= min_size positions) is there
    r.trail_limit = num;
    if (r.trail) {
        DVS_CUDA_TRY(cudaStreamWaitEvent(r.st, r.trail->first_ready, 0));
        r.trail_limit = std::min(r.trail->limit0, num);
        if (r.mode != DVS_MODE_NMOST || r.trail_limit < r.min_size)  // nothing to gain / not enough rows yet
            DVS_TRY(wait_counted(r));
    }
    r.valid.resize(f->nrec);
    r.err.resize(f->nrec);
    r.err_total.resize(f->nrec);
    DVS_TRY(read_flags(r, r.trail_limit));

    std::vector<unsigned> init;  // records.rs:299-305: first min_size records, failures dropped
    for (uint32_t i = 0; i < r.min_size; ++i)
        if (r.valid[order[i]]) init.push_back(order[i]);
    if (init.empty()) {
        set_error("records cannot be empty");  // records.rs:28-30
        return DVS_ERR_VALUE;
    }
    if (init.size() <= 1) {
        set_error("must have > 1 KmerSeq");  // records.rs:227-230
        return DVS_ERR_VALUE;
    }
    // (duplicates in the initial set: the reference's Vec keeps both rows; so does this one)

    r.grow_mode = (r.mode != DVS_MODE_NMOST);
    // max modes with max_size below the initial size (e.g. max_size < min_size, which only the reference's
    // CLI rejects, cli.py:311): `size == max_size` never holds, so the set keeps growing as in
    // records.rs:427-451 - every buffer is then sized for all `num` records
    const bool unbounded = r.grow_mode && r.max_size < (uint32_t)init.size();
    r.cap = (unbounded ? num : std::max<unsigned>(std::max(r.min_size, r.max_size), (unsigned)init.size())) + 1;
    r.n = (unsigned)init.size();
    if constexpr (kByOwner<RS>) DVS_TRY(shard_prepare(r, init));
    else if constexpr (SelRun<RS>::Src::kSparse) DVS_TRY(sparse_state_fits(r));
    DVS_TRY(r.A.alloc(r.dim, r.cap));
    if (r.grow_mode) DVS_TRY(r.B.alloc(r.dim, r.cap));
    DVS_TRY(r.is_member.alloc(f->nrec));
    DVS_TRY(r.d_order.alloc(num));
    DVS_TRY(r.d_init.alloc(init.size()));
    DVS_CUDA_TRY(cudaMemsetAsync(r.is_member.p, 0, f->nrec, r.st));
    DVS_CUDA_TRY(cudaMemcpyAsync(r.d_order.p, order, num * sizeof(unsigned), cudaMemcpyHostToDevice, r.st));
    DVS_CUDA_TRY(cudaMemcpyAsync(r.d_init.p, init.data(), init.size() * sizeof(unsigned), cudaMemcpyHostToDevice, r.st));
    k_set_members<<<(unsigned)((init.size() + 255) / 256), 256, 0, r.st>>>(r.is_member.p, r.d_init.p, r.n, 1);
    DVS_LAUNCHED(ctx);
    r.pt.emplace(ctx, DVS_PHASE_SELECT);
    r.sel = Selector<RS>{ctx, f, r.dim, r.st, (SelScal*)ctx->pinned};
    DVS_TRY(r.sel.build(*r.cur, r.d_init.p, r.n, -1));
    r.window_max = std::max(64u, (unsigned)ctx->sm_count * 12u);
    if constexpr (kByOwner<RS>) r.window_max *= r.world;  // each rank scores its share of the window
    r.cursor = r.min_size;
    // DVS_SELECT_EXACT_ONLY=1 disables the bounded-error fast path (tests compare both)
    const char* exact_env = getenv("DVS_SELECT_EXACT_ONLY");
    r.use_fast = !(exact_env && exact_env[0] == '1');

    // DVS_SELECT_PERSIST=0: host-driven rounds, =1: the global-state persistent kernel; default: SM-replicated
    // rounds when the state fits in shared memory.  Host-driven rounds also run where cooperative launches do not.
    // DVS_SELECT_GRID: CTAs of the persistent kernels (tests run several ranks on ONE GPU: their kernels must be
    // co-resident, so each takes a share of the SMs).  Sparse rows take the host-driven rounds: one evaluation of a
    // 4^12-element vector is far too long for a round of the persistent kernels to pay off.
    if constexpr (SelRun<RS>::Src::kSparse) {
        r.use_persist = r.sm_ok = false;
        DVS_TRY(sparse_smem_setup());
    } else {
    const char* grid_env = getenv("DVS_SELECT_GRID");
    const unsigned grid_cap = grid_env && atoi(grid_env) > 0 ? (unsigned)atoi(grid_env) : 0xFFFFFFFFu;
    const char* per_env = getenv("DVS_SELECT_PERSIST");
    int coop = 0, per_sm = 0, per_sm2 = 0;
    cudaDeviceGetAttribute(&coop, cudaDevAttrCooperativeLaunch, ctx->device);
    if (coop && cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, k_sel_persist, kFastThreads, 0) != cudaSuccess)
        per_sm = 0;
    r.use_persist = r.use_fast && coop && per_sm > 0 && !(per_env && per_env[0] == '0');
    r.persist_grid = std::min((unsigned)ctx->sm_count * (unsigned)std::min(per_sm, 2), std::max(1u, std::min(grid_cap, 0x7FFFFFFFu)));
    r.sm_ok = r.use_persist && !(per_env && per_env[0] == '1') && r.dim <= kSmMaxDim;
    if (r.sm_ok) {
        r.sm_ok = cudaFuncSetAttribute(k_sel_persist_sm_full, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                       (int)sizeof(SmShared)) == cudaSuccess &&
                  cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm2, k_sel_persist_sm_full, kFastThreads,
                                                                sizeof(SmShared)) == cudaSuccess &&
                  per_sm2 > 0;
        (void)cudaGetLastError();
    }
    r.sm_grid = std::min(std::min<unsigned>((unsigned)ctx->sm_count, kSmMaxGrid), grid_cap);
    if (r.sm_ok) {
        DVS_TRY(r.d_spart.alloc(2 * kSmMaxGrid));
        DVS_TRY(r.d_upart.alloc(kSmMaxN + 1));
        DVS_TRY(r.d_dpart.alloc(3));  // the leader's broadcasts: scan decision (double buffered), update result
    }
    }
    // batched grow attempts (see k_grow_eval): scratch for a window of candidates; DVS_SELECT_GROW_BATCH=0
    // keeps one host-driven attempt per candidate
    const char* gb_env = getenv("DVS_SELECT_GROW_BATCH");
    r.use_grow_batch = r.use_fast && r.grow_mode && !(gb_env && gb_env[0] == '0');
    // (rows scored by their owner: the filter's windows stay those of one GPU, because where they end decides which
    // candidates the filter hands to the host path, and with that the exact evaluations)
    r.grow_window_max = kByOwner<RS> ? 64u : 64 * r.world;
    if (r.use_grow_batch && r.n != r.max_size) {
        DVS_TRY(r.fresh.alloc(r.dim, r.cap));
        DVS_TRY(r.d_gparts.alloc((size_t)r.grow_window_max * (r.cap + 3)));
        DVS_TRY(r.d_gmd.alloc((size_t)r.grow_window_max * r.cap));
        DVS_TRY(r.d_gmb.alloc((size_t)r.grow_window_max * r.cap));
        DVS_TRY(r.d_gscratch.alloc(r.grow_window_max));  // (indexed by the window offset)
        DVS_TRY(r.d_ginteresting.alloc(1));
    }
    return DVS_OK;
}

// max while the set grows: evaluate a window of grow attempts on the device and move the cursor to the first
// candidate that could be adopted (the host path then decides it), past the window when none can
template <class RS>
static int grow_filter(SelRun<RS>& r) {
    if (r.filter_bypass > 0) {
        --r.filter_bypass;
        r.single_candidate = true;  // straight to the host path for this candidate
        return DVS_OK;
    }
    dvs_ctx* ctx = r.ctx;
    const RS* f = r.f;
    SelState* cur = r.cur;
    const unsigned n = r.n, cursor = r.cursor, world = r.world;
    if (!r.fresh_valid || r.fresh_n != n || r.fresh_of != cur || r.fresh_which != cur->which) {
        DVS_TRY(r.sel.sum(r.fresh, cur->members(), n, -1));
        r.fresh_valid = true;
        r.fresh_n = n;
        r.fresh_of = cur;
        r.fresh_which = cur->which;
    }
    const unsigned W = std::min(r.grow_window, r.num - cursor);
    DVS_CUDA_TRY(cudaMemsetAsync(r.d_ginteresting.p, 0xFF, sizeof(unsigned), r.st));
    // candidate-sharded: this GPU evaluates the window candidates c with (cursor + c) % world == rank; with rows kept
    // by their owner, every candidate of the window whose row it holds (the mask cand_valid)
    const unsigned cw = kByOwner<RS> ? 1u : world;
    const unsigned gc0 = kByOwner<RS> ? 0u : (r.rank + world - cursor % world) % world;
    const unsigned Wloc = W > gc0 ? (W - gc0 + cw - 1) / cw : 0;
    if (Wloc) {
        k_grow_eval<<<dim3(n + 3, Wloc), kFastThreads, stage_bytes<typename SelRun<RS>::Src>(2), r.st>>>(
            r.sel.rows(), r.dim, cur->S(), cur->members(), cur->sc.p, r.fresh.S(), cand_valid(f), r.is_member.p, r.d_order.p,
            cursor, r.d_gparts.p, gc0, cw);
        DVS_LAUNCHED(ctx);
        k_grow_decide<<<Wloc, kFastThreads, 0, r.st>>>(f->entropy.p, r.dim, cur->members(), cur->sc.p, r.fresh.sc.p,
                                                       cand_valid(f), r.is_member.p, r.d_order.p, cursor, r.d_gparts.p,
                                                       r.d_gmd.p, r.d_gmb.p, r.cap, r.d_gscratch.p, r.d_ginteresting.p,
                                                       r.mode == DVS_MODE_MAX_COV ? 1 : 0, gc0, cw);
        DVS_LAUNCHED(ctx);
    }
    if (world > 1) DVS_TRY(comm_min_u32(ctx, r.comm, r.d_ginteresting.p, r.d_ginteresting.p));
    unsigned* h_fi = reinterpret_cast<unsigned*>(reinterpret_cast<char*>(ctx->pinned) + sizeof(SelScal));
    DVS_CUDA_TRY(cudaMemcpyAsync(h_fi, r.d_ginteresting.p, sizeof(unsigned), cudaMemcpyDeviceToHost, r.st));
    DVS_CUDA_TRY(cudaStreamSynchronize(r.st));
    const unsigned fi = *h_fi;
    if (fi == kNone) {  // the whole window was certainly rejected
        r.cursor += W;
        r.grow_window = std::min(r.grow_window * 2u, r.grow_window_max);
        return DVS_OK;
    }
    r.grow_window = std::max(4u, std::min(r.grow_window_max, 2u * (fi - cursor + 1u)));
    if (fi == cursor) {
        if (++r.filter_streak >= 2) r.filter_bypass = 1u << std::min(r.filter_streak - 2u, 3u);
    } else {
        r.filter_streak = 0;
    }
    r.cursor = fi;  // everything before it is certainly rejected; the host path takes this one
    r.single_candidate = true;
    return DVS_OK;
}

// DVS_SELECT_TRACE: CTA 0's phase timeline of the first rounds, appended as text to the file it names;
// DVS_SELECT_TRACE_ALL (SM-replicated kernel): every CTA's, raw u64 [256 rounds][8 slots][256 CTAs]
static int write_trace(const unsigned long long* d_trace, size_t len, bool all, bool use_sm, const char* path) {
    std::vector<unsigned long long> tr(len);
    DVS_CUDA_TRY(cudaMemcpy(tr.data(), d_trace, len * sizeof(unsigned long long), cudaMemcpyDeviceToHost));
    if (all) {
        if (FILE* fp = fopen(path, "wb")) {
            fwrite(tr.data(), sizeof(unsigned long long), len, fp);
            fclose(fp);
        }
        return DVS_OK;
    }
    if (FILE* fp = fopen(path, "a")) {
        const int slots = use_sm ? kSmTraceSlots : 4, used = use_sm ? 7 : 4;
        fprintf(fp, use_sm ? "# round scan_ns gather_ns decide_ns update_ns gather2_ns finalize_ns next_ns (CTA 0)\n"
                           : "# round scan_ns wait1_ns update_ns wait2_ns (CTA 0; wait = grid barrier incl. the slowest CTA)\n");
        for (int q = 0; (q + 1) * slots < 2048 && tr[slots * (q + 1)]; ++q) {
            fprintf(fp, "%d", q);
            for (int p = 0; p + 1 < used; ++p) fprintf(fp, " %llu", tr[slots * q + p + 1] - tr[slots * q + p]);
            fprintf(fp, " %llu\n", tr[slots * (q + 1)] - tr[slots * q + used - 1]);
        }
        fclose(fp);
    }
    return DVS_OK;
}

// every remaining replacing round in one launch, until the rounds finish or halt for the host (`halted`: an
// undecided candidate or state, which the host resolves exactly).  The SM-replicated kernel runs while the state
// fits its shared memory, k_sel_persist otherwise.  Trailing the counting, the SM-replicated kernel takes
// DVS_TRAIL_SMS whole SMs and returns when everything has been published; anything else waits for the counting.
template <class RS>
static int persist_rounds(SelRun<RS>& r, bool& halted) {
    dvs_ctx* ctx = r.ctx;
    const RS* f = r.f;
    SelState* cur = r.cur;
    const unsigned world = r.world;
    const bool use_sm = r.sm_ok && r.n <= kSmMaxN;
    const bool trailing = r.trail_limit < r.num && use_sm && world == 1;
    if (!trailing) DVS_TRY(wait_counted(r));
    const unsigned grid = trailing ? std::min(r.sm_grid, trail_sms(ctx->sm_count)) : (use_sm ? r.sm_grid : r.persist_grid);
    k_sel_set_dev<<<1, 1, 0, r.st>>>(cur->sc.p, r.cursor, std::min(r.window, grid * world), grid * world, r.num,
                                     r.accepts, (unsigned)cur->which);
    if (r.comm) {
        r.shard.tag_base = (unsigned)((++r.comm->sel_tag_base) << 20);
        DVS_TRY(comm_host_rendezvous(ctx, r.comm));  // (ranks sharing one GPU only)
    }
    DVS_LAUNCHED(ctx);
    const double* a_F = f->freqs.p;
    const double* a_H = f->entropy.p;
    uint64_t a_dim = r.dim;
    double *a_S0 = cur->Sbuf[0].p, *a_S1 = cur->Sbuf[1].p;
    unsigned *a_M0 = cur->membuf[0].p, *a_M1 = cur->membuf[1].p;
    uint8_t* a_mem = r.is_member.p;
    double *a_md = cur->mdelta.p, *a_mb = cur->mbound.p;
    SelScal* a_sc = cur->sc.p;
    const uint8_t* a_valid = f->valid.p;
    const unsigned* a_order = r.d_order.p;
    unsigned a_rounds = world > 1 ? 0xFFFF0u : 0x7fffffffu;  // (exchange tags of one launch are 20 bits)
    unsigned long long* a_trace = nullptr;
    DevBuf<unsigned long long> d_trace;
    const char* tr_env = getenv("DVS_SELECT_TRACE");
    const char* tra_env = getenv("DVS_SELECT_TRACE_ALL");
    int a_trace_all = (use_sm && tra_env && tra_env[0]) ? 1 : 0;
    const char* trace_path = a_trace_all ? tra_env : (tr_env && tr_env[0] ? tr_env : nullptr);
    const size_t trace_len = a_trace_all ? (size_t)256 * kSmTraceSlots * kSmMaxGrid : 2048;
    if (trace_path) {
        DVS_TRY(d_trace.alloc(trace_len));
        DVS_CUDA_TRY(cudaMemsetAsync(d_trace.p, 0, trace_len * sizeof(unsigned long long), r.st));
        a_trace = d_trace.p;
    }
    if (use_sm) {
        unsigned a_dim32 = (unsigned)r.dim;
        double* a_S = cur->S();
        unsigned* a_M = cur->members();
        SmPart *a_sp = r.d_spart.p, *a_up = r.d_upart.p, *a_dp = r.d_dpart.p;
        DVS_CUDA_TRY(cudaMemsetAsync(r.d_dpart.p, 0, 3 * sizeof(SmPart), r.st));
        // exchange tags restart at 1 in every launch
        DVS_CUDA_TRY(cudaMemsetAsync(r.d_spart.p, 0, 2 * kSmMaxGrid * sizeof(SmPart), r.st));
        DVS_CUDA_TRY(cudaMemsetAsync(r.d_upart.p, 0, (kSmMaxN + 1) * sizeof(SmPart), r.st));
        const unsigned* a_ready = trailing ? r.trail->d_ready : nullptr;
        unsigned a_limit0 = r.trail_limit;
        if (trailing) {
            if (!ctx->stream_hi) {
                int lo_p = 0, hi_p = 0;
                DVS_CUDA_TRY(cudaDeviceGetStreamPriorityRange(&lo_p, &hi_p));
                DVS_CUDA_TRY(cudaStreamCreateWithPriority(&ctx->stream_hi, cudaStreamNonBlocking, hi_p));
                DVS_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_hi_in, cudaEventDisableTiming));
                DVS_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_hi_out, cudaEventDisableTiming));
            }
            // 512 threads x 128 registers: one CTA fills an SM's register file, so these CTAs take whole SMs - the
            // ones the counting CTAs of the launch in flight leave when it ends (the higher stream priority puts them
            // ahead of the next counting launch's CTAs)
            DVS_CUDA_TRY(cudaEventRecord(ctx->ev_hi_in, r.st));
            DVS_CUDA_TRY(cudaStreamWaitEvent(ctx->stream_hi, ctx->ev_hi_in, 0));
            k_sel_persist_sm_full<<<grid, kFastThreads, sizeof(SmShared), ctx->stream_hi>>>(
                a_F, a_H, a_dim32, a_S, a_M, a_mem, a_md, a_mb, a_sc, a_valid, a_order, a_sp, a_up, a_dp, a_trace,
                a_trace_all, r.shard, a_ready, a_limit0);
            DVS_CUDA_TRY(cudaGetLastError());
            DVS_CUDA_TRY(cudaEventRecord(ctx->ev_hi_out, ctx->stream_hi));
            DVS_CUDA_TRY(cudaStreamWaitEvent(r.st, ctx->ev_hi_out, 0));
        } else {
            void* args[] = {&a_F, &a_H, &a_dim32, &a_S, &a_M, &a_mem, &a_md, &a_mb, &a_sc, &a_valid, &a_order,
                            &a_sp, &a_up, &a_dp, &a_trace, &a_trace_all, &r.shard, &a_ready, &a_limit0};
            DVS_CUDA_TRY(cudaLaunchCooperativeKernel((void*)k_sel_persist_sm_full, dim3(grid), dim3(kFastThreads), args,
                                                     sizeof(SmShared), r.st));
        }
    } else {
        // DVS_SELECT_SLICES (A/B measurements): 0 = one CTA per candidate / member slot, 1 = candidates of a short
        // window are cut into slices (default), 2 = member slots of the update too (measured slower: a slice
        // repeats the slot's set-up and pays a fence + ticket, 55 us against 33 us per update at k = 8, n = 100)
        const char* sl_env = getenv("DVS_SELECT_SLICES");
        unsigned a_slice_mode = sl_env ? (unsigned)atoi(sl_env) : 1u;
        if (!r.d_slparts.p && a_slice_mode) {
            const size_t slots = std::max<size_t>(grid, (size_t)r.cap + 1);
            DVS_TRY(r.d_slparts.alloc(slots * kMaxSlices));
            DVS_TRY(r.d_slticks.alloc(slots));
            DVS_CUDA_TRY(cudaMemsetAsync(r.d_slticks.p, 0, slots * sizeof(unsigned), r.st));
        }
        SlicePart* a_parts = r.d_slparts.p;
        unsigned* a_ticks = r.d_slticks.p;
        void* args[] = {&a_F, &a_H, &a_dim, &a_S0, &a_S1, &a_M0, &a_M1, &a_mem, &a_md, &a_mb, &a_sc, &a_valid,
                        &a_order, &a_rounds, &a_trace, &r.shard, &a_parts, &a_ticks, &a_slice_mode};
        DVS_CUDA_TRY(cudaLaunchCooperativeKernel((void*)k_sel_persist, dim3(grid), dim3(kFastThreads), args, 0, r.st));
    }
    ctx->launches++;
    DVS_TRY(r.sel.read(*cur));
    if (a_trace) DVS_TRY(write_trace(a_trace, trace_len, a_trace_all, use_sm, trace_path));
    const SelScal hd = *r.sel.h_sc;
    if (hd.panic) return panic_error(hd);
    if (trailing) {
        ctx->last_trail_accepts += hd.accepts - r.accepts;
        ++ctx->last_trail_launches;
        std::vector<unsigned> smid(grid);
        DVS_CUDA_TRY(cudaMemcpyAsync(smid.data(), r.trail->d_ready + kTrailSmidOff, grid * sizeof(unsigned),
                                     cudaMemcpyDeviceToHost, r.st));
        DVS_CUDA_TRY(cudaStreamSynchronize(r.st));
        std::sort(smid.begin(), smid.end());
        const unsigned distinct = (unsigned)(std::unique(smid.begin(), smid.end()) - smid.begin());
        ctx->last_trail_sms = std::min(ctx->last_trail_sms, distinct);
        r.trail_limit = std::max(r.trail_limit, std::min(hd.limit, r.num));
    }
    r.cursor = hd.cursor;
    r.window = hd.window;
    r.accepts = hd.accepts;
    cur->which = (int)hd.which;
    halted = hd.halt != 0;
    if (halted) DVS_TRY(r.sel.reset_scan(*cur));
    return DVS_OK;
}

// one host-driven round: score a window of candidates, decide undecided candidates and states exactly, and let
// the first acceptance replace the lowest record (records.rs:111-118).  While the set grows (max), the accepted
// candidate is left in `grow_row` for grow_attempt instead, with the scan's scalars in `h`.
template <class RS>
static int host_window(SelRun<RS>& r, int& grow_row, SelScal& h) {
    const RS* f = r.f;
    SelState* cur = r.cur;
    grow_row = -1;
    if (!r.use_persist || r.cursor >= r.trail_limit) DVS_TRY(wait_counted(r));  // (host rounds do not trail)
    const unsigned count = r.single_candidate ? 1u : std::min(r.window, r.trail_limit - r.cursor);
    r.single_candidate = false;
    unsigned pos = kNone;
    if (r.use_fast) {
        DVS_TRY(r.sel.scan_fast(*cur, r.is_member.p, r.d_order.p, r.cursor, count));
        DVS_TRY(agree_scan(r));
        DVS_TRY(r.sel.read(*cur));
        h = *r.sel.h_sc;
        if (h.panic) return panic_error(h);
        if (h.state_unsure) {
            // the last fast update could not certify lowest_index / a sum check: redo it exactly and
            // re-score the window against the now certain state
            DVS_TRY(r.sel.update(*cur, r.n));
            ++r.exact_evals;
            return DVS_OK;
        }
        if (h.first_unsure < h.first_true) {
            // an undecided candidate comes before the first certain acceptance: decide it exactly
            const unsigned pu = h.first_unsure;
            if (!h.exact) DVS_TRY(r.sel.update(*cur, r.n));
            DVS_TRY(r.sel.scan(*cur, f, r.is_member.p, r.d_order.p, pu, 1, nullptr));  // (decided by its owner)
            DVS_TRY(agree_scan(r));
            DVS_TRY(r.sel.read(*cur));
            h = *r.sel.h_sc;
            ++r.exact_evals;
            if (h.panic) return panic_error(h);
            if (h.first_panic == pu) {
                set_error("cannot calculate entropy as frequency vector total !=1.0 (candidate at position %u)", pu);
                return DVS_ERR_VALUE;
            }
            if (h.first_true != pu) {  // rejected by the exact evaluation: carry on after it
                DVS_TRY(r.sel.reset_scan(*cur));
                r.cursor = pu + 1;
                return DVS_OK;
            }
            pos = pu;
        } else if (h.first_true != kNone) {
            pos = h.first_true;
        }
    } else {
        DVS_TRY(r.sel.scan(*cur, f, r.is_member.p, r.d_order.p, r.cursor, count, nullptr));
        DVS_TRY(agree_scan(r));
        DVS_TRY(r.sel.read(*cur));
        h = *r.sel.h_sc;
        if (h.panic) return panic_error(h);
        if (h.first_panic != kNone && h.first_panic <= h.first_true) {
            set_error("cannot calculate entropy as frequency vector total !=1.0 (candidate at position %u)",
                      h.first_panic);
            return DVS_ERR_VALUE;
        }
        pos = h.first_true;
    }
    if (pos == kNone) {
        r.cursor += count;
        r.window = std::min(r.window * 2, r.window_max);
        return DVS_OK;
    }
    const unsigned row = r.order[pos];
    r.window = std::max(64u, std::min(r.window_max, 2 * (pos - r.cursor + 1)));
    r.cursor = pos + 1;
    if (r.grow_mode && r.n != r.max_size) {
        grow_row = (int)row;
        return DVS_OK;
    }
    unsigned low_row = 0;
    if constexpr (kByOwner<RS>) {
        DVS_TRY(take_row(r, row));
        DVS_TRY(member_row(r, h.lowest, low_row));
    }
    DVS_TRY(r.use_fast ? r.sel.replace_fast(*cur, r.n, row, r.is_member.p) : r.sel.replace(*cur, r.n, row, r.is_member.p));
    drop_row(r, low_row);
    ++r.accepts;
    return DVS_OK;
}

// records.rs:434-451: nw = clone(); nw.push(rec); keep whichever has the larger statistic.  First tried with the
// bounded-error kernels: the comparison is decided from them only when it holds for every admissible error;
// otherwise both states are evaluated by the exact kernel.  `h`: the scalars of the current state.
template <class RS>
static int grow_attempt(SelRun<RS>& r, unsigned row, SelScal h) {
    const bool use_cov = (r.mode == DVS_MODE_MAX_COV);
    auto adopt = [&]() -> int {
        std::swap(r.cur, r.alt);
        ++r.n;
        ++r.accepts;
        uint8_t one = 1;
        DVS_CUDA_TRY(cudaMemcpyAsync(r.is_member.p + row, &one, 1, cudaMemcpyHostToDevice, r.st));
        DVS_CUDA_TRY(cudaStreamSynchronize(r.st));
        return DVS_OK;
    };
    auto discard = [&]() -> int {
        drop_row(r, row);
        return r.sel.reset_scan(*r.cur);  // re-arm the min-index reduction of `cur`
    };
    DVS_TRY(take_row(r, row));
    if (r.use_fast && !h.state_unsure) {
        DVS_TRY(r.sel.build_fast(*r.alt, r.cur->members(), r.n, (int)row));
        DVS_TRY(r.sel.read(*r.alt));
        const SelScal hf = *r.sel.h_sc;
        if (hf.panic) return panic_error(hf);
        if (!hf.state_unsure) {
            const double sa_f = use_cov ? h.cov : h.stdv, ba = h.exact ? 0.0 : (use_cov ? h.cov_bound : h.std_bound);
            const double sb_f = use_cov ? hf.cov : hf.stdv, bb = use_cov ? hf.cov_bound : hf.std_bound;
            if (sb_f - bb > sa_f + ba) return adopt();
            if (sb_f + bb < sa_f - ba) return discard();
        }
    }
    if (r.use_fast) ++r.exact_evals;
    if (!h.exact) {
        DVS_TRY(r.sel.update(*r.cur, r.n));
        DVS_TRY(r.sel.read(*r.cur));
        h = *r.sel.h_sc;
        if (h.panic) return panic_error(h);
    }
    DVS_TRY(r.sel.build(*r.alt, r.cur->members(), r.n, (int)row));
    DVS_TRY(r.sel.read(*r.alt));
    const SelScal hb = *r.sel.h_sc;
    if (hb.panic) return panic_error(hb);
    const double sa = use_cov ? h.cov : h.stdv;
    const double sb = use_cov ? hb.cov : hb.stdv;
    if (sb > sa) return adopt();
    return discard();
}

// the panic check of the records that were not published when a trailing selection started, the exact
// re-evaluation of the final state (reported numbers are exact), and the copies out
template <class RS>
static int select_finish(SelRun<RS>& r) {
    dvs_ctx* ctx = r.ctx;
    if (r.trail) {
        DVS_CUDA_TRY(cudaStreamWaitEvent(r.st, r.trail->count_done, 0));
        DVS_TRY(read_flags(r, r.num));
    }
    DVS_TRY(r.sel.read(*r.cur));
    if (!r.sel.h_sc->exact || r.sel.h_sc->state_unsure) DVS_TRY(r.sel.update(*r.cur, r.n));
    ctx->last_exact_evals = r.exact_evals;
    DVS_TRY(r.sel.read(*r.cur));
    const SelScal h = *r.sel.h_sc;
    if (h.panic) return panic_error(h);
    if (r.sel_idx)
        DVS_CUDA_TRY(cudaMemcpyAsync(r.sel_idx, r.cur->members(), r.n * sizeof(unsigned), cudaMemcpyDeviceToHost, r.st));
    if (r.sel_delta)
        DVS_CUDA_TRY(cudaMemcpyAsync(r.sel_delta, r.cur->mdelta.p, r.n * sizeof(double), cudaMemcpyDeviceToHost, r.st));
    DVS_CUDA_TRY(cudaStreamSynchronize(r.st));
    if (r.stats5) {
        r.stats5[0] = h.total_jsd;
        r.stats5[1] = h.mean;
        r.stats5[2] = h.stdv;
        r.stats5[3] = h.cov;
        r.stats5[4] = h.E;
    }
    *r.size_out = r.n;
    ctx->last_accepts = r.accepts;
    if (r.world > 1) DVS_TRY(comm_check_error(ctx, r.comm, "dvs_select_sharded"));
    return DVS_OK;
}

// comm == nullptr: one GPU.  Otherwise every rank calls this with the same rows (a kfreqs made by
// dvs_count_kmers_sharded / dvs_kfreqs_allgather), the same order and the same arguments: the state and
// every host-side decision are replicated (identical inputs, identical kernels), while the windows of
// candidates are scored candidate-sharded with an all-reduce(min) of the first interesting position.
template <class RS>
static int select_core(dvs_ctx* ctx, dvs_comm* comm, const RS* f, const uint32_t* order, uint32_t num, int mode,
                       uint32_t min_size, uint32_t max_size, uint32_t* sel_idx, double* sel_delta, double* stats5,
                       uint32_t* size_out, const TrailArgs* trail = nullptr) {
    SelRun<RS> r{ctx, comm, f, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5, size_out, trail};
    DVS_TRY(select_setup(r));
    while (r.cursor < num) {
        const bool growing = r.grow_mode && r.n != r.max_size;  // max below its size: candidates join the set
        if (growing && r.use_grow_batch && !r.single_candidate) {
            DVS_TRY(grow_filter(r));  // batched grow attempts isolate the next candidate worth one
            continue;
        }
        if constexpr (!SelRun<RS>::Src::kSparse) {  // (sparse rows: host-driven rounds only)
            if (!growing && r.use_persist) {  // replacing rounds on the device, until they finish or halt
                bool halted = false;
                DVS_TRY(persist_rounds(r, halted));
                if (!halted) continue;
                if (r.cursor >= num) break;
            }
        }
        // host-driven: the rounds themselves without persistent kernels (DVS_SELECT_PERSIST=0, exact-only,
        // no cooperative launch), a halted round's exact decision, and every candidate of a growing set
        int grow_row = -1;
        SelScal h;
        DVS_TRY(host_window(r, grow_row, h));
        if (grow_row >= 0) DVS_TRY(grow_attempt(r, (unsigned)grow_row, h));
    }
    return select_finish(r);
}

int select_with_trail(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* order, uint32_t num, int mode, uint32_t min_size,
                      uint32_t max_size, uint32_t* sel_idx, double* sel_delta, double* stats5, uint32_t* size_out,
                      const TrailArgs* trail) {
    return select_core(ctx, nullptr, f, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5, size_out, trail);
}

}  // namespace dvs

using namespace dvs;

struct dvs_summed {
    int device = 0;
    const dvs_kfreqs* f = nullptr;
    SelState st;
    unsigned n = 0;
};

extern "C" {

int dvs_select(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* order, uint32_t num, int mode, uint32_t min_size,
               uint32_t max_size, uint32_t* sel_idx, double* sel_delta, double* stats5, uint32_t* size_out) {
    return select_core(ctx, nullptr, f, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5, size_out);
}

int dvs_select_sharded(dvs_ctx* ctx, dvs_comm* comm, const dvs_kfreqs* f_all, const uint32_t* order, uint32_t num,
                       int mode, uint32_t min_size, uint32_t max_size, uint32_t* sel_idx, double* sel_delta,
                       double* stats5, uint32_t* size_out) {
    if (!comm || !comm->connected) {
        set_error("dvs_select_sharded: the communicator is not connected");
        return DVS_ERR_ARG;
    }
    return select_core(ctx, comm->world > 1 ? comm : nullptr, f_all, order, num, mode, min_size, max_size, sel_idx,
                       sel_delta, stats5, size_out);
}

int dvs_select_sparse(dvs_ctx* ctx, const dvs_ksparse* sp, const uint32_t* order, uint32_t num, int mode,
                      uint32_t min_size, uint32_t max_size, uint32_t* sel_idx, double* sel_delta, double* stats5,
                      uint32_t* size_out) {
    if (sp && !sp->has_entropy) {
        set_error("dvs_select_sparse: the rows were counted without entropies (dvs_count_kmers_sparse with want_entropy = 0)");
        return DVS_ERR_ARG;
    }
    if (sp && sp->dim % kSpLowBins != 0) {
        set_error("dvs_select_sparse: 4^k = %llu is not a whole number of %u-bin buckets", (unsigned long long)sp->dim,
                  kSpLowBins);
        return DVS_ERR_ARG;
    }
    return select_core(ctx, nullptr, sp, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5, size_out);
}

int dvs_select_sparse_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_ksparse* local, const uint32_t* nrec_per_rank,
                              const uint32_t* order, uint32_t num, int mode, uint32_t min_size, uint32_t max_size,
                              uint32_t* sel_idx, double* sel_delta, double* stats5, uint32_t* size_out) {
    if (ctx) {
        ctx->last_rows_fetched = 0;
        ctx->last_bytes_fetched = 0;
    }
    if (!ctx || !c || !local || !nrec_per_rank || !c->connected) {
        set_error("%s: bad argument / communicator not connected", kShardName);
        return DVS_ERR_ARG;
    }
    if (c->world == 1)
        return dvs_select_sparse(ctx, local, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5, size_out);
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    const int W = c->world, me = c->rank;
    // 1. what every rank tells the others; the checks below see the same data everywhere, so all return the same status
    struct Meta {
        uint64_t nrec, k, has_entropy, max_len, npr[kCommMaxWorld];
    };
    std::vector<Meta> m(W);
    {
        Meta x;
        memset(&x, 0, sizeof x);
        x.nrec = local->nrec;
        x.k = (uint64_t)local->k;
        x.has_entropy = (local->has_entropy || local->nrec == 0) ? 1 : 0;  // (no records: no entropy pass to ask for)
        for (uint32_t q = 0; q < local->nrec; ++q)
            x.max_len = std::max(x.max_len, local->h_offsets[q + 1] - local->h_offsets[q]);
        for (int q = 0; q < W; ++q) x.npr[q] = nrec_per_rank[q];
        DevBuf<Meta> d_in, d_all;
        DVS_TRY(d_in.alloc(1));
        DVS_TRY(d_all.alloc(W));
        DVS_CUDA_TRY(cudaMemcpyAsync(d_in.p, &x, sizeof x, cudaMemcpyHostToDevice, st));
        std::vector<uint64_t> bytes(W, sizeof(Meta));
        DVS_TRY(dvs_comm_allgatherv(ctx, c, d_in.p, bytes.data(), d_all.p));
        DVS_CUDA_TRY(cudaMemcpyAsync(m.data(), d_all.p, W * sizeof(Meta), cudaMemcpyDeviceToHost, st));
        DVS_CUDA_TRY(cudaStreamSynchronize(st));
    }
    SparseShard s;
    s.comm = c;
    s.local = local;
    s.k = local->k;
    s.dim = local->dim;
    s.nb = local->nb;
    s.rank_base.assign(W + 1, 0);
    uint64_t n64 = 0;
    for (int r = 0; r < W; ++r) {
        if (!m[r].has_entropy) {
            set_error("%s: rank %d counted its rows without entropies (dvs_count_kmers_sparse with want_entropy = 0)",
                      kShardName, r);
            return DVS_ERR_ARG;
        }
        if (m[r].k != m[0].k) {
            set_error("%s: rank %d counted k=%llu, rank 0 k=%llu", kShardName, r, (unsigned long long)m[r].k,
                      (unsigned long long)m[0].k);
            return DVS_ERR_ARG;
        }
        for (int q = 0; q < W; ++q)
            if (m[q].npr[r] != m[r].nrec) {
                set_error("%s: rank %d passed nrec_per_rank[%d] = %llu, but rank %d holds %llu records", kShardName, q, r,
                          (unsigned long long)m[q].npr[r], r, (unsigned long long)m[r].nrec);
                return DVS_ERR_ARG;
            }
        s.rank_base[r] = (uint32_t)n64;
        n64 += m[r].nrec;
        s.slot_len = std::max(s.slot_len, m[r].max_len);
    }
    if (n64 >= (1ull << 31)) {
        set_error("%s: %llu records are too many", kShardName, (unsigned long long)n64);
        return DVS_ERR_ARG;
    }
    s.nrec = (uint32_t)n64;
    s.rank_base[W] = s.nrec;
    const uint64_t need = shard_window_need(s.nrec, s.slot_len, s.nb);
    if (need > c->window_bytes) {
        set_error("%s: the per-record scalars of %u records and the outbox of one row of up to %llu entries need a window "
                  "of %llu bytes, the window has %llu (shard.window_bytes_for_sparse_select)",
                  kShardName, s.nrec, (unsigned long long)s.slot_len, (unsigned long long)need,
                  (unsigned long long)c->window_bytes);
        return DVS_ERR_ARG;
    }
    // 2. the per-record scalars of every record, in rank-major order; the owned mask; where the rows live
    {
        const uint32_t nl = local->nrec, base = s.rank_base[me];
        DVS_TRY(s.valid.alloc(s.nrec));
        DVS_TRY(s.err.alloc(s.nrec));
        DVS_TRY(s.owned.alloc(s.nrec));
        DVS_TRY(s.err_total.alloc(s.nrec));
        DVS_TRY(s.entropy.alloc(s.nrec));
        DVS_TRY(s.totals.alloc(s.nrec));
        DVS_TRY(s.where.alloc(s.nrec));
        DevBuf<uint64_t> d_len, d_lens;
        DVS_TRY(d_len.alloc(nl));
        DVS_TRY(d_lens.alloc(s.nrec));
        std::vector<uint64_t> len(nl);
        for (uint32_t q = 0; q < nl; ++q) len[q] = local->h_offsets[q + 1] - local->h_offsets[q];
        DVS_CUDA_TRY(cudaMemcpyAsync(d_len.p, len.data(), nl * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
        std::vector<uint64_t> b1(W), b8(W);
        for (int r = 0; r < W; ++r) {
            b1[r] = m[r].nrec;
            b8[r] = m[r].nrec * 8;
        }
        DVS_TRY(dvs_comm_allgatherv(ctx, c, local->valid.p, b1.data(), s.valid.p));
        DVS_TRY(dvs_comm_allgatherv(ctx, c, local->err.p, b1.data(), s.err.p));
        DVS_TRY(dvs_comm_allgatherv(ctx, c, local->err_total.p, b8.data(), s.err_total.p));
        DVS_TRY(dvs_comm_allgatherv(ctx, c, local->entropy.p, b8.data(), s.entropy.p));
        DVS_TRY(dvs_comm_allgatherv(ctx, c, local->totals.p, b8.data(), s.totals.p));
        DVS_TRY(dvs_comm_allgatherv(ctx, c, d_len.p, b8.data(), d_lens.p));
        s.lens.resize(s.nrec);
        DVS_CUDA_TRY(cudaMemcpyAsync(s.lens.data(), d_lens.p, s.nrec * sizeof(uint64_t), cudaMemcpyDeviceToHost, st));
        DVS_CUDA_TRY(cudaMemsetAsync(s.owned.p, 0, s.nrec, st));
        if (nl) DVS_CUDA_TRY(cudaMemcpyAsync(s.owned.p + base, local->valid.p, nl, cudaMemcpyDeviceToDevice, st));
        s.h_where.assign(s.nrec, kAbsentRow);
        for (uint32_t q = 0; q < nl; ++q) s.h_where[base + q] = q;
        DVS_CUDA_TRY(cudaMemcpyAsync(s.where.p, s.h_where.data(), s.nrec * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
        DVS_CUDA_TRY(cudaStreamSynchronize(st));
        s.refs.assign(s.nrec, 0);
    }
    // 3. the outbox (symmetric heap: the same size on every rank), the selection, the status of all ranks
    DVS_TRY(comm_heap_alloc(c, shard_row_layout(s.slot_len, s.nb).bytes, &s.outbox));
    const int rc = select_core(ctx, c, &s, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5, size_out);
    ctx->last_rows_fetched = s.fetched;
    ctx->last_bytes_fetched = s.fetched_bytes;
    const int all = agree_status(ctx, c, rc);  // (also: no rank still pulls from an outbox)
    comm_heap_free(c, s.outbox);
    return all;
}

int dvs_debug_fast_terms(dvs_ctx* ctx, const double* a, const double* b, double* m, double* l, int32_t* special,
                         uint64_t n) {
    if (n == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    DevBuf<double> da, db, dm, dl;
    DevBuf<int> ds;
    DVS_TRY(da.alloc(n));
    DVS_TRY(db.alloc(n));
    DVS_TRY(dm.alloc(n));
    DVS_TRY(dl.alloc(n));
    DVS_TRY(ds.alloc(n));
    DVS_CUDA_TRY(cudaMemcpyAsync(da.p, a, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    DVS_CUDA_TRY(cudaMemcpyAsync(db.p, b, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    k_debug_fast_terms<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(da.p, db.p, dm.p, dl.p, ds.p, n);
    DVS_LAUNCHED(ctx);
    DVS_CUDA_TRY(cudaMemcpyAsync(m, dm.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaMemcpyAsync(l, dl.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaMemcpyAsync(special, ds.p, n * sizeof(int), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DVS_OK;
}

uint32_t dvs_select_last_accepts(dvs_ctx* ctx) { return ctx->last_accepts; }
uint32_t dvs_select_last_exact_evals(dvs_ctx* ctx) { return ctx->last_exact_evals; }
uint32_t dvs_select_last_rows_fetched(dvs_ctx* ctx) { return ctx->last_rows_fetched; }
uint64_t dvs_select_last_bytes_fetched(dvs_ctx* ctx) { return ctx->last_bytes_fetched; }
uint32_t dvs_select_last_trail_accepts(dvs_ctx* ctx) { return ctx->last_trail_accepts; }
uint32_t dvs_select_last_trail_launches(dvs_ctx* ctx) { return ctx->last_trail_launches; }
uint32_t dvs_select_last_trail_sms(dvs_ctx* ctx) { return ctx->last_trail_launches ? ctx->last_trail_sms : 0; }

int dvs_summed_create(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* members, uint32_t n, dvs_summed** out) {
    if (!ctx || !f || !out || (!members && n)) {
        set_error("dvs_summed_create: NULL argument");
        return DVS_ERR_ARG;
    }
    if (n == 0) {
        set_error("records cannot be empty");
        return DVS_ERR_VALUE;
    }
    if (n <= 1) {
        set_error("must have > 1 KmerSeq");
        return DVS_ERR_VALUE;
    }
    for (uint32_t i = 0; i < n; ++i)
        if (members[i] >= f->nrec) {
            set_error("dvs_summed_create: member %u out of range", members[i]);
            return DVS_ERR_ARG;
        }
    DVS_CUDA_TRY(dvs::enter(ctx));
    auto* s = new dvs_summed();
    s->device = ctx->device;
    s->f = f;
    s->n = n;
    int rc = s->st.alloc(f->dim, n + 1);
    DevBuf<unsigned> d_m;
    if (rc == DVS_OK) rc = d_m.alloc(n);
    if (rc == DVS_OK) {
        cudaError_t e = cudaMemcpyAsync(d_m.p, members, n * sizeof(unsigned), cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) {
            set_error("member upload failed: %s", cudaGetErrorString(e));
            rc = DVS_ERR_CUDA;
        }
    }
    Selector<dvs_kfreqs> sel{ctx, f, f->dim, ctx->stream, (SelScal*)ctx->pinned};
    if (rc == DVS_OK) rc = sel.build(s->st, d_m.p, n, -1);
    if (rc == DVS_OK) rc = sel.read(s->st);
    if (rc == DVS_OK && sel.h_sc->panic) rc = panic_error(*sel.h_sc);
    if (rc != DVS_OK) {
        dvs_summed_free(s);
        return rc;
    }
    *out = s;
    return DVS_OK;
}

int dvs_summed_delta_jsd(dvs_ctx* ctx, dvs_summed* s, const dvs_kfreqs* q, uint32_t q_row, int is_member,
                         double* out) {
    if (!ctx || !s || !q || !out || q_row >= q->nrec || q->dim != s->f->dim) {
        set_error("dvs_summed_delta_jsd: bad argument");
        return DVS_ERR_ARG;
    }
    if (is_member) {  // records.rs:71-73
        *out = 0.0;
        return DVS_OK;
    }
    DVS_CUDA_TRY(dvs::enter(ctx));
    Selector<dvs_kfreqs> sel{ctx, s->f, s->f->dim, ctx->stream, (SelScal*)ctx->pinned};
    DevBuf<double> d_out;
    DVS_TRY(d_out.alloc(1));
    // a window of one candidate at position == row (order == nullptr); validity is the caller's business
    DVS_TRY(sel.scan_raw(s->st, q->freqs.p, q->entropy.p, q_row, d_out.p));
    DVS_CUDA_TRY(cudaMemcpyAsync(out, d_out.p, sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_TRY(sel.read(s->st));
    const SelScal h = *sel.h_sc;
    if (h.first_panic != kNone) {
        set_error("cannot calculate entropy as frequency vector total !=1.0");
        return DVS_ERR_VALUE;
    }
    return DVS_OK;
}

int dvs_summed_delta_jsd_batch(dvs_ctx* ctx, dvs_summed* s, const dvs_kfreqs* q, const uint8_t* is_member_or_null,
                               double* out) {
    if (!ctx || !s || !q || !out || q->dim != s->f->dim) {
        set_error("dvs_summed_delta_jsd_batch: bad argument");
        return DVS_ERR_ARG;
    }
    const uint32_t nq = q->nrec;
    if (nq == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    Selector<dvs_kfreqs> sel{ctx, s->f, s->f->dim, ctx->stream, (SelScal*)ctx->pinned};
    DevBuf<double> d_out;
    DevBuf<uint8_t> d_mem;
    DVS_TRY(d_out.alloc(nq));
    DVS_TRY(d_mem.alloc(nq));
    std::vector<uint8_t> h_mem(nq, 0), h_valid(nq);
    if (is_member_or_null)
        for (uint32_t i = 0; i < nq; ++i) h_mem[i] = is_member_or_null[i] ? 1 : 0;
    DVS_CUDA_TRY(cudaMemcpyAsync(d_mem.p, h_mem.data(), nq, cudaMemcpyHostToDevice, ctx->stream));
    DVS_CUDA_TRY(cudaMemsetAsync(d_out.p, 0, nq * sizeof(double), ctx->stream));
    DVS_TRY(sel.reset_scan(s->st));
    // one CTA per query row; position == row (order == nullptr); invalid / member rows are skipped
    k_sel_scan<<<nq, kEntThreads, kEntSmemBytes, ctx->stream>>>(DenseRows{s->f->freqs.p}, s->f->entropy.p, s->f->dim, s->st.S(),
                                                                 s->st.members(), s->st.sc.p, q->freqs.p,
                                                                 q->entropy.p, q->valid.p, d_mem.p, nullptr, 0u,
                                                                 d_out.p);
    DVS_LAUNCHED(ctx);
    DVS_CUDA_TRY(cudaMemcpyAsync(out, d_out.p, nq * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaMemcpyAsync(h_valid.data(), q->valid.p, nq, cudaMemcpyDeviceToHost, ctx->stream));
    DVS_TRY(sel.read(s->st));
    const SelScal h = *sel.h_sc;
    DVS_TRY(sel.reset_scan(s->st));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (h.first_panic != kNone) {
        set_error("cannot calculate entropy as frequency vector total !=1.0 (query %u)", h.first_panic);
        return DVS_ERR_VALUE;
    }
    for (uint32_t i = 0; i < nq; ++i)
        if (!h_valid[i]) out[i] = std::numeric_limits<double>::quiet_NaN();
    return DVS_OK;
}

int dvs_summed_result(dvs_ctx* ctx, dvs_summed* s, uint32_t* sel_idx, double* sel_delta, double* stats5,
                      uint32_t* size_out, uint32_t* lowest_out) {
    DVS_CUDA_TRY(dvs::enter(ctx));
    Selector<dvs_kfreqs> sel{ctx, s->f, s->f->dim, ctx->stream, (SelScal*)ctx->pinned};
    DVS_TRY(sel.read(s->st));
    const SelScal h = *sel.h_sc;
    if (sel_idx)
        DVS_CUDA_TRY(cudaMemcpyAsync(sel_idx, s->st.members(), s->n * sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
    if (sel_delta)
        DVS_CUDA_TRY(cudaMemcpyAsync(sel_delta, s->st.mdelta.p, s->n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    if (stats5) {
        stats5[0] = h.total_jsd;
        stats5[1] = h.mean;
        stats5[2] = h.stdv;
        stats5[3] = h.cov;
        stats5[4] = h.E;
    }
    if (size_out) *size_out = s->n;
    if (lowest_out) *lowest_out = h.lowest;
    return DVS_OK;
}

void dvs_summed_free(dvs_summed* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    delete s;
}

}  // extern "C"
