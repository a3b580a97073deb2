// select_fast.cuh — bounded-error selection kernels: term evaluation, scan / update / replace, cooperative rounds
// Part of select.cu (included inside namespace dvs, after the exact kernels); split out for readability only.
#pragma once

// ------------------------------------------------------------------------------- fast path ----
// The exact kernels above cost one dependent FP64 add per element (~30 us per 4^6-element
// entropy).  Most decisions are nowhere near a tie, so they are first attempted with a PARALLEL
// evaluation whose distance from the reference's value is rigorously bounded:
//   * the frequencies m_i are formed with the same IEEE operations, so they are identical;
//   * each term -m*log2(m) differs from the reference's by <= 3 ulp (two <1-ulp log2s, one product);
//   * a pairwise (tree) sum of D terms is within (ceil(log2 D)+3) u A of the real sum A' of the
//     computed terms, the reference's sequential sum within (D-1) u A        (u = 2^-53, A = sum|term|);
// so |e_fast - e_ref| <= (D + 64) * 1.2e-16 * A =: bound.  A decision is taken from the fast value
// only when it holds for every value in [fast - bound, fast + bound]; otherwise the position is
// reported as "unsure" and the exact kernel decides.  The reference's sum-to-one check
// |t_ref - 1| <= D*EPS is certified from the tree sum t (|t - T| <= 16u, |t_ref - T| <= (D-1)u):
// it cannot fail when |t - 1| <= 0.45*D*EPS; otherwise: unsure.  Selected sets, their order and all
// reported numbers are therefore still the exact path's (the final state is always re-evaluated
// exactly); only the work is reduced.
constexpr int kFastThreads = 512;

struct FastSum {
    double e, t, a;  // entropy, total, sum |term|
    int bad;         // a negative / NaN frequency was seen (reference yields NaN): cannot be bounded
};

// elements [lo, hi) of a vector (the SM-replicated selection kernel splits one vector over several CTAs).
// `stage(base)`: a row source's staging hook, called by every thread before each pass of 8 x kFastThreads elements
template <class Elem, class Stage = NoStage>
__device__ FastSum block_entropy_span(uint64_t lo, uint64_t dim, Elem elem, Stage stage = Stage()) {
    __shared__ double s_part[3][kFastThreads / 32];
    __shared__ int s_bad[kFastThreads / 32];
    double e0 = 0.0, e1 = 0.0, t0 = 0.0, t1 = 0.0, a0 = 0.0, a1 = 0.0;
    int bad = 0;
    // 8 elements per thread per pass: all frequencies (global loads + divides) are formed before the
    // first log2 so one memory latency is exposed per pass, not one per element
    constexpr int kBatch = 8;
    for (uint64_t base = lo; base < dim; base += (uint64_t)kBatch * kFastThreads) {
        stage(base);
        double x[kBatch];
#pragma unroll
        for (int q = 0; q < kBatch; ++q) {
            const uint64_t i = base + threadIdx.x + (uint64_t)q * kFastThreads;
            x[q] = i < dim ? elem(i) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < kBatch; q += 2) {
            const double x0 = x[q], x1 = x[q + 1];
            if (!(x0 == 0.0)) {
                bad |= !(x0 > 0.0);
                const double tm = __dmul_rn(-x0, log2(x0));
                e0 += tm; a0 += fabs(tm); t0 += x0;
            }
            if (!(x1 == 0.0)) {
                bad |= !(x1 > 0.0);
                const double tm = __dmul_rn(-x1, log2(x1));
                e1 += tm; a1 += fabs(tm); t1 += x1;
            }
        }
    }
    double e = e0 + e1, t = t0 + t1, a = a0 + a1;
    for (int o = 16; o; o >>= 1) {
        e += __shfl_xor_sync(0xffffffffu, e, o);
        t += __shfl_xor_sync(0xffffffffu, t, o);
        a += __shfl_xor_sync(0xffffffffu, a, o);
        bad |= __shfl_xor_sync(0xffffffffu, bad, o);
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        s_part[0][w] = e; s_part[1][w] = t; s_part[2][w] = a; s_bad[w] = bad;
    }
    __syncthreads();
    FastSum r{0.0, 0.0, 0.0, 0};
    for (int q = 0; q < kFastThreads / 32; ++q) {
        r.e += s_part[0][q]; r.t += s_part[1][q]; r.a += s_part[2][q]; r.bad |= s_bad[q];
    }
    __syncthreads();
    return r;
}
template <class Elem, class Stage = NoStage>
__device__ __forceinline__ FastSum block_entropy_fast(uint64_t dim, Elem elem, Stage stage = Stage()) {
    return block_entropy_span(0, dim, elem, stage);
}

// ---- the same sums with instruction-level parallelism (SM-replicated rounds) ----
// block_entropy_span evaluates one element at a time: CUDA's ddiv and log2 are ~50 dependent FP64
// instructions behind their own branches, and with 4 warps per scheduler at ~14 cycles per dependent
// FP64 instruction the FP64 pipe idles most of the time (measured 0.47 us per element per thread).
// Here every step is branch-free straight-line code over 8 elements per thread, so 8 chains interleave:
//   * x / b by div_exact (entropy.cuh): reciprocal + two fused-remainder steps, = __ddiv_rn bit for bit;
//   * log2 by the table-driven path of the glibc restatement (dvs_log2_main): the reference's own bits,
//     so a term -m*log2(m) is now IDENTICAL to the reference's, not merely within 3 ulp.
// Inputs that the glibc algorithm sends down its other paths (m within ~4 % of 1, subnormals) or that
// make the reference's value NaN raise `bad`, which the callers already treat as "undecided".
// m is usable by the table path (and was divided exactly) iff 2^-900 <= m < 0x1.ea4afp-1: one unsigned
// compare on its high word; negative, NaN, inf, zero, subnormal and "near 1 or above" all fall outside.
// (Below 2^-900 the fused remainders of div_exact could underflow; k-mer frequencies are >= ~1e-10.)
__device__ __forceinline__ bool fast_term_ok(double m) {
    return (uint32_t)__double2hiint(m) - 0x07b00000u < 0x3feea4afu - 0x07b00000u;
}

template <bool CLAMP, int BATCH, int NT = kFastThreads, class Num, class Stage = NoStage>
__device__ FastSum block_entropy_ilp(unsigned lo, unsigned hi, Num num, const FastDiv dv,
                                     const double2* __restrict__ ltab, Stage stage = Stage()) {
    __shared__ double s_part[3][NT / 32];
    __shared__ int s_bad[NT / 32];
    double e0 = 0.0, e1 = 0.0, t0 = 0.0, t1 = 0.0, a0 = 0.0, a1 = 0.0;
    bool bad = false;
    for (unsigned base = lo; base < hi; base += BATCH * NT) {
        stage(base);
        double x[BATCH], l[BATCH];
#pragma unroll
        for (int q = 0; q < BATCH; ++q) {
            const unsigned i = base + threadIdx.x + (unsigned)q * NT;
            x[q] = i < hi ? num(i) : 0.0;
        }
#pragma unroll
        for (int q = 0; q < BATCH; ++q) {
            double m = div_exact(x[q], dv);
            if (CLAMP) m = (m <= kEps) ? 0.0 : m;
            x[q] = m;
        }
#pragma unroll
        for (int q = 0; q < BATCH; ++q) {
            int ignored = 0;
            l[q] = dvs_log2_main(x[q], ltab, ignored);
        }
#pragma unroll
        for (int q = 0; q < BATCH; ++q) {
            const bool ok = fast_term_ok(x[q]);
            bad |= !ok && !(x[q] == 0.0);
            const double tm = ok ? __dmul_rn(-x[q], l[q]) : 0.0;
            if (q & 1) {
                e1 += tm; a1 += fabs(tm); t1 += x[q];
            } else {
                e0 += tm; a0 += fabs(tm); t0 += x[q];
            }
        }
    }
    double e = e0 + e1, t = t0 + t1, a = a0 + a1;
    int badi = bad ? 1 : 0;
    for (int o = 16; o; o >>= 1) {
        e += __shfl_xor_sync(0xffffffffu, e, o);
        t += __shfl_xor_sync(0xffffffffu, t, o);
        a += __shfl_xor_sync(0xffffffffu, a, o);
        badi |= __shfl_xor_sync(0xffffffffu, badi, o);
    }
    const int w = threadIdx.x >> 5;
    if ((threadIdx.x & 31) == 0) {
        s_part[0][w] = e; s_part[1][w] = t; s_part[2][w] = a; s_bad[w] = badi;
    }
    __syncthreads();
    FastSum r{0.0, 0.0, 0.0, 0};
    for (int q = 0; q < NT / 32; ++q) {
        r.e += s_part[0][q]; r.t += s_part[1][q]; r.a += s_part[2][q]; r.bad |= s_bad[q];
    }
    __syncthreads();
    return r;
}

// The same evaluation for the kernels that keep their state in global memory (host-driven rounds, the
// cooperative kernel, the batched grow attempts — the k >= 7 paths): m_i =
// num(i) / divisor, optionally clamped (<= EPS -> 0).  Stages the log2 table itself; divisors beyond the
// range the exact division was verified for, and vectors longer than 2^30, take the one-element-at-a-time
// form with __ddiv_rn (same values either way).  Both forms take passes of 8 x kFastThreads = 4,096 elements, which
// is one bucket of a sparse row: `stage` is the row source's hook (select.cu).
template <bool CLAMP, class Num, class Stage = NoStage>
__device__ FastSum block_entropy_div(uint64_t dim, Num num, double divisor, Stage stage = Stage()) {
    if (dim > (1ull << 30) || !(divisor >= 1.0 && divisor <= 4096.0)) {  // block-uniform
        return block_entropy_fast(dim, [&](uint64_t i) {
            const double m = __ddiv_rn(num(i), divisor);
            return (CLAMP && m <= kEps) ? 0.0 : m;
        }, stage);
    }
    __shared__ double2 s_ltab_div[64];
    dvs_log2_stage_table(s_ltab_div);
    __syncthreads();
    return block_entropy_ilp<CLAMP, 8>(0u, (unsigned)dim, num, make_fast_div(divisor), s_ltab_div, stage);
}

// Each thread first sums dim/kFastThreads elements sequentially, then the partials are tree-summed:
// |sum_fast - real sum| <= (dim/kFastThreads + 12) u A, the reference's sequential sum is within
// (dim - 1) u A, and the per-term differences add 6 u A; 1.2e-16 > u = 2^-53 absorbs second-order terms.
// `depth`: additional sequential additions on top of the tree (partials of a vector split over CTAs)
__device__ __forceinline__ double fast_slack(uint64_t dim, double depth = 0.0) {
    return (double)(dim / kFastThreads) + 12.0 + depth;
}
__device__ __forceinline__ double fast_bound(uint64_t dim, double a, double extra, double depth = 0.0) {
    return ((double)dim + fast_slack(dim, depth) + 16.0) * 1.2e-16 * (a + fabs(extra) + 1.0);
}
// reference check: |t_ref - 1| <= dim*EPS = 2 dim u.  |t_ref - T| <= (dim-1) u, |t - T| <= slack u (T ~ 1),
// so the check cannot fail when |t - 1| <= (dim + 1 - slack) u; for tiny dim this is never certified
// and the (then trivially cheap) exact kernel decides.
__device__ __forceinline__ bool fast_total_ok(uint64_t dim, double t, double depth = 0.0) {
    const double lim = ((double)dim + 1.0 - fast_slack(dim, depth) - 2.0) * 1.1102230246251565e-16;
    return lim > 0.0 && fabs(t - 1.0) <= lim;
}

// Block-cooperative end of a fast update (run by every thread of the LAST CTA to finish):
// delta_j = total - jsd_j, argmin (lowest index wins ties) and the certainty test
// "member `low` is smaller than every other member for all admissible errors".  Returns 1 when the
// argmin could not be certified.  (A single thread walking n global values costs n L2 latencies.)
// GLOBAL: the arrays live in global memory and were written by other CTAs (read through L2); otherwise
// they are this CTA's own shared-memory copies.
template <bool GLOBAL = true>
__device__ __forceinline__ unsigned finalize_fast_block(double* mdelta, const double* mbound, unsigned n, double total,
                                                        double total_bound, unsigned* low_out) {
    auto ld = [](const double* p) { return GLOBAL ? __ldcg(p) : *p; };
    __shared__ double s_mn[kFastThreads / 32], s_mb[kFastThreads / 32];
    __shared__ unsigned s_ix[kFastThreads / 32];
    __shared__ double s_best, s_bestb;
    __shared__ unsigned s_besti;
    double mn = 1e300, mb = 0.0;
    unsigned ix = kNone;
    for (unsigned t = threadIdx.x; t < n; t += blockDim.x) {
        const double d = total - ld(&mdelta[t]);
        mdelta[t] = d;
        if (d < mn || (d == mn && t < ix)) {
            mn = d;
            mb = ld(&mbound[t]);
            ix = t;
        }
    }
    for (int o = 16; o; o >>= 1) {
        const double omn = __shfl_xor_sync(0xffffffffu, mn, o), omb = __shfl_xor_sync(0xffffffffu, mb, o);
        const unsigned oix = __shfl_xor_sync(0xffffffffu, ix, o);
        if (omn < mn || (omn == mn && oix < ix)) {
            mn = omn; mb = omb; ix = oix;
        }
    }
    if ((threadIdx.x & 31) == 0) {
        s_mn[threadIdx.x >> 5] = mn; s_mb[threadIdx.x >> 5] = mb; s_ix[threadIdx.x >> 5] = ix;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        for (unsigned w = 1; w < blockDim.x / 32; ++w)
            if (s_mn[w] < mn || (s_mn[w] == mn && s_ix[w] < ix)) {
                mn = s_mn[w]; mb = s_mb[w]; ix = s_ix[w];
            }
        s_best = mn; s_bestb = mb; s_besti = (ix == kNone) ? 0u : ix;
    }
    __syncthreads();
    mn = s_best; mb = s_bestb;
    const unsigned low = s_besti;
    int unsure = 0;
    for (unsigned t = threadIdx.x; t < n; t += blockDim.x)
        if (t != low && !(mn + mb + 2.0 * kEps < mdelta[t] - ld(&mbound[t]))) unsure = 1;
    if (!(mn + mb + total_bound < 1e6)) unsure = 1;  // the reference's `min_delta_jsd = 1e6` initial value
    unsure = __syncthreads_or(unsure);
    *low_out = low;
    return (unsigned)unsure;
}

// block-wide sum / max of one double per thread (all threads get the result)
__device__ __forceinline__ double block_sum_fast(double v) {
    __shared__ double s_red[kFastThreads / 32];
    __shared__ double s_out;
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (unsigned w = 0; w < blockDim.x / 32; ++w) t += s_red[w];
        s_out = t;
    }
    __syncthreads();
    const double r = s_out;
    __syncthreads();
    return r;
}
__device__ __forceinline__ double block_max_fast(double v) {
    __shared__ double s_red[kFastThreads / 32];
    __shared__ double s_out;
    for (int o = 16; o; o >>= 1) v = fmax(v, __shfl_xor_sync(0xffffffffu, v, o));
    if ((threadIdx.x & 31) == 0) s_red[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = s_red[0];
        for (unsigned w = 1; w < blockDim.x / 32; ++w) t = fmax(t, s_red[w]);
        s_out = t;
    }
    __syncthreads();
    const double r = s_out;
    __syncthreads();
    return r;
}

// mean / std / cov of the (approximate) member deltas with rigorous distance bounds to the values
// the reference computes (src/records.rs:153-172).  delta_j is within mbound_j (+ the common
// total_bound, which cancels in the deviations) of the reference's; std is 1-Lipschitz in the
// deviations scaled by 1/sqrt(n-1), the sequential sums add <= (n+8) u relative error.
__device__ __forceinline__ void stats_fast_block(const double* mdelta, const double* mbound, unsigned n,
                                                 double total_bound, SelScal* sc) {
    double sd = 0.0, bmx = 0.0, amx = 0.0;
    for (unsigned t = threadIdx.x; t < n; t += blockDim.x) {
        const double d = mdelta[t];
        sd += d;
        bmx = fmax(bmx, __ldcg(&mbound[t]));
        amx = fmax(amx, fabs(d));
    }
    const double nd = (double)n;
    const double mean = block_sum_fast(sd) / nd;
    bmx = block_max_fast(bmx);
    amx = block_max_fast(amx);
    double ss = 0.0;
    for (unsigned t = threadIdx.x; t < n; t += blockDim.x) {
        const double d = mdelta[t] - mean;
        ss += d * d;
    }
    const double sdev = sqrt(block_sum_fast(ss) / (nd - 1.0));
    if (threadIdx.x == 0) {
        const double u = 1.2e-16, scale = amx + fabs(mean);
        const double b_mean = bmx + total_bound + (nd + 8.0) * u * scale;
        const double b_std = 1.5 * (bmx + 4.0 * u * scale) + (nd + 8.0) * u * sdev;
        const double cov = sdev / mean;
        double b_cov = 1e300;
        if (fabs(mean) > 2.0 * b_mean) b_cov = (b_std + fabs(cov) * b_mean) / (fabs(mean) - b_mean) + 8.0 * u * fabs(cov);
        sc->mean = mean;
        sc->stdv = sdev;
        sc->cov = cov;
        sc->std_bound = b_std;
        sc->cov_bound = b_cov;
    }
}

// The mutable selection state (S, member list, is_member, scalars) is read with ld.global.cg inside the
// bodies below: the persistent kernel keeps CTAs alive across rounds, where a line cached in L1 during
// an earlier round would be stale.  Rows of F / H / valid / order never change and use the default path.
struct ScanScal {
    double E, total_jsd, total_bound;
    unsigned n, low_row;
};

// fast increases_jsd of the candidate at position `pos`; first_true / first_unsure by atomicMin
template <class Src>
__device__ __forceinline__ void scan_fast_body(const Src src, const double* __restrict__ H, uint64_t dim,
                                               const double* __restrict__ S, SelScal* sc, const ScanScal& q,
                                               const uint8_t* __restrict__ valid,
                                               const uint8_t* __restrict__ is_member,
                                               const unsigned* __restrict__ order, unsigned pos) {
    const unsigned row = order[pos];
    if (!valid[row] || __ldcg(is_member + row)) return;
    const double nd = (double)q.n;
    auto v = src.view(stage_smem<Src>());
    const auto fl = v.row(0, q.low_row, dim);
    const auto fc = v.row(1, row, dim);
    FastSum h = block_entropy_div<false>(
        dim, [&](uint64_t i) { return __dadd_rn(__dsub_rn(__ldcg(S + i), fl[i]), fc[i]); }, nd, stager(v));
    if (threadIdx.x == 0) {
        const double mean_entropy = __ddiv_rn(__dadd_rn(__dsub_rn(q.E, H[q.low_row]), H[row]), nd);
        const double d = h.e - mean_entropy;
        const double b = fast_bound(dim, h.a, mean_entropy);
        const double thr = q.total_jsd + kEps, tb = q.total_bound + 4.0 * kEps;
        if (h.bad || !fast_total_ok(dim, h.t) || !(d == d)) {
            atomicMin(&sc->first_unsure, pos);
        } else if (d - b > thr + tb) {
            atomicMin(&sc->first_true, pos);
        } else if (!(d + b < thr - tb)) {
            atomicMin(&sc->first_unsure, pos);
        }
    }
}

__device__ __forceinline__ ScanScal load_scan_scal(const SelScal* sc, const unsigned* members) {
    ScanScal q;
    q.E = __ldcg(&sc->E);
    q.total_jsd = __ldcg(&sc->total_jsd);
    q.total_bound = __ldcg(&sc->total_bound);
    q.n = __ldcg(&sc->n);
    q.low_row = __ldcg(members + __ldcg(&sc->lowest));
    return q;
}

// host-driven window: one CTA per position pos0 + blockIdx.x
template <class Src>
__global__ void __launch_bounds__(kFastThreads)
k_sel_scan_fast(const Src src, const double* __restrict__ H, uint64_t dim, const double* __restrict__ S,
                const unsigned* __restrict__ members, SelScal* sc, const uint8_t* __restrict__ valid,
                const uint8_t* __restrict__ is_member, const unsigned* __restrict__ order, unsigned pos0) {
    const ScanScal q = load_scan_scal(sc, members);
    scan_fast_body(src, H, dim, S, sc, q, valid, is_member, order, pos0 + blockIdx.x);
}

// fast total_jsd + get_lowest_record_index: same shape as k_sel_update.  Leaves approximate
// total_jsd (with total_bound) and mdelta, and lowest_index only if it is certain.
template <class Src>
__global__ void __launch_bounds__(kFastThreads)
k_sel_update_fast(const Src src, const double* __restrict__ H, uint64_t dim,
                  const double* __restrict__ S, const unsigned* __restrict__ members, double* __restrict__ mdelta,
                  double* __restrict__ mbound, SelScal* sc) {
    __shared__ unsigned s_last;
    const unsigned j = blockIdx.x, n = sc->n;
    const double nd = (double)n;
    if (j == n) {
        FastSum h = block_entropy_div<false>(dim, [&](uint64_t i) { return S[i]; }, nd);
        if (threadIdx.x == 0) {
            const double me = __ddiv_rn(sc->E, nd);
            sc->total_jsd = h.e - me;
            sc->total_bound = fast_bound(dim, h.a, me);
            if (h.bad || !fast_total_ok(dim, h.t)) atomicExch(&sc->state_unsure, 1u);
        }
    } else {
        const unsigned row = members[j];
        const double div = __dsub_rn(nd, 1.0);
        auto v = src.view(stage_smem<Src>());
        const auto f = v.row(0, row, dim);
        FastSum h = block_entropy_div<true>(dim, [&](uint64_t i) { return __dsub_rn(S[i], f[i]); }, div, stager(v));
        if (threadIdx.x == 0) {
            const double mean_entropy = __ddiv_rn(__dsub_rn(sc->E, H[row]), div);
            mdelta[j] = h.e - mean_entropy;
            mbound[j] = fast_bound(dim, h.a, mean_entropy);
            if (h.bad || !fast_total_ok(dim, h.t)) atomicExch(&sc->state_unsure, 1u);
        }
    }
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(&sc->ticket, 1u) == n) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {  // block-uniform
        __threadfence();
        const double total = __ldcg(&sc->total_jsd), tb = __ldcg(&sc->total_bound);
        unsigned low = 0;
        const unsigned unsure = finalize_fast_block(mdelta, mbound, n, total, tb, &low);
        stats_fast_block(mdelta, mbound, n, tb, sc);
        if (threadIdx.x == 0) {
            sc->lowest = low;
            if (unsure) atomicExch(&sc->state_unsure, 1u);
            sc->exact = 0;
            sc->ticket = 0;
            sc->first_true = kNone;
            sc->first_panic = kNone;
            sc->first_unsure = kNone;
        }
    }
}

// replace_lowest + total_jsd + get_lowest_record_index in ONE launch (fast path).  Every CTA forms
// the updated sums S'[i] = clamp(S[i] - f_low[i]) + f_c[i] on the fly from the OLD buffers (same
// operations as k_sel_replace_vec, so S' is bitwise the reference's); CTA n also stores S' and the
// last CTA to finish stores the new member list / scalars into the other buffer set.
// dev_pos != kNone: device-driven round; the last CTA also advances cursor / window / accepts / which.
template <class Src>
__device__ __forceinline__ void replace_update_fast_body(
    const Src src, const double* __restrict__ H, uint64_t dim, const double* __restrict__ S_in,
    double* __restrict__ S_out, const unsigned* __restrict__ m_in, unsigned* __restrict__ m_out,
    uint8_t* __restrict__ is_member, double* __restrict__ mdelta, double* __restrict__ mbound, SelScal* sc,
    unsigned cand_row, unsigned dev_pos, unsigned dev_cursor, unsigned j, unsigned n, unsigned low, double E_old) {
    __shared__ unsigned s_last;
    const double nd = (double)n;
    const unsigned low_row = __ldcg(m_in + low);
    auto v = src.view(stage_smem<Src>());
    const auto fl = v.row(0, low_row, dim);
    const auto fc = v.row(1, cand_row, dim);
    const double E_new = __dadd_rn(__dsub_rn(E_old, H[low_row]), H[cand_row]);  // records.rs:101,129
    auto s_new = [&](uint64_t i) {
        double s = __dsub_rn(__ldcg(S_in + i), fl[i]);
        if (s <= kEps) s = 0.0;
        return __dadd_rn(s, fc[i]);
    };
    if (j == n) {
        FastSum h = block_entropy_div<false>(dim, [&](uint64_t i) {
            const double s = s_new(i);
            S_out[i] = s;
            return s;
        }, nd, stager(v));
        if (threadIdx.x == 0) {
            const double me = __ddiv_rn(E_new, nd);
            sc->total_jsd = h.e - me;
            sc->total_bound = fast_bound(dim, h.a, me);
            if (h.bad || !fast_total_ok(dim, h.t)) atomicExch(&sc->state_unsure, 1u);
        }
    } else {
        // member j of the list after Vec::remove(low) + push(cand)
        const unsigned row = j < low ? __ldcg(m_in + j) : (j + 1 < n ? __ldcg(m_in + j + 1) : cand_row);
        const double div = __dsub_rn(nd, 1.0);
        const auto f = v.row(2, row, dim);
        FastSum h = block_entropy_div<true>(dim, [&](uint64_t i) { return __dsub_rn(s_new(i), f[i]); }, div, stager(v));
        if (threadIdx.x == 0) {
            const double mean_entropy = __ddiv_rn(__dsub_rn(E_new, H[row]), div);
            mdelta[j] = h.e - mean_entropy;
            mbound[j] = fast_bound(dim, h.a, mean_entropy);
            if (h.bad || !fast_total_ok(dim, h.t)) atomicExch(&sc->state_unsure, 1u);
        }
    }
    if (threadIdx.x == 0) {
        __threadfence();
        s_last = (atomicAdd(&sc->ticket, 1u) == n) ? 1u : 0u;
    }
    __syncthreads();
    if (s_last) {  // block-uniform: the whole last CTA finishes the round
        __threadfence();
        for (unsigned t = threadIdx.x; t < n; t += blockDim.x)
            m_out[t] = t < low ? __ldcg(m_in + t) : (t + 1 < n ? __ldcg(m_in + t + 1) : cand_row);
        const double total = __ldcg(&sc->total_jsd), tb = __ldcg(&sc->total_bound);
        unsigned lo2 = 0;
        const unsigned unsure = finalize_fast_block(mdelta, mbound, n, total, tb, &lo2);
        if (dev_pos == kNone) stats_fast_block(mdelta, mbound, n, tb, sc);  // only max-mode callers read them
        if (threadIdx.x == 0) {
            is_member[low_row] = 0;
            is_member[cand_row] = 1;
            sc->E = E_new;
            sc->lowest = lo2;
            if (unsure) atomicExch(&sc->state_unsure, 1u);
            sc->exact = 0;
            sc->ticket = 0;
            sc->first_true = kNone;
            sc->first_panic = kNone;
            sc->first_unsure = kNone;
            if (dev_pos != kNone) {
                sc->window = max(64u, min(__ldcg(&sc->window_max), 2u * (dev_pos - dev_cursor + 1u)));
                sc->cursor = dev_pos + 1u;
                sc->accepts = __ldcg(&sc->accepts) + 1u;
                sc->which = __ldcg(&sc->which) ^ 1u;
            }
        }
    }
}

template <class Src>
__global__ void __launch_bounds__(kFastThreads)
k_sel_replace_update_fast(const Src src, const double* __restrict__ H, uint64_t dim,
                          const double* __restrict__ S_in, double* __restrict__ S_out,
                          const unsigned* __restrict__ m_in, unsigned* __restrict__ m_out,
                          uint8_t* __restrict__ is_member, double* __restrict__ mdelta, double* __restrict__ mbound,
                          SelScal* sc, unsigned cand_row) {
    replace_update_fast_body(src, H, dim, S_in, S_out, m_in, m_out, is_member, mdelta, mbound, sc, cand_row, kNone, 0u,
                             blockIdx.x, sc->n, sc->lowest, sc->E);
}

// ---- sliced evaluation for the cooperative kernel (vectors that do not fit shared memory: k >= 7) ----
// With one CTA per candidate / member slot the rounds are THROUGHPUT bound at 4^8 elements: a round scans ~60
// candidates and updates n + 1 = 101 slots on 296 resident CTAs, i.e. a fifth / a third of the GPU works for the
// 51 us / 58 us one vector costs one CTA (tools/trace_select.py --k 8).  Here a vector is cut into P <= 8 slices that
// different CTAs evaluate; each publishes its partial sums, and the CTA that arrives last at the vector's ticket adds
// them in slice order and does what the unsliced body does with the sum.  The P - 1 extra sequential additions
// enter the error bounds as `depth` (fast_slack), exactly as in the SM-replicated kernel.
struct __align__(16) SlicePart {
    double e, t, a;
    int bad, pad;
};
constexpr unsigned kMaxSlices = 8;

__device__ __forceinline__ void slice_publish(SlicePart* p, const FastSum& h) {
    __stcg(&p->e, h.e);
    __stcg(&p->t, h.t);
    __stcg(&p->a, h.a);
    __stcg(&p->bad, h.bad);
}
__device__ __forceinline__ FastSum slice_combine(const SlicePart* part, unsigned P) {
    FastSum r{__ldcg(&part[0].e), __ldcg(&part[0].t), __ldcg(&part[0].a), __ldcg(&part[0].bad)};
    for (unsigned s = 1; s < P; ++s) {
        r.e += __ldcg(&part[s].e);
        r.t += __ldcg(&part[s].t);
        r.a += __ldcg(&part[s].a);
        r.bad |= __ldcg(&part[s].bad);
    }
    return r;
}
// thread 0 of the CTA: publish slice s; true (with the combined sums in h) for the last of the P CTAs to arrive
__device__ __forceinline__ bool slice_arrive(SlicePart* part, unsigned* tick, unsigned s, unsigned P, FastSum& h) {
    slice_publish(part + s, h);
    __threadfence();
    if (atomicAdd(tick, 1u) != P - 1u) return false;
    __threadfence();
    *tick = 0u;  // (next use is behind a grid barrier)
    h = slice_combine(part, P);
    return true;
}

// scan_fast_body for slice s of P of the candidate at `pos`
__device__ __forceinline__ void scan_sliced_body(const double* __restrict__ F, const double* __restrict__ H, uint64_t dim,
                                                 const double* __restrict__ S, SelScal* sc, const ScanScal& q,
                                                 const uint8_t* __restrict__ valid, const uint8_t* __restrict__ is_member,
                                                 const unsigned* __restrict__ order, unsigned pos, unsigned s, unsigned P,
                                                 SlicePart* part, unsigned* tick) {
    __shared__ double2 s_ltab_sl[64];
    const unsigned row = order[pos];
    if (!valid[row] || __ldcg(is_member + row)) return;  // (the same for every slice: no ticket is taken)
    dvs_log2_stage_table(s_ltab_sl);
    __syncthreads();
    const double nd = (double)q.n;
    const double* fl = F + (size_t)q.low_row * dim;
    const double* fc = F + (size_t)row * dim;
    const unsigned lo = (unsigned)(dim * s / P), hi = (unsigned)(dim * (s + 1) / P);
    FastSum h = block_entropy_ilp<false, 8>(
        lo, hi, [&](unsigned i) { return __dadd_rn(__dsub_rn(__ldcg(S + i), fl[i]), fc[i]); }, make_fast_div(nd), s_ltab_sl);
    if (threadIdx.x == 0 && slice_arrive(part, tick, s, P, h)) {
        const double depth = (double)P;
        const double mean_entropy = __ddiv_rn(__dadd_rn(__dsub_rn(q.E, H[q.low_row]), H[row]), nd);
        const double d = h.e - mean_entropy;
        const double b = fast_bound(dim, h.a, mean_entropy, depth);
        const double thr = q.total_jsd + kEps, tb = q.total_bound + 4.0 * kEps;
        if (h.bad || !fast_total_ok(dim, h.t, depth) || !(d == d)) {
            atomicMin(&sc->first_unsure, pos);
        } else if (d - b > thr + tb) {
            atomicMin(&sc->first_true, pos);
        } else if (!(d + b < thr - tb)) {
            atomicMin(&sc->first_unsure, pos);
        }
    }
}

// replace_update_fast_body (device-driven form) for slice s of P of member slot j
__device__ __forceinline__ void replace_update_sliced_body(
    const double* __restrict__ F, const double* __restrict__ H, uint64_t dim, const double* __restrict__ S_in,
    double* __restrict__ S_out, const unsigned* __restrict__ m_in, unsigned* __restrict__ m_out,
    uint8_t* __restrict__ is_member, double* __restrict__ mdelta, double* __restrict__ mbound, SelScal* sc,
    unsigned cand_row, unsigned dev_pos, unsigned dev_cursor, unsigned j, unsigned s, unsigned P, unsigned n, unsigned low,
    double E_old, SlicePart* part, unsigned* tick) {
    __shared__ unsigned s_last_sl;
    __shared__ double2 s_ltab_up[64];
    dvs_log2_stage_table(s_ltab_up);
    __syncthreads();
    const double nd = (double)n, depth = (double)P;
    const unsigned low_row = __ldcg(m_in + low);
    const double* fl = F + (size_t)low_row * dim;
    const double* fc = F + (size_t)cand_row * dim;
    const double E_new = __dadd_rn(__dsub_rn(E_old, H[low_row]), H[cand_row]);  // records.rs:101,129
    auto s_new = [&](unsigned i) {
        double v = __dsub_rn(__ldcg(S_in + i), fl[i]);
        if (v <= kEps) v = 0.0;
        return __dadd_rn(v, fc[i]);
    };
    const unsigned lo = (unsigned)(dim * s / P), hi = (unsigned)(dim * (s + 1) / P);
    const unsigned row = j == n ? 0u : (j < low ? __ldcg(m_in + j) : (j + 1 < n ? __ldcg(m_in + j + 1) : cand_row));
    FastSum h;
    if (j == n) {
        h = block_entropy_ilp<false, 8>(lo, hi, [&](unsigned i) {
            const double v = s_new(i);
            S_out[i] = v;
            return v;
        }, make_fast_div(nd), s_ltab_up);
    } else {
        const double* f = F + (size_t)row * dim;
        h = block_entropy_ilp<true, 8>(lo, hi, [&](unsigned i) { return __dsub_rn(s_new(i), f[i]); },
                                       make_fast_div(__dsub_rn(nd, 1.0)), s_ltab_up);
    }
    if (threadIdx.x == 0) {
        unsigned last = 0;
        if (slice_arrive(part, tick, s, P, h)) {
            if (j == n) {
                const double me = __ddiv_rn(E_new, nd);
                sc->total_jsd = h.e - me;
                sc->total_bound = fast_bound(dim, h.a, me, depth);
            } else {
                const double mean_entropy = __ddiv_rn(__dsub_rn(E_new, H[row]), __dsub_rn(nd, 1.0));
                mdelta[j] = h.e - mean_entropy;
                mbound[j] = fast_bound(dim, h.a, mean_entropy, depth);
            }
            if (h.bad || !fast_total_ok(dim, h.t, depth)) atomicExch(&sc->state_unsure, 1u);
            __threadfence();
            last = (atomicAdd(&sc->ticket, 1u) == n) ? 1u : 0u;
        }
        s_last_sl = last;
    }
    __syncthreads();
    if (s_last_sl) {  // block-uniform: the whole last CTA finishes the round (as in replace_update_fast_body)
        __threadfence();
        for (unsigned t = threadIdx.x; t < n; t += blockDim.x)
            m_out[t] = t < low ? __ldcg(m_in + t) : (t + 1 < n ? __ldcg(m_in + t + 1) : cand_row);
        const double total = __ldcg(&sc->total_jsd), tb = __ldcg(&sc->total_bound);
        unsigned lo2 = 0;
        const unsigned unsure = finalize_fast_block(mdelta, mbound, n, total, tb, &lo2);
        if (threadIdx.x == 0) {
            is_member[low_row] = 0;
            is_member[cand_row] = 1;
            sc->E = E_new;
            sc->lowest = lo2;
            if (unsure) atomicExch(&sc->state_unsure, 1u);
            sc->exact = 0;
            sc->ticket = 0;
            sc->first_true = kNone;
            sc->first_panic = kNone;
            sc->first_unsure = kNone;
            sc->window = max(64u, min(__ldcg(&sc->window_max), 2u * (dev_pos - dev_cursor + 1u)));
            sc->cursor = dev_pos + 1u;
            sc->accepts = __ldcg(&sc->accepts) + 1u;
            sc->which = __ldcg(&sc->which) ^ 1u;
        }
    }
}

// All device-driven rounds in ONE cooperative launch: the CTAs stay resident, a round is
//   scan (one candidate per CTA and pass) | grid barrier | accept: fused replace + update over n+1 member
//   slots, or advance / halt | grid barrier
// The kernel carries cursor / window / accepts / which in the scalar block and halts for the host when the
// first interesting candidate or the state cannot be decided within the error bound; the host then resolves
// it exactly and launches again.  Against two launches per round this removes the launch and block
// scheduling latency of ~2 x 350 dependent kernels per nmost run and loads the round's scalars once per
// CTA instead of through chains of dependent global loads.
struct RoundScal {
    ScanScal q;
    unsigned lowest, which, cursor, count, window, stop, ft, fu, su;
};

__global__ void __launch_bounds__(kFastThreads)
k_sel_persist(const double* __restrict__ F, const double* __restrict__ H, uint64_t dim, double* S0, double* S1,
              unsigned* M0, unsigned* M1, uint8_t* is_member, double* mdelta, double* mbound, SelScal* sc,
              const uint8_t* __restrict__ valid, const unsigned* __restrict__ order, unsigned max_rounds,
              unsigned long long* trace, const ShardArgs sh, SlicePart* parts, unsigned* ticks, unsigned slice_mode) {
    cg::grid_group grid = cg::this_grid();
    __shared__ RoundScal rs;
    __shared__ unsigned s_xft, s_xfu, s_xdead;
    const unsigned world = (unsigned)sh.world, rank = (unsigned)sh.rank;
    // DVS_SELECT_TRACE: CTA 0 stamps %globaltimer at the four phase boundaries of the first rounds
    auto stamp = [&](unsigned round, int slot) {
        if (trace && blockIdx.x == 0 && threadIdx.x == 0 && round < 512) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            trace[round * 4 + slot] = t;
        }
    };
    for (unsigned round = 0; round < max_rounds; ++round) {
        stamp(round, 0);
        if (threadIdx.x == 0) {
            const unsigned cursor = __ldcg(&sc->cursor), num = __ldcg(&sc->num), window = __ldcg(&sc->window);
            rs.stop = __ldcg(&sc->halt) || cursor >= num;
            rs.cursor = cursor;
            rs.window = window;
            rs.count = cursor < num ? min(window, num - cursor) : 0u;
            rs.which = __ldcg(&sc->which);
            rs.lowest = __ldcg(&sc->lowest);
            rs.q = load_scan_scal(sc, rs.which ? M1 : M0);
        }
        __syncthreads();
        if (rs.stop) break;  // grid-uniform: every CTA read the same scalar block
        const unsigned which = rs.which, cursor = rs.cursor, count = rs.count, n = rs.q.n;
        const ScanScal q = rs.q;
        // candidate-sharded over the GPUs: this one scores the window positions p with p % world == rank
        const unsigned woff = (rank + world - cursor % world) % world;
        // (slicing needs the exact-division / table range of block_entropy_div and room for the partial sums)
        const bool slice_ok = parts && dim <= (1ull << 30) && n >= 2u && n <= 4096u;
        const unsigned nloc = count > woff ? (count - woff + world - 1u) / world : 0u;
        unsigned P = 1;
        if (slice_ok)
            while (P < kMaxSlices && nloc * P * 2u <= gridDim.x) P *= 2u;
        if (P == 1u) {
            for (unsigned c = woff + world * blockIdx.x; c < count; c += world * gridDim.x)
                scan_fast_body(DenseRows{F}, H, dim, which ? S1 : S0, sc, q, valid, is_member, order, cursor + c);
        } else if (blockIdx.x < nloc * P) {  // slice s of this GPU's candidate c of the window
            const unsigned c = blockIdx.x / P, s = blockIdx.x % P;
            scan_sliced_body(F, H, dim, which ? S1 : S0, sc, q, valid, is_member, order, cursor + woff + world * c, s, P,
                             parts + (size_t)c * kMaxSlices, ticks + c);
        }
        stamp(round, 1);
        grid.sync();
        if (world > 1u) {  // all-reduce(min) of {first_true, first_unsure} over NVLink by CTA 0 (select_sm.cuh)
            if (blockIdx.x == 0) {
                if (threadIdx.x == 0) {
                    s_xft = kNone;
                    s_xfu = kNone;
                    s_xdead = 0;
                }
                __syncthreads();
                shard_exchange_min(sh, round + 1u, __ldcg(&sc->first_true), __ldcg(&sc->first_unsure), &s_xft, &s_xfu,
                                   &s_xdead);
                __syncthreads();
                if (threadIdx.x == 0) {
                    if (s_xdead) {
                        sc->panic = 2u;
                        sc->halt = 1u;
                        s_xft = kNone;
                        s_xfu = 0u;
                    }
                    sc->first_true = s_xft;
                    sc->first_unsure = s_xfu;
                    __threadfence();
                }
            }
            grid.sync();
        }
        stamp(round, 2);
        if (threadIdx.x == 0) {
            rs.ft = __ldcg(&sc->first_true);
            rs.fu = __ldcg(&sc->first_unsure);
            rs.su = __ldcg(&sc->state_unsure);
        }
        __syncthreads();
        const unsigned ft = rs.ft, fu = rs.fu, su = rs.su;
        if (!su && !(fu < ft) && ft != kNone) {
            const unsigned cand_row = order[ft];
            // slices per member slot: the P in {1, 2, 4, 8} with the fewest (waves of CTAs) / P
            unsigned Pu = 1;
            if (slice_ok && slice_mode >= 2u) {
                unsigned best = (n + gridDim.x) / gridDim.x * kMaxSlices;  // waves at P = 1, in units of 1/8 vector
                for (unsigned Pc = 2; Pc <= kMaxSlices; Pc *= 2u) {
                    const unsigned waves = ((n + 1u) * Pc + gridDim.x - 1u) / gridDim.x, cost = waves * (kMaxSlices / Pc);
                    if (cost < best) {
                        best = cost;
                        Pu = Pc;
                    }
                }
            }
            if (Pu == 1u) {
                for (unsigned j = blockIdx.x; j <= n; j += gridDim.x)
                    replace_update_fast_body(DenseRows{F}, H, dim, which ? S1 : S0, which ? S0 : S1, which ? M1 : M0, which ? M0 : M1,
                                             is_member, mdelta, mbound, sc, cand_row, ft, cursor, j, n, rs.lowest, q.E);
            } else {
                for (unsigned u = blockIdx.x; u < (n + 1u) * Pu; u += gridDim.x) {
                    const unsigned j = u / Pu, s = u % Pu;
                    replace_update_sliced_body(F, H, dim, which ? S1 : S0, which ? S0 : S1, which ? M1 : M0,
                                               which ? M0 : M1, is_member, mdelta, mbound, sc, cand_row, ft, cursor, j, s,
                                               Pu, n, rs.lowest, q.E, parts + (size_t)j * kMaxSlices, ticks + j);
                }
            }
        } else if (blockIdx.x == 0 && threadIdx.x == 0) {
            if (su || fu < ft) {
                sc->halt = 1u;
            } else {  // empty window
                sc->cursor = cursor + count;
                sc->window = min(rs.window * 2u, __ldcg(&sc->window_max));
            }
        }
        stamp(round, 3);
        grid.sync();
    }
}

