// select_grow.cuh — batched grow attempts of `max` (k_grow_eval, k_grow_decide)
// Part of select.cu (included inside namespace dvs, after the exact kernels); split out for readability only.
#pragma once

// ------------------------------------------------------------------ batched grow attempts (max) ----
// While a `max` selection is below max_size every candidate that increases the JSD costs the reference a
// `clone()` + `push` and a comparison of std / cov (records.rs:434-451), and the candidate is DISCARDED
// when the statistic does not improve — the state is unchanged.  On the benchmark set almost every
// candidate is of that kind (stdev 5..10 over 10.5k genomes: 4 adoptions), and one host-driven attempt
// costs ~210 us.  As with the windowed scan, a window of candidates is therefore evaluated concurrently
// against the same state: for each candidate the scan predicate and, for the grown set, H(S'/(n+1)) and the
// n+1 leave-one-out entropies (one CTA each, same operations as k_sel_sum + k_sel_update_fast), then the
// bounded statistic.  A candidate is skipped only if it CERTAINLY does not increase the JSD or CERTAINLY
// does not improve the statistic; the first candidate that is anything else is handed to the existing
// host path (which adopts it, or decides it exactly).  Decisions are unchanged, only certain discards
// are taken in bulk.
template <class Src>
__global__ void __launch_bounds__(kFastThreads)
k_grow_eval(const Src src, uint64_t dim, const double* __restrict__ S_cur,
            const unsigned* __restrict__ members, const SelScal* __restrict__ sc_cur,
            const double* __restrict__ S_fresh, const uint8_t* __restrict__ valid,
            const uint8_t* __restrict__ is_member, const unsigned* __restrict__ order, unsigned cursor,
            FastSum* __restrict__ parts, unsigned c0, unsigned cstride) {
    // (c0, cstride): the window candidates this GPU evaluates (candidate-sharded `max`, all of them on one GPU)
    const unsigned c = c0 + cstride * blockIdx.y, t = blockIdx.x, n = sc_cur->n;
    const unsigned row = order[cursor + c];
    if (!valid[row] || is_member[row]) return;
    auto v = src.view(stage_smem<Src>());
    const auto fc = v.row(0, row, dim);
    const double nd = (double)n;
    FastSum h;
    if (t == 0) {  // increases_jsd against the current state (records.rs:70-92)
        const auto fl = v.row(1, members[sc_cur->lowest], dim);
        h = block_entropy_div<false>(dim, [&](uint64_t i) { return __dadd_rn(__dsub_rn(S_cur[i], fl[i]), fc[i]); }, nd, stager(v));
    } else if (t == 1) {  // total of the grown set: clone() re-sums in member order, push adds the candidate
        const double nd1 = __dadd_rn(nd, 1.0);
        h = block_entropy_div<false>(dim, [&](uint64_t i) { return __dadd_rn(S_fresh[i], fc[i]); }, nd1, stager(v));
    } else {  // leave-one-out of member j of the grown set (j == n: the candidate itself)
        const unsigned j = t - 2;
        const auto f = v.row(1, j < n ? members[j] : row, dim);
        h = block_entropy_div<true>(dim, [&](uint64_t i) { return __dsub_rn(__dadd_rn(S_fresh[i], fc[i]), f[i]); }, nd, stager(v));
    }
    if (threadIdx.x == 0) parts[(size_t)c * (n + 3) + t] = h;
}

__global__ void __launch_bounds__(kFastThreads)
k_grow_decide(const double* __restrict__ H, uint64_t dim, const unsigned* __restrict__ members,
              const SelScal* __restrict__ sc_cur, const SelScal* __restrict__ sc_fresh,
              const uint8_t* __restrict__ valid, const uint8_t* __restrict__ is_member,
              const unsigned* __restrict__ order, unsigned cursor, const FastSum* __restrict__ parts,
              double* __restrict__ md, double* __restrict__ mb, unsigned cap, SelScal* __restrict__ scratch,
              unsigned* __restrict__ first_interesting, int use_cov, unsigned c0, unsigned cstride) {
    __shared__ int s_dec;
    const unsigned c = c0 + cstride * blockIdx.x, pos = cursor + c, n = sc_cur->n;
    const unsigned row = order[pos];
    if (!valid[row] || is_member[row]) return;  // skipped silently, like the scan
    const FastSum* P = parts + (size_t)c * (n + 3);
    const double nd = (double)n;
    if (threadIdx.x == 0) {
        const FastSum h = P[0];
        const unsigned low_row = members[sc_cur->lowest];
        const double me = __ddiv_rn(__dadd_rn(__dsub_rn(sc_cur->E, H[low_row]), H[row]), nd);
        const double d = h.e - me, b = fast_bound(dim, h.a, me);
        const double thr = sc_cur->total_jsd + kEps, tb = sc_cur->total_bound + 4.0 * kEps;
        int dec = 2;  // 0: certainly not increasing, 1: certainly increasing, 2: undecided
        if (!sc_cur->state_unsure && !h.bad && fast_total_ok(dim, h.t) && d == d) {
            if (d - b > thr + tb) dec = 1;
            else if (d + b < thr - tb) dec = 0;
        }
        s_dec = dec;
    }
    __syncthreads();
    const int dec = s_dec;
    if (dec == 0) return;
    if (dec == 2) {
        if (threadIdx.x == 0) atomicMin(first_interesting, pos);
        return;
    }
    // the grown set's total, member deltas and statistic (same forms as k_sel_update_fast)
    const double nd1 = __dadd_rn(nd, 1.0);
    const double E_try = __dadd_rn(sc_fresh->E, H[row]);
    const FastSum tot = P[1];
    const double me_t = __ddiv_rn(E_try, nd1);
    const double total_try = tot.e - me_t, tbound = fast_bound(dim, tot.a, me_t);
    int unsure = (tot.bad || !fast_total_ok(dim, tot.t)) ? 1 : 0;
    double* mdc = md + (size_t)c * cap;
    double* mbc = mb + (size_t)c * cap;
    for (unsigned j = threadIdx.x; j <= n; j += blockDim.x) {
        const FastSum hj = P[2 + j];
        const double Hj = j < n ? H[members[j]] : H[row];
        const double me = __ddiv_rn(__dsub_rn(E_try, Hj), nd);
        mdc[j] = total_try - (hj.e - me);
        mbc[j] = fast_bound(dim, hj.a, me);
        if (hj.bad || !fast_total_ok(dim, hj.t)) unsure = 1;
    }
    unsure = __syncthreads_or(unsure);
    if (unsure) {
        if (threadIdx.x == 0) atomicMin(first_interesting, pos);
        return;
    }
    stats_fast_block(mdc, mbc, n + 1, tbound, scratch + c);
    __syncthreads();
    if (threadIdx.x == 0) {
        const SelScal* g = scratch + c;
        const double sa = use_cov ? sc_cur->cov : sc_cur->stdv;
        const double ba = sc_cur->exact ? 0.0 : (use_cov ? sc_cur->cov_bound : sc_cur->std_bound);
        const double sb = use_cov ? g->cov : g->stdv, bb = use_cov ? g->cov_bound : g->std_bound;
        if (!(sb + bb < sa - ba)) atomicMin(first_interesting, pos);  // not a certain discard (NaN included)
    }
}

