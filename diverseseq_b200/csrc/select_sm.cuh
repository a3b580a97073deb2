// select_sm.cuh — SM-replicated persistent selection rounds (k_sel_persist_sm)
// Part of select.cu (included inside namespace dvs, after the exact kernels); split out for readability only.
#pragma once

// ---------------------------------------------------------------- SM-replicated selection rounds ----
// k_sel_persist still pays ~10 dependent L2 round trips per round (scalar block, member list, ticket,
// last-CTA tail) and two cooperative-groups barriers.  For vectors that fit in shared memory (dim <= 4096,
// i.e. k <= 6) the whole selection state is instead REPLICATED in every SM:
//   shared memory: S, member rows and their entropies, per-member delta / bound, and the (row, valid,
//   entropy) of the next 512 positions of `order` (their rows are prefetched into L2 when the chunk is
//   staged);   registers: E, total_jsd, lowest, cursor, window.  (The global is_member map is only
//   brought up to date when the kernel ends.)
// Per round only 32-byte partial sums cross the L2, and they carry their own arrival flag, so there is no
// separate grid barrier:
//   scan    CTA b scores slice p = b % P of candidate c = b / P of the window (P = 4, 2 or 1 CTAs per
//           candidate, so a short window still uses every SM) and publishes {e, t, a, bad | tag} as two
//           self-validating 128-bit stores (tag = number of the exchange); CTAs without a candidate
//           publish an empty slot;
//   decide  the leader (CTA 0) polls all G slots until their tags match (one one-way latency after the
//           last writer), combines the partials in order, finds the first certain acceptance / first
//           undecided candidate and broadcasts them in one tagged 128-bit store that every other CTA polls;
//   accept  CTA j computes the leave-one-out entropy of member j (CTA n: H(S'/n)) and publishes its partial,
//           every CTA forms S' = clamp(S - f_lowest) + f_cand and the new member list in shared memory;
//   final   the leader gathers the n + 1 partials, forms the member deltas and the certified argmin and
//           broadcasts {total_jsd, total_bound, lowest, unsure}.
// (Letting every CTA poll every slot and decide redundantly was measured at 2.2 us per exchange against
// 1.3 us for the leader form — 148 x 148 pollers — tools/microbench/gridsync_bench.cu.)
// Slot reuse is safe without resets: the leader only broadcasts scan decision x after EVERY CTA has
// published its slot of exchange x, i.e. after every CTA has consumed all earlier broadcasts, and two
// update exchanges are always separated by a scan exchange; scan slots are double buffered.
// Arithmetic, bounds and the halt protocol are those of the kernels above (the partial sums only add
// P - 1 sequential additions, covered by `depth`; `a` travels as a float rounded UP, which only widens a
// bound), so decisions are identical; CTA 0 writes the state back to global memory when the rounds end or
// halt for the host.
constexpr unsigned kSmMaxDim = 4096, kSmMaxN = 1024, kSmMaxGrid = 256, kSmChunk = 4 * kFastThreads;
constexpr double kSmDepth = 4.0;

struct __align__(16) SmPart {
    unsigned long long w[4];  // {e, bad<<32 | tag}, {t, float_ru(a)<<32 | tag}
};

template <unsigned MAXN, unsigned CHUNK>
struct SmSharedT {
    double S[kSmMaxDim];
    double mH[2][MAXN + 1];
    double md[MAXN + 1];
    double mb[MAXN + 1];
    unsigned members[2][MAXN + 1];
    double cH[CHUNK];
    unsigned crow[CHUNK];
    unsigned char cvalid[CHUNK];
    double pe[kSmMaxGrid], pt[kSmMaxGrid], pa[kSmMaxGrid];
    unsigned char pbad[kSmMaxGrid], wskip[kSmMaxGrid];
    unsigned ft, fu, unsure, xft, xfu, dead, limit;
    double2 ltab[64];  // glibc log2 table {1/c, log2 c}
};
using SmShared = SmSharedT<kSmMaxN, kSmChunk>;  // ~105 KB

__device__ __forceinline__ void sm_st128(void* p, unsigned long long lo, unsigned long long hi) {
    asm volatile("{ .reg .b128 v; mov.b128 v, {%1, %2}; st.relaxed.gpu.global.b128 [%0], v; }" ::"l"(p), "l"(lo), "l"(hi)
                 : "memory");
}
__device__ __forceinline__ void sm_ld128(const void* p, unsigned long long& lo, unsigned long long& hi) {
    asm volatile("{ .reg .b128 v; ld.relaxed.gpu.global.b128 v, [%2]; mov.b128 {%0, %1}, v; }"
                 : "=l"(lo), "=l"(hi)
                 : "l"(p)
                 : "memory");
}
__device__ __forceinline__ void sm_publish(SmPart* slot, const FastSum& h, unsigned tag) {
    sm_st128(&slot->w[0], (unsigned long long)__double_as_longlong(h.e), ((unsigned long long)(h.bad ? 1u : 0u) << 32) | tag);
    sm_st128(&slot->w[2], (unsigned long long)__double_as_longlong(h.t),
             ((unsigned long long)__float_as_uint(__double2float_ru(h.a)) << 32) | tag);
}
__device__ __forceinline__ FastSum sm_gather(const SmPart* slot, unsigned tag) {
    unsigned long long w0, w1, w2, w3;
    do sm_ld128(&slot->w[0], w0, w1); while ((unsigned)w1 != tag);
    do sm_ld128(&slot->w[2], w2, w3); while ((unsigned)w3 != tag);
    return FastSum{__longlong_as_double((long long)w0), __longlong_as_double((long long)w2),
                   (double)__uint_as_float((unsigned)(w3 >> 32)), (int)(w1 >> 32)};
}

// finalize_fast_block on this CTA's shared-memory copies, with the cross-warp step done redundantly by
// every thread (one barrier less, no serial tail on thread 0)
template <int NT>
__device__ __forceinline__ unsigned sm_finalize(double* md, const double* mb_, unsigned n, double total,
                                                double total_bound, unsigned* low_out) {
    __shared__ double s_mn[NT / 32], s_mb[NT / 32];
    __shared__ unsigned s_ix[NT / 32];
    double mn = 1e300, mb = 0.0;
    unsigned ix = kNone;
    for (unsigned t = threadIdx.x; t < n; t += blockDim.x) {
        const double d = total - md[t];
        md[t] = d;
        if (d < mn || (d == mn && t < ix)) {
            mn = d; mb = mb_[t]; ix = t;
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
    mn = s_mn[0]; mb = s_mb[0]; ix = s_ix[0];
#pragma unroll
    for (unsigned w = 1; w < NT / 32; ++w) {
        const double wmn = s_mn[w];
        const unsigned wix = s_ix[w];
        if (wmn < mn || (wmn == mn && wix < ix)) {
            mn = wmn; mb = s_mb[w]; ix = wix;
        }
    }
    const unsigned low = (ix == kNone) ? 0u : ix;
    int unsure = 0;
    for (unsigned t = threadIdx.x; t < n; t += blockDim.x)
        if (t != low && !(mn + mb + 2.0 * kEps < md[t] - mb_[t])) unsure = 1;
    if (!(mn + mb + total_bound < 1e6)) unsure = 1;  // the reference's `min_delta_jsd = 1e6` initial value
    unsure = __syncthreads_or(unsure);  // (also fences s_mn / s_mb / s_ix for the next call)
    *low_out = low;
    return (unsigned)unsure;
}

constexpr int kSmTraceSlots = 8;
constexpr unsigned kTrailSmidOff = 64;  // words behind the ready word: %smid of every CTA of the last trailing launch

// One CTA of NT = 512 threads owns its SM.  In the TRAILING form (dvs_count_select) the kernel examines a position
// only once the record's row has been published (`ready_pos`), so the rounds trail the counting.
template <int NT, int MINB, unsigned MAXN, unsigned CHUNK>
__global__ void __launch_bounds__(NT, MINB)
k_sel_persist_sm_t(const double* __restrict__ F, const double* __restrict__ H, unsigned dim, double* S_glob,
                 unsigned* M_glob, uint8_t* is_member, double* mdelta_g, double* mbound_g, SelScal* sc,
                 const uint8_t* __restrict__ valid, const unsigned* __restrict__ order, SmPart* spart, SmPart* upart,
                 SmPart* dpart, unsigned long long* trace, int trace_all, const ShardArgs sh,
                 const unsigned* ready_pos, unsigned limit0) {
    // ready_pos != NULL: TRAILING mode.  Positions below *ready_pos (a device word that only grows, written in stream
    // order behind the kernels that produce the rows) may be examined; `limit` is the value all CTAs agree on: the
    // leader samples the word when it takes a round's decision and broadcasts it with the decision, so every CTA
    // sizes the next window from the same number.  Window sizes never change a decision (only the first acceptance
    // of a window is applied, the rest is re-scored), so the result does not depend on the timing.  The kernel
    // returns to the host when everything has been published (the stand-alone kernel finishes the job).
    extern __shared__ __align__(16) unsigned char sm_raw[];
    SmSharedT<MAXN, CHUNK>& sm = *reinterpret_cast<SmSharedT<MAXN, CHUNK>*>(sm_raw);
    const unsigned tid = threadIdx.x, b = blockIdx.x, G = gridDim.x;
    if (ready_pos && tid == 0) {  // placement record of the trailing launch (dvs_select_last_trail_sms)
        unsigned smid;
        asm volatile("mov.u32 %0, %%smid;" : "=r"(smid));
        const_cast<unsigned*>(ready_pos)[kTrailSmidOff + b] = smid;
    }
    unsigned tr_round = 0;
    // DVS_SELECT_TRACE: CTA 0's timeline of the first 256 rounds; DVS_SELECT_TRACE_ALL: every CTA's
    auto stamp = [&](int slot) {
        if (trace && tid == 0 && tr_round < 256 && (b == 0 || trace_all)) {
            unsigned long long t;
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
            if (trace_all)
                trace[((size_t)tr_round * kSmTraceSlots + slot) * kSmMaxGrid + b] = t;
            else
                trace[tr_round * kSmTraceSlots + slot] = t;
        }
    };

    // ---- every CTA loads the state the host / the previous kernels left in global memory ----
    const unsigned n = sc->n, num = sc->num;
    const double nd = (double)n, div = __dsub_rn(nd, 1.0);
    const FastDiv div_n = make_fast_div(nd), div_n1 = make_fast_div(div);
    double E = sc->E, total_jsd = sc->total_jsd, total_bound = sc->total_bound;
    unsigned lowest = sc->lowest, cursor = sc->cursor, window = sc->window, accepts = sc->accepts;
    unsigned state_unsure = sc->state_unsure, halt = state_unsure ? 1u : 0u, mw = 0;
    bool touched = false;  // an acceptance happened in this launch: md / mb / total are this kernel's
    dvs_log2_stage_table(sm.ltab);
    for (unsigned i = tid; i < dim; i += NT) sm.S[i] = S_glob[i];
    for (unsigned j = tid; j < n; j += NT) {
        const unsigned r = M_glob[j];
        sm.members[0][j] = r;
        sm.mH[0][j] = H[r];
    }
    __syncthreads();
    const unsigned world = (unsigned)sh.world, rank = (unsigned)sh.rank, Gw = G * world;
    const unsigned wmin = max(1u, Gw / 4u);
    if (tid == 0) sm.dead = 0;
    // loop-invariant factors of fast_bound / fast_total_ok (same expressions, same rounding)
    const double kb0 = ((double)dim + fast_slack(dim) + 16.0) * 1.2e-16;
    const double kb4 = ((double)dim + fast_slack(dim, kSmDepth) + 16.0) * 1.2e-16;
    const double lim0 = ((double)dim + 1.0 - fast_slack(dim) - 2.0) * 1.1102230246251565e-16;
    const double lim4 = ((double)dim + 1.0 - fast_slack(dim, kSmDepth) - 2.0) * 1.1102230246251565e-16;
    auto total_ok = [](double t, double lim) { return lim > 0.0 && fabs(t - 1.0) <= lim; };
    unsigned xs = 0, xu = 0;       // scan / update exchanges so far (= tags)
    unsigned cbase = 0, cend = 0;  // positions [cbase, cend) of `order` are staged in shared memory
    unsigned limit = ready_pos ? min(limit0, num) : num;  // positions below it may be examined

    while (!halt && cursor < num) {
        stamp(0);
        if (xs >= 0xFFFF0u) {  // exchange tags of one launch are 20 bits: let the host start a new launch
            halt = 1;
            break;
        }
        if (ready_pos && limit >= num) break;  // everything is published: hand over to the stand-alone kernel
        window = max(1u, min(window, min(Gw, CHUNK)));
        const unsigned P = (dim >= 2048u && window * 4u <= Gw) ? 4u : ((dim >= 2048u && window * 2u <= Gw) ? 2u : 1u);
        const unsigned count = min(window, limit - cursor);
        // this GPU's candidates: window positions p with p % world == rank, i.e. offsets woff + world * i
        const unsigned woff = (rank + world - cursor % world) % world;
        const unsigned nloc = count > woff ? (count - woff + world - 1u) / world : 0u;
        if (cursor < cbase || cursor + count > cend) {  // stage the next chunk of positions (CTA-uniform)
            __syncthreads();
            cbase = cursor;
            cend = min(limit, cbase + CHUNK);
            for (unsigned q = tid; cbase + q < cend; q += NT) {
                const unsigned row = order[cbase + q];
                sm.crow[q] = row;
                // (through L2: in trailing mode a neighbouring entry of the same line may have been cached before
                // its record was published)
                sm.cvalid[q] = __ldcg(valid + row);
                sm.cH[q] = __ldcg(H + row);
            }
            // ... and pull the rows this GPU will score towards L2, one 128-byte line per prefetch, dealt over the CTAs
            for (unsigned r = (rank + world - cbase % world) % world + world * b; r < cend - cbase; r += world * G) {
                const double* fr = F + (size_t)order[cbase + r] * dim;
                for (unsigned l = tid * 16u; l < dim; l += NT * 16u)
                    asm volatile("prefetch.global.L2 [%0];" ::"l"(fr + l));
            }
            __syncthreads();
        }
        const unsigned coff = cursor - cbase;
        if (tid == 0) {
            sm.ft = kNone;
            sm.fu = kNone;
        }
        for (unsigned q = tid; q < nloc; q += NT) sm.wskip[q] = sm.cvalid[coff + woff + world * q] ? 0 : 1;
        // ---- scan: slice p of candidate c ----
        ++xs;
        SmPart* const sbuf = spart + (xs & 1u) * kSmMaxGrid;
        const unsigned c = b / P, p = b % P;  // c: index among this GPU's candidates of the window
        const unsigned cw = woff + world * c;  // ... and its offset inside the window
        const double* fl = F + (size_t)sm.members[mw][lowest] * dim;
        if (c < nloc && sm.cvalid[coff + cw]) {  // CTA-uniform (a member's score is published but never read)
            const double* fc = F + (size_t)sm.crow[coff + cw] * dim;
            const unsigned lo = (unsigned)(((uint64_t)dim * p) / P), hi = (unsigned)(((uint64_t)dim * (p + 1)) / P);
            auto num = [&](unsigned i) { return __dadd_rn(__dsub_rn(sm.S[i], fl[i]), fc[i]); };
            const FastSum h = P == 4u   ? block_entropy_ilp<false, 2, NT>(lo, hi, num, div_n, sm.ltab)
                              : P == 2u ? block_entropy_ilp<false, 4, NT>(lo, hi, num, div_n, sm.ltab)
                                        : block_entropy_ilp<false, 8, NT>(lo, hi, num, div_n, sm.ltab);
            if (tid == 0) sm_publish(sbuf + b, h, xs);
        } else if (tid == 0) {
            // every CTA publishes in every scan exchange: the leader's wait for all G slots is what bounds
            // how far any CTA can lag, i.e. what makes the reuse of all exchange slots safe
            sm_publish(sbuf + b, FastSum{0.0, 0.0, 0.0, 0}, xs);
        }
        stamp(1);
        // ---- gather + decision by the leader (CTA 0), broadcast of {first_true, first_unsure} ----
        // (an all-to-all gather — every CTA polling every slot — costs 2.2 us per exchange on 148 SMs, the
        // leader form 1.3 us: tools/microbench/gridsync_bench.cu)
        SmPart* const dslot = dpart + (xs & 1u);
        if (b == 0) {
            // a candidate that is already a member is skipped (records.rs:76-78): the replicated member list
            // is the ground truth, searched while the partials are still in flight (thread j holds member j
            // and walks the window)
            __syncthreads();  // wskip initialised (a CTA without a candidate has not passed a barrier yet)
            for (unsigned j = tid; j < n; j += NT) {
                const unsigned r = sm.members[mw][j];
                for (unsigned cc = 0; cc < nloc; ++cc)
                    if (sm.crow[coff + woff + world * cc] == r) sm.wskip[cc] = 1;
            }
            __syncthreads();
            for (unsigned q = tid; q < G; q += NT) {
                const FastSum g = sm_gather(sbuf + q, xs);
                if (q < nloc * P && !sm.wskip[q / P]) {
                    sm.pe[q] = g.e; sm.pt[q] = g.t; sm.pa[q] = g.a; sm.pbad[q] = (unsigned char)g.bad;
                }
            }
            __syncthreads();
            stamp(2);
            for (unsigned lc = tid; lc < nloc; lc += NT) {
                if (sm.wskip[lc]) continue;
                FastSum h{sm.pe[lc * P], sm.pt[lc * P], sm.pa[lc * P], sm.pbad[lc * P]};
                for (unsigned q = 1; q < P; ++q) {
                    h.e += sm.pe[lc * P + q]; h.t += sm.pt[lc * P + q]; h.a += sm.pa[lc * P + q];
                    h.bad |= sm.pbad[lc * P + q];
                }
                const unsigned pos = cursor + woff + world * lc;
                const double mean_entropy =
                    div_exact(__dadd_rn(__dsub_rn(E, sm.mH[mw][lowest]), sm.cH[pos - cbase]), div_n);
                const double d = h.e - mean_entropy;
                const double bd = (P > 1u ? kb4 : kb0) * (h.a + fabs(mean_entropy) + 1.0);
                const double thr = total_jsd + kEps, tb = total_bound + 4.0 * kEps;
                if (h.bad || !total_ok(h.t, P > 1u ? lim4 : lim0) || !(d == d)) {
                    atomicMin(&sm.fu, pos);
                } else if (d - bd > thr + tb) {
                    atomicMin(&sm.ft, pos);
                } else if (!(d + bd < thr - tb)) {
                    atomicMin(&sm.fu, pos);
                }
            }
            __syncthreads();
            if (world > 1u) {  // the leaders' all-reduce(min) over NVLink
                const unsigned lft = sm.ft, lfu = sm.fu;
                __syncthreads();
                shard_exchange_min(sh, xs, lft, lfu, &sm.ft, &sm.fu, &sm.dead);
                __syncthreads();
                if (sm.dead) {  // a peer is gone: stop everything (the host reports the error)
                    if (tid == 0) {
                        sm.ft = kNone;
                        sm.fu = 0u;
                        sc->panic = 2u;
                    }
                    __syncthreads();
                }
            }
            if (tid == 0) {
                unsigned nl = limit;
                if (ready_pos) nl = max(limit, min(num, *reinterpret_cast<const volatile unsigned*>(ready_pos)));
                sm.limit = nl;
                sm_st128(&dslot->w[0], ((unsigned long long)sm.fu << 32) | sm.ft, ((unsigned long long)nl << 32) | xs);
            }
            __syncthreads();  // sm.limit
        } else {
            if (tid == 0) {
                unsigned long long w0, w1;
                do sm_ld128(&dslot->w[0], w0, w1); while ((unsigned)w1 != xs);
                sm.ft = (unsigned)w0;
                sm.fu = (unsigned)(w0 >> 32);
                sm.limit = (unsigned)(w1 >> 32);
            }
            stamp(2);
            __syncthreads();
        }
        const unsigned ft = sm.ft, fu = sm.fu;
        const unsigned next_limit = sm.limit;
        __syncthreads();
        stamp(3);
        if (fu < ft) {  // the first interesting candidate is undecided: the host resolves it exactly
            halt = 1;
            break;
        }
        if (ft == kNone) {  // empty window (or, trailing, nothing published beyond the cursor yet)
            cursor += count;
            if (count) window = min(window * 2u, Gw);
            limit = next_limit;
            stamp(4); stamp(5); stamp(6);
            ++tr_round;
            continue;
        }
        // ---- accept: replace_lowest + leave-one-out update ----
        const unsigned cand = sm.crow[ft - cbase];
        const double Hc = sm.cH[ft - cbase];
        const double E_new = __dadd_rn(__dsub_rn(E, sm.mH[mw][lowest]), Hc);  // records.rs:101,129
        const double* fc = F + (size_t)cand * dim;
        auto member_after = [&](unsigned j) {  // Vec::remove(lowest) + push(cand)
            return j < lowest ? sm.members[mw][j] : (j + 1 < n ? sm.members[mw][j + 1] : cand);
        };
        auto s_new = [&](unsigned i) {
            double s = __dsub_rn(sm.S[i], fl[i]);
            if (s <= kEps) s = 0.0;
            return __dadd_rn(s, fc[i]);
        };
        ++xu;
        bool have_S = false;
        for (unsigned j = b; j <= n; j += G) {
            FastSum h;
            if (j == n) {
                h = block_entropy_ilp<false, 8, NT>(0u, dim, [&](unsigned i) {
                    const double s = have_S ? sm.S[i] : s_new(i);
                    if (!have_S) sm.S[i] = s;
                    return s;
                }, div_n, sm.ltab);
            } else {
                const double* f = F + (size_t)member_after(j) * dim;
                h = block_entropy_ilp<true, 8, NT>(0u, dim, [&](unsigned i) {
                    const double s = have_S ? sm.S[i] : s_new(i);
                    if (!have_S) sm.S[i] = s;
                    return __dsub_rn(s, f[i]);
                }, div_n1, sm.ltab);
            }
            if (tid == 0) sm_publish(upart + j, h, xu);
            have_S = true;
        }
        if (!have_S)
            for (unsigned i = tid; i < dim; i += NT) sm.S[i] = s_new(i);
        stamp(4);
        // ---- every CTA: new member list; the leader: deltas + certified argmin, broadcast ----
        for (unsigned t = tid; t < n; t += NT) {
            sm.members[mw ^ 1][t] = member_after(t);
            sm.mH[mw ^ 1][t] = t < lowest ? sm.mH[mw][t] : (t + 1 < n ? sm.mH[mw][t + 1] : Hc);
        }
        if (tid == 0) sm.unsure = 0;
        __syncthreads();
        mw ^= 1;
        E = E_new;
        unsigned lo2 = 0, unsure = 0;
        SmPart* const fslot = dpart + 2;
        if (b == 0) {
            int uns = 0;
            for (unsigned t = tid; t <= n; t += NT) {
                const FastSum g = sm_gather(upart + t, xu);
                if (t == n) {
                    sm.pe[0] = g.e; sm.pa[0] = g.a;  // (scan staging is free again)
                } else {
                    const double mean_entropy = div_exact(__dsub_rn(E, sm.mH[mw][t]), div_n1);
                    sm.md[t] = g.e - mean_entropy;
                    sm.mb[t] = kb0 * (g.a + fabs(mean_entropy) + 1.0);
                }
                if (g.bad || !total_ok(g.t, lim0)) uns = 1;
            }
            if (uns) sm.unsure = 1;  // benign race: every writer stores 1
            __syncthreads();
            stamp(5);
            const double me = div_exact(E, div_n);
            total_jsd = sm.pe[0] - me;
            total_bound = kb0 * (sm.pa[0] + fabs(me) + 1.0);
            unsure = sm_finalize<NT>(sm.md, sm.mb, n, total_jsd, total_bound, &lo2);
            unsure |= sm.unsure;
            if (tid == 0) {
                sm_st128(&fslot->w[0], (unsigned long long)__double_as_longlong(total_jsd), ((unsigned long long)lo2 << 32) | xu);
                sm_st128(&fslot->w[2], (unsigned long long)__double_as_longlong(total_bound),
                         ((unsigned long long)unsure << 32) | xu);
            }
        } else {
            if (tid == 0) {
                unsigned long long w0, w1, w2, w3;
                do sm_ld128(&fslot->w[0], w0, w1); while ((unsigned)w1 != xu);
                do sm_ld128(&fslot->w[2], w2, w3); while ((unsigned)w3 != xu);
                sm.pe[0] = __longlong_as_double((long long)w0);
                sm.pa[0] = __longlong_as_double((long long)w2);
                sm.ft = (unsigned)(w1 >> 32);
                sm.unsure = (unsigned)(w3 >> 32);
            }
            __syncthreads();
            stamp(5);
            total_jsd = sm.pe[0];
            total_bound = sm.pa[0];
            lo2 = sm.ft;
            unsure = sm.unsure;
            __syncthreads();
        }
        lowest = lo2;
        touched = true;
        limit = next_limit;
        window = max(wmin, min(Gw, 2u * (ft - cursor + 1u)));
        cursor = ft + 1u;
        ++accepts;
        stamp(6);
        ++tr_round;
        if (unsure) {  // the argmin / a sum check could not be certified: the host redoes the update exactly
            state_unsure = 1;
            halt = 1;
            break;
        }
    }
    stamp(0);

    // ---- CTA 0 hands the state back in the layout the other kernels and the host loop use ----
    if (b == 0) {
        __syncthreads();
        if (touched) {
            for (unsigned i = tid; i < dim; i += NT) S_glob[i] = sm.S[i];
            for (unsigned j = tid; j < n; j += NT) is_member[M_glob[j]] = 0;  // the set at entry
            __syncthreads();
            for (unsigned j = tid; j < n; j += NT) {
                const unsigned r = sm.members[mw][j];
                M_glob[j] = r;
                is_member[r] = 1;
                mdelta_g[j] = sm.md[j];
                mbound_g[j] = sm.mb[j];
            }
        }
        if (tid == 0) {
            if (touched) {
                sc->E = E;
                sc->total_jsd = total_jsd;
                sc->total_bound = total_bound;
                sc->lowest = lowest;
                sc->exact = 0;
            }
            sc->state_unsure = state_unsure;
            sc->ticket = 0;
            sc->first_true = kNone;
            sc->first_panic = kNone;
            sc->first_unsure = kNone;
            sc->cursor = cursor;
            sc->window = window;
            sc->accepts = accepts;
            sc->halt = halt;
            sc->limit = limit;
        }
    }
}

