// sparse.cu — k-mer counting into SPARSE (index, count) rows for tables that cannot be held as dense rows
// (9 <= k <= 12, num_states = 4: 4^12 bins x 8 B = 134 MB per record dense, 10.5k genomes = 1.4 TB).
//
// Same counting semantics as count.cu (/root/reference/src/record.rs:41-84); the output of a record is the list
// of its DISTINCT k-mers in ascending index order with their counts - exactly the non-zero entries of the
// reference's dense vector, so frequencies and the sequential-order entropy (record.rs:86-106, zeros are skipped
// there too) follow bit for bit.  Algorithmic bytes: L + 8 D_r per record (SURVEY.md §8d: 8.1 B/bp at k=12).
//
// A 4^12-bin table (64 MB as u32) fits neither shared memory nor, for more than one record at a time, the L2, and
// global RED.ADD into it runs at ~190 Gbp/s (DRAM-sector / L2-atomic bound, profiles/r1_hist_microbench.txt).
// Instead the keys are radix-partitioned so that every histogram lives in shared memory:
//   pass 0  k_sp_hist       per 32 KB item of sequence: shared-memory histogram of the key's HIGH bits (its
//                           bucket: 4^(k-6) buckets) -> item_hist[item][bucket] (u16)
//   scan    k_sp_scan       per record: prefix over its items and over the buckets -> where every (item, bucket)
//                           run goes, bucket_ptr[record][bucket]
//   pass 1  k_sp_partition  per item again: keys are placed bucket-sorted in a shared-memory stage (one ATOMS per
//                           key on a per-bucket cursor) and leave as contiguous runs: the LOW 12 bits (u16) of
//                           every key, grouped by bucket, in a 2 B/key scratch array (L2 resident per record)
//   pass 2  k_sp_bucket     per (record, bucket): 4096-bin shared-memory histogram of its low halves, non-zero
//                           bins emitted in order as (index, count); the slots between a bucket's distinct count
//                           and its key count are zero-filled (count 0 = "no entry", skipped by every consumer)
// Every sequence byte is read twice (the second time mostly from L2), a key costs three shared-memory atomics,
// and the 2-byte scratch is written and read once.
#include <stdlib.h>
#include <string.h>

#include <algorithm>

#include "common.cuh"
#include "entropy.cuh"
#include "sparse.cuh"

namespace dvs {

constexpr uint32_t kSpItemBytes = 32768;  // <= 32768 k-mers per item: u16 item histograms cannot overflow
constexpr int kSpThreads = 1024;
constexpr int kSpBucketThreads = 256;

struct SpItem {
    uint64_t begin, end;  // 16-byte aligned absolute byte range
    uint32_t rec, pad;
};

__device__ __forceinline__ uint32_t sp_pack4(uint32_t w) { return (w * 0x40100401u) >> 24; }
__device__ __forceinline__ uint32_t sp_pack16(uint4 v) {
    return (sp_pack4(v.x) << 24) | (sp_pack4(v.y) << 16) | (sp_pack4(v.z) << 8) | sp_pack4(v.w);
}

// f(key) for every valid k-mer whose LAST byte lies in the item (2 k-bit key, first base most significant)
template <class F>
__device__ __forceinline__ void sp_for_each_kmer(const uint8_t* __restrict__ seqs, const SpItem& w, uint64_t start,
                                                 uint64_t end, int k, uint32_t mask, F f) {
    for (uint64_t a = w.begin + (uint64_t)threadIdx.x * 16; a < w.end; a += (uint64_t)blockDim.x * 16) {
        const uint4 cur = __ldg(reinterpret_cast<const uint4*>(seqs + a));
        const uint4 prev = __ldg(reinterpret_cast<const uint4*>(seqs + a - 16));  // front pad keeps this in bounds
        const uint32_t any = cur.x | cur.y | cur.z | cur.w | prev.x | prev.y | prev.z | prev.w;
        if (((any & 0xFCFCFCFCu) == 0) && a >= start + 16 && a + 16 <= end) {
            const uint32_t pc = sp_pack16(cur), pp = sp_pack16(prev);
#pragma unroll
            for (int j = 0; j < 15; ++j) f(__funnelshift_r(pc, pp, 2 * (15 - j)) & mask);
            f(pc & mask);
        } else {
            const uint32_t wv[8] = {prev.x, prev.y, prev.z, prev.w, cur.x, cur.y, cur.z, cur.w};
            uint32_t run = 0, v = 0;
#pragma unroll 1
            for (int i = 0; i < 32; ++i) {
                const uint64_t p = a - 16 + i;
                uint32_t b = (wv[i >> 2] >> (8 * (i & 3))) & 0xFFu;
                if (p < start || p >= end) b = 0xFFu;
                if (b >= 4u) {
                    run = 0;
                    v = 0;
                } else {
                    v = ((v << 2) | b) & mask;
                    ++run;
                    if (i >= 16 && run >= (uint32_t)k) f(v);
                }
            }
        }
    }
}

// block-wide exclusive scan of one value per thread (kSpThreads or fewer threads, all must call)
__device__ __forceinline__ uint32_t sp_block_exscan(uint32_t v, uint32_t* s_warp /* >= 33 words */, uint32_t* total) {
    const unsigned lane = threadIdx.x & 31, wid = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    uint32_t inc = v;
    for (int o = 1; o < 32; o <<= 1) {
        const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= (unsigned)o) inc += t;
    }
    if (lane == 31) s_warp[wid] = inc;
    __syncthreads();
    if (wid == 0) {
        uint32_t x = lane < nw ? s_warp[lane] : 0u, xi = x;
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, xi, o);
            if (lane >= (unsigned)o) xi += t;
        }
        s_warp[lane] = xi - x;
        if (lane == 31) s_warp[32] = xi;
    }
    __syncthreads();
    const uint32_t r = s_warp[wid] + inc - v;
    *total = s_warp[32];
    __syncthreads();
    return r;
}

__global__ void __launch_bounds__(kSpThreads)
k_sp_hist(const uint8_t* __restrict__ seqs, const uint64_t* __restrict__ offsets, const SpItem* __restrict__ items,
          uint32_t nitems, int k, uint32_t nb, uint16_t* __restrict__ item_hist) {
    extern __shared__ uint32_t sp_smem[];
    uint32_t* hist = sp_smem;
    const uint32_t mask = (1u << (2 * k)) - 1u;
    for (uint32_t it = blockIdx.x; it < nitems; it += gridDim.x) {
        const SpItem w = items[it];
        for (uint32_t b = threadIdx.x; b < nb; b += kSpThreads) hist[b] = 0;
        __syncthreads();
        sp_for_each_kmer(seqs, w, offsets[w.rec], offsets[w.rec + 1], k, mask,
                         [&](uint32_t key) { atomicAdd(&hist[key >> kSpLowBits], 1u); });
        __syncthreads();
        for (uint32_t b = threadIdx.x; b < nb; b += kSpThreads) item_hist[(size_t)it * nb + b] = (uint16_t)hist[b];
        __syncthreads();
    }
}

// one CTA per record: bucket totals over its items, exclusive scan over the buckets, then the offset (inside the
// record's region) of every (item, bucket) run
__global__ void __launch_bounds__(kSpThreads)
k_sp_scan(const uint16_t* __restrict__ item_hist, const uint32_t* __restrict__ rec_item_begin, uint32_t nb,
          uint32_t* __restrict__ item_off, uint32_t* __restrict__ bucket_ptr, uint64_t* __restrict__ totals,
          uint8_t* __restrict__ valid) {
    __shared__ uint32_t s_warp[34];
    const uint32_t rec = blockIdx.x, i0 = rec_item_begin[rec], i1 = rec_item_begin[rec + 1];
    const uint32_t per = (nb + kSpThreads - 1) / kSpThreads;  // consecutive buckets per thread (<= 4)
    const uint32_t b0 = threadIdx.x * per;
    uint32_t tot[4] = {0, 0, 0, 0};
    for (uint32_t it = i0; it < i1; ++it)
        for (uint32_t q = 0; q < per; ++q)
            if (b0 + q < nb) {
                const size_t at = (size_t)it * nb + b0 + q;
                item_off[at] = tot[q];  // offset inside the bucket, completed below
                tot[q] += item_hist[at];
            }
    uint32_t mine = 0;
    for (uint32_t q = 0; q < per; ++q) mine += tot[q];
    uint32_t total = 0;
    uint32_t base = sp_block_exscan(mine, s_warp, &total);
    uint32_t bstart[4];
    for (uint32_t q = 0; q < per; ++q) {
        bstart[q] = base;
        if (b0 + q < nb) bucket_ptr[(size_t)rec * (nb + 1) + b0 + q] = base;
        base += tot[q];
    }
    if (threadIdx.x == 0) {
        bucket_ptr[(size_t)rec * (nb + 1) + nb] = total;
        totals[rec] = total;
        valid[rec] = total ? 1 : 0;
    }
    for (uint32_t it = i0; it < i1; ++it)
        for (uint32_t q = 0; q < per; ++q)
            if (b0 + q < nb) item_off[(size_t)it * nb + b0 + q] += bstart[q];
}

__global__ void __launch_bounds__(kSpThreads)
k_sp_partition(const uint8_t* __restrict__ seqs, const uint64_t* __restrict__ offsets, const SpItem* __restrict__ items,
               uint32_t nitems, int k, uint32_t nb, const uint16_t* __restrict__ item_hist,
               const uint32_t* __restrict__ item_off, uint16_t* __restrict__ lowbuf) {
    extern __shared__ uint32_t sp_smem[];
    __shared__ uint32_t s_warp[34];
    uint32_t* stage = sp_smem;                 // [kSpItemBytes] bucket-sorted keys of the item
    uint32_t* lcur = stage + kSpItemBytes;     // [nb] cursor inside the stage
    uint32_t* goff = lcur + nb;                // [nb] (first slot of this item's run in the record's region) - (its stage slot)
    const uint32_t mask = (1u << (2 * k)) - 1u;
    const uint32_t per = (nb + kSpThreads - 1) / kSpThreads, b0 = threadIdx.x * per;
    for (uint32_t it = blockIdx.x; it < nitems; it += gridDim.x) {
        const SpItem w = items[it];
        const uint64_t start = offsets[w.rec], end = offsets[w.rec + 1];
        uint32_t cnt[4] = {0, 0, 0, 0}, mine = 0;
        for (uint32_t q = 0; q < per; ++q)
            if (b0 + q < nb) {
                cnt[q] = item_hist[(size_t)it * nb + b0 + q];
                mine += cnt[q];
                goff[b0 + q] = item_off[(size_t)it * nb + b0 + q];
            }
        uint32_t n = 0;
        uint32_t base = sp_block_exscan(mine, s_warp, &n);
        for (uint32_t q = 0; q < per; ++q)
            if (b0 + q < nb) {
                lcur[b0 + q] = base;
                goff[b0 + q] -= base;  // stage slot e of bucket b goes to slot goff[b] + e of the record's region
                base += cnt[q];
            }
        __syncthreads();
        sp_for_each_kmer(seqs, w, start, end, k, mask, [&](uint32_t key) {
            const uint32_t slot = atomicAdd(&lcur[key >> kSpLowBits], 1u);
            stage[slot] = key;
        });
        __syncthreads();
        uint16_t* dst = lowbuf + start;  // the record's region starts at its byte offset (#k-mers <= #bytes)
        for (uint32_t e = threadIdx.x; e < n; e += kSpThreads) {
            const uint32_t key = stage[e], b = key >> kSpLowBits;
            dst[goff[b] + e] = (uint16_t)(key & (kSpLowBins - 1u));  // (mod 2^32: goff may have wrapped)
        }
        __syncthreads();
    }
}

__global__ void __launch_bounds__(kSpBucketThreads)
k_sp_bucket(const uint16_t* __restrict__ lowbuf, const uint64_t* __restrict__ offsets, const uint32_t* __restrict__ bucket_ptr,
            uint32_t nrec, uint32_t nb, uint32_t* __restrict__ out_idx, uint32_t* __restrict__ out_cnt,
            uint32_t* __restrict__ bucket_nnz, const uint64_t* __restrict__ list, const uint32_t* __restrict__ list_count) {
    __shared__ __align__(16) uint32_t hist[kSpLowBins];
    __shared__ uint32_t s_warp[34];
    // list == NULL: every (record, bucket) pair; otherwise the listed pairs only (buckets too large for 16-bit bins)
    const uint64_t npairs = list ? (uint64_t)*list_count : (uint64_t)nrec * nb;
    constexpr uint32_t kBinsPer = kSpLowBins / kSpBucketThreads;  // 16 consecutive bins per thread
    for (uint64_t q = blockIdx.x; q < npairs; q += gridDim.x) {
        const uint64_t p = list ? list[q] : q;
        const uint32_t rec = (uint32_t)(p / nb), b = (uint32_t)(p % nb);
        const uint32_t* bp = bucket_ptr + (size_t)rec * (nb + 1);
        const uint32_t s0 = bp[b], n = bp[b + 1] - s0;
        if (n == 0) {  // CTA-uniform
            if (threadIdx.x == 0) bucket_nnz[p] = 0;
            continue;
        }
        const uint64_t base = offsets[rec] + s0;
        uint4* h4 = reinterpret_cast<uint4*>(hist);
        for (uint32_t i = threadIdx.x; i < kSpLowBins / 4; i += kSpBucketThreads) h4[i] = make_uint4(0, 0, 0, 0);
        __syncthreads();
        for (uint32_t e = threadIdx.x; e < n; e += kSpBucketThreads) atomicAdd(&hist[lowbuf[base + e]], 1u);
        __syncthreads();
        uint32_t c[kBinsPer], mine = 0;
#pragma unroll
        for (uint32_t q = 0; q < kBinsPer; q += 4) {
            const uint4 v = h4[(threadIdx.x * kBinsPer + q) / 4];
            c[q] = v.x; c[q + 1] = v.y; c[q + 2] = v.z; c[q + 3] = v.w;
        }
#pragma unroll
        for (uint32_t q = 0; q < kBinsPer; ++q) mine += c[q] ? 1u : 0u;
        uint32_t nnz = 0;
        uint32_t pos = sp_block_exscan(mine, s_warp, &nnz);
#pragma unroll
        for (uint32_t q = 0; q < kBinsPer; ++q)
            if (c[q]) {
                out_idx[base + pos] = (b << kSpLowBits) | (threadIdx.x * kBinsPer + q);
                out_cnt[base + pos] = c[q];
                ++pos;
            }
        for (uint32_t e = nnz + threadIdx.x; e < n; e += kSpBucketThreads) {  // unused slots of the bucket: "no entry"
            out_idx[base + e] = 0xFFFFFFFFu;
            out_cnt[base + e] = 0u;
        }
        if (threadIdx.x == 0) bucket_nnz[p] = nnz;
        __syncthreads();
    }
}

// pass 2, warp form: ONE WARP per (record, bucket) - no block barriers, 8 KB of shared memory per warp (4,096 bins
// as 16-bit halves of 2,048 words, safe while the bucket has fewer than 65,536 keys; larger buckets are listed and
// left to k_sp_bucket).  The bins are walked one word per lane and iteration, so that the 32 lanes hold 64
// consecutive bins and the non-zero ones are compacted with two ballots: consecutive lanes write consecutive
// output slots (coalesced), and no counting pre-pass is needed.
constexpr int kSpWarpsPerCta = 8;
__global__ void __launch_bounds__(32 * kSpWarpsPerCta)
k_sp_bucket_warp(const uint16_t* __restrict__ lowbuf, const uint64_t* __restrict__ offsets,
                 const uint32_t* __restrict__ bucket_ptr, uint32_t nrec, uint32_t nb, uint32_t* __restrict__ out_idx,
                 uint32_t* __restrict__ out_cnt, uint32_t* __restrict__ bucket_nnz, uint64_t* __restrict__ big_list,
                 uint32_t* __restrict__ big_count, const uint64_t* __restrict__ list,
                 const uint32_t* __restrict__ list_count) {
    extern __shared__ __align__(16) uint32_t sp_wsmem[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    uint32_t* h = sp_wsmem + warp * (kSpLowBins / 2);
    // list == NULL: every (record, bucket) pair; otherwise the pairs k_sp_bucket_bits left
    const uint64_t npairs = list ? (uint64_t)*list_count : (uint64_t)nrec * nb;
    const uint32_t lt = (1u << lane) - 1u;
    const int nb_log2 = __ffs(nb) - 1;
    for (uint64_t q = (uint64_t)blockIdx.x * kSpWarpsPerCta + warp; q < npairs; q += (uint64_t)gridDim.x * kSpWarpsPerCta) {
        const uint64_t p = list ? list[q] : q;
        const uint32_t rec = (uint32_t)(p >> nb_log2), b = (uint32_t)p & (nb - 1u);  // (nb = 4^(k-6))
        const uint32_t* bp = bucket_ptr + (size_t)rec * (nb + 1);
        const uint32_t s0 = bp[b], n = bp[b + 1] - s0;
        if (n == 0) {
            if (lane == 0) bucket_nnz[p] = 0;
            continue;
        }
        if (n > 65535u) {  // a 16-bit half could overflow: the CTA kernel with 32-bit bins takes this bucket
            if (lane == 0) big_list[atomicAdd(big_count, 1u)] = p;
            continue;
        }
        const uint64_t base = offsets[rec] + s0;
        uint4* h4 = reinterpret_cast<uint4*>(h);
#pragma unroll 4
        for (uint32_t i = lane; i < kSpLowBins / 8; i += 32) h4[i] = make_uint4(0, 0, 0, 0);
        __syncwarp();
        for (uint32_t e = lane; e < n; e += 32) {
            const uint32_t key = lowbuf[base + e];
            atomicAdd(&h[key >> 1], (key & 1u) ? 0x10000u : 1u);
        }
        __syncwarp();
        uint32_t run = 0;
        const uint32_t idx_hi = b << kSpLowBits;
#pragma unroll 4
        for (uint32_t i = 0; i < kSpLowBins / 64; ++i) {
            const uint32_t wd = i * 32 + lane, v = h[wd];
            const uint32_t lo = v & 0xFFFFu, hi = v >> 16;
            const uint32_t mlo = __ballot_sync(0xffffffffu, lo != 0), mhi = __ballot_sync(0xffffffffu, hi != 0);
            uint32_t pos = run + __popc(mlo & lt) + __popc(mhi & lt);
            if (lo) {
                out_idx[base + pos] = idx_hi | (2 * wd);
                out_cnt[base + pos] = lo;
                ++pos;
            }
            if (hi) {
                out_idx[base + pos] = idx_hi | (2 * wd + 1);
                out_cnt[base + pos] = hi;
            }
            run += __popc(mlo) + __popc(mhi);
        }
        for (uint32_t e = run + lane; e < n; e += 32) {  // unused slots of the bucket: "no entry"
            out_idx[base + e] = 0xFFFFFFFFu;
            out_cnt[base + e] = 0u;
        }
        if (lane == 0) bucket_nnz[p] = run;
        __syncwarp();
    }
}

// pass 2, bitmap form - for the SPARSELY occupied buckets of k = 11, 12 (a bucket of ~1,000 keys over 4,096 bins:
// three quarters of the keys are the only one of their bin).  Walking 4,096 counters for 1,000 keys made
// k_sp_bucket_warp instruction bound (4.2 warp instructions per key); here a warp
//   1. sets the bit of every key in a 4,096-bit occupancy bitmap (atomicOr),
//   2. forms the prefix of the bitmap's word popcounts: rank(bin) = pre[word] + popc(bits below) is the position of
//      the bin among the distinct ones,
//   3. reads the keys again (L1 hits) and, for each, stores the bin at its rank in a 16-bit stage and adds one to a
//      16-bit count stage at that rank (every occurrence writes the same bin: no "first occurrence" logic),
//   4. writes the row from the two stages with coalesced stores.
// All loops are warp-uniform.  Buckets with more than kSpBitsMaxDistinct distinct keys (or 65,535 keys) are listed
// for k_sp_bucket_warp.
constexpr uint32_t kSpBitsMaxDistinct = 2048;
constexpr int kSpBitsWarps = 8;
struct __align__(16) SpBitsWarp {
    uint32_t bm[kSpLowBins / 32];
    uint32_t pre[kSpLowBins / 32];
    uint32_t cnt[kSpBitsMaxDistinct / 2];  // 16-bit halves
    uint16_t idx[kSpBitsMaxDistinct];
};
__global__ void __launch_bounds__(32 * kSpBitsWarps)
k_sp_bucket_bits(const uint16_t* __restrict__ lowbuf, const uint64_t* __restrict__ offsets,
                 const uint32_t* __restrict__ bucket_ptr, uint32_t nrec, uint32_t nb, uint32_t* __restrict__ out_idx,
                 uint32_t* __restrict__ out_cnt, uint32_t* __restrict__ bucket_nnz, uint64_t* __restrict__ mid_list,
                 uint32_t* __restrict__ mid_count) {
    extern __shared__ __align__(16) unsigned char sp_bits_raw[];
    const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    SpBitsWarp& sw = reinterpret_cast<SpBitsWarp*>(sp_bits_raw)[warp];
    const uint64_t npairs = (uint64_t)nrec * nb, stride = (uint64_t)gridDim.x * kSpBitsWarps;
    const int nb_log2 = __ffs(nb) - 1;
    // (s0, n, record base) of a pair; the next pair's are fetched while the current one is processed
    auto fetch = [&](uint64_t p, uint32_t& s0, uint32_t& n, uint64_t& rbase) {
        if (p < npairs) {
            const uint32_t rec = (uint32_t)(p >> nb_log2), b = (uint32_t)p & (nb - 1u);  // (nb = 4^(k-6))
            const uint32_t* bp = bucket_ptr + (size_t)rec * (nb + 1);
            s0 = __ldg(bp + b);
            n = __ldg(bp + b + 1) - s0;
            rbase = __ldg(offsets + rec);
        }
    };
    uint64_t p = (uint64_t)blockIdx.x * kSpBitsWarps + warp;
    uint32_t s0 = 0, n = 0, s0_next = 0, n_next = 0;
    uint64_t rbase = 0, rbase_next = 0;
    fetch(p, s0, n, rbase);
    for (; p < npairs; p += stride, s0 = s0_next, n = n_next, rbase = rbase_next) {
        fetch(p + stride, s0_next, n_next, rbase_next);
        if (n == 0) {
            if (lane == 0) bucket_nnz[p] = 0;
            continue;
        }
        if (n > 65535u) {  // (warp-uniform) a 16-bit count could overflow
            if (lane == 0) mid_list[atomicAdd(mid_count, 1u)] = p;
            continue;
        }
        const uint64_t base = rbase + s0;
        const uint16_t* __restrict__ src = lowbuf + base;
        uint32_t* __restrict__ oi = out_idx + base;
        uint32_t* __restrict__ oc = out_cnt + base;
        reinterpret_cast<uint4*>(sw.bm)[lane] = make_uint4(0, 0, 0, 0);
        __syncwarp();
        // (the loops are kept compact on purpose: a fully unrolled, register-resident variant ran into instruction
        // cache misses - stall_no_instruction 5.8 per issue - and was slower)
        // batches of 256 keys (8 per lane); the next batch is loaded before the current one is used, and the last,
        // partial batch is a predicated one (0xFFFFFFFF = no key): one exposed memory latency per bucket instead of
        // one per batch plus one per 32 keys of the remainder
        auto load8 = [&](uint32_t e0, uint32_t (&kk)[8]) {
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                const uint32_t e = e0 + lane + 32u * q;
                kk[q] = e < n ? (uint32_t)__ldg(src + e) : 0xFFFFFFFFu;
            }
        };
        uint32_t ka[8], kb[8];
        load8(0, ka);
        for (uint32_t e0 = 0; e0 < n; e0 += 256) {
            load8(e0 + 256, kb);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                if (ka[q] != 0xFFFFFFFFu) atomicOr(&sw.bm[ka[q] >> 5], 1u << (ka[q] & 31u));
                ka[q] = kb[q];
            }
        }
        __syncwarp();
        // rank of every bitmap word among the distinct bins
        const uint4 m4 = reinterpret_cast<const uint4*>(sw.bm)[lane];
        const uint32_t c0 = __popc(m4.x), c1 = __popc(m4.y), c2 = __popc(m4.z), c3 = __popc(m4.w);
        const uint32_t mine = c0 + c1 + c2 + c3;
        uint32_t inc = mine;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= (uint32_t)o) inc += t;
        }
        const uint32_t nnz = __shfl_sync(0xffffffffu, inc, 31), excl = inc - mine;
        if (nnz > kSpBitsMaxDistinct) {  // (warp-uniform)
            if (lane == 0) mid_list[atomicAdd(mid_count, 1u)] = p;
            __syncwarp();
            continue;
        }
        reinterpret_cast<uint4*>(sw.pre)[lane] = make_uint4(excl, excl + c0, excl + c0 + c1, excl + c0 + c1 + c2);
        for (uint32_t i = lane; i < (nnz + 7) / 8; i += 32) reinterpret_cast<uint4*>(sw.cnt)[i] = make_uint4(0, 0, 0, 0);
        __syncwarp();
        auto place = [&](uint32_t key) {
            const uint32_t w = key >> 5;
            const uint32_t r = sw.pre[w] + __popc(sw.bm[w] & ((1u << (key & 31u)) - 1u));
            sw.idx[r] = (uint16_t)key;
            atomicAdd(&sw.cnt[r >> 1], (r & 1u) ? 0x10000u : 1u);
        };
        load8(0, ka);  // (L1 hits)
        for (uint32_t e0 = 0; e0 < n; e0 += 256) {
            load8(e0 + 256, kb);
#pragma unroll
            for (int q = 0; q < 8; ++q) {
                if (ka[q] != 0xFFFFFFFFu) place(ka[q]);
                ka[q] = kb[q];
            }
        }
        __syncwarp();
        const uint32_t idx_hi = ((uint32_t)p & (nb - 1u)) << kSpLowBits;
        // two entries per lane and step, from the first slot that is 8-byte aligned in the output
        const uint16_t* cnt16 = reinterpret_cast<const uint16_t*>(sw.cnt);
        const uint32_t first = (uint32_t)base & 1u;
        if (first && lane == 0) {
            oi[0] = idx_hi | sw.idx[0];
            oc[0] = cnt16[0];
        }
        const uint32_t pairs = (nnz - first) >> 1;
        for (uint32_t q = lane; q < pairs; q += 32) {
            const uint32_t a = first + 2u * q;
            *reinterpret_cast<uint2*>(oi + a) = make_uint2(idx_hi | sw.idx[a], idx_hi | sw.idx[a + 1]);
            *reinterpret_cast<uint2*>(oc + a) = make_uint2(cnt16[a], cnt16[a + 1]);
        }
        if (((nnz - first) & 1u) && lane == 0) {
            oi[nnz - 1] = idx_hi | sw.idx[nnz - 1];
            oc[nnz - 1] = cnt16[nnz - 1];
        }
        for (uint32_t q = nnz + lane; q < n; q += 32) {  // unused slots of the bucket: "no entry"
            oi[q] = 0xFFFFFFFFu;
            oc[q] = 0u;
        }
        if (lane == 0) bucket_nnz[p] = nnz;
        __syncwarp();
    }
}

// distinct k-mers per record
__global__ void k_sp_nnz(const uint32_t* __restrict__ bucket_nnz, uint32_t nb, uint64_t* __restrict__ nnz) {
    __shared__ unsigned long long s_sum;
    if (threadIdx.x == 0) s_sum = 0;
    __syncthreads();
    unsigned long long part = 0;
    for (uint32_t b = threadIdx.x; b < nb; b += blockDim.x) part += bucket_nnz[(size_t)blockIdx.x * nb + b];
    for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_sum, part);
    __syncthreads();
    if (threadIdx.x == 0) nnz[blockIdx.x] = s_sum;
}

// exact entropy of every record from its sparse row: the reference's sequential sum over the non-zero
// frequencies in index order (slots with count 0 are x == 0.0, skipped like the zeros of the dense vector)
__global__ void __launch_bounds__(kEntThreads)
k_sp_entropy(const uint32_t* __restrict__ out_cnt, const uint64_t* __restrict__ offsets, const uint64_t* __restrict__ totals,
             uint64_t dim, double* __restrict__ entropy, uint8_t* __restrict__ err, double* __restrict__ err_total) {
    extern __shared__ __align__(16) double ent_smem[];
    const uint32_t r = blockIdx.x;
    const uint64_t total_u = totals[r];
    if (total_u == 0) {
        if (threadIdx.x == 0) {
            entropy[r] = 0.0;
            err[r] = 0;
            err_total[r] = 0.0;
        }
        return;
    }
    const uint32_t* c = out_cnt + offsets[r];
    const FastDiv dv = make_fast_div((double)total_u);
    EntropyResult h = block_entropy_exact(total_u, [&](uint64_t i) {
        const uint32_t v = c[i];
        return v ? div_exact((double)v, dv) : 0.0;
    }, ent_smem);
    if (threadIdx.x == 0) {
        entropy[r] = h.e;
        err[r] = entropy_total_bad(h.t, dim) ? 1 : 0;  // the reference's check uses the DENSE length (record.rs:101-104)
        err_total[r] = h.t;
    }
}

// one record's row without the empty slots (download path)
__global__ void __launch_bounds__(kSpThreads)
k_sp_compact(const uint32_t* __restrict__ out_idx, const uint32_t* __restrict__ out_cnt, const uint32_t* __restrict__ bucket_ptr,
             const uint32_t* __restrict__ bucket_nnz, uint64_t rec_base, uint32_t nb, uint32_t* __restrict__ idx,
             uint32_t* __restrict__ cnt) {
    __shared__ uint32_t s_warp[34];
    __shared__ uint32_t s_run;
    if (threadIdx.x == 0) s_run = 0;
    __syncthreads();
    for (uint32_t b0 = 0; b0 < nb; b0 += kSpThreads) {  // one bucket per thread and pass
        const uint32_t b = b0 + threadIdx.x;
        const uint32_t n = b < nb ? bucket_nnz[b] : 0u;
        uint32_t tot = 0;
        const uint32_t at = s_run + sp_block_exscan(n, s_warp, &tot);
        if (n) {
            const uint64_t src = rec_base + bucket_ptr[b];
            for (uint32_t e = 0; e < n; ++e) {
                idx[at + e] = out_idx[src + e];
                cnt[at + e] = out_cnt[src + e];
            }
        }
        __syncthreads();
        if (threadIdx.x == 0) s_run += tot;
        __syncthreads();
    }
}

}  // namespace dvs

using namespace dvs;

extern "C" {

int dvs_count_kmers_sparse(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, int want_entropy, dvs_ksparse** out) {
    if (!ctx || !s || !out) {
        set_error("dvs_count_kmers_sparse: NULL argument");
        return DVS_ERR_ARG;
    }
    if (num_states != 4 || k < 9 || k > 12) {
        set_error("dvs_count_kmers_sparse: supported for num_states = 4 and 9 <= k <= 12 (got k=%d, num_states=%d); "
                  "smaller tables are dense (dvs_count_kmers)", k, num_states);
        return DVS_ERR_ARG;
    }
    for (uint32_t r = 0; r < s->nrec; ++r)
        if (s->h_offsets[r + 1] - s->h_offsets[r] >= (1ULL << 32)) {
            set_error("dvs_count_kmers_sparse: record %u has 2^32 bases or more", r);
            return DVS_ERR_ARG;
        }
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    auto* sp = new dvs_ksparse();
    sp->device = ctx->device;
    sp->nrec = s->nrec;
    sp->k = k;
    sp->dim = 1ull << (2 * k);
    sp->nb = 1u << (2 * k - kSpLowBits);
    sp->slots = s->total;
    sp->h_offsets = s->h_offsets;
    const uint32_t nb = sp->nb, nrec = s->nrec;
    auto fail = [&](int rc) {
        dvs_ksparse_free(sp);
        return rc;
    };
    // items: 32 KB pieces of every record (record-major)
    std::vector<SpItem> items;
    std::vector<uint32_t> rec_item_begin(nrec + 1, 0);
    for (uint32_t r = 0; r < nrec; ++r) {
        rec_item_begin[r] = (uint32_t)items.size();
        const uint64_t b = s->h_offsets[r], e = s->h_offsets[r + 1];
        if (e <= b) continue;
        const uint64_t a0 = b & ~15ULL, a1 = (e + 15) & ~15ULL;
        for (uint64_t a = a0; a < a1; a += kSpItemBytes) items.push_back({a, std::min<uint64_t>(a + kSpItemBytes, a1), r, 0});
    }
    rec_item_begin[nrec] = (uint32_t)items.size();
    if (items.size() > 0x7FFFFFFFull) {
        set_error("dvs_count_kmers_sparse: too many work items");
        return fail(DVS_ERR_ARG);
    }
    const uint32_t nitems = (uint32_t)items.size();
    const size_t n1 = std::max<uint32_t>(nrec, 1);
    DevBuf<SpItem> d_items;
    DevBuf<uint32_t> d_rib, d_item_off;
    DevBuf<uint16_t> d_item_hist, d_low;
    int rc = d_items.alloc(std::max<uint32_t>(nitems, 1));
    if (rc == DVS_OK) rc = d_rib.alloc(nrec + 1);
    if (rc == DVS_OK) rc = d_item_hist.alloc((size_t)std::max<uint32_t>(nitems, 1) * nb);
    if (rc == DVS_OK) rc = d_item_off.alloc((size_t)std::max<uint32_t>(nitems, 1) * nb);
    if (rc == DVS_OK) rc = d_low.alloc(std::max<uint64_t>(s->total, 1) + 16);
    if (rc == DVS_OK) rc = sp->offsets.alloc(nrec + 1);
    if (rc == DVS_OK) rc = sp->idx.alloc(std::max<uint64_t>(s->total, 1));
    if (rc == DVS_OK) rc = sp->cnt.alloc(std::max<uint64_t>(s->total, 1));
    if (rc == DVS_OK) rc = sp->bucket_ptr.alloc(n1 * (nb + 1));
    if (rc == DVS_OK) rc = sp->bucket_nnz.alloc(n1 * nb);
    if (rc == DVS_OK) rc = sp->totals.alloc(n1);
    if (rc == DVS_OK) rc = sp->nnz.alloc(n1);
    if (rc == DVS_OK) rc = sp->entropy.alloc(n1);
    if (rc == DVS_OK) rc = sp->err_total.alloc(n1);
    if (rc == DVS_OK) rc = sp->valid.alloc(n1);
    if (rc == DVS_OK) rc = sp->err.alloc(n1);
    if (rc != DVS_OK) return fail(rc);
#define TRY_P(expr)                                                    \
    do {                                                               \
        cudaError_t _e = (expr);                                       \
        if (_e != cudaSuccess) {                                       \
            set_error("%s failed: %s", #expr, cudaGetErrorString(_e)); \
            return fail(DVS_ERR_CUDA);                                 \
        }                                                              \
    } while (0)
    TRY_P(cudaMemcpyAsync(d_items.p, items.data(), (size_t)nitems * sizeof(SpItem), cudaMemcpyHostToDevice, st));
    TRY_P(cudaMemcpyAsync(d_rib.p, rec_item_begin.data(), (nrec + 1) * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    TRY_P(cudaMemcpyAsync(sp->offsets.p, s->h_offsets.data(), (nrec + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, st));
    TRY_P(cudaMemsetAsync(sp->err.p, 0, n1, st));
    TRY_P(cudaMemsetAsync(sp->entropy.p, 0, n1 * sizeof(double), st));
    if (nrec && nitems) {
        PhaseTimer pt(ctx, DVS_PHASE_SPARSE);
        const size_t smem_hist = (size_t)nb * 4, smem_part = ((size_t)kSpItemBytes + 2 * (size_t)nb) * 4;
        TRY_P(cudaFuncSetAttribute(k_sp_partition, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_part));
        const unsigned g_hist = (unsigned)std::min<size_t>(nitems, (size_t)ctx->sm_count * 2);
        const unsigned g_part = (unsigned)std::min<size_t>(nitems, (size_t)ctx->sm_count);
        k_sp_hist<<<g_hist, kSpThreads, smem_hist, st>>>(s->data(), s->offsets.p, d_items.p, nitems, k, nb, d_item_hist.p);
        ctx->launches++;
        TRY_P(cudaGetLastError());
        k_sp_scan<<<nrec, kSpThreads, 0, st>>>(d_item_hist.p, d_rib.p, nb, d_item_off.p, sp->bucket_ptr.p, sp->totals.p,
                                               sp->valid.p);
        ctx->launches++;
        TRY_P(cudaGetLastError());
        k_sp_partition<<<g_part, kSpThreads, smem_part, st>>>(s->data(), s->offsets.p, d_items.p, nitems, k, nb,
                                                              d_item_hist.p, d_item_off.p, d_low.p);
        ctx->launches++;
        TRY_P(cudaGetLastError());
        const uint64_t npairs = (uint64_t)nrec * nb;
        // DVS_SPARSE_CTA_BUCKETS=1: the CTA-per-bucket kernel for everything (A/B measurements)
        const char* cta_env = getenv("DVS_SPARSE_CTA_BUCKETS");
        if (cta_env && cta_env[0] == '1') {
            const unsigned g_b = (unsigned)std::min<uint64_t>(npairs, (uint64_t)ctx->sm_count * 8 * 4);
            k_sp_bucket<<<g_b, kSpBucketThreads, 0, st>>>(d_low.p, sp->offsets.p, sp->bucket_ptr.p, nrec, nb, sp->idx.p,
                                                          sp->cnt.p, sp->bucket_nnz.p, nullptr, nullptr);
            ctx->launches++;
            TRY_P(cudaGetLastError());
        } else {
            // a bucket of more than 65,535 keys needs >= 65,536 k-mers that share their first k - 6 bases in one record
            DevBuf<uint64_t> d_big;
            DevBuf<uint32_t> d_nbig;
            const uint64_t big_cap = std::max<uint64_t>(s->total / 65536 + nrec, 1);
            if (d_big.alloc(big_cap) != DVS_OK || d_nbig.alloc(1) != DVS_OK) return fail(DVS_ERR_CUDA);
            TRY_P(cudaMemsetAsync(d_nbig.p, 0, sizeof(uint32_t), st));
            const size_t smem_w = (size_t)kSpWarpsPerCta * (kSpLowBins / 2) * sizeof(uint32_t);
            TRY_P(cudaFuncSetAttribute(k_sp_bucket_warp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_w));
            const unsigned g_w = (unsigned)std::min<uint64_t>((npairs + kSpWarpsPerCta - 1) / kSpWarpsPerCta,
                                                              (uint64_t)ctx->sm_count * 3 * 4);
            // sparsely occupied buckets (k >= 11: 4^k bins against ~L keys) go through the bitmap kernel first;
            // DVS_SPARSE_BITS=0 keeps the counter-walking warp kernel for everything (A/B measurements)
            const char* bits_env = getenv("DVS_SPARSE_BITS");
            const bool use_bits = k >= 11 && !(bits_env && bits_env[0] == '0');
            DevBuf<uint64_t> d_mid;
            DevBuf<uint32_t> d_nmid;
            if (use_bits) {
                if (d_mid.alloc(std::max<uint64_t>(npairs, 1)) != DVS_OK || d_nmid.alloc(1) != DVS_OK) return fail(DVS_ERR_CUDA);
                TRY_P(cudaMemsetAsync(d_nmid.p, 0, sizeof(uint32_t), st));
                const size_t smem_b = (size_t)kSpBitsWarps * sizeof(SpBitsWarp);
                TRY_P(cudaFuncSetAttribute(k_sp_bucket_bits, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_b));
                const unsigned g_b = (unsigned)std::min<uint64_t>((npairs + kSpBitsWarps - 1) / kSpBitsWarps,
                                                                  (uint64_t)ctx->sm_count * 2 * 4);
                k_sp_bucket_bits<<<g_b, 32 * kSpBitsWarps, smem_b, st>>>(d_low.p, sp->offsets.p, sp->bucket_ptr.p, nrec, nb,
                                                                         sp->idx.p, sp->cnt.p, sp->bucket_nnz.p, d_mid.p,
                                                                         d_nmid.p);
                ctx->launches++;
                TRY_P(cudaGetLastError());
            }
            k_sp_bucket_warp<<<g_w, 32 * kSpWarpsPerCta, smem_w, st>>>(d_low.p, sp->offsets.p, sp->bucket_ptr.p, nrec, nb,
                                                                       sp->idx.p, sp->cnt.p, sp->bucket_nnz.p, d_big.p,
                                                                       d_nbig.p, use_bits ? d_mid.p : nullptr,
                                                                       use_bits ? d_nmid.p : nullptr);
            ctx->launches++;
            TRY_P(cudaGetLastError());
            k_sp_bucket<<<(unsigned)std::min<uint64_t>(big_cap, (uint64_t)ctx->sm_count * 8), kSpBucketThreads, 0, st>>>(
                d_low.p, sp->offsets.p, sp->bucket_ptr.p, nrec, nb, sp->idx.p, sp->cnt.p, sp->bucket_nnz.p, d_big.p, d_nbig.p);
            ctx->launches++;
            TRY_P(cudaGetLastError());
        }
        k_sp_nnz<<<nrec, 256, 0, st>>>(sp->bucket_nnz.p, nb, sp->nnz.p);
        ctx->launches++;
        TRY_P(cudaGetLastError());
        pt.stop();
        if (want_entropy) {
            k_sp_entropy<<<nrec, kEntThreads, kEntSmemBytes, st>>>(sp->cnt.p, sp->offsets.p, sp->totals.p, sp->dim,
                                                                   sp->entropy.p, sp->err.p, sp->err_total.p);
            ctx->launches++;
            TRY_P(cudaGetLastError());
            sp->has_entropy = true;
        }
    } else if (nrec) {
        TRY_P(cudaMemsetAsync(sp->totals.p, 0, n1 * sizeof(uint64_t), st));
        TRY_P(cudaMemsetAsync(sp->nnz.p, 0, n1 * sizeof(uint64_t), st));
        TRY_P(cudaMemsetAsync(sp->valid.p, 0, n1, st));
        TRY_P(cudaMemsetAsync(sp->bucket_nnz.p, 0, n1 * nb * sizeof(uint32_t), st));
        TRY_P(cudaMemsetAsync(sp->bucket_ptr.p, 0, n1 * (nb + 1) * sizeof(uint32_t), st));
    }
    TRY_P(cudaStreamSynchronize(st));  // the host item list dies here
#undef TRY_P
    *out = sp;
    return DVS_OK;
}

uint32_t dvs_ksparse_nrec(const dvs_ksparse* sp) { return sp->nrec; }

int dvs_ksparse_stats(dvs_ctx* ctx, const dvs_ksparse* sp, uint64_t* nnz, uint64_t* totals, double* entropy,
                      uint8_t* valid) {
    if (!ctx || !sp) {
        set_error("dvs_ksparse_stats: NULL argument");
        return DVS_ERR_ARG;
    }
    if (entropy && !sp->has_entropy) {
        set_error("dvs_ksparse_stats: entropies were not requested (want_entropy = 0)");
        return DVS_ERR_ARG;
    }
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    const size_t n = sp->nrec;
    if (n == 0) return DVS_OK;
    std::vector<uint8_t> err(n);
    std::vector<double> et(n);
    if (nnz) DVS_CUDA_TRY(cudaMemcpyAsync(nnz, sp->nnz.p, n * 8, cudaMemcpyDeviceToHost, st));
    if (totals) DVS_CUDA_TRY(cudaMemcpyAsync(totals, sp->totals.p, n * 8, cudaMemcpyDeviceToHost, st));
    if (entropy) DVS_CUDA_TRY(cudaMemcpyAsync(entropy, sp->entropy.p, n * 8, cudaMemcpyDeviceToHost, st));
    if (valid) DVS_CUDA_TRY(cudaMemcpyAsync(valid, sp->valid.p, n, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaMemcpyAsync(err.data(), sp->err.p, n, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaMemcpyAsync(et.data(), sp->err_total.p, n * 8, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    if (entropy)
        for (size_t r = 0; r < n; ++r)
            if (err[r]) {
                set_error("cannot calculate entropy as frequency vector total %.17g!=1.0", et[r]);
                return DVS_ERR_VALUE;
            }
    return DVS_OK;
}

int dvs_ksparse_download(dvs_ctx* ctx, const dvs_ksparse* sp, uint32_t rec, uint32_t* idx, uint32_t* cnt, uint64_t cap,
                         uint64_t* nnz_out) {
    if (!ctx || !sp || rec >= sp->nrec || !nnz_out) {
        set_error("dvs_ksparse_download: bad argument");
        return DVS_ERR_ARG;
    }
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    uint64_t nnz = 0;
    DVS_CUDA_TRY(cudaMemcpyAsync(&nnz, sp->nnz.p + rec, 8, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    *nnz_out = nnz;
    if (!idx && !cnt) return DVS_OK;
    if (cap < nnz) {
        set_error("dvs_ksparse_download: capacity %llu < %llu distinct k-mers", (unsigned long long)cap,
                  (unsigned long long)nnz);
        return DVS_ERR_ARG;
    }
    if (nnz == 0) return DVS_OK;
    DevBuf<uint32_t> d_idx, d_cnt;
    DVS_TRY(d_idx.alloc(nnz));
    DVS_TRY(d_cnt.alloc(nnz));
    k_sp_compact<<<1, kSpThreads, 0, st>>>(sp->idx.p, sp->cnt.p, sp->bucket_ptr.p + (size_t)rec * (sp->nb + 1),
                                           sp->bucket_nnz.p + (size_t)rec * sp->nb, sp->h_offsets[rec], sp->nb, d_idx.p,
                                           d_cnt.p);
    DVS_LAUNCHED(ctx);
    if (idx) DVS_CUDA_TRY(cudaMemcpyAsync(idx, d_idx.p, nnz * 4, cudaMemcpyDeviceToHost, st));
    if (cnt) DVS_CUDA_TRY(cudaMemcpyAsync(cnt, d_cnt.p, nnz * 4, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    return DVS_OK;
}

void dvs_ksparse_free(dvs_ksparse* sp) {
    if (!sp) return;
    cudaSetDevice(sp->device);
    delete sp;
}

}  // extern "C"
