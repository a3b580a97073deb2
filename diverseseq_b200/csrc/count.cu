// k-mer counting -> frequency rows -> exact entropies.
//
// Replaces SeqRecord::to_kcounts / to_kmerseq and entropy of the reference
// (/root/reference/src/record.rs:31-84, 124-141, 86-106).
//
// Counting semantics (record.rs:41-84 == run-length form, SURVEY.md appendix A): a k-mer ending
// at position p is counted iff the k bytes p-k+1..p all lie inside the record and are
// < num_states; its bin is the base-num_states value of those bytes, first byte most significant.
//
// Kernel shape: sequence bytes stream from HBM with coalesced 16-byte loads (thread t owns the
// 16-byte block t of an 8 KB stripe; the k-1 byte halo comes from the preceding 16-byte block,
// an L1 hit).  For num_states == 4 a block of 16 valid bases is packed to 32 bits with four
// integer multiplies and each k-mer index is one funnel shift + mask.  Bins live in a
// shared-memory histogram (u32) when num_states^k * 4 B fits; otherwise the bin range is split
// into `nparts` shared-memory passes (k=8) or, for larger tables, updated with global RED.ADD.
// Work is (record, part, 16B-aligned byte range) items pulled from a global queue by persistent
// CTAs, so long records are split across CTAs and merged with one global atomic per non-empty bin.
#include <stdlib.h>

#include <algorithm>

#include <functional>

#include "comm.cuh"
#include "common.cuh"
#include "fused.cuh"
#include "entropy.cuh"

namespace dvs {

struct CountWork {
    uint64_t begin;  // 16-byte aligned absolute byte range [begin, end) inside seqset data
    uint64_t end;
    uint32_t rec;
    uint32_t part;
};

constexpr int kCountThreads = 512;
constexpr int kPrefetch = 4;  // 512-byte steps in flight per warp

__device__ __forceinline__ uint32_t pack4(uint32_t w) {
    // bytes b0..b3 (memory order, each 0..3) -> b0<<6 | b1<<4 | b2<<2 | b3
    return (w * 0x40100401u) >> 24;
}
__device__ __forceinline__ uint32_t pack16(uint4 v) {
    return (pack4(v.x) << 24) | (pack4(v.y) << 16) | (pack4(v.z) << 8) | pack4(v.w);
}

__device__ __forceinline__ uint4 ldg16(const uint8_t* p) { return __ldg(reinterpret_cast<const uint4*>(p)); }

// ---- generic kernel (any num_states): per-byte path only ----------------------------------------
// SMEM: bins [part*part_bins, (part+1)*part_bins) in shared memory; else global atomics.
template <bool SMEM>
__global__ void __launch_bounds__(kCountThreads)
k_count_generic(const uint8_t* __restrict__ seqs, const uint64_t* __restrict__ offsets,
                const CountWork* __restrict__ work, uint32_t nwork, uint32_t* __restrict__ next_item, int k,
                uint32_t num_states, uint64_t dim, uint32_t part_bins, uint32_t* __restrict__ counts) {
    extern __shared__ uint32_t hist[];
    __shared__ uint32_t s_item;
    const int tid = threadIdx.x;
    for (;;) {
        if (tid == 0) s_item = atomicAdd(next_item, 1u);
        __syncthreads();
        const uint32_t item = s_item;
        if (item >= nwork) break;
        const CountWork w = work[item];
        const uint64_t start = offsets[w.rec], end = offsets[w.rec + 1];
        const uint32_t part_base = w.part * part_bins;
        uint32_t* grow = counts + (size_t)w.rec * dim;
        if (SMEM) {
            for (uint32_t i = tid; i < part_bins; i += kCountThreads) hist[i] = 0;
            __syncthreads();
        }
        for (uint64_t a = w.begin + (uint64_t)tid * 16; a < w.end; a += (uint64_t)kCountThreads * 16) {
            const uint4 cur = ldg16(seqs + a);
            const uint4 prev = ldg16(seqs + a - 16);  // front pad keeps a-16 inside the allocation
            const uint32_t wv[8] = {prev.x, prev.y, prev.z, prev.w, cur.x, cur.y, cur.z, cur.w};
            uint32_t run = 0;
            uint64_t idx = 0;
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                const uint64_t p = a - 16 + i;
                uint32_t b = (wv[i >> 2] >> (8 * (i & 3))) & 0xFFu;
                if (p < start || p >= end) b = 0xFFu;
                if (b >= num_states) {
                    run = 0;
                    idx = 0;
                } else {
                    idx = (idx * num_states + b) % dim;
                    ++run;
                    if (i >= 16 && run >= (uint32_t)k) {
                        if (SMEM) {
                            uint32_t local = (uint32_t)idx - part_base;
                            if (local < part_bins) atomicAdd(&hist[local], 1u);
                        } else {
                            atomicAdd(&grow[idx], 1u);
                        }
                    }
                }
            }
        }
        if (SMEM) {
            __syncthreads();
            for (uint32_t i = tid; i < part_bins; i += kCountThreads) {
                uint32_t c = hist[i];
                if (c && (uint64_t)part_base + i < dim) atomicAdd(&grow[part_base + i], c);
            }
        }
        __syncthreads();  // s_item / hist reuse
    }
}

// ---- num_states == 4 kernel ------------------------------------------------------------------------
// MODE 0: shared-memory histogram of 4^k bins, one ATOMS per k-mer            (k = 7)
// MODE 1: as 0 but only bins of part `w.part` (several passes over the bytes)   (k = 8)
// MODE 2: global RED.ADD into the record's row                                  (k >= 9)
// MODE 3: SUPER-K-MERS: histogram the (k+1)-mers ending at ODD positions (4^(k+1) bins); each one
//         carries two k-mers (its prefix and its suffix), so the ATOMS count halves.  (k+1)-windows
//         that contain an invalid byte / cross the record start fall back to a small side histogram
//         of single k-mers.  The flush folds both into k-mer counts:
//         cnt[x] = side[x] + sum_b h[(x<<2)|b] + sum_a h[(a<<2k)|x].             (k <= 6)
// Each warp walks a contiguous span of its work item in 512-byte steps (lane l owns bytes
// [16l,16l+16)); the k-byte halo of lane l is the packed block of lane l-1 (warp shuffle), lane 0
// keeps lane 31's block of the previous step, so every sequence byte is loaded exactly once.
constexpr int MODE_SMEM = 0, MODE_SMEM_PARTS = 1, MODE_GLOBAL = 2, MODE_SUPER = 3, MODE_SUPER3 = 4;

// 16 packed bases from 16 bytes: four multiplies put each word's 8 bits in its top byte, three
// PRMTs gather the top bytes (first base most significant)
__device__ __forceinline__ uint32_t pack16p(uint4 v) {
    const uint32_t p0 = v.x * 0x40100401u, p1 = v.y * 0x40100401u, p2 = v.z * 0x40100401u, p3 = v.w * 0x40100401u;
    const uint32_t hi = __byte_perm(p1, p0, 0x7300);  // byte3 = p0.b3, byte2 = p1.b3
    const uint32_t lo = __byte_perm(p3, p2, 0x0073);  // byte1 = p2.b3, byte0 = p3.b3
    return __byte_perm(lo, hi, 0x7610);
}

// Bank scrambling of the shared-memory tables.  The bank of a bin is its low 5 index bits = the last 2.5
// bases, whose distribution is as skewed as the genome's composition, so ATOMS bank conflicts grow with the
// skew (ncu: 4.9 wavefronts per instruction on the benchmark set vs 2.6 for uniform bins).  Storing bin
// `idx` at slot `idx ^ (idx >> 5)` (a bijection) folds the next 2.5 bases into the bank bits.
__device__ __forceinline__ uint32_t scr_word(uint32_t idx) { return idx ^ (idx >> 5); }

template <int MODE, int THREADS>
__global__ void __launch_bounds__(THREADS)
k_count(const uint8_t* __restrict__ seqs, const uint64_t* __restrict__ offsets, const CountWork* __restrict__ work,
        uint32_t nwork, uint32_t* __restrict__ next_item, int k, uint64_t dim, uint32_t part_bins,
        uint32_t* __restrict__ counts, const uint32_t* __restrict__ nwork_dev) {
    extern __shared__ uint32_t hist[];
    __shared__ uint32_t s_item;
    if (nwork_dev) nwork = *nwork_dev;  // retry pass of k_count_s3: the list length only exists on the device
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = THREADS / 32;
    constexpr uint32_t kFull = 0xffffffffu;
    const int kk = (MODE == MODE_SUPER) ? k + 1 : k;                       // bases per histogrammed word
    const uint32_t mask = (kk >= 16) ? 0xFFFFFFFFu : ((1u << (2 * kk)) - 1u);
    const uint32_t mask4 = mask << 2;                                       // same, as a byte offset
    const uint32_t mask_k = (k >= 16) ? 0xFFFFFFFFu : ((1u << (2 * k)) - 1u);
    const uint32_t hist_words = (MODE == MODE_SUPER) ? (uint32_t)(dim * 4 + dim)
                                                     : (MODE == MODE_SMEM_PARTS ? part_bins + 1 : part_bins);
    uint32_t* side = hist + dim * 4;  // MODE_SUPER only: single k-mer histogram after the (k+1)-mer table
    char* const hist_b = reinterpret_cast<char*>(hist);

    for (;;) {
        if (tid == 0) s_item = atomicAdd(next_item, 1u);
        __syncthreads();
        const uint32_t item = s_item;
        if (item >= nwork) break;
        const CountWork w = work[item];
        const uint64_t start = offsets[w.rec], end = offsets[w.rec + 1];
        const uint32_t part_base = (MODE == MODE_SMEM_PARTS) ? w.part * part_bins : 0u;
        uint32_t* grow = counts + (size_t)w.rec * dim;
        if (MODE != MODE_GLOBAL) {
            for (uint32_t i = tid; i < hist_words; i += THREADS) hist[i] = 0;
            __syncthreads();
        }
        // idx4 = 4 * bin: one k-mer (MODE 0/1/2) or one (k+1)-mer (MODE 3)
        auto bump4 = [&](uint32_t idx4) {
            if (MODE == MODE_SMEM || MODE == MODE_SUPER) {
                idx4 ^= (idx4 >> 5) & ~3u;
                atomicAdd(reinterpret_cast<uint32_t*>(hist_b + idx4), 1u);
            } else if (MODE == MODE_SMEM_PARTS) {
                // branch-free: bins of the other part wrap to huge offsets and are clamped onto one
                // dummy word behind the table (same-address ATOMS are merged by the hardware)
                uint32_t local4 = idx4 - (part_base << 2);
                local4 ^= (local4 >> 5) & ~3u;  // (garbage for foreign bins, clamped next)
                local4 = min(local4, part_bins << 2);
                atomicAdd(reinterpret_cast<uint32_t*>(hist_b + local4), 1u);
            } else {
                atomicAdd(&grow[idx4 >> 2], 1u);
            }
        };

        // item-relative 32-bit coordinates (items are <= 1 MB): bytes [rs, re) belong to the record
        const uint32_t item_len = (uint32_t)(w.end - w.begin);
        const uint32_t rs = start > w.begin ? (uint32_t)min(start - w.begin, (uint64_t)item_len) : 0u;
        const uint32_t re = end < w.end ? (end > w.begin ? (uint32_t)(end - w.begin) : 0u) : item_len;
        // this warp's contiguous span of the item, walked in 512-byte steps
        const uint32_t span = ((item_len + kWarps - 1) / kWarps + 511u) & ~511u;
        const uint32_t r0 = min(item_len, (uint32_t)warp * span);
        const uint32_t r1 = min(item_len, r0 + span);
        const uint8_t* base = seqs + w.begin;
        uint32_t carry_pc = 0;
        bool carry_ok = false;
        // register ring of kPrefetch steps in flight per lane: with 32 warps/SM one step ahead leaves
        // only ~16 KB outstanding per SM, well short of what 6.5 TB/s x ~0.8 us latency needs (~35 KB)
        uint4 ring[kPrefetch];
#pragma unroll
        for (int u = 0; u < kPrefetch; ++u) {
            const uint32_t a = r0 + 512u * u + 16 * lane;
            ring[u] = (a < r1) ? ldg16(base + a) : make_uint4(~0u, ~0u, ~0u, ~0u);
        }
        if (r0 < r1) {
            // halo of lane 0 for the first step: the 16 bytes before the span
            const uint4 h = ldg16(base + r0 - 16);  // front pad keeps this inside the allocation
            const uint64_t a0 = w.begin + r0;
            carry_ok = (((h.x | h.y | h.z | h.w) & 0xFCFCFCFCu) == 0) && (a0 >= start + 16) && (a0 <= end);
            carry_pc = pack16p(h);
        }
        for (uint32_t rbase = r0; rbase < r1; rbase += 512u * kPrefetch) {
#pragma unroll
          for (int u = 0; u < kPrefetch; ++u) {
            const uint32_t r = rbase + 512u * u;
            if (r >= r1) break;  // warp-uniform
            const uint32_t a = r + 16 * lane;
            const uint4 cur = ring[u];
            // refill this slot with the step kPrefetch ahead
            ring[u] = (a + 512u * kPrefetch < r1) ? ldg16(base + a + 512u * kPrefetch) : make_uint4(~0u, ~0u, ~0u, ~0u);
            const bool ok = (((cur.x | cur.y | cur.z | cur.w) & 0xFCFCFCFCu) == 0) && (a >= rs) && (a + 16 <= re) && (a < r1);
            const uint32_t pc = pack16p(cur);
            uint32_t pp = __shfl_up_sync(kFull, pc, 1);
            if (lane == 0) pp = carry_pc;
            const uint32_t okmask = __ballot_sync(kFull, ok);
            const bool all_fast = (okmask == kFull) && carry_ok;  // warp-uniform: the common case
            if (all_fast) {
                if (MODE == MODE_SUPER) {
#pragma unroll
                    for (int j = 1; j < 15; j += 2) bump4(__funnelshift_r(pc, pp, 2 * (15 - j) - 2) & mask4);
                    bump4((pc << 2) & mask4);
                } else {
#pragma unroll
                    for (int j = 0; j < 15; ++j) bump4(__funnelshift_r(pc, pp, 2 * (15 - j) - 2) & mask4);
                    bump4((pc << 2) & mask4);
                }
            } else if (a < r1) {
                const bool prev_ok = lane == 0 ? carry_ok : ((okmask >> (lane - 1)) & 1u) != 0;
                if (ok && prev_ok) {
                    if (MODE == MODE_SUPER) {
#pragma unroll
                        for (int j = 1; j < 16; j += 2) bump4((__funnelshift_r(pc, pp, 2 * (15 - j)) & mask) << 2);
                    } else {
#pragma unroll
                        for (int j = 0; j < 16; ++j) bump4((__funnelshift_r(pc, pp, 2 * (15 - j)) & mask) << 2);
                    }
                } else {
                    // per-byte path: invalid bytes or record edges inside [a-16, a+16)
                    const uint4 prev = ldg16(base + a - 16);
                    const uint32_t wv[8] = {prev.x, prev.y, prev.z, prev.w, cur.x, cur.y, cur.z, cur.w};
                    uint32_t run = 0, idx = 0, run_even = 0, idx_even = 0;
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        const uint64_t p = w.begin + a + i - 16;  // absolute position (halo bytes may precede the item)
                        uint32_t bb = (wv[i >> 2] >> (8 * (i & 3))) & 0xFFu;
                        if (p < start || p >= end) bb = 0xFFu;
                        if (bb >= 4u) {
                            run = 0;
                            idx = 0;
                        } else {
                            idx = ((idx << 2) | bb) & mask;
                            ++run;
                        }
                        if (i < 16) continue;
                        if (MODE != MODE_SUPER) {
                            if (run >= (uint32_t)k) bump4(idx << 2);
                        } else if ((i & 1) == 0) {  // even position: decided together with its odd partner
                            run_even = run;
                            idx_even = idx;
                        } else if (run >= (uint32_t)(k + 1)) {
                            bump4(idx << 2);  // both k-mers valid: one (k+1)-mer
                        } else {              // fall back to single k-mers in the side table
                            if (run_even >= (uint32_t)k) atomicAdd(&side[idx_even & mask_k], 1u);
                            if (run >= (uint32_t)k) atomicAdd(&side[idx & mask_k], 1u);
                        }
                    }
                }
            }
            carry_pc = __shfl_sync(kFull, pc, 31);
            carry_ok = (okmask >> 31) != 0;
          }
        }
        if (MODE != MODE_GLOBAL) {
            __syncthreads();
            if (MODE == MODE_SUPER) {
                for (uint32_t x = tid; x < (uint32_t)dim; x += THREADS) {
                    uint32_t c = side[x];
#pragma unroll
                    for (uint32_t b = 0; b < 4; ++b) {  // x is the prefix k-mer
                        const uint32_t y = (x << 2) | b;
                        c += hist[scr_word(y)];
                    }
#pragma unroll
                    for (uint32_t a4 = 0; a4 < 4; ++a4) {  // x is the suffix k-mer
                        const uint32_t y = (a4 << (2 * k)) | x;
                        c += hist[scr_word(y)];
                    }
                    if (c) atomicAdd(&grow[x], c);
                }
            } else {
                for (uint32_t i = tid; i < part_bins; i += THREADS) {
                    uint32_t c = hist[scr_word(i)];
                    if (c && (uint64_t)part_base + i < dim) atomicAdd(&grow[part_base + i], c);
                }
            }
        }
        __syncthreads();  // s_item / hist reuse
    }
}

// ---- MODE_SUPER3: (k+2)-mers at every third position, 16-bit packed counters ------------------------------
// The k-mer kernels above sit on the shared-memory atomic rate (~3.5 bank-conflict wavefronts per ATOMS, the
// expectation for 32 random banks), so the lever is fewer atomics per base.  Here every lane histograms, for its
// 16-base block, the five (k+2)-mers ending at block positions 2, 5, 8, 11, 14 - each carries the three k-mers
// ending at its last three positions - plus the single k-mer ending at position 15 in a small side table:
// 6 ATOMS per 16 bases instead of 8, all at compile-time shifts of the packed window pp:pc (the triplets are
// local to the lane's block, so there is no phase to track and no triplet ever spans a block boundary, a record
// boundary or two work items).  4^(k+2) counters only fit shared memory as 16-bit halves of 32-bit words (k = 6:
// 128 KB); a half can overflow after 65,535 hits in one work item, which is detected exactly at the flush: every
// overflow (carry into the neighbour half or out of the word) lowers the sum of all halves, so
// sum == number of increments  <=>  no overflow.  An item that fails the check is not added; it is appended to a
// retry list and recounted by the 32-bit (k+1)-mer kernel.  Blocks that contain an invalid byte, a record edge,
// or follow such a block count their k-mers one by one in the side table (the reference's run-length rule).
// 32 contiguous bytes per lane and step (one LDG.256; a warp walks 1 KB per step): the per-step overhead -
// validity test, halo shuffle, ballot, loop control - is shared by two 16-base blocks, and the second block's
// halo is the lane's own first block.  Work items start on 32-byte boundaries for this kernel.
__device__ __forceinline__ void ldg32(const uint8_t* p, uint32_t (&v)[8]) {
    asm volatile("ld.global.nc.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(v[0]), "=r"(v[1]), "=r"(v[2]), "=r"(v[3]), "=r"(v[4]), "=r"(v[5]), "=r"(v[6]), "=r"(v[7])
                 : "l"(p));
}
__device__ __forceinline__ uint32_t pack16w(uint32_t x, uint32_t y, uint32_t z, uint32_t w) {
    return pack16p(make_uint4(x, y, z, w));
}

template <int THREADS, int PF>
__global__ void __launch_bounds__(THREADS, 1)
k_count_s3(const uint8_t* __restrict__ seqs, const uint64_t* __restrict__ offsets, const CountWork* __restrict__ work,
           uint32_t nwork, uint32_t* __restrict__ next_item, int k, uint64_t dim, uint32_t* __restrict__ counts,
           CountWork* __restrict__ retry, uint32_t* __restrict__ retry_count) {
    extern __shared__ uint32_t hist[];  // [4^(k+2) / 2] packed halves, then side[4^k]
    __shared__ uint32_t s_item, s_sum, s_inc;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    constexpr int kWarps = THREADS / 32;
    constexpr uint32_t kFull = 0xffffffffu, kStep = 1024u;
    const int kk = k + 2;
    const uint32_t mask = (1u << (2 * kk)) - 1u;  // kk <= 8
    const uint32_t mask_k = (1u << (2 * k)) - 1u;
    const uint32_t hwords = (uint32_t)(dim * 8);  // 4^(k+2) / 2
    uint32_t* side = hist + hwords;
    char* const hist_b = reinterpret_cast<char*>(hist);
    char* const side_b = reinterpret_cast<char*>(side);
    const uint32_t offmask = mask << 1 & ~3u, sidemask4 = mask_k << 2;
    const uint32_t lane32 = 32u * (uint32_t)lane;

    for (;;) {
        if (tid == 0) {
            s_item = atomicAdd(next_item, 1u);
            s_sum = 0;
            s_inc = 0;
        }
        __syncthreads();
        const uint32_t item = s_item;
        if (item >= nwork) break;
        const CountWork w = work[item];
        const uint64_t start = offsets[w.rec], end = offsets[w.rec + 1];
        uint32_t* grow = counts + (size_t)w.rec * dim;
        {
            uint4* h4 = reinterpret_cast<uint4*>(hist);
            const uint32_t n4 = (hwords + (uint32_t)dim) / 4;  // both multiples of 4 for k >= 1
            for (uint32_t i = tid; i < n4; i += THREADS) h4[i] = make_uint4(0, 0, 0, 0);
        }
        __syncthreads();
        uint32_t n_fast = 0;  // fast 16-base blocks of this thread: 5 (k+2)-mer increments each
        // v = (k+2)-mer << 1 with garbage above bit 2kk: byte offset of its counter word in bits [2kk:2], half in bit 1
        auto bump_v = [&](uint32_t v) {
            atomicAdd(reinterpret_cast<uint32_t*>(hist_b + (v & offmask)), (v & 2u) ? 0x10000u : 1u);
        };
        // the five (k+2)-mers ending at block positions 2, 5, 8, 11, 14 and the k-mer ending at position 15
        auto fast_block = [&](uint32_t pc, uint32_t pp) {
#pragma unroll
            for (int t = 0; t < 5; ++t) bump_v(__funnelshift_r(pc, pp, 25 - 6 * t));
            atomicAdd(reinterpret_cast<uint32_t*>(side_b + ((pc << 2) & sidemask4)), 1u);
        };

        const uint32_t item_len = (uint32_t)(w.end - w.begin);
        const uint32_t rs = start > w.begin ? (uint32_t)min(start - w.begin, (uint64_t)item_len) : 0u;
        const uint32_t re = end < w.end ? (end > w.begin ? (uint32_t)(end - w.begin) : 0u) : item_len;
        const uint32_t span = ((item_len + kWarps - 1) / kWarps + kStep - 1u) & ~(kStep - 1u);
        const uint32_t r0 = min(item_len, (uint32_t)warp * span);
        const uint32_t r1 = min(item_len, r0 + span);
        const uint8_t* base = seqs + w.begin;
        const uint32_t safe_hi = min(re, r1);
        uint32_t carry_pc = 0;
        bool carry_ok = false;
        uint32_t ring[PF][8];
#pragma unroll
        for (int u = 0; u < PF; ++u) {
            const uint32_t a = r0 + kStep * u + lane32;
            if (a < r1) ldg32(base + a, ring[u]);
            else {
#pragma unroll
                for (int q = 0; q < 8; ++q) ring[u][q] = ~0u;
            }
        }
        if (r0 < r1) {
            const uint4 h = ldg16(base + r0 - 16);
            const uint64_t a0 = w.begin + r0;
            carry_ok = (((h.x | h.y | h.z | h.w) & 0xFCFCFCFCu) == 0) && (a0 >= start + 16) && (a0 <= end);
            carry_pc = pack16p(h);
        }
        for (uint32_t rbase = r0; rbase < r1; rbase += kStep * PF) {
#pragma unroll
          for (int u = 0; u < PF; ++u) {
            const uint32_t r = rbase + kStep * u;
            if (r >= r1) break;  // warp-uniform
            const uint32_t a = r + lane32;
            uint32_t any = ring[u][0] | ring[u][1] | ring[u][2] | ring[u][3] | ring[u][4] | ring[u][5] | ring[u][6] | ring[u][7];
            // interior steps (warp-uniform test): the whole KB lies inside the record and the span, so only the
            // bytes themselves can invalidate a lane's 32 bases
            bool ok = (any & 0xFCFCFCFCu) == 0;
            if (!(r >= rs && r + kStep <= safe_hi)) ok = ok && (a >= rs) && (a + 32 <= safe_hi);
            const uint32_t pc0 = pack16w(ring[u][0], ring[u][1], ring[u][2], ring[u][3]);
            const uint32_t pc1 = pack16w(ring[u][4], ring[u][5], ring[u][6], ring[u][7]);
            // refill the slot only now: the raw bytes are dead from here on (the per-byte path re-reads them)
            {
                const uint32_t an = a + kStep * PF;
                if (an < r1) ldg32(base + an, ring[u]);
                else {
#pragma unroll
                    for (int q = 0; q < 8; ++q) ring[u][q] = ~0u;
                }
            }
            uint32_t pp0 = __shfl_up_sync(kFull, pc1, 1);
            if (lane == 0) pp0 = carry_pc;
            const uint32_t okmask = __ballot_sync(kFull, ok);
            bool fast = okmask == kFull && carry_ok;  // warp-uniform: the common case
            if (!fast) {
                const bool prev_ok = lane == 0 ? carry_ok : ((okmask >> (lane - 1)) & 1u) != 0;
                fast = ok && prev_ok;
            }
            if (fast) {
                fast_block(pc0, pp0);
                fast_block(pc1, pc0);
                n_fast += 2;
            } else if (a < r1) {
                // per-byte path: every k-mer ending in this lane's bytes (inside the item), one by one, side table
                const uint4 q0 = ldg16(base + a - 16), q1 = ldg16(base + a), q2 = ldg16(base + a + 16);
                const uint32_t wv[12] = {q0.x, q0.y, q0.z, q0.w, q1.x, q1.y, q1.z, q1.w, q2.x, q2.y, q2.z, q2.w};
                uint32_t run = 0, idx = 0;
#pragma unroll 4
                for (int i = 0; i < 48; ++i) {
                    const uint64_t p = w.begin + a + i - 16;
                    uint32_t bb = (wv[i >> 2] >> (8 * (i & 3))) & 0xFFu;
                    if (p < start || p >= end) bb = 0xFFu;
                    if (bb >= 4u) {
                        run = 0;
                        idx = 0;
                    } else {
                        idx = ((idx << 2) | bb) & mask_k;
                        ++run;
                        if (i >= 16 && a + i - 16 < r1 && run >= (uint32_t)k) atomicAdd(&side[idx], 1u);
                    }
                }
            }
            carry_pc = __shfl_sync(kFull, pc1, 31);
            carry_ok = (okmask >> 31) != 0;
          }
        }
        __syncthreads();
        // fold: cnt[x] = side[x] + sum of the (k+2)-mers that hold x at offset 0, 1 or 2
        uint32_t pre_sum = 0;
        for (uint32_t x = tid; x < (uint32_t)dim; x += THREADS) {
            uint32_t c = side[x], pre = 0;
#pragma unroll
            for (uint32_t t = 0; t < 8; ++t) {  // x first: y = x * 16 + (0..15) = 8 whole words
                const uint32_t v = hist[(x << 3) | t];
                pre += (v & 0xFFFFu) + (v >> 16);
            }
            c += pre;
            pre_sum += pre;
#pragma unroll
            for (uint32_t a4 = 0; a4 < 4; ++a4) {  // x in the middle: y = a | x | b
#pragma unroll
                for (uint32_t t = 0; t < 2; ++t) {
                    const uint32_t v = hist[(a4 << (2 * k + 1)) | (x << 1) | t];
                    c += (v & 0xFFFFu) + (v >> 16);
                }
            }
#pragma unroll
            for (uint32_t t = 0; t < 16; ++t) {  // x last: y = t * 4^k + x
                const uint32_t v = hist[(t << (2 * k - 1)) | (x >> 1)];
                c += (x & 1u) ? (v >> 16) : (v & 0xFFFFu);
            }
            side[x] = c;  // thread-private slot until the overflow check has passed
        }
        uint32_t n_inc = 5u * n_fast;
#pragma unroll
        for (int o = 16; o; o >>= 1) {
            pre_sum += __shfl_xor_sync(kFull, pre_sum, o);
            n_inc += __shfl_xor_sync(kFull, n_inc, o);
        }
        if (lane == 0) {
            atomicAdd(&s_sum, pre_sum);
            atomicAdd(&s_inc, n_inc);
        }
        __syncthreads();
        if (s_sum == s_inc) {
            for (uint32_t x = tid; x < (uint32_t)dim; x += THREADS) {
                const uint32_t c = side[x];
                if (c) atomicAdd(&grow[x], c);
            }
        } else if (tid == 0) {
            retry[atomicAdd(retry_count, 1u)] = w;
        }
        __syncthreads();  // s_item / hist reuse
    }
}

// one block per record: total, validity, frequency row, exact entropy
__global__ void __launch_bounds__(kEntThreads)
k_freq_entropy(const uint32_t* __restrict__ counts, uint64_t dim, double* __restrict__ freqs,
               uint64_t* __restrict__ totals, double* __restrict__ entropy, uint8_t* __restrict__ valid,
               uint8_t* __restrict__ err, double* __restrict__ err_total, const uint32_t* __restrict__ rec_list) {
    extern __shared__ __align__(16) double ent_smem[];
    __shared__ unsigned long long s_total;
    const uint32_t r = rec_list ? rec_list[blockIdx.x] : blockIdx.x;  // (records counted in a caller-given sequence)
    const uint32_t* c = counts + (size_t)r * dim;
    double* f = freqs + (size_t)r * dim;
    if (threadIdx.x == 0) s_total = 0ULL;
    __syncthreads();
    unsigned long long part = 0;
    for (uint64_t i = threadIdx.x; i < dim; i += blockDim.x) part += c[i];
    for (int o = 16; o; o >>= 1) part += __shfl_xor_sync(0xffffffffu, part, o);
    if ((threadIdx.x & 31) == 0) atomicAdd(&s_total, part);
    __syncthreads();
    const unsigned long long total_u = s_total;
    const double total = (double)total_u;  // `sum::<usize>() as f64`
    if (total_u == 0ULL) {
        for (uint64_t i = threadIdx.x; i < dim; i += blockDim.x) f[i] = __ddiv_rn((double)c[i], total);  // NaN row
        if (threadIdx.x == 0) {
            totals[r] = 0;
            entropy[r] = 0.0;
            valid[r] = 0;
            err[r] = 0;
            err_total[r] = 0.0;
        }
        return;
    }
    // count / total by div_exact (= IEEE division, entropy.cuh); the row is stored by the same pass
    const FastDiv dv = make_fast_div(total);
    EntropyResult h = block_entropy_exact(dim, [&](uint64_t i) {
        const double x = div_exact((double)c[i], dv);
        f[i] = x;
        return x;
    }, ent_smem);
    if (threadIdx.x == 0) {
        totals[r] = total_u;
        entropy[r] = h.e;
        valid[r] = 1;
        bool bad = entropy_total_bad(h.t, dim);
        err[r] = bad ? 1 : 0;
        err_total[r] = h.t;
    }
}

// rows supplied by the caller: entropy as KmerSeq::new computes it (record.rs:157-168)
__global__ void __launch_bounds__(kEntThreads)
k_rows_entropy(const double* __restrict__ freqs, uint64_t dim, double* __restrict__ entropy,
               uint8_t* __restrict__ err, double* __restrict__ err_total, int write_entropy) {
    extern __shared__ __align__(16) double ent_smem[];
    const uint32_t r = blockIdx.x;
    const double* f = freqs + (size_t)r * dim;
    EntropyResult h = block_entropy_exact(dim, [&](uint64_t i) { return f[i]; }, ent_smem);
    if (threadIdx.x == 0) {
        if (write_entropy) entropy[r] = h.e;
        bool bad = entropy_total_bad(h.t, dim);
        err[r] = bad ? 1 : 0;
        err_total[r] = h.t;
    }
}

// device gather of whole rows (+ their scalars): one CTA per output row
__global__ void k_take_rows(const double* __restrict__ F, const double* __restrict__ H, const uint8_t* __restrict__ V,
                            const uint8_t* __restrict__ E, const double* __restrict__ ET, uint64_t dim,
                            const uint32_t* __restrict__ rows, double* __restrict__ Fo, double* __restrict__ Ho,
                            uint8_t* __restrict__ Vo, uint8_t* __restrict__ Eo, double* __restrict__ ETo) {
    const uint32_t i = blockIdx.x, r = rows[i];
    const double* src = F + (size_t)r * dim;
    double* dst = Fo + (size_t)i * dim;
    for (uint64_t c = threadIdx.x; c < dim; c += blockDim.x) dst[c] = src[c];
    if (threadIdx.x == 0) {
        Ho[i] = H[r];
        Vo[i] = V[r];
        Eo[i] = E[r];
        ETo[i] = ET[r];
    }
}

__global__ void k_log2(const double* x, double* y, uint64_t n) {
    uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) y[i] = dvs_log2(x[i]);
}

static bool pow_dim(int num_states, int k, uint64_t* dim) {
    uint64_t d = 1;
    for (int i = 0; i < k; ++i) {
        d *= (uint64_t)num_states;
        if (d > (1ULL << 32)) return false;
    }
    *dim = d;
    return true;
}

static int kfreqs_alloc(dvs_ctx* ctx, uint32_t nrec, uint64_t dim, bool with_counts, dvs_kfreqs** out) {
    DVS_CUDA_TRY(dvs::enter(ctx));
    auto* f = new dvs_kfreqs();
    f->device = ctx->device;
    f->nrec = nrec;
    f->dim = dim;
    f->has_counts = with_counts;
    int rc = DVS_OK;
    if (with_counts) rc = f->counts.alloc((size_t)nrec * dim);
    if (rc == DVS_OK) rc = f->freqs.alloc((size_t)nrec * dim);
    if (rc == DVS_OK) rc = f->totals.alloc(nrec);
    if (rc == DVS_OK) rc = f->entropy.alloc(nrec);
    if (rc == DVS_OK) rc = f->valid.alloc(nrec);
    if (rc == DVS_OK) rc = f->err.alloc(nrec);
    if (rc == DVS_OK) rc = f->err_total.alloc(nrec);
    if (rc != DVS_OK) {
        delete f;
        return rc;
    }
    *out = f;
    return DVS_OK;
}

}  // namespace dvs

using namespace dvs;

extern "C" {

// Where the rows of the local records go, and what happens after each chunk of records.  Plain counting:
// the kfreqs' own arrays, one chunk.  Sharded counting (dvs_count_kmers_sharded): the arrays of the
// all-ranks kfreqs inside the peer window at this rank's row offset, several chunks, and after every chunk
// its rows are pushed to the peers on the side stream while the next chunk is being counted.
struct CountDest {
    double* freqs;
    uint64_t* totals;
    double* entropy;
    uint8_t* valid;
    uint8_t* err;
    double* err_total;
    uint32_t chunks;                                   // >= 1
    std::function<int(uint32_t, uint32_t)> after_chunk;  // (first record, end record) of the chunk just enqueued
    // optional: the sequence in which the records are counted (a permutation of 0..nrec-1; chunk c covers
    // rec_seq[rb..re)) - dvs_count_select counts in the selection's examination order so that the rounds can trail
    const uint32_t* rec_seq = nullptr;
    const uint32_t* weights = nullptr;  // [chunks] relative chunk sizes (NULL: equal)
};

static int count_core(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, uint32_t* d_counts, uint64_t dim,
                      const CountDest& dst) {
    cudaStream_t st = ctx->stream;
#define TRY_F(expr)                                                          \
    do {                                                                     \
        cudaError_t _e = (expr);                                             \
        if (_e != cudaSuccess) {                                             \
            set_error("%s failed: %s", #expr, cudaGetErrorString(_e));       \
            return DVS_ERR_CUDA;                                             \
        }                                                                    \
    } while (0)

    TRY_F(cudaMemsetAsync(d_counts, 0, (size_t)s->nrec * dim * sizeof(uint32_t), st));

    // ---- histogram placement ----
    const bool ns4 = (num_states == 4);
    const size_t max_hist_bytes = std::min<size_t>(ctx->smem_optin > 4096 ? ctx->smem_optin - 2048 : 0, 128 * 1024 + 16);
    uint32_t nparts = 1, part_bins = (uint32_t)std::min<uint64_t>(dim, 1u << 31);
    int mode = MODE_SMEM;
    size_t hist_bytes = (size_t)dim * 4;
    // (k+2)-mers at every third position in 16-bit packed counters (k_count_s3) for k = 4..6: a third fewer
    // shared atomics than the (k+1)-mer kernel.  DVS_COUNT_S3=0 selects the (k+1)-mer kernel instead.
    const char* s3_env = getenv("DVS_COUNT_S3");
    const bool want_s3 = !(s3_env && s3_env[0] == '0');
    if (ns4 && want_s3 && k >= 4 && dim * 36 + 2048 <= ctx->smem_optin && dim * 36 <= 160 * 1024) {
        // (k+2)-mers at every third position, 16-bit packed counters + side table: k = 4..6 -> at most 144 KB.
        // Smaller k would overflow the 16-bit halves routinely (4^(k+2) bins share the item's increments).
        mode = MODE_SUPER3;
        hist_bytes = (size_t)dim * 36;
    } else if (ns4 && dim * 20 <= 96 * 1024) {  // (k+1)-mer table + side table: k <= 6 -> at most 80 KB
        mode = MODE_SUPER;
        hist_bytes = (size_t)dim * 20;
    } else if (dim * 4 > max_hist_bytes) {
        uint64_t bins_per = max_hist_bytes / 4;
        uint64_t np = (dim + bins_per - 1) / bins_per;
        if (np <= 2) {
            mode = MODE_SMEM_PARTS;
            nparts = (uint32_t)np;
            part_bins = (uint32_t)((dim + np - 1) / np);
            hist_bytes = (size_t)part_bins * 4 + 16;  // + the dummy word that absorbs the other part's bins
        } else {
            mode = MODE_GLOBAL;
            hist_bytes = 0;
        }
    }
    const bool smem = (mode != MODE_GLOBAL);

    // ---- work list: (record, part, aligned range) ----
    int ctas_per_sm = 4;
    if (smem) ctas_per_sm = (int)std::max<size_t>(1, std::min<size_t>(4, (ctx->smem_optin + 1024) / (hist_bytes + 1024)));
    const uint32_t grid = (uint32_t)(ctx->sm_count * ctas_per_sm);
    const int threads4 = (mode == MODE_SMEM_PARTS || mode == MODE_SUPER3) ? 1024 : kCountThreads;
    uint64_t chunk = 1 << 20;
    {
        // aim for >= 8 items per CTA, multiples of the 8 KB stripe.  Every item pays a zero + flush of its
        // table, so big tables (k >= 7) take up to 2-8 MB per item, small ones 64 KB .. 1 MB
        // global atomics per item at flush time (none for MODE_GLOBAL, which updates the row directly)
        const uint64_t flush_bins =
            (mode == MODE_GLOBAL) ? 0 : (mode == MODE_SUPER ? dim : (mode == MODE_SUPER3 ? dim * 16 : part_bins));
        const uint64_t max_chunk = flush_bins >= 32768 ? (8u << 20) : (flush_bins >= 16384 ? (2u << 20) : (1u << 20));
        uint64_t want_items = (uint64_t)grid * 8 * dst.chunks;
        uint64_t c = (s->total + want_items - 1) / std::max<uint64_t>(want_items, 1);
        c = std::max<uint64_t>(64 << 10, std::min<uint64_t>(c, max_chunk));
        chunk = (c + 8191) / 8192 * 8192;
        // MODE_GLOBAL with rows larger than a fraction of L2 (k >= 11: 16 MB+): the RED.ADDs only run at
        // L2 speed while the row being updated is L2 resident, so keep the whole grid on ~1 record at a
        // time with 8 KB items (measured at k=12: 37 Gbp/s with 9 rows in flight, DRAM sector bound)
        if (mode == MODE_GLOBAL && dim * 4 >= (16u << 20)) chunk = 8192;
    }
    DevBuf<uint32_t> d_rec_seq;
    if (dst.rec_seq) {
        if (d_rec_seq.alloc(std::max<uint32_t>(s->nrec, 1)) != DVS_OK) return DVS_ERR_CUDA;
        TRY_F(cudaMemcpyAsync(d_rec_seq.p, dst.rec_seq, (size_t)s->nrec * sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    }
    const bool same_seq = dst.rec_seq ? (s->work_seq.size() == s->nrec &&
                                         std::equal(s->work_seq.begin(), s->work_seq.end(), dst.rec_seq))
                                      : s->work_seq.empty();
    if (s->work_chunk != chunk || s->work_nparts != nparts || !s->work_cache.p || !same_seq) {
        std::vector<CountWork> work;
        s->work_item_begin.assign(s->nrec + 1, 0);
        for (uint32_t q = 0; q < s->nrec; ++q) {
            const uint32_t r = dst.rec_seq ? dst.rec_seq[q] : q;  // items are grouped by position in the counting sequence
            s->work_item_begin[q] = (uint32_t)work.size();
            uint64_t b = s->h_offsets[r], e = s->h_offsets[r + 1];
            if (e <= b) continue;
            uint64_t a0 = b & ~31ULL, a1 = (e + 15) & ~15ULL;  // (32-byte aligned starts: k_count_s3 loads 32 bytes per lane)
            for (uint64_t a = a0; a < a1; a += chunk)
                for (uint32_t p = 0; p < nparts; ++p) work.push_back({a, std::min(a + chunk, a1), r, p});
        }
        if (work.size() > 0xFFFFFFF0ull) {
            dvs::set_error("too many counting work items");
            return DVS_ERR_ARG;
        }
        s->work_item_begin[s->nrec] = (uint32_t)work.size();
        s->work_chunk = 0;
        if (s->work_cache.alloc(work.size() * sizeof(CountWork)) != DVS_OK) return DVS_ERR_CUDA;
        // pageable source: the copy is staged before the call returns, so `work` may die here
        TRY_F(cudaMemcpyAsync(s->work_cache.p, work.data(), work.size() * sizeof(CountWork), cudaMemcpyHostToDevice, st));
        s->work_chunk = chunk;
        s->work_nparts = nparts;
        s->work_items = (uint32_t)work.size();
        if (dst.rec_seq)
            s->work_seq.assign(dst.rec_seq, dst.rec_seq + s->nrec);  // (the list is cached per counting sequence)
        else
            s->work_seq.clear();
    }
    const CountWork* d_work_all = reinterpret_cast<const CountWork*>(s->work_cache.p);
    const uint32_t nchunks = std::max<uint32_t>(1, std::min<uint32_t>(dst.chunks, std::max<uint32_t>(s->nrec, 1)));
    DevBuf<uint32_t> d_next, d_rc;
    DevBuf<CountWork> d_retry;
    if (d_next.alloc(nchunks) != DVS_OK) return DVS_ERR_CUDA;
    TRY_F(cudaMemsetAsync(d_next.p, 0, nchunks * sizeof(uint32_t), st));
    if (mode == MODE_SUPER3) {
        if (d_retry.alloc(std::max<uint32_t>(s->work_items, 1)) != DVS_OK || d_rc.alloc(2 * nchunks) != DVS_OK)
            return DVS_ERR_CUDA;
        TRY_F(cudaMemsetAsync(d_rc.p, 0, 2 * nchunks * sizeof(uint32_t), st));
    }
    // several chunks: one timer around the whole loop (it then includes the small freq/entropy launches)
    PhaseTimer pt_all(nchunks > 1 ? ctx : nullptr, DVS_PHASE_COUNT_KERNEL);
    struct TimingGuard {  // (the per-launch timers below stay silent while the loop timer runs)
        dvs_ctx* c;
        bool saved;
        ~TimingGuard() { c->timing = saved; }
    } timing_guard{ctx, ctx->timing};
    if (nchunks > 1) ctx->timing = false;
    const bool chunk_ev = nchunks > 1 && timing_guard.saved && nchunks <= 64;
    ctx->n_chunk_ev = 0;
    if (chunk_ev)
        for (uint32_t i = 0; i < 2 * nchunks; ++i)
            if (!ctx->ev_chunk[i]) TRY_F(cudaEventCreate(&ctx->ev_chunk[i]));
    // chunk c covers positions [chunk_first(c), chunk_first(c + 1)) of the counting sequence: equal shares unless the
    // caller gives weights
    uint64_t wsum = 0;
    for (uint32_t c = 0; c < nchunks && dst.weights; ++c) wsum += dst.weights[c];
    auto chunk_first = [&](uint32_t c) -> uint32_t {
        if (!dst.weights || !wsum) return (uint32_t)((uint64_t)s->nrec * c / nchunks);
        uint64_t acc = 0;
        for (uint32_t i = 0; i < c; ++i) acc += dst.weights[i];
        return (uint32_t)((unsigned __int128)s->nrec * acc / wsum);
    };
    for (uint32_t ch = 0; ch < nchunks; ++ch) {
        const uint32_t rb = chunk_first(ch), re = chunk_first(ch + 1);
        const uint32_t ib = s->work_item_begin[rb], ie = s->work_item_begin[re];
        const CountWork* d_work = d_work_all + ib;
        const uint32_t n_work = ie - ib;
        uint32_t* d_nx = d_next.p + ch;
        if (n_work) {
            const uint32_t g = (uint32_t)std::min<size_t>(grid, n_work);
            auto set_smem = [&](auto kern) -> cudaError_t {
                return hist_bytes > 48 * 1024
                           ? cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_bytes)
                           : cudaSuccess;
            };
            auto launch4 = [&](auto kern) -> cudaError_t {
                cudaError_t e = set_smem(kern);
                if (e != cudaSuccess) return e;
                kern<<<g, threads4, hist_bytes, st>>>(s->data(), s->offsets.p, d_work, n_work, d_nx, k, dim, part_bins,
                                                      d_counts, nullptr);
                ctx->launches++;
                return cudaGetLastError();
            };
            auto launch_generic = [&](auto kern) -> cudaError_t {
                cudaError_t e = set_smem(kern);
                if (e != cudaSuccess) return e;
                kern<<<g, kCountThreads, hist_bytes, st>>>(s->data(), s->offsets.p, d_work, n_work, d_nx, k,
                                                           (uint32_t)num_states, dim, part_bins, d_counts);
                ctx->launches++;
                return cudaGetLastError();
            };
            cudaError_t e;
            PhaseTimer pt(ctx, DVS_PHASE_COUNT_KERNEL);
            if (chunk_ev) cudaEventRecord(ctx->ev_chunk[2 * ctx->n_chunk_ev], st);
            if (!ns4)
                e = smem ? launch_generic(k_count_generic<true>) : launch_generic(k_count_generic<false>);
            else if (mode == MODE_SUPER3) {
                // main pass + retry pass (items whose 16-bit halves overflowed, recounted with 32-bit counters).
                // The 8-mer table spreads over 32,768 words: bank scrambling would cost two instructions per atomic
                // and buy nothing here.  1024 threads x 3 KB-steps in flight per warp (8.78 ms on the bench set;
                // 2 steps 8.97 ms, 512 threads x 4 steps 9.03 ms)
                auto s3 = k_count_s3<1024, 3>;
                auto rk = k_count<MODE_SUPER, 512>;
                TRY_F(cudaFuncSetAttribute(s3, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)hist_bytes));
                const size_t retry_bytes = (size_t)dim * 20;
                if (retry_bytes > 48 * 1024)
                    TRY_F(cudaFuncSetAttribute(rk, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)retry_bytes));
                uint32_t* rc2 = d_rc.p + 2 * ch;
                s3<<<g, 1024, hist_bytes, st>>>(s->data(), s->offsets.p, d_work, n_work, d_nx, k, dim, d_counts,
                                                d_retry.p + ib, rc2);
                ctx->launches++;
                e = cudaGetLastError();
                if (e == cudaSuccess) {
                    const uint32_t g2 = (uint32_t)std::min<size_t>((size_t)ctx->sm_count * 2, n_work);
                    rk<<<g2, 512, retry_bytes, st>>>(s->data(), s->offsets.p, d_retry.p + ib, 0u, rc2 + 1, k, dim,
                                                     (uint32_t)dim, d_counts, rc2);
                    ctx->launches++;
                    e = cudaGetLastError();
                }
            } else if (mode == MODE_SUPER)
                e = launch4(k_count<MODE_SUPER, 512>);
            else if (mode == MODE_SMEM)
                e = launch4(k_count<MODE_SMEM, 512>);
            else if (mode == MODE_SMEM_PARTS)  // one 128 KB CTA per SM: 1024 threads keep 32 warps resident
                e = launch4(k_count<MODE_SMEM_PARTS, 1024>);
            else
                e = launch4(k_count<MODE_GLOBAL, 512>);
            pt.stop();
            if (chunk_ev) cudaEventRecord(ctx->ev_chunk[2 * ctx->n_chunk_ev++ + 1], st);
            if (e != cudaSuccess) {
                set_error("k_count launch failed: %s", cudaGetErrorString(e));
                return DVS_ERR_CUDA;
            }
        }
        if (re > rb) {
            PhaseTimer pt(ctx, DVS_PHASE_FREQ_ENTROPY);
            if (dst.rec_seq)
                k_freq_entropy<<<re - rb, kEntThreads, kEntSmemBytes, st>>>(d_counts, dim, dst.freqs, dst.totals, dst.entropy,
                                                                            dst.valid, dst.err, dst.err_total, d_rec_seq.p + rb);
            else
                k_freq_entropy<<<re - rb, kEntThreads, kEntSmemBytes, st>>>(
                    d_counts + (size_t)rb * dim, dim, dst.freqs + (size_t)rb * dim, dst.totals + rb, dst.entropy + rb,
                    dst.valid + rb, dst.err + rb, dst.err_total + rb, nullptr);
            ctx->launches++;
            TRY_F(cudaGetLastError());
        }
        if (dst.after_chunk) DVS_TRY(dst.after_chunk(rb, re));
    }
    ctx->timing = timing_guard.saved;
    pt_all.stop();
#undef TRY_F
    return DVS_OK;
}

static int count_args_ok(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, const void* out, uint64_t* dim) {
    if (!ctx || !s || !out) {
        set_error("dvs_count_kmers: NULL argument");
        return DVS_ERR_ARG;
    }
    if (k == 0) {
        set_error("k cannot be 0");  // record.rs:126
        return DVS_ERR_VALUE;
    }
    if (k < 0 || k > 16 || num_states < 1 || num_states > 255) {
        set_error("dvs_count_kmers: unsupported k=%d / num_states=%d (need 1<=k<=16, 1<=num_states<=255)", k,
                  num_states);
        return DVS_ERR_ARG;
    }
    if (!pow_dim(num_states, k, dim)) {
        set_error("dvs_count_kmers: num_states^k = %d^%d does not fit a dense u32-indexed table", num_states, k);
        return DVS_ERR_ARG;
    }
    // per-bin counters are u32 (the reference counts in usize): a bin cannot exceed the number of k-mers
    // of its record, so records below 2^32 bases can never wrap; longer ones are refused, not miscounted
    for (uint32_t r = 0; r < s->nrec; ++r)
        if (s->h_offsets[r + 1] - s->h_offsets[r] >= (1ULL << 32)) {
            set_error("dvs_count_kmers: record %u has %llu bases; records of 2^32 bases or more are not supported "
                      "(32-bit bin counters)", r, (unsigned long long)(s->h_offsets[r + 1] - s->h_offsets[r]));
            return DVS_ERR_ARG;
        }
    return DVS_OK;
}

static int dense_rows_fit(double need, const char* what, uint32_t nrec, uint64_t dim) {
    size_t free_b = 0, total_b = 0;
    // cudaMemGetInfo costs milliseconds and pooled blocks count as "used": only ask when it can matter
    if (need > 8e9) DVS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    if (need > 8e9 && need > 0.9 * (double)free_b) {
        set_error("%s: dense rows need %.1f GB (nrec=%u, dim=%llu) but only %.1f GB are free", what, need / 1e9, nrec,
                  (unsigned long long)dim, free_b / 1e9);
        return DVS_ERR_ARG;
    }
    return DVS_OK;
}

int dvs_count_kmers(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, dvs_kfreqs** out) {
    uint64_t dim = 0;
    DVS_TRY(count_args_ok(ctx, s, k, num_states, out, &dim));
    DVS_CUDA_TRY(dvs::enter(ctx));
    DVS_TRY(dense_rows_fit((double)s->nrec * (double)dim * 12.0, "dvs_count_kmers", s->nrec, dim));
    dvs_kfreqs* f = nullptr;
    DVS_TRY(kfreqs_alloc(ctx, s->nrec, dim, true, &f));
    f->k = k;
    f->num_states = num_states;
    CountDest dst{f->freqs.p, f->totals.p, f->entropy.p, f->valid.p, f->err.p, f->err_total.p, 1, nullptr};
    int rc = count_core(ctx, s, k, num_states, f->counts.p, dim, dst);
    if (rc != DVS_OK) {
        dvs_kfreqs_free(f);
        return rc;
    }
    // (no synchronisation: the work list is cached in the seqset and every scratch buffer is released in
    // stream order, so the caller's next call can be enqueued while the counting is still running)
    *out = f;
    return DVS_OK;
}

// ---- counting with the selection rounds trailing it (one GPU) ---------------------------------------------
__global__ void k_set_word(unsigned* w, unsigned v) { *w = v; }

// The records are counted on a second stream in `order`'s sequence, `chunks` launches; after each one the number of
// positions whose rows / entropies / flags exist is published in a device word, and the nmost rounds (select.cu:
// the SM-replicated kernel on DVS_TRAIL_SMS SMs of its own) only examine positions below it.  The result is
// the one dvs_count_kmers + dvs_select give (same kernels' arithmetic; tests/test_gpu_fused.py).
int dvs_count_select(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, const uint32_t* order, uint32_t num,
                     int mode, uint32_t min_size, uint32_t max_size, uint32_t chunks, dvs_kfreqs** out,
                     uint32_t* sel_idx, double* sel_delta, double* stats5, uint32_t* size_out) {
    uint64_t dim = 0;
    DVS_TRY(count_args_ok(ctx, s, k, num_states, out, &dim));
    if ((!order && num) || !size_out) {
        set_error("dvs_count_select: NULL argument");
        return DVS_ERR_ARG;
    }
    for (uint32_t i = 0; i < num; ++i)
        if (order[i] >= s->nrec) {
            set_error("dvs_count_select: order[%u]=%u out of range (nrec=%u)", i, order[i], s->nrec);
            return DVS_ERR_ARG;
        }
    DVS_CUDA_TRY(dvs::enter(ctx));
    DVS_TRY(dense_rows_fit((double)s->nrec * (double)dim * 12.0, "dvs_count_select", s->nrec, dim));
    if (!ctx->stream2) {
        DVS_CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream2, cudaStreamNonBlocking));
        DVS_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_first, cudaEventDisableTiming));
        DVS_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_count_done, cudaEventDisableTiming));
        DVS_CUDA_TRY(cudaEventCreateWithFlags(&ctx->ev_fork, cudaEventDisableTiming));
        DVS_CUDA_TRY(cudaMalloc(&ctx->d_ready, 4096));
    }
    dvs_kfreqs* f = nullptr;
    DVS_TRY(kfreqs_alloc(ctx, s->nrec, dim, true, &f));
    f->k = k;
    f->num_states = num_states;

    // counting sequence: the records in order of first appearance in `order`, then the ones it does not name
    std::vector<uint32_t> seq, seqpos(s->nrec, 0xFFFFFFFFu);
    seq.reserve(s->nrec);
    for (uint32_t i = 0; i < num; ++i)
        if (seqpos[order[i]] == 0xFFFFFFFFu) {
            seqpos[order[i]] = (uint32_t)seq.size();
            seq.push_back(order[i]);
        }
    for (uint32_t r = 0; r < s->nrec; ++r)
        if (seqpos[r] == 0xFFFFFFFFu) {
            seqpos[r] = (uint32_t)seq.size();
            seq.push_back(r);
        }
    // need[i] = records (in sequence) that must be counted before positions 0..i are all there (non-decreasing)
    std::vector<uint32_t> need(num);
    for (uint32_t i = 0, m = 0; i < num; ++i) {
        m = std::max(m, seqpos[order[i]] + 1);
        need[i] = m;
    }
    auto ready_after = [&](uint32_t re) {  // positions published once seq[0..re) is counted
        return (uint32_t)(std::upper_bound(need.begin(), need.end(), re) - need.begin());
    };
    // chunk sizes: DVS_TRAIL_WEIGHTS="w0,w1,..." (relative sizes, also sets the number of chunks) for measurements
    std::vector<uint32_t> weights;
    if (const char* w_env = getenv("DVS_TRAIL_WEIGHTS")) {
        for (const char* p = w_env; *p;) {
            char* end = nullptr;
            const unsigned long v = strtoul(p, &end, 10);
            if (end == p) break;
            weights.push_back((uint32_t)std::max<unsigned long>(v, 1));
            p = *end ? end + 1 : end;
        }
        if (weights.size() >= 2 && weights.size() <= 64) chunks = (uint32_t)weights.size();
        else weights.clear();
    }
    if (chunks == 0 && weights.empty()) {
        // default: six launches, the middle ones large, the last ones small - the selection can take its SMs at the
        // end of the second launch and little is left to examine once the counting has finished (measured on the
        // bench set with 36 selection SMs: 12.34 ms/step; equal chunks 12.61; 7 chunks 12.44-12.50)
        weights = {3, 4, 4, 3, 2, 1};
        chunks = 6;
    }
    chunks = std::min<uint32_t>(chunks, 64);
    // the first chunk has to hold the initial set
    auto first_chunk_end = [&]() -> uint32_t {
        if (weights.size() != chunks) return (uint32_t)((uint64_t)s->nrec / chunks);
        uint64_t ws = 0;
        for (uint32_t w : weights) ws += w;
        return (uint32_t)((uint64_t)s->nrec * weights[0] / ws);
    };
    while (chunks > 1 && ready_after(first_chunk_end()) < std::max<uint32_t>(min_size, 1)) {
        --chunks;
        weights.clear();
    }
    // (only beside k_count_s3: k = 4..6 over 4 states)
    const char* s3_env = getenv("DVS_COUNT_S3");
    const bool s3 = num_states == 4 && k >= 4 && k <= 6 && !(s3_env && s3_env[0] == '0');
    const bool trail = chunks > 1 && mode == DVS_MODE_NMOST && num > 0 && s3;
    // DVS_TRAIL=0 (A/B measurements): same chunked counting, but the selection starts when it has finished
    const char* trail_env = getenv("DVS_TRAIL");
    const bool trail_rounds = !(trail_env && trail_env[0] == '0');

    cudaStream_t main_st = ctx->stream;
    int rc;
    if (!trail) {  // nothing to overlap: the two calls back to back
        CountDest dst{f->freqs.p, f->totals.p, f->entropy.p, f->valid.p, f->err.p, f->err_total.p, 1, nullptr};
        rc = count_core(ctx, s, k, num_states, f->counts.p, dim, dst);
        if (rc == DVS_OK)
            rc = dvs::select_with_trail(ctx, f, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5,
                                        size_out, nullptr);
    } else {
        dvs::TrailArgs ta{ctx->d_ready, 0, ctx->ev_first, ctx->ev_count_done};
        DVS_CUDA_TRY(cudaMemsetAsync(ctx->d_ready, 0, sizeof(unsigned), main_st));
        DVS_CUDA_TRY(cudaEventRecord(ctx->ev_fork, main_st));
        DVS_CUDA_TRY(cudaStreamWaitEvent(ctx->stream2, ctx->ev_fork, 0));
        CountDest dst{f->freqs.p, f->totals.p, f->entropy.p, f->valid.p, f->err.p, f->err_total.p, chunks, nullptr};
        dst.rec_seq = seq.data();
        if (weights.size() == chunks) dst.weights = weights.data();
        bool first = true;
        cudaStream_t side = ctx->stream2;
        dst.after_chunk = [&](uint32_t, uint32_t re) -> int {
            const uint32_t rdy = ready_after(re);
            k_set_word<<<1, 1, 0, side>>>(ctx->d_ready, rdy);
            DVS_CUDA_TRY(cudaGetLastError());
            if (first) {
                first = false;
                ta.limit0 = rdy;
                DVS_CUDA_TRY(cudaEventRecord(ctx->ev_first, side));
            }
            return DVS_OK;
        };
        ctx->stream = side;  // count_core and its scratch buffers live on the second stream
        dvs::tl_stream = side;
        rc = count_core(ctx, s, k, num_states, f->counts.p, dim, dst);
        cudaError_t e1 = first ? cudaEventRecord(ctx->ev_first, side) : cudaSuccess;  // (never leave a waiter behind)
        cudaError_t e2 = cudaEventRecord(ctx->ev_count_done, side);
        ctx->stream = main_st;
        dvs::tl_stream = main_st;
        if (rc == DVS_OK && (e1 != cudaSuccess || e2 != cudaSuccess)) {
            set_error("dvs_count_select: cudaEventRecord failed");
            rc = DVS_ERR_CUDA;
        }
        if (rc == DVS_OK && !trail_rounds) cudaStreamWaitEvent(main_st, ctx->ev_count_done, 0);
        if (rc == DVS_OK)
            rc = dvs::select_with_trail(ctx, f, order, num, mode, min_size, max_size, sel_idx, sel_delta, stats5,
                                        size_out, trail_rounds ? &ta : nullptr);
        cudaStreamWaitEvent(main_st, ctx->ev_count_done, 0);  // join, whatever happened
        if (getenv("DVS_TRAIL_DEBUG") && ctx->timing) {  // per-launch counting times of this call
            cudaStreamSynchronize(main_st);
            fprintf(stderr, "[dvs] count launches (ms):");
            for (uint32_t c = 0; c < ctx->n_chunk_ev; ++c) {
                float ms = 0.f;
                cudaEventElapsedTime(&ms, ctx->ev_chunk[2 * c], ctx->ev_chunk[2 * c + 1]);
                fprintf(stderr, " %.3f", ms);
            }
            fprintf(stderr, "  trailing launches %u, fewest SMs %u, accepts while counting %u\n", ctx->last_trail_launches,
                    ctx->last_trail_launches ? ctx->last_trail_sms : 0, ctx->last_trail_accepts);
        }
    }
    if (rc != DVS_OK) {
        cudaStreamSynchronize(main_st);
        dvs_kfreqs_free(f);
        return rc;
    }
    *out = f;
    return DVS_OK;
}

// ---- rows of all ranks in one kfreqs: storage in the symmetric heap of the peer window --------------------
struct AllRows {
    dvs_kfreqs* f = nullptr;
    uint64_t off_freqs = 0, off_ent = 0, off_et = 0, off_tot = 0, off_valid = 0, off_err = 0;  // inside the block
    uint32_t row0 = 0, total = 0;
};

static int allrows_alloc(dvs_ctx* ctx, dvs_comm* c, const uint32_t* nrec_per_rank, uint64_t dim, AllRows* a) {
    uint64_t total = 0;
    for (int r = 0; r < c->world; ++r) {
        if (r == c->rank) a->row0 = (uint32_t)total;
        total += nrec_per_rank[r];
    }
    if (total > 0xFFFFFFF0ull) {
        set_error("too many records in total");
        return DVS_ERR_ARG;
    }
    a->total = (uint32_t)total;
    auto up = [](uint64_t x) { return (x + 255) & ~255ull; };
    const uint64_t n = std::max<uint64_t>(total, 1);
    a->off_freqs = 0;
    a->off_ent = up(n * dim * 8);
    a->off_et = a->off_ent + up(n * 8);
    a->off_tot = a->off_et + up(n * 8);
    a->off_valid = a->off_tot + up(n * 8);
    a->off_err = a->off_valid + up(n);
    const uint64_t bytes = a->off_err + up(n);
    uint64_t hoff = 0;
    DVS_TRY(comm_heap_alloc(c, bytes, &hoff));
    auto* f = new dvs_kfreqs();
    f->device = ctx->device;
    f->nrec = a->total;
    f->dim = dim;
    f->has_counts = false;
    f->heap = c;
    f->heap_off = hoff;
    uint8_t* base = c->window + hoff;
    f->freqs.borrow(reinterpret_cast<double*>(base + a->off_freqs), n * dim);
    f->entropy.borrow(reinterpret_cast<double*>(base + a->off_ent), n);
    f->err_total.borrow(reinterpret_cast<double*>(base + a->off_et), n);
    f->totals.borrow(reinterpret_cast<uint64_t*>(base + a->off_tot), n);
    f->valid.borrow(base + a->off_valid, n);
    f->err.borrow(base + a->off_err, n);
    a->f = f;
    return DVS_OK;
}

// push rows [rb, re) of this rank (already in place in its own window) to the same place in every peer's window
static int allrows_push(dvs_comm* c, const AllRows& a, uint32_t rb, uint32_t re, bool scalars) {
    if (re <= rb) return DVS_OK;
    const uint64_t dim = a.f->dim, hoff = a.f->heap_off;
    const size_t g0 = (size_t)a.row0 + rb, cnt = re - rb;
    // fork from `side` (which is behind the rows' producer): one stream per peer, joined back into `side`
    DVS_CUDA_TRY(cudaEventRecord(c->ev_fan, c->side));
    for (int d = 1; d < c->world; ++d) {
        const int r = (c->rank + d) % c->world;
        uint8_t* pb = c->peer[r] + hoff;
        const uint8_t* mb = c->window + hoff;
        cudaStream_t ps = c->peer_stream[d];
        DVS_CUDA_TRY(cudaStreamWaitEvent(ps, c->ev_fan, 0));
        auto cp = [&](uint64_t off, size_t elem) {
            return cudaMemcpyAsync(pb + off + g0 * elem, mb + off + g0 * elem, cnt * elem, cudaMemcpyDeviceToDevice, ps);
        };
        DVS_CUDA_TRY(cp(a.off_freqs, dim * 8));
        if (scalars) {
            DVS_CUDA_TRY(cp(a.off_ent, 8));
            DVS_CUDA_TRY(cp(a.off_et, 8));
            DVS_CUDA_TRY(cp(a.off_tot, 8));
            DVS_CUDA_TRY(cp(a.off_valid, 1));
            DVS_CUDA_TRY(cp(a.off_err, 1));
        }
        DVS_CUDA_TRY(cudaEventRecord(c->peer_ev[d], ps));
        DVS_CUDA_TRY(cudaStreamWaitEvent(c->side, c->peer_ev[d], 0));
    }
    return DVS_OK;
}

static int sharded_args_ok(dvs_ctx* ctx, dvs_comm* c, const uint32_t* nrec_per_rank, uint32_t mine, const void* out) {
    if (!ctx || !c || !nrec_per_rank || !out) {
        set_error("sharded call: NULL argument");
        return DVS_ERR_ARG;
    }
    if (!c->connected) {
        set_error("sharded call: the communicator is not connected (dvs_comm_connect)");
        return DVS_ERR_ARG;
    }
    if (nrec_per_rank[c->rank] != mine) {
        set_error("sharded call: nrec_per_rank[%d] = %u but this rank holds %u records", c->rank, nrec_per_rank[c->rank], mine);
        return DVS_ERR_ARG;
    }
    return DVS_OK;
}

int dvs_count_kmers_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_seqset* s, int k, int num_states,
                            const uint32_t* nrec_per_rank, dvs_kfreqs** out_all) {
    uint64_t dim = 0;
    DVS_TRY(count_args_ok(ctx, s, k, num_states, out_all, &dim));
    DVS_TRY(sharded_args_ok(ctx, c, nrec_per_rank, s->nrec, out_all));
    DVS_CUDA_TRY(dvs::enter(ctx));
    DVS_TRY(dense_rows_fit((double)s->nrec * (double)dim * 4.0, "dvs_count_kmers_sharded", s->nrec, dim));
    AllRows a;
    DVS_TRY(allrows_alloc(ctx, c, nrec_per_rank, dim, &a));
    a.f->k = k;
    a.f->num_states = num_states;
    auto fail = [&](int rc) {
        cudaStreamSynchronize(c->side);
        dvs_kfreqs_free(a.f);
        return rc;
    };
    DevBuf<uint32_t> counts;
    if (counts.alloc((size_t)s->nrec * dim) != DVS_OK) return fail(DVS_ERR_CUDA);
    // every rank has left its previous use of this heap block before anybody writes into it
    int rc = comm_push_begin(ctx, c);
    if (rc == DVS_OK) rc = comm_barrier(ctx, c);
    if (rc != DVS_OK) return fail(rc);
    const char* ch_env = getenv("DVS_SHARD_CHUNKS");
    // every launch costs the counting ~0.12 ms (2 GPUs: 3 chunks 9.52 ms, 4: 9.60, 8: 10.11, 12: 10.79), while what the last
    // chunk leaves to push - 1/chunks of the rows to world - 1 peers - is exposed: few chunks, a few more with more peers
    // (chunks tapering towards the end were measured too: the small last launches balance badly, 10.27 ms at 4)
    const int dflt_chunks = c->world <= 2 ? 4 : 6;
    const uint32_t chunks = c->world == 1 ? 1u : (uint32_t)std::max(1, std::min(64, ch_env ? atoi(ch_env) : dflt_chunks));
    const size_t r0 = a.row0;
    CountDest dst{a.f->freqs.p + r0 * dim, a.f->totals.p + r0, a.f->entropy.p + r0, a.f->valid.p + r0, a.f->err.p + r0,
                  a.f->err_total.p + r0, chunks, nullptr};
    dst.after_chunk = [&](uint32_t rb, uint32_t re) -> int {
        // rows [rb, re) are final once the stream gets here: push them behind an event, on the copy engines,
        // while the next chunk is counted
        DVS_CUDA_TRY(cudaEventRecord(c->ev_ready, ctx->stream));
        DVS_CUDA_TRY(cudaStreamWaitEvent(c->side, c->ev_ready, 0));
        return allrows_push(c, a, rb, re, true);
    };
    rc = count_core(ctx, s, k, num_states, counts.p, dim, dst);
    if (rc == DVS_OK) rc = comm_push_commit(ctx, c);
    if (rc == DVS_OK) rc = comm_push_wait(ctx, c);
    if (rc == DVS_OK) rc = comm_check_error_async(ctx, c, "dvs_count_kmers_sharded");
    if (rc != DVS_OK) return fail(rc);
    *out_all = a.f;
    return DVS_OK;
}

int dvs_kfreqs_allgather(dvs_ctx* ctx, dvs_comm* c, const dvs_kfreqs* f, const uint32_t* nrec_per_rank,
                         dvs_kfreqs** out_all) {
    if (!f) {
        set_error("dvs_kfreqs_allgather: NULL argument");
        return DVS_ERR_ARG;
    }
    DVS_TRY(sharded_args_ok(ctx, c, nrec_per_rank, f->nrec, out_all));
    DVS_CUDA_TRY(dvs::enter(ctx));
    AllRows a;
    DVS_TRY(allrows_alloc(ctx, c, nrec_per_rank, f->dim, &a));
    a.f->k = f->k;
    a.f->num_states = f->num_states;
    auto fail = [&](int rc) {
        cudaStreamSynchronize(c->side);
        dvs_kfreqs_free(a.f);
        return rc;
    };
    cudaStream_t st = ctx->stream;
    int rc = comm_push_begin(ctx, c);
    if (rc == DVS_OK) rc = comm_barrier(ctx, c);
    if (rc != DVS_OK) return fail(rc);
    const size_t r0 = a.row0, n = f->nrec;
    cudaError_t e = cudaSuccess;
    if (n) {
        e = cudaMemcpyAsync(a.f->freqs.p + r0 * f->dim, f->freqs.p, n * f->dim * 8, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(a.f->entropy.p + r0, f->entropy.p, n * 8, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(a.f->err_total.p + r0, f->err_total.p, n * 8, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(a.f->totals.p + r0, f->totals.p, n * 8, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(a.f->valid.p + r0, f->valid.p, n, cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess) e = cudaMemcpyAsync(a.f->err.p + r0, f->err.p, n, cudaMemcpyDeviceToDevice, st);
    }
    if (e == cudaSuccess) e = cudaEventRecord(c->ev_ready, st);
    if (e == cudaSuccess) e = cudaStreamWaitEvent(c->side, c->ev_ready, 0);
    if (e != cudaSuccess) {
        set_error("dvs_kfreqs_allgather: %s", cudaGetErrorString(e));
        return fail(DVS_ERR_CUDA);
    }
    rc = allrows_push(c, a, 0, f->nrec, true);
    if (rc == DVS_OK) rc = comm_push_commit(ctx, c);
    if (rc == DVS_OK) rc = comm_push_wait(ctx, c);
    if (rc == DVS_OK) rc = comm_check_error_async(ctx, c, "dvs_kfreqs_allgather");
    if (rc != DVS_OK) return fail(rc);
    *out_all = a.f;
    return DVS_OK;
}

int dvs_kfreqs_from_rows(dvs_ctx* ctx, const double* rows, const double* entropies_or_null, uint32_t nrec,
                         uint64_t dim, dvs_kfreqs** out) {
    if (!ctx || !rows || !out || dim == 0) {
        set_error("dvs_kfreqs_from_rows: bad argument");
        return DVS_ERR_ARG;
    }
    dvs_kfreqs* f = nullptr;
    DVS_TRY(kfreqs_alloc(ctx, nrec, dim, false, &f));
    cudaStream_t st = ctx->stream;
    cudaError_t e = cudaSuccess;
    if (nrec) {
        e = cudaMemcpyAsync(f->freqs.p, rows, (size_t)nrec * dim * sizeof(double), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess && entropies_or_null)
            e = cudaMemcpyAsync(f->entropy.p, entropies_or_null, nrec * sizeof(double), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(f->valid.p, 1, nrec, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(f->totals.p, 0, nrec * sizeof(uint64_t), st);
        if (e == cudaSuccess) {
            k_rows_entropy<<<nrec, kEntThreads, kEntSmemBytes, st>>>(f->freqs.p, dim, f->entropy.p, f->err.p,
                                                                     f->err_total.p, entropies_or_null ? 0 : 1);
            ctx->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (e != cudaSuccess) {
        set_error("dvs_kfreqs_from_rows failed: %s", cudaGetErrorString(e));
        dvs_kfreqs_free(f);
        return DVS_ERR_CUDA;
    }
    *out = f;
    return DVS_OK;
}

int dvs_kfreqs_device_ptrs(const dvs_kfreqs* f, void** freqs, void** entropies, void** valid) {
    if (freqs) *freqs = f->freqs.p;
    if (entropies) *entropies = f->entropy.p;
    if (valid) *valid = f->valid.p;
    return DVS_OK;
}

int dvs_kfreqs_from_device(dvs_ctx* ctx, const void* d_rows, const void* d_entropies, const void* d_valid,
                           uint32_t nrec, uint64_t dim, dvs_kfreqs** out) {
    if (!ctx || !d_rows || !out || dim == 0) {
        set_error("dvs_kfreqs_from_device: bad argument");
        return DVS_ERR_ARG;
    }
    dvs_kfreqs* f = nullptr;
    DVS_TRY(kfreqs_alloc(ctx, nrec, dim, false, &f));
    cudaStream_t st = ctx->stream;
    cudaError_t e = cudaSuccess;
    if (nrec) {
        e = cudaMemcpyAsync(f->freqs.p, d_rows, (size_t)nrec * dim * sizeof(double), cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess && d_entropies)
            e = cudaMemcpyAsync(f->entropy.p, d_entropies, nrec * sizeof(double), cudaMemcpyDeviceToDevice, st);
        if (e == cudaSuccess)
            e = d_valid ? cudaMemcpyAsync(f->valid.p, d_valid, nrec, cudaMemcpyDeviceToDevice, st)
                        : cudaMemsetAsync(f->valid.p, 1, nrec, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(f->err.p, 0, nrec, st);
        if (e == cudaSuccess) e = cudaMemsetAsync(f->err_total.p, 0, nrec * sizeof(double), st);
        if (e == cudaSuccess) e = cudaMemsetAsync(f->totals.p, 0, nrec * sizeof(uint64_t), st);
        if (e == cudaSuccess && !d_entropies) {
            k_rows_entropy<<<nrec, kEntThreads, kEntSmemBytes, st>>>(f->freqs.p, dim, f->entropy.p, f->err.p,
                                                                     f->err_total.p, 1);
            ctx->launches++;
            e = cudaGetLastError();
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    }
    if (e != cudaSuccess) {
        set_error("dvs_kfreqs_from_device failed: %s", cudaGetErrorString(e));
        dvs_kfreqs_free(f);
        return DVS_ERR_CUDA;
    }
    *out = f;
    return DVS_OK;
}

int dvs_kfreqs_take_rows(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* rows, uint32_t n, dvs_kfreqs** out) {
    if (!ctx || !f || !out || (!rows && n)) {
        set_error("dvs_kfreqs_take_rows: bad argument");
        return DVS_ERR_ARG;
    }
    for (uint32_t i = 0; i < n; ++i)
        if (rows[i] >= f->nrec) {
            set_error("dvs_kfreqs_take_rows: row %u out of range", rows[i]);
            return DVS_ERR_ARG;
        }
    dvs_kfreqs* g = nullptr;
    DVS_TRY(kfreqs_alloc(ctx, n, f->dim, false, &g));
    g->k = f->k;
    g->num_states = f->num_states;
    cudaStream_t st = ctx->stream;
    cudaError_t e = cudaSuccess;
    DevBuf<uint32_t> d_rows;
    if (n) {
        if (d_rows.alloc(n) != DVS_OK) {
            dvs_kfreqs_free(g);
            return DVS_ERR_CUDA;
        }
        e = cudaMemcpyAsync(d_rows.p, rows, n * sizeof(uint32_t), cudaMemcpyHostToDevice, st);
        if (e == cudaSuccess) {
            k_take_rows<<<n, 256, 0, st>>>(f->freqs.p, f->entropy.p, f->valid.p, f->err.p, f->err_total.p, f->dim,
                                           d_rows.p, g->freqs.p, g->entropy.p, g->valid.p, g->err.p, g->err_total.p);
            ctx->launches++;
            e = cudaGetLastError();
        }
    }
    if (e == cudaSuccess) e = cudaMemsetAsync(g->totals.p, 0, (size_t)std::max<uint32_t>(n, 1) * sizeof(uint64_t), st);
    if (e == cudaSuccess) e = cudaStreamSynchronize(st);
    if (e != cudaSuccess) {
        set_error("dvs_kfreqs_take_rows failed: %s", cudaGetErrorString(e));
        dvs_kfreqs_free(g);
        return DVS_ERR_CUDA;
    }
    *out = g;
    return DVS_OK;
}

uint32_t dvs_kfreqs_nrec(const dvs_kfreqs* f) { return f->nrec; }
uint64_t dvs_kfreqs_dim(const dvs_kfreqs* f) { return f->dim; }

int dvs_kfreqs_download(dvs_ctx* ctx, const dvs_kfreqs* f, uint32_t first, uint32_t count, uint64_t* counts,
                        double* freqs, double* entropies, uint8_t* valid) {
    if (first + (uint64_t)count > f->nrec) {
        set_error("dvs_kfreqs_download: range out of bounds");
        return DVS_ERR_ARG;
    }
    if (count == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    const size_t n = (size_t)count * f->dim;
    std::vector<uint32_t> tmp;
    if (counts) {
        if (!f->has_counts) {
            set_error("dvs_kfreqs_download: this kfreqs was built from rows and holds no counts");
            return DVS_ERR_ARG;
        }
        tmp.resize(n);
        DVS_CUDA_TRY(cudaMemcpyAsync(tmp.data(), f->counts.p + (size_t)first * f->dim, n * sizeof(uint32_t),
                                     cudaMemcpyDeviceToHost, st));
    }
    if (freqs)
        DVS_CUDA_TRY(cudaMemcpyAsync(freqs, f->freqs.p + (size_t)first * f->dim, n * sizeof(double),
                                     cudaMemcpyDeviceToHost, st));
    if (entropies)
        DVS_CUDA_TRY(cudaMemcpyAsync(entropies, f->entropy.p + first, count * sizeof(double), cudaMemcpyDeviceToHost, st));
    if (valid) DVS_CUDA_TRY(cudaMemcpyAsync(valid, f->valid.p + first, count, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    if (counts)
        for (size_t i = 0; i < n; ++i) counts[i] = tmp[i];
    return DVS_OK;
}

void dvs_kfreqs_free(dvs_kfreqs* f) {
    if (!f) return;
    cudaSetDevice(f->device);
    // rows held in a peer window: the block goes back to the symmetric heap (the communicator must still be alive)
    if (f->heap) comm_heap_free(f->heap, f->heap_off);
    delete f;
}

int dvs_count_kmers_host(dvs_ctx* ctx, const uint8_t* seqs, const uint64_t* offsets, uint32_t nrec, int k,
                         int num_states, uint64_t* counts, double* freqs, double* entropies, uint8_t* valid) {
    dvs_seqset* s = nullptr;
    DVS_TRY(dvs_seqset_upload(ctx, seqs, offsets, nrec, &s));
    dvs_kfreqs* f = nullptr;
    int rc = dvs_count_kmers(ctx, s, k, num_states, &f);
    if (rc == DVS_OK) rc = dvs_kfreqs_download(ctx, f, 0, nrec, counts, freqs, entropies, valid);
    dvs_kfreqs_free(f);
    dvs_seqset_free(s);
    return rc;
}

int dvs_debug_log2(dvs_ctx* ctx, const double* x, double* y, uint64_t n) {
    if (n == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    DevBuf<double> dx, dy;
    DVS_TRY(dx.alloc(n));
    DVS_TRY(dy.alloc(n));
    DVS_CUDA_TRY(cudaMemcpyAsync(dx.p, x, n * sizeof(double), cudaMemcpyHostToDevice, ctx->stream));
    k_log2<<<(unsigned)((n + 255) / 256), 256, 0, ctx->stream>>>(dx.p, dy.p, n);
    DVS_LAUNCHED(ctx);
    DVS_CUDA_TRY(cudaMemcpyAsync(y, dy.p, n * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DVS_OK;
}

int dvs_debug_entropy(dvs_ctx* ctx, const double* rows, uint32_t nrec, uint64_t dim, double* out, uint8_t* err) {
    dvs_kfreqs* f = nullptr;
    DVS_TRY(dvs_kfreqs_from_rows(ctx, rows, nullptr, nrec, dim, &f));
    int rc = DVS_OK;
    cudaError_t e = cudaMemcpyAsync(out, f->entropy.p, nrec * sizeof(double), cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess && err) e = cudaMemcpyAsync(err, f->err.p, nrec, cudaMemcpyDeviceToHost, ctx->stream);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        set_error("dvs_debug_entropy failed: %s", cudaGetErrorString(e));
        rc = DVS_ERR_CUDA;
    }
    dvs_kfreqs_free(f);
    return rc;
}

}  // extern "C"
