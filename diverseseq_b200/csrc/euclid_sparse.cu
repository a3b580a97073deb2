// Euclidean distance matrix over SPARSE k-mer rows (dvs_count_kmers_sparse, 9 <= k <= 12): the dense rows of
// dvs_euclid_distances take 4^k x 12 bytes per record (201 MB at k=12) and 2 x 4^k flops per pair whatever the
// records share; here a pair costs one product per k-mer the two records share.
//
// Exact integer Gram form (DESIGN.md §5.11).  Record a has counts c_a and T_a = sum c_a < 2^32 valid k-mers, its
// frequencies are c_a / T_a.  With X_ab = sum_i c_a,i c_b,i and Q_a = X_aa (both < 2^64, exact in u64):
//     d_ab^2 = N_ab / (T_a T_b)^2,   N_ab = T_b^2 Q_a + T_a^2 Q_b - 2 T_a T_b X_ab = sum_i (c_a,i T_b - c_b,i T_a)^2
// N_ab is an exact unsigned 128-bit integer while T_a T_b < 2^63, so d = sqrt((double)N) / ((double)T_a (double)T_b)
// is within a few ulps of the true distance and exactly 0.0 for copies and proportional rows.  The reference
// computes the norm over ROUNDED frequencies fl(c / T) instead; the two differ by up to
// u sqrt(2 (|a|^2 + |b|^2)) absolute, so pairs with N < kXsTau (T_b^2 Q_a + T_a^2 Q_b) - i.e.
// d^2 < kXsTau (|a|^2 + |b|^2) - and pairs with T_a T_b >= 2^63 are recomputed by a difference-form pair kernel
// over the rounded frequencies (k_xs_pairs).
//
//   k_xs_self    Q_a of every record
//   k_xs_gram    X over the lower-triangle tiles of 8 rows (I) x 64 rows (J), a range of buckets per CTA: the I rows'
//                entries of a bucket are scattered into a shared table tab[bin][8] (u32 counts, 128 KB), every J
//                entry then reads the 8 counts of its bin with two LDS.128 and adds 8 u32 x u32 products
//                (IMAD.WIDE.U32) to u64 sums; bucket ranges are combined by u64 atomicAdd (integers: any order
//                gives the same bits)
//   k_xs_finish  N -> d, symmetric store, zero diagonal, NaN for records without a valid k-mer, the fallback list
//   k_xs_pairs   sum (fl(c_a/T_a) - fl(c_b/T_b))^2 over the union of two rows, bucket by bucket (one warp per pair)
// Every pair is computed by the same tile and the same code whatever the row range, so partial-range calls
// return the same bits as the whole matrix.
//
// dvs_euclid_distances_sparse_sharded runs the same kernels over two row sets: the I rows of this rank and the J rows
// of one peer, copied out of the peer's window (rectangular tiles: k_xs_gram<true>, k_xs_finish with rect = 1).  X
// and Q are exact integers and k_xs_finish / k_xs_pairs give a pair the same bits in either orientation, so every
// entry equals the single-GPU call's.
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "comm.cuh"
#include "common.cuh"
#include "sparse.cuh"

namespace dvs {

constexpr uint32_t kXsI = 8;                       // I rows per tile = u32 counts per table bin
constexpr uint32_t kXsWarps = 16;
constexpr uint32_t kXsThreads = 32 * kXsWarps;
constexpr uint32_t kXsJPerWarp = 4;
constexpr uint32_t kXsJ = kXsWarps * kXsJPerWarp;  // J rows per tile
constexpr size_t kXsSmemBytes = (size_t)kSpLowBins * kXsI * sizeof(uint32_t);
constexpr double kXsTau = 1e-13;                   // >= 8 u^2 / 1e-18 = 9.9e-14 (DESIGN.md §5.11)
constexpr uint32_t kXsFlagCap = 1u << 24;

struct XsTile {
    uint32_t ib, jc;  // I rows [8 ib, 8 ib + 8), J rows [64 jc, 64 jc + 64); 64 jc <= 8 ib + 7 unless rectangular
};

// one set of sparse rows as the kernels read them: a dvs_ksparse, a copy of a peer's rows, or rows [first, ...) of
// either (the per-row arrays start at row `first`; idx / cnt are addressed through offsets)
struct XsRows {
    const uint32_t* idx;
    const uint32_t* cnt;
    const uint64_t* offsets;
    const uint32_t* bucket_ptr;
    const uint32_t* bucket_nnz;
    const uint64_t* totals;
    uint32_t n, base;  // rows in the set, global index of its row 0
};

__global__ void __launch_bounds__(256)
k_xs_self(const uint32_t* __restrict__ cnt, const uint64_t* __restrict__ offsets, const uint32_t* __restrict__ bucket_ptr,
          uint32_t nb, unsigned long long* __restrict__ Q) {
    __shared__ unsigned long long s_w[8];
    const uint32_t r = blockIdx.x;
    const uint32_t* c = cnt + offsets[r];
    const uint32_t m = bucket_ptr[(size_t)r * (nb + 1) + nb];  // slots of the record (unused ones hold count 0)
    unsigned long long s = 0;
    for (uint32_t e = threadIdx.x; e < m; e += blockDim.x) s += (unsigned long long)c[e] * c[e];
    for (int o = 16; o; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (uint32_t w = 0; w < blockDim.x / 32; ++w) t += s_w[w];
        Q[r] = t;
    }
}

// X[tile][8][64] += the tile's products over buckets [range * bper, (range + 1) * bper).  kRect: the J rows are
// the set `J` (all rows of the tile, no triangle), otherwise they are the I rows (lower triangle) and `J` is unused.
template <bool kRect>
__global__ void __launch_bounds__(kXsThreads, 1)
k_xs_gram(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ cnt, const uint64_t* __restrict__ offsets,
          const uint32_t* __restrict__ bucket_ptr, const uint32_t* __restrict__ bucket_nnz, uint32_t n, uint32_t nb,
          const XsTile* __restrict__ tiles, uint32_t ntiles, uint32_t bper, unsigned long long* __restrict__ X,
          const XsRows J) {
    const uint32_t* __restrict__ j_idx = kRect ? J.idx : idx;
    const uint32_t* __restrict__ j_cnt = kRect ? J.cnt : cnt;
    const uint32_t* __restrict__ j_bptr = kRect ? J.bucket_ptr : bucket_ptr;
    const uint32_t* __restrict__ j_bnnz = kRect ? J.bucket_nnz : bucket_nnz;
    extern __shared__ __align__(16) uint32_t xs_tab[];  // [kSpLowBins][kXsI]
    const uint4* tab4 = reinterpret_cast<const uint4*>(xs_tab);
    // bucket-major grid: the CTAs resident at one time work on the same buckets, so the J slices come from L2
    const uint32_t tile = blockIdx.x % ntiles, range = blockIdx.x / ntiles;
    const XsTile tt = tiles[tile];
    const uint32_t b0 = range * bper, b1 = min(nb, b0 + bper);
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    for (uint32_t q = threadIdx.x; q < kSpLowBins * kXsI / 4; q += kXsThreads)
        reinterpret_cast<uint4*>(xs_tab)[q] = make_uint4(0, 0, 0, 0);
    // warps 0..7 own I row 8 ib + warp (densify / reset); every warp owns J rows 64 jc + warp + 16 q
    const uint32_t irow = tt.ib * kXsI + warp;
    const bool i_ok = warp < kXsI && irow < n;
    const uint64_t i_base = i_ok ? offsets[irow] : 0;
    const uint32_t i_last = min(n - 1, tt.ib * kXsI + kXsI - 1);
    uint32_t jrow[kXsJPerWarp];
    uint64_t j_base[kXsJPerWarp];
    bool j_ok[kXsJPerWarp];
#pragma unroll
    for (uint32_t q = 0; q < kXsJPerWarp; ++q) {
        jrow[q] = tt.jc * kXsJ + warp + kXsWarps * q;
        j_ok[q] = kRect ? jrow[q] < J.n : jrow[q] <= i_last;  // (pairs j > i of diagonal tiles are not stored)
        j_base[q] = j_ok[q] ? (kRect ? J.offsets : offsets)[jrow[q]] : 0;
    }
    unsigned long long acc[kXsJPerWarp][kXsI];
#pragma unroll
    for (uint32_t q = 0; q < kXsJPerWarp; ++q)
#pragma unroll
        for (uint32_t r = 0; r < kXsI; ++r) acc[q][r] = 0;
    __syncthreads();
    for (uint32_t b = b0; b < b1; ++b) {
        uint64_t is = 0;
        uint32_t im = 0;
        if (i_ok) {
            is = i_base + bucket_ptr[(size_t)irow * (nb + 1) + b];
            im = bucket_nnz[(size_t)irow * nb + b];
            for (uint32_t e = lane; e < im; e += 32) xs_tab[(idx[is + e] & (kSpLowBins - 1u)) * kXsI + warp] = cnt[is + e];
        }
        __syncthreads();
#pragma unroll
        for (uint32_t q = 0; q < kXsJPerWarp; ++q) {
            if (!j_ok[q]) continue;
            const uint64_t js = j_base[q] + j_bptr[(size_t)jrow[q] * (nb + 1) + b];
            const uint32_t jm = j_bnnz[(size_t)jrow[q] * nb + b];
            // batches of 4 entries per lane: the loads of a batch are issued before any of them is used
            for (uint32_t e0 = 0; e0 < jm; e0 += 128) {
                uint32_t lo[4], c[4];
#pragma unroll
                for (uint32_t u = 0; u < 4; ++u) {
                    const uint32_t e = e0 + lane + 32 * u;
                    lo[u] = e < jm ? __ldg(j_idx + js + e) & (kSpLowBins - 1u) : 0u;
                    c[u] = e < jm ? __ldg(j_cnt + js + e) : 0u;
                }
#pragma unroll
                for (uint32_t u = 0; u < 4; ++u) {
                    if (c[u] == 0) continue;
                    const uint4 v0 = tab4[lo[u] * 2], v1 = tab4[lo[u] * 2 + 1];
                    const unsigned long long cc = c[u];
                    acc[q][0] += cc * v0.x; acc[q][1] += cc * v0.y; acc[q][2] += cc * v0.z; acc[q][3] += cc * v0.w;
                    acc[q][4] += cc * v1.x; acc[q][5] += cc * v1.y; acc[q][6] += cc * v1.z; acc[q][7] += cc * v1.w;
                }
            }
        }
        __syncthreads();
        if (i_ok) {
            for (uint32_t e = lane; e < im; e += 32) xs_tab[(idx[is + e] & (kSpLowBins - 1u)) * kXsI + warp] = 0u;
            __syncwarp();  // the same warp scatters the next bucket of this row
        }
    }
    unsigned long long* xt = X + (size_t)tile * kXsI * kXsJ;
#pragma unroll
    for (uint32_t q = 0; q < kXsJPerWarp; ++q) {
        if (!j_ok[q]) continue;
#pragma unroll
        for (uint32_t r = 0; r < kXsI; ++r) {
            unsigned long long v = acc[q][r];
            for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (lane == r && v) atomicAdd(xt + r * kXsJ + warp + kXsWarps * q, v);
        }
    }
}

__device__ __forceinline__ double xs_u128_to_double(unsigned __int128 v) {
    const uint64_t hi = (uint64_t)(v >> 64), lo = (uint64_t)v;
    return hi ? __dadd_rn(__dmul_rn((double)hi, 18446744073709551616.0), (double)lo) : (double)lo;
}

// stores d at (i, j) and (j, i) (global indices) of every output where those rows are in [row_begin, row_end)
__device__ __forceinline__ void xs_store(const EuOuts& outs, uint32_t n, uint32_t row_begin, uint32_t row_end,
                                         uint32_t i, uint32_t j, double d) {
    for (int o = 0; o < outs.count; ++o) {
        if (i >= row_begin && i < row_end) outs.p[o][(size_t)(i - row_begin) * n + j] = d;
        if (i != j && j >= row_begin && j < row_end) outs.p[o][(size_t)(j - row_begin) * n + i] = d;
    }
}

// tile rows i of the I set (Qi, Ti: ni rows, global index ibase + i) against tile columns j of the J set.  rect = 0:
// the two sets are one and only j <= i is a pair; the list holds (i, j) as set-local indices.
__global__ void __launch_bounds__(kXsI * kXsJ)
k_xs_finish(const unsigned long long* __restrict__ X, const unsigned long long* __restrict__ Qi,
            const unsigned long long* __restrict__ Qj, const uint64_t* __restrict__ Ti, const uint64_t* __restrict__ Tj,
            const XsTile* __restrict__ tiles, uint32_t ni, uint32_t nj, uint32_t ibase, uint32_t jbase, int rect,
            uint32_t n, uint32_t row_begin, uint32_t row_end, const EuOuts outs, uint2* __restrict__ flagged,
            uint32_t flag_cap, uint32_t* __restrict__ flag_count) {
    const XsTile tt = tiles[blockIdx.x];
    const uint32_t r = threadIdx.x / kXsJ, c = threadIdx.x % kXsJ;
    const uint32_t i = tt.ib * kXsI + r, j = tt.jc * kXsJ + c;
    if (i >= ni || j >= nj || (!rect && j > i)) return;
    double d = 0.0;
    if (rect || i != j) {
        const uint64_t ta = Ti[i], tb = Tj[j];
        if (ta == 0 || tb == 0) {
            d = __longlong_as_double(0x7FF8000000000000LL);  // NaN: frequencies 0 / 0 (the dense rows' NaN row)
        } else {
            const uint64_t tab = ta * tb;  // < 2^64
            bool exact = tab < (1ull << 63);
            if (exact) {
                const unsigned long long x = X[(size_t)blockIdx.x * kXsI * kXsJ + threadIdx.x];
                const unsigned __int128 p = (unsigned __int128)(tb * tb) * Qi[i] + (unsigned __int128)(ta * ta) * Qj[j];
                const unsigned __int128 nn = p - (unsigned __int128)(2 * tab) * x;  // = sum (c_a T_b - c_b T_a)^2 >= 0
                if (nn != 0) {
                    const double nd = xs_u128_to_double(nn);
                    exact = nd >= kXsTau * xs_u128_to_double(p);
                    d = __ddiv_rn(__dsqrt_rn(nd), __dmul_rn((double)ta, (double)tb));
                }
            }
            if (!exact) {  // recomputed in difference form by k_xs_pairs
                const uint32_t at = atomicAdd(flag_count, 1u);
                if (at < flag_cap) flagged[at] = make_uint2(i, j);
                return;
            }
        }
    }
    xs_store(outs, n, row_begin, row_end, ibase + i, jbase + j, d);
}

// difference form over the rounded frequencies, one warp per pair (a of set A, b of set B): lane l merges the two
// rows' slices of buckets l, l + 32, ... (both ascending); the 32 partial sums are added by a fixed butterfly, so a
// pair gives the same bits whatever its position in the list, its orientation or the sets it is read from.
// out_list != NULL: d of pair p goes to out_list[p] (test hook), otherwise to the outputs.
__global__ void __launch_bounds__(256)
k_xs_pairs(const XsRows A, const XsRows B, uint32_t nb, const uint2* __restrict__ pairs, uint32_t np, uint32_t n,
           uint32_t row_begin, uint32_t row_end, const EuOuts outs, double* __restrict__ out_list) {
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t p = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); p < np; p += gridDim.x * (blockDim.x / 32)) {
        const uint2 ij = pairs[p];
        const uint32_t a = ij.x, b = ij.y;
        const double ta = (double)A.totals[a], tb = (double)B.totals[b];  // (exact: < 2^32)
        double acc = 0.0;
        for (uint32_t bk = lane; bk < nb; bk += 32) {
            const uint64_t sa = A.offsets[a] + A.bucket_ptr[(size_t)a * (nb + 1) + bk];
            const uint64_t sb = B.offsets[b] + B.bucket_ptr[(size_t)b * (nb + 1) + bk];
            const uint32_t na = A.bucket_nnz[(size_t)a * nb + bk], nbb = B.bucket_nnz[(size_t)b * nb + bk];
            uint32_t x = 0, y = 0;
            while (x < na || y < nbb) {
                const uint32_t ka = x < na ? A.idx[sa + x] : 0xFFFFFFFFu, kb = y < nbb ? B.idx[sb + y] : 0xFFFFFFFFu;
                const bool ua = ka <= kb, ub = kb <= ka;
                const double fa = ua ? __ddiv_rn((double)A.cnt[sa + x], ta) : 0.0;
                const double fb = ub ? __ddiv_rn((double)B.cnt[sb + y], tb) : 0.0;
                x += ua;
                y += ub;
                const double df = __dsub_rn(fa, fb);
                acc = __dadd_rn(acc, __dmul_rn(df, df));
            }
        }
        for (int o = 16; o; o >>= 1) acc = __dadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, o));
        if (lane == 0) {
            const uint32_t ga = A.base + a, gb = B.base + b;
            double d = __dsqrt_rn(acc);
            if (ga == gb) d = 0.0;
            else if (A.totals[a] == 0 || B.totals[b] == 0) d = __longlong_as_double(0x7FF8000000000000LL);
            if (out_list) out_list[p] = d;
            else xs_store(outs, n, row_begin, row_end, ga, gb, d);
        }
    }
}

// lower-triangle tiles that hold a pair with a row in [row_begin, row_end)
static std::vector<XsTile> xs_tiles_for_rows(uint32_t n, uint32_t row_begin, uint32_t row_end) {
    std::vector<XsTile> tiles;
    const uint32_t ni = (n + kXsI - 1) / kXsI;
    for (uint32_t ib = 0; ib < ni; ++ib) {
        const uint32_t i0 = ib * kXsI, i1 = std::min(n, i0 + kXsI);
        const bool i_in = i0 < row_end && i1 > row_begin;
        for (uint32_t jc = 0; jc * kXsJ < i1; ++jc) {
            const uint32_t j0 = jc * kXsJ, j1 = std::min(i1, j0 + kXsJ);
            if (i_in || (j0 < row_end && j1 > row_begin)) tiles.push_back({ib, jc});
        }
    }
    return tiles;
}

// all tiles of I rows [0, ni) x J rows [0, nj) (a block of pairs between two row sets)
static std::vector<XsTile> xs_tiles_rect(uint32_t ni, uint32_t nj) {
    std::vector<XsTile> tiles;
    for (uint32_t ib = 0; ib * kXsI < ni; ++ib)
        for (uint32_t jc = 0; jc * kXsJ < nj; ++jc) tiles.push_back({ib, jc});
    return tiles;
}

static XsRows xs_rows(const dvs_ksparse* sp) {
    return {sp->idx.p, sp->cnt.p, sp->offsets.p, sp->bucket_ptr.p, sp->bucket_nnz.p, sp->totals.p, sp->nrec, 0};
}

// rows [first, first + count) of a set
static XsRows xs_subset(XsRows r, uint32_t nb, uint32_t first, uint32_t count) {
    r.offsets += first;
    r.bucket_ptr += (size_t)first * (nb + 1);
    r.bucket_nnz += (size_t)first * nb;
    r.totals += first;
    r.n = count;
    r.base += first;
    return r;
}

// buckets per CTA: the J slices of one bucket range of all rows (`entries` in all) should stay in L2 (~32 MB of
// entries) while every (tile, range) CTA that reads them runs, and there should be a few CTAs per SM
static uint32_t xs_bucket_range(uint64_t entries, uint32_t nb, uint64_t ntiles, int sm_count) {
    const double per_bucket_bytes = 8.0 * (double)entries / (double)nb;  // all rows, one bucket
    uint32_t bper = nb;
    while (bper > 1 && per_bucket_bytes * bper > 32e6) bper >>= 1;
    while (bper > 1 && ntiles * ((nb + bper - 1) / bper) < 4ull * sm_count) bper >>= 1;
    return bper;
}

static int xs_launch_pairs(dvs_ctx* ctx, const XsRows& a, const XsRows& b, uint32_t nb, const uint2* d_pairs,
                           uint32_t npairs, uint32_t n, uint32_t row_begin, uint32_t row_end, const EuOuts& outs,
                           double* out_list) {
    const unsigned grid = (unsigned)std::min<uint32_t>((npairs + 7) / 8, (uint32_t)ctx->sm_count * 16);
    k_xs_pairs<<<grid, 256, 0, ctx->stream>>>(a, b, nb, d_pairs, npairs, n, row_begin, row_end, outs, out_list);
    DVS_LAUNCHED(ctx);
    return DVS_OK;
}

static EuOuts xs_one_out(double* out) {
    EuOuts o;
    memset(&o, 0, sizeof o);
    o.p[0] = out;
    o.count = out ? 1 : 0;
    return o;
}

}  // namespace dvs

using namespace dvs;

extern "C" int dvs_euclid_distances_sparse(dvs_ctx* ctx, const dvs_ksparse* sp, uint32_t row_begin, uint32_t row_end,
                                           double* dist) {
    // the counter describes this call whatever its outcome; after a list overflow it holds the overflowing count
    if (ctx) ctx->last_euclid_fallback_pairs = 0;
    if (!ctx || !sp || !dist || row_begin > row_end || row_end > sp->nrec) {
        set_error("dvs_euclid_distances_sparse: bad argument");
        return DVS_ERR_ARG;
    }
    const uint32_t n = sp->nrec, nb = sp->nb;
    const size_t nrows = row_end - row_begin;
    if (nrows == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    const std::vector<XsTile> tiles = xs_tiles_for_rows(n, row_begin, row_end);
    const uint32_t ntiles = (uint32_t)tiles.size();
    // the matrix is written in place when `dist` is device memory of this GPU
    cudaPointerAttributes pa;
    const bool on_device = cudaPointerGetAttributes(&pa, dist) == cudaSuccess && pa.device == ctx->device &&
                           (pa.type == cudaMemoryTypeDevice || pa.type == cudaMemoryTypeManaged);
    cudaGetLastError();
    const uint64_t tile_pairs = (uint64_t)ntiles * kXsI * kXsJ;
    const uint32_t flag_cap = (uint32_t)std::min<uint64_t>(tile_pairs, kXsFlagCap);
    const uint64_t need = tile_pairs * 8 + (on_device ? 0 : (uint64_t)nrows * n * 8) + (uint64_t)flag_cap * 8 +
                          (uint64_t)n * 16 + (uint64_t)ntiles * sizeof(XsTile);
    size_t free_b = 0, total_b = 0;
    DVS_CUDA_TRY(cudaMemGetInfo(&free_b, &total_b));
    if (need > free_b) {
        set_error("dvs_euclid_distances_sparse: rows [%u, %u) x %u columns need %.2f GB of device memory, %.2f GB are "
                  "free; ask for fewer rows at a time (row_begin, row_end)%s", row_begin, row_end, n, need / 1e9,
                  free_b / 1e9, on_device ? "" : " or pass a device output");
        return DVS_ERR_ARG;
    }
    std::vector<uint64_t> h_nnz(n);
    DVS_CUDA_TRY(cudaMemcpyAsync(h_nnz.data(), sp->nnz.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    uint64_t entries = 0;
    for (uint64_t v : h_nnz) entries += v;
    const uint32_t bper = xs_bucket_range(entries, nb, ntiles, ctx->sm_count);
    const uint32_t nranges = (nb + bper - 1) / bper;
    if ((uint64_t)ntiles * nranges > 0x7FFFFFFFull) {
        set_error("dvs_euclid_distances_sparse: %u records are too many for one call", n);
        return DVS_ERR_ARG;
    }
    DevBuf<XsTile> d_tiles;
    DevBuf<unsigned long long> d_X, d_Q;
    DevBuf<uint2> d_flag;
    DevBuf<uint32_t> d_cnt;
    DevBuf<double> d_out;
    DVS_TRY(d_tiles.alloc(ntiles));
    DVS_TRY(d_X.alloc(tile_pairs));
    DVS_TRY(d_Q.alloc(n));
    DVS_TRY(d_flag.alloc(flag_cap));
    DVS_TRY(d_cnt.alloc(1));
    double* out = dist;
    if (!on_device) {
        DVS_TRY(d_out.alloc(nrows * n));
        out = d_out.p;
    }
    const XsRows all = xs_rows(sp);
    const EuOuts outs = xs_one_out(out);
    DVS_CUDA_TRY(cudaMemcpyAsync(d_tiles.p, tiles.data(), ntiles * sizeof(XsTile), cudaMemcpyHostToDevice, st));
    DVS_CUDA_TRY(cudaMemsetAsync(d_X.p, 0, tile_pairs * 8, st));
    DVS_CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, sizeof(uint32_t), st));
    DVS_CUDA_TRY(cudaFuncSetAttribute(k_xs_gram<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXsSmemBytes));
    PhaseTimer pt(ctx, DVS_PHASE_EUCLID_SPARSE);
    k_xs_self<<<n, 256, 0, st>>>(sp->cnt.p, sp->offsets.p, sp->bucket_ptr.p, nb, d_Q.p);
    DVS_LAUNCHED(ctx);
    k_xs_gram<false><<<ntiles * nranges, kXsThreads, kXsSmemBytes, st>>>(
        sp->idx.p, sp->cnt.p, sp->offsets.p, sp->bucket_ptr.p, sp->bucket_nnz.p, n, nb, d_tiles.p, ntiles, bper, d_X.p,
        all);
    DVS_LAUNCHED(ctx);
    k_xs_finish<<<ntiles, kXsI * kXsJ, 0, st>>>(d_X.p, d_Q.p, d_Q.p, sp->totals.p, sp->totals.p, d_tiles.p, n, n, 0, 0,
                                                0, n, row_begin, row_end, outs, d_flag.p, flag_cap, d_cnt.p);
    DVS_LAUNCHED(ctx);
    uint32_t h_cnt = 0;
    DVS_CUDA_TRY(cudaMemcpyAsync(&h_cnt, d_cnt.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    ctx->last_euclid_fallback_pairs = h_cnt;
    if (h_cnt > flag_cap) {
        set_error("dvs_euclid_distances_sparse: %u pairs need the difference form, more than the %u one call can list; "
                  "ask for fewer rows at a time", h_cnt, flag_cap);
        return DVS_ERR_VALUE;
    }
    if (h_cnt) DVS_TRY(xs_launch_pairs(ctx, all, all, nb, d_flag.p, h_cnt, n, row_begin, row_end, outs, nullptr));
    pt.stop();
    if (!on_device)
        DVS_CUDA_TRY(cudaMemcpyAsync(dist, out, nrows * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    return DVS_OK;
}

// ---- multi-GPU: rows stay with the rank that counted them ------------------------------------------------------

namespace dvs {

// what every rank tells the others before anything else (dvs_comm_allgatherv)
struct XsMeta {
    uint64_t nrec, k, slots;
    uint64_t half_slot;           // first slot of local row ceil(nrec / 2) (relative to the first row's)
    uint64_t entries_lo, entries_hi;  // distinct k-mers of rows [0, ceil(nrec / 2)) and of the rest
    uint64_t npr[kCommMaxWorld];  // the nrec_per_rank this rank was given
};

// byte layout of one rank's staged rows; every rank stages at the largest shard's sizes, so its heap allocations
// stay in step with the peers'.  The same layout holds the copy of one peer's rows.
struct XsStage {
    uint64_t idx, cnt, offsets, bucket_ptr, bucket_nnz, totals, bytes;
};

static uint64_t xs_align(uint64_t b) { return (b + 255) & ~255ull; }

static XsStage xs_stage_layout(uint64_t max_n, uint64_t max_slots, uint32_t nb) {
    XsStage s;
    uint64_t o = 0;
    s.idx = o;
    o += xs_align(max_slots * 4);
    s.cnt = o;
    o += xs_align(max_slots * 4);
    s.offsets = o;
    o += xs_align((max_n + 1) * 8);
    s.bucket_ptr = o;
    o += xs_align(max_n * (nb + 1) * 4);
    s.bucket_nnz = o;
    o += xs_align(max_n * nb * 4);
    s.totals = o;
    o += xs_align(max_n * 8);
    s.bytes = std::max<uint64_t>(o, 256);
    return s;
}

// window bytes the call needs: control words + staged rows (none on one rank: nobody would read them) + the n x n
// matrix (shard.window_bytes_for_sparse)
static uint64_t xs_window_need(int world, uint64_t max_n, uint64_t max_slots, uint32_t nb, uint64_t n) {
    return kCommCtrlBytes + (world > 1 ? xs_stage_layout(max_n, max_slots, nb).bytes : 0) +
           std::max<uint64_t>(xs_align(n * n * 8), 256);
}

static XsRows xs_rows_at(uint8_t* base, const XsStage& L, uint32_t n, uint32_t global_base) {
    return {reinterpret_cast<const uint32_t*>(base + L.idx), reinterpret_cast<const uint32_t*>(base + L.cnt),
            reinterpret_cast<const uint64_t*>(base + L.offsets), reinterpret_cast<const uint32_t*>(base + L.bucket_ptr),
            reinterpret_cast<const uint32_t*>(base + L.bucket_nnz), reinterpret_cast<const uint64_t*>(base + L.totals),
            n, global_base};
}

// one block of pairs this rank computes: its rows [i0, i0 + ni) against rows [j0, j0 + nj) of rank q (q == rank:
// the lower triangle of its own rows)
struct XsBlock {
    int q;
    uint32_t i0, ni, j0, nj;
    uint64_t entries;  // distinct k-mers of the rows involved
    std::vector<XsTile> tiles;
};

// the prescribed ownership: a pair of ranks p != q at distance d = (q - p) mod W is computed by p for d < W/2, by q
// for d > W/2; at d = W/2 rank r = min(p, q) takes its rows below ceil(n_r / 2) and rank r + W/2 the rest
static std::vector<XsBlock> xs_blocks(int me, int W, const std::vector<XsMeta>& m) {
    std::vector<XsBlock> out;
    const uint32_t n_me = (uint32_t)m[me].nrec;
    if (n_me) out.push_back({me, 0, n_me, 0, n_me, m[me].entries_lo + m[me].entries_hi, xs_tiles_for_rows(n_me, 0, n_me)});
    for (int d = 1; 2 * d <= W; ++d) {
        const int q = (me + d) % W;
        const uint32_t n_q = (uint32_t)m[q].nrec;
        XsBlock b{q, 0, n_me, 0, n_q, 0, {}};
        uint64_t e_i = m[me].entries_lo + m[me].entries_hi, e_j = m[q].entries_lo + m[q].entries_hi;
        if (2 * d == W) {
            if (me < q) {
                b.ni = (n_me + 1) / 2;
                e_i = m[me].entries_lo;
            } else {
                b.j0 = (n_q + 1) / 2;
                b.nj = n_q - b.j0;
                e_j = m[q].entries_hi;
            }
        }
        if (!b.ni || !b.nj) continue;
        b.entries = e_i + e_j;
        b.tiles = xs_tiles_rect(b.ni, b.nj);
        out.push_back(std::move(b));
    }
    return out;
}

// copies rows [j0, n) of rank q's staged rows (at `src` in its window, rows at their staged positions) into `dst`
static cudaError_t xs_copy_rows(uint8_t* dst, const uint8_t* src, const XsStage& L, const XsMeta& mq, uint32_t j0,
                                uint32_t nb, cudaStream_t st) {
    const uint64_t n = mq.nrec, s0 = j0 ? mq.half_slot : 0;
    const uint64_t pieces[5][3] = {{L.idx + s0 * 4, (mq.slots - s0) * 4, 0},
                                   {L.cnt + s0 * 4, (mq.slots - s0) * 4, 0},
                                   {L.offsets + j0 * 8ull, (n + 1 - j0) * 8, 0},
                                   {L.bucket_ptr + j0 * (nb + 1ull) * 4, (n - j0) * (nb + 1) * 4, 0},
                                   {L.bucket_nnz + j0 * (uint64_t)nb * 4, (n - j0) * nb * 4, 0}};
    for (const auto& pc : pieces)
        if (pc[1]) {
            cudaError_t e = cudaMemcpyAsync(dst + pc[0], src + pc[0], pc[1], cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) return e;
        }
    return (n - j0) ? cudaMemcpyAsync(dst + L.totals + j0 * 8ull, src + L.totals + j0 * 8ull, (n - j0) * 8,
                                      cudaMemcpyDeviceToDevice, st)
                    : cudaSuccess;
}

// this rank's blocks, after every rank has staged its rows.  *listed: pairs listed for the difference form over all
// blocks (may exceed the cap: then no pair kernel runs and the caller reports the overflow)
static int xs_sharded_blocks(dvs_ctx* ctx, dvs_comm* c, const dvs_ksparse* local, const std::vector<XsMeta>& m,
                             const std::vector<uint32_t>& base, const XsStage& L, uint64_t stage_off,
                             const EuOuts& outs, uint32_t n, uint32_t* listed) {
    cudaStream_t st = ctx->stream;
    const int me = c->rank, W = c->world;
    const uint32_t nb = local->nb;
    std::vector<XsBlock> blocks = xs_blocks(me, W, m);
    *listed = 0;
    if (blocks.empty()) return DVS_OK;
    uint64_t max_tiles = 0, tile_pairs = 0;
    for (const XsBlock& b : blocks) {
        max_tiles = std::max<uint64_t>(max_tiles, b.tiles.size());
        tile_pairs += (uint64_t)b.tiles.size() * kXsI * kXsJ;
    }
    const uint32_t flag_cap = (uint32_t)std::min<uint64_t>(tile_pairs, kXsFlagCap);
    uint64_t max_n = 0;
    for (const XsMeta& x : m) max_n = std::max<uint64_t>(max_n, x.nrec);
    DevBuf<uint8_t> d_peer;
    DevBuf<XsTile> d_tiles;
    DevBuf<unsigned long long> d_X, d_Qi, d_Qj;
    DevBuf<uint2> d_flag;
    DevBuf<uint32_t> d_cnt;
    DVS_TRY(d_peer.alloc(W > 1 ? L.bytes : 1));
    DVS_TRY(d_tiles.alloc(max_tiles));
    DVS_TRY(d_X.alloc(max_tiles * kXsI * kXsJ));
    DVS_TRY(d_Qi.alloc(m[me].nrec));
    DVS_TRY(d_Qj.alloc(max_n));
    DVS_TRY(d_flag.alloc(flag_cap));
    DVS_TRY(d_cnt.alloc(1));
    DVS_CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, sizeof(uint32_t), st));
    DVS_CUDA_TRY(cudaFuncSetAttribute(k_xs_gram<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXsSmemBytes));
    DVS_CUDA_TRY(cudaFuncSetAttribute(k_xs_gram<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXsSmemBytes));
    XsRows mine = xs_rows(local);
    mine.base = base[me];
    const XsRows peer_all = xs_rows_at(d_peer.p, L, 0, 0);
    ctx->euclid_rows_ms = 0.0;
    PhaseTimer pt(ctx, DVS_PHASE_EUCLID_SPARSE);
    k_xs_self<<<m[me].nrec, 256, 0, st>>>(local->cnt.p, local->offsets.p, local->bucket_ptr.p, nb, d_Qi.p);
    DVS_LAUNCHED(ctx);
    uint32_t done = 0;  // pairs listed by the blocks before this one
    for (const XsBlock& b : blocks) {
        const bool cross = b.q != me;
        const XsRows I = xs_subset(mine, nb, b.i0, b.ni);
        XsRows J = I;
        if (cross) {
            // the staged rows do not change before the final barrier of the call: no barrier per step
            if (ctx->timing) cudaEventRecord(ctx->ev_start[DVS_PHASE_EUCLID_SPARSE_ROWS], st);
            DVS_CUDA_TRY(xs_copy_rows(d_peer.p, c->peer[b.q] + stage_off, L, m[b.q], b.j0, nb, st));
            if (ctx->timing) cudaEventRecord(ctx->ev_stop[DVS_PHASE_EUCLID_SPARSE_ROWS], st);
            XsRows all_q = peer_all;
            all_q.n = (uint32_t)m[b.q].nrec;
            all_q.base = base[b.q];
            J = xs_subset(all_q, nb, b.j0, b.nj);
            k_xs_self<<<b.nj, 256, 0, st>>>(J.cnt, J.offsets, J.bucket_ptr, nb, d_Qj.p);
            DVS_LAUNCHED(ctx);
        }
        const uint32_t ntiles = (uint32_t)b.tiles.size();
        const uint32_t bper = xs_bucket_range(b.entries, nb, ntiles, ctx->sm_count);
        const uint32_t nranges = (nb + bper - 1) / bper;
        if ((uint64_t)ntiles * nranges > 0x7FFFFFFFull) {
            set_error("dvs_euclid_distances_sparse_sharded: %u x %u records are too many for one block", b.ni, b.nj);
            return DVS_ERR_ARG;
        }
        DVS_CUDA_TRY(cudaMemcpyAsync(d_tiles.p, b.tiles.data(), ntiles * sizeof(XsTile), cudaMemcpyHostToDevice, st));
        DVS_CUDA_TRY(cudaMemsetAsync(d_X.p, 0, (size_t)ntiles * kXsI * kXsJ * 8, st));
        if (cross)
            k_xs_gram<true><<<ntiles * nranges, kXsThreads, kXsSmemBytes, st>>>(
                I.idx, I.cnt, I.offsets, I.bucket_ptr, I.bucket_nnz, I.n, nb, d_tiles.p, ntiles, bper, d_X.p, J);
        else
            k_xs_gram<false><<<ntiles * nranges, kXsThreads, kXsSmemBytes, st>>>(
                I.idx, I.cnt, I.offsets, I.bucket_ptr, I.bucket_nnz, I.n, nb, d_tiles.p, ntiles, bper, d_X.p, J);
        DVS_LAUNCHED(ctx);
        const unsigned long long* Qi = d_Qi.p + b.i0;
        const unsigned long long* Qj = cross ? d_Qj.p : Qi;
        k_xs_finish<<<ntiles, kXsI * kXsJ, 0, st>>>(d_X.p, Qi, Qj, I.totals, J.totals, d_tiles.p, I.n, J.n, I.base,
                                                    J.base, cross ? 1 : 0, n, 0, n, outs, d_flag.p, flag_cap, d_cnt.p);
        DVS_LAUNCHED(ctx);
        uint32_t h_cnt = 0;
        DVS_CUDA_TRY(cudaMemcpyAsync(&h_cnt, d_cnt.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
        DVS_CUDA_TRY(cudaStreamSynchronize(st));
        *listed = h_cnt;
        if (cross && ctx->timing) {
            float ms = 0.0f;
            if (cudaEventElapsedTime(&ms, ctx->ev_start[DVS_PHASE_EUCLID_SPARSE_ROWS],
                                     ctx->ev_stop[DVS_PHASE_EUCLID_SPARSE_ROWS]) == cudaSuccess)
                ctx->euclid_rows_ms += ms;
        }
        // this block's pairs are listed at [done, h_cnt); they read the peer copy, which the next step overwrites
        if (h_cnt <= flag_cap && h_cnt > done)
            DVS_TRY(xs_launch_pairs(ctx, I, J, nb, d_flag.p + done, h_cnt - done, n, 0, n, outs, nullptr));
        done = h_cnt;
    }
    pt.stop();
    return DVS_OK;
}

}  // namespace dvs

extern "C" int dvs_euclid_distances_sparse_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_ksparse* local,
                                                   const uint32_t* nrec_per_rank, double* dist) {
    static const char* kName = "dvs_euclid_distances_sparse_sharded";
    if (ctx) ctx->last_euclid_fallback_pairs = 0;
    if (!ctx || !c || !local || !nrec_per_rank || !dist || !c->connected) {
        set_error("%s: bad argument / communicator not connected", kName);
        return DVS_ERR_ARG;
    }
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    const int W = c->world, me = c->rank;
    ctx->euclid_rows_ms = -1.0;
    // 1. metadata of every rank; the checks below see the same data on every rank, so all return the same status
    std::vector<XsMeta> m(W);
    {
        XsMeta x;
        memset(&x, 0, sizeof x);
        const uint32_t nl = local->nrec, h = (nl + 1) / 2;
        x.nrec = nl;
        x.k = (uint64_t)local->k;
        x.slots = local->h_offsets[nl] - local->h_offsets[0];
        x.half_slot = local->h_offsets[h] - local->h_offsets[0];
        if (nl) {
            std::vector<uint64_t> h_nnz(nl);
            DVS_CUDA_TRY(cudaMemcpyAsync(h_nnz.data(), local->nnz.p, (size_t)nl * 8, cudaMemcpyDeviceToHost, st));
            DVS_CUDA_TRY(cudaStreamSynchronize(st));
            for (uint32_t r = 0; r < nl; ++r) (r < h ? x.entries_lo : x.entries_hi) += h_nnz[r];
        }
        for (int r = 0; r < W; ++r) x.npr[r] = nrec_per_rank[r];
        DevBuf<XsMeta> d_in, d_all;
        DVS_TRY(d_in.alloc(1));
        DVS_TRY(d_all.alloc(W));
        DVS_CUDA_TRY(cudaMemcpyAsync(d_in.p, &x, sizeof x, cudaMemcpyHostToDevice, st));
        std::vector<uint64_t> bytes(W, sizeof(XsMeta));
        DVS_TRY(dvs_comm_allgatherv(ctx, c, d_in.p, bytes.data(), d_all.p));
        DVS_CUDA_TRY(cudaMemcpyAsync(m.data(), d_all.p, W * sizeof(XsMeta), cudaMemcpyDeviceToHost, st));
        DVS_CUDA_TRY(cudaStreamSynchronize(st));
    }
    std::vector<uint32_t> base(W + 1, 0);
    uint64_t n64 = 0, max_n = 0, max_slots = 0;
    for (int r = 0; r < W; ++r) {
        if (m[r].k != m[0].k) {
            set_error("%s: rank %d counted k=%llu, rank 0 k=%llu", kName, r, (unsigned long long)m[r].k,
                      (unsigned long long)m[0].k);
            return DVS_ERR_ARG;
        }
        for (int s = 0; s < W; ++s)
            if (m[s].npr[r] != m[r].nrec) {
                set_error("%s: rank %d passed nrec_per_rank[%d] = %llu, but rank %d holds %llu records", kName, s, r,
                          (unsigned long long)m[s].npr[r], r, (unsigned long long)m[r].nrec);
                return DVS_ERR_ARG;
            }
        base[r] = (uint32_t)n64;
        n64 += m[r].nrec;
        max_n = std::max(max_n, m[r].nrec);
        max_slots = std::max(max_slots, m[r].slots);
    }
    if (n64 >= (1ull << 31)) {
        set_error("%s: %llu records are too many", kName, (unsigned long long)n64);
        return DVS_ERR_ARG;
    }
    const uint32_t n = (uint32_t)n64, nb = local->nb;
    base[W] = n;
    if (n == 0) return DVS_OK;
    const uint64_t need = xs_window_need(W, max_n, max_slots, nb, n);
    if (need > c->window_bytes) {
        set_error("%s: the staged rows and the %u x %u matrix need a window of %llu bytes, the window has %llu "
                  "(shard.window_bytes_for_sparse)", kName, n, n, (unsigned long long)need,
                  (unsigned long long)c->window_bytes);
        return DVS_ERR_ARG;
    }
    // 2. symmetric heap: staged rows (W > 1), matrix (the same sizes on every rank)
    const bool staged = W > 1;
    const XsStage L = xs_stage_layout(max_n, max_slots, nb);
    uint64_t soff = 0, moff = 0;
    if (staged) DVS_TRY(comm_heap_alloc(c, L.bytes, &soff));
    int rc = comm_heap_alloc(c, (uint64_t)n * n * 8, &moff);
    if (rc != DVS_OK) {
        if (staged) comm_heap_free(c, soff);
        return rc;
    }
    // from here on every rank goes through the final barrier and the all-reduce whatever happens
    cudaError_t e = cudaSuccess;
    if (staged) {
        uint8_t* w = c->window + soff;
        const XsMeta& x = m[me];
        const uint64_t s0 = local->h_offsets[0];
        std::vector<uint64_t> rebased(x.nrec + 1);
        for (uint64_t r = 0; r <= x.nrec; ++r) rebased[r] = local->h_offsets[r] - s0;
        if (x.slots) {
            e = cudaMemcpyAsync(w + L.idx, local->idx.p + s0, x.slots * 4, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(w + L.cnt, local->cnt.p + s0, x.slots * 4, cudaMemcpyDeviceToDevice, st);
        }
        if (e == cudaSuccess)
            e = cudaMemcpyAsync(w + L.offsets, rebased.data(), (x.nrec + 1) * 8, cudaMemcpyHostToDevice, st);
        if (x.nrec) {
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(w + L.bucket_ptr, local->bucket_ptr.p, x.nrec * (nb + 1) * 4,
                                    cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(w + L.bucket_nnz, local->bucket_nnz.p, x.nrec * nb * 4, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess)
                e = cudaMemcpyAsync(w + L.totals, local->totals.p, x.nrec * 8, cudaMemcpyDeviceToDevice, st);
        }
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);  // (the host offsets above)
    }
    if (e != cudaSuccess) {
        set_error("%s: staging the rows: %s", kName, cudaGetErrorString(e));
        rc = DVS_ERR_CUDA;
    }
    int brc = comm_barrier(ctx, c);  // every rank's rows are staged, nobody still reads an older block
    if (rc == DVS_OK) rc = brc;
    uint32_t listed = 0;
    if (rc == DVS_OK) {
        EuOuts outs;
        memset(&outs, 0, sizeof outs);
        for (int r = 0; r < W; ++r) outs.p[r] = reinterpret_cast<double*>(c->peer[(me + r) % W] + moff);
        outs.count = W;
        rc = xs_sharded_blocks(ctx, c, local, m, base, L, soff, outs, n, &listed);
    }
    ctx->last_euclid_fallback_pairs = listed;
    const bool overflow = rc == DVS_OK && listed > kXsFlagCap;
    // 3. every distance has landed in every window; the worst status of any rank decides for all (a failure of the
    // CUDA runtime before a bad argument before a list overflow)
    enum : uint32_t { kCuda = 0, kArg = 1, kValue = 2, kOk = 3 };
    const uint32_t mine_st = overflow || rc == DVS_ERR_VALUE ? kValue : rc == DVS_OK ? kOk : rc == DVS_ERR_ARG ? kArg : kCuda;
    uint32_t h_st[2] = {mine_st, kCuda};
    DevBuf<uint32_t> d_st;
    int rc2 = d_st.alloc(2);
    if (rc2 == DVS_OK && (e = cudaMemcpyAsync(d_st.p, h_st, sizeof h_st, cudaMemcpyHostToDevice, st)) != cudaSuccess)
        rc2 = DVS_ERR_CUDA;
    if (rc2 == DVS_OK) rc2 = comm_barrier(ctx, c);
    if (rc2 == DVS_OK) rc2 = comm_min_u32(ctx, c, d_st.p, d_st.p + 1);
    if (rc2 == DVS_OK && ((e = cudaMemcpyAsync(h_st, d_st.p, sizeof h_st, cudaMemcpyDeviceToHost, st)) != cudaSuccess ||
                          (e = cudaStreamSynchronize(st)) != cudaSuccess))
        rc2 = DVS_ERR_CUDA;
    if (rc2 == DVS_OK) rc2 = comm_check_error(ctx, c, kName);
    if (rc2 == DVS_OK && h_st[1] == kOk) {
        e = cudaMemcpyAsync(dist, c->window + moff, (size_t)n * n * sizeof(double), cudaMemcpyDefault, st);
        if (e == cudaSuccess) e = cudaStreamSynchronize(st);
        if (e != cudaSuccess) {
            set_error("%s: copying the matrix out: %s", kName, cudaGetErrorString(e));
            rc2 = DVS_ERR_CUDA;
        }
    }
    comm_heap_free(c, moff);
    if (staged) comm_heap_free(c, soff);
    if (rc2 != DVS_OK) {  // (the ranks could not agree on a status)
        if (e != cudaSuccess && rc2 == DVS_ERR_CUDA) set_error("%s: %s", kName, cudaGetErrorString(e));
        return rc2;
    }
    const uint32_t all_st = h_st[1];
    if (all_st == kOk) return DVS_OK;
    if (all_st == kValue && overflow)
        set_error("%s: %u pairs of rank %d need the difference form, more than the %u one rank can list", kName, listed,
                  me, kXsFlagCap);
    else if (all_st == kValue)
        set_error("%s: more pairs of another rank need the difference form than the %u one rank can list", kName,
                  kXsFlagCap);
    else if (all_st != mine_st)  // (otherwise this rank's own message stands)
        set_error("%s: the call failed on another rank (%s)", kName,
                  all_st == kArg ? "bad argument or too many records" : "CUDA error");
    return all_st == kValue ? DVS_ERR_VALUE : all_st == kArg ? DVS_ERR_ARG : DVS_ERR_CUDA;
}

extern "C" int dvs_debug_euclid_sparse_pairs(dvs_ctx* ctx, const dvs_ksparse* sp, const uint32_t* pairs, uint32_t n,
                                             double* out) {
    if (!ctx || !sp || (n && (!pairs || !out))) {
        set_error("dvs_debug_euclid_sparse_pairs: bad argument");
        return DVS_ERR_ARG;
    }
    for (uint64_t q = 0; q < 2ull * n; ++q)
        if (pairs[q] >= sp->nrec) {
            set_error("dvs_debug_euclid_sparse_pairs: record %u out of range (%u records)", pairs[q], sp->nrec);
            return DVS_ERR_ARG;
        }
    if (n == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    DevBuf<uint2> d_pairs;
    DevBuf<double> d_out;
    DVS_TRY(d_pairs.alloc(n));
    DVS_TRY(d_out.alloc(n));
    DVS_CUDA_TRY(cudaMemcpyAsync(d_pairs.p, pairs, (size_t)n * sizeof(uint2), cudaMemcpyHostToDevice, st));
    const XsRows all = xs_rows(sp);
    DVS_TRY(xs_launch_pairs(ctx, all, all, sp->nb, d_pairs.p, n, sp->nrec, 0, 0, xs_one_out(nullptr), d_out.p));
    DVS_CUDA_TRY(cudaMemcpyAsync(out, d_out.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    return DVS_OK;
}
