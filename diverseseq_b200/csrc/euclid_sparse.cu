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
#include <math.h>
#include <string.h>

#include <algorithm>
#include <vector>

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
    uint32_t ib, jc;  // I rows [8 ib, 8 ib + 8), J rows [64 jc, 64 jc + 64), 64 jc <= 8 ib + 7
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

// X[tile][8][64] += the tile's products over buckets [range * bper, (range + 1) * bper)
__global__ void __launch_bounds__(kXsThreads, 1)
k_xs_gram(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ cnt, const uint64_t* __restrict__ offsets,
          const uint32_t* __restrict__ bucket_ptr, const uint32_t* __restrict__ bucket_nnz, uint32_t n, uint32_t nb,
          const XsTile* __restrict__ tiles, uint32_t ntiles, uint32_t bper, unsigned long long* __restrict__ X) {
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
        j_ok[q] = jrow[q] <= i_last;  // (pairs j > i of the diagonal tiles are computed and not stored)
        j_base[q] = j_ok[q] ? offsets[jrow[q]] : 0;
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
            const uint64_t js = j_base[q] + bucket_ptr[(size_t)jrow[q] * (nb + 1) + b];
            const uint32_t jm = bucket_nnz[(size_t)jrow[q] * nb + b];
            // batches of 4 entries per lane: the loads of a batch are issued before any of them is used
            for (uint32_t e0 = 0; e0 < jm; e0 += 128) {
                uint32_t lo[4], c[4];
#pragma unroll
                for (uint32_t u = 0; u < 4; ++u) {
                    const uint32_t e = e0 + lane + 32 * u;
                    lo[u] = e < jm ? __ldg(idx + js + e) & (kSpLowBins - 1u) : 0u;
                    c[u] = e < jm ? __ldg(cnt + js + e) : 0u;
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

// stores d at (i, j) and (j, i) where those rows are in [row_begin, row_end)
__device__ __forceinline__ void xs_store(double* __restrict__ out, uint32_t n, uint32_t row_begin, uint32_t row_end,
                                         uint32_t i, uint32_t j, double d) {
    if (i >= row_begin && i < row_end) out[(size_t)(i - row_begin) * n + j] = d;
    if (i != j && j >= row_begin && j < row_end) out[(size_t)(j - row_begin) * n + i] = d;
}

__global__ void __launch_bounds__(kXsI * kXsJ)
k_xs_finish(const unsigned long long* __restrict__ X, const unsigned long long* __restrict__ Q,
            const uint64_t* __restrict__ T, const XsTile* __restrict__ tiles, uint32_t n, uint32_t row_begin,
            uint32_t row_end, double* __restrict__ out, uint2* __restrict__ flagged, uint32_t flag_cap,
            uint32_t* __restrict__ flag_count) {
    const XsTile tt = tiles[blockIdx.x];
    const uint32_t r = threadIdx.x / kXsJ, c = threadIdx.x % kXsJ;
    const uint32_t i = tt.ib * kXsI + r, j = tt.jc * kXsJ + c;
    if (i >= n || j > i) return;
    double d = 0.0;
    if (i != j) {
        const uint64_t ta = T[i], tb = T[j];
        if (ta == 0 || tb == 0) {
            d = __longlong_as_double(0x7FF8000000000000LL);  // NaN: frequencies 0 / 0 (the dense rows' NaN row)
        } else {
            const uint64_t tab = ta * tb;  // < 2^64
            bool exact = tab < (1ull << 63);
            if (exact) {
                const unsigned long long x = X[(size_t)blockIdx.x * kXsI * kXsJ + threadIdx.x];
                const unsigned __int128 p = (unsigned __int128)(tb * tb) * Q[i] + (unsigned __int128)(ta * ta) * Q[j];
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
    xs_store(out, n, row_begin, row_end, i, j, d);
}

// difference form over the rounded frequencies, one warp per pair: lane l merges the two rows' slices of buckets
// l, l + 32, ... (both ascending); the 32 partial sums are added by a fixed butterfly, so a pair gives the same bits
// whatever its position in the list or its orientation.  out_list != NULL: d of pair p goes to out_list[p]
// (test hook), otherwise to the matrix.
__global__ void __launch_bounds__(256)
k_xs_pairs(const uint32_t* __restrict__ idx, const uint32_t* __restrict__ cnt, const uint64_t* __restrict__ offsets,
           const uint32_t* __restrict__ bucket_ptr, const uint32_t* __restrict__ bucket_nnz, const uint64_t* __restrict__ T,
           uint32_t nb, uint32_t n, const uint2* __restrict__ pairs, const uint32_t* __restrict__ npairs,
           uint32_t row_begin, uint32_t row_end, double* __restrict__ out, double* __restrict__ out_list) {
    const uint32_t np = *npairs;
    const uint32_t lane = threadIdx.x & 31u;
    for (uint32_t p = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); p < np; p += gridDim.x * (blockDim.x / 32)) {
        const uint2 ij = pairs[p];
        const uint32_t a = ij.x, b = ij.y;
        const double ta = (double)T[a], tb = (double)T[b];  // (exact: < 2^32)
        double acc = 0.0;
        for (uint32_t bk = lane; bk < nb; bk += 32) {
            const uint64_t sa = offsets[a] + bucket_ptr[(size_t)a * (nb + 1) + bk];
            const uint64_t sb = offsets[b] + bucket_ptr[(size_t)b * (nb + 1) + bk];
            const uint32_t na = bucket_nnz[(size_t)a * nb + bk], nbb = bucket_nnz[(size_t)b * nb + bk];
            uint32_t x = 0, y = 0;
            while (x < na || y < nbb) {
                const uint32_t ka = x < na ? idx[sa + x] : 0xFFFFFFFFu, kb = y < nbb ? idx[sb + y] : 0xFFFFFFFFu;
                const bool ua = ka <= kb, ub = kb <= ka;
                const double fa = ua ? __ddiv_rn((double)cnt[sa + x], ta) : 0.0;
                const double fb = ub ? __ddiv_rn((double)cnt[sb + y], tb) : 0.0;
                x += ua;
                y += ub;
                const double df = __dsub_rn(fa, fb);
                acc = __dadd_rn(acc, __dmul_rn(df, df));
            }
        }
        for (int o = 16; o; o >>= 1) acc = __dadd_rn(acc, __shfl_xor_sync(0xffffffffu, acc, o));
        if (lane == 0) {
            double d = __dsqrt_rn(acc);
            if (a == b) d = 0.0;
            else if (T[a] == 0 || T[b] == 0) d = __longlong_as_double(0x7FF8000000000000LL);
            if (out_list) out_list[p] = d;
            else xs_store(out, n, row_begin, row_end, a, b, d);
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

static int xs_launch_pairs(dvs_ctx* ctx, const dvs_ksparse* sp, const uint2* d_pairs, const uint32_t* d_count,
                           uint32_t npairs, uint32_t row_begin, uint32_t row_end, double* out, double* out_list) {
    const unsigned grid = (unsigned)std::min<uint32_t>((npairs + 7) / 8, (uint32_t)ctx->sm_count * 16);
    k_xs_pairs<<<grid, 256, 0, ctx->stream>>>(sp->idx.p, sp->cnt.p, sp->offsets.p, sp->bucket_ptr.p, sp->bucket_nnz.p,
                                              sp->totals.p, sp->nb, sp->nrec, d_pairs, d_count, row_begin, row_end, out,
                                              out_list);
    DVS_LAUNCHED(ctx);
    return DVS_OK;
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
    // buckets per CTA: the J slices of one bucket range of all rows should stay in L2 (~32 MB of entries) while
    // every (tile, range) CTA that reads them runs, and there should be a few CTAs per SM
    std::vector<uint64_t> h_nnz(n);
    DVS_CUDA_TRY(cudaMemcpyAsync(h_nnz.data(), sp->nnz.p, (size_t)n * 8, cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    uint64_t entries = 0;
    for (uint64_t v : h_nnz) entries += v;
    const double per_bucket_bytes = 8.0 * (double)entries / (double)nb;  // all rows, one bucket
    uint32_t bper = nb;
    while (bper > 1 && per_bucket_bytes * bper > 32e6) bper >>= 1;
    while (bper > 1 && (uint64_t)ntiles * ((nb + bper - 1) / bper) < 4ull * ctx->sm_count) bper >>= 1;
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
    DVS_CUDA_TRY(cudaMemcpyAsync(d_tiles.p, tiles.data(), ntiles * sizeof(XsTile), cudaMemcpyHostToDevice, st));
    DVS_CUDA_TRY(cudaMemsetAsync(d_X.p, 0, tile_pairs * 8, st));
    DVS_CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, sizeof(uint32_t), st));
    DVS_CUDA_TRY(cudaFuncSetAttribute(k_xs_gram, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kXsSmemBytes));
    PhaseTimer pt(ctx, DVS_PHASE_EUCLID_SPARSE);
    k_xs_self<<<n, 256, 0, st>>>(sp->cnt.p, sp->offsets.p, sp->bucket_ptr.p, nb, d_Q.p);
    DVS_LAUNCHED(ctx);
    k_xs_gram<<<ntiles * nranges, kXsThreads, kXsSmemBytes, st>>>(sp->idx.p, sp->cnt.p, sp->offsets.p, sp->bucket_ptr.p,
                                                                  sp->bucket_nnz.p, n, nb, d_tiles.p, ntiles, bper, d_X.p);
    DVS_LAUNCHED(ctx);
    k_xs_finish<<<ntiles, kXsI * kXsJ, 0, st>>>(d_X.p, d_Q.p, sp->totals.p, d_tiles.p, n, row_begin, row_end, out,
                                                d_flag.p, flag_cap, d_cnt.p);
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
    if (h_cnt) DVS_TRY(xs_launch_pairs(ctx, sp, d_flag.p, d_cnt.p, h_cnt, row_begin, row_end, out, nullptr));
    pt.stop();
    if (!on_device)
        DVS_CUDA_TRY(cudaMemcpyAsync(dist, out, nrows * n * sizeof(double), cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    return DVS_OK;
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
    DevBuf<uint32_t> d_n;
    DevBuf<double> d_out;
    DVS_TRY(d_pairs.alloc(n));
    DVS_TRY(d_n.alloc(1));
    DVS_TRY(d_out.alloc(n));
    DVS_CUDA_TRY(cudaMemcpyAsync(d_pairs.p, pairs, (size_t)n * sizeof(uint2), cudaMemcpyHostToDevice, st));
    DVS_CUDA_TRY(cudaMemcpyAsync(d_n.p, &n, sizeof(uint32_t), cudaMemcpyHostToDevice, st));
    DVS_TRY(xs_launch_pairs(ctx, sp, d_pairs.p, d_n.p, n, 0, 0, nullptr, d_out.p));
    DVS_CUDA_TRY(cudaMemcpyAsync(out, d_out.p, (size_t)n * sizeof(double), cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    return DVS_OK;
}
