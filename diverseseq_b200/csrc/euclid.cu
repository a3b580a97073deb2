// Euclidean distance matrix over k-mer frequency rows.
//
// Replaces euclidean_distances / euclidean_distance (/root/reference/diverse_seq/distance.py:294-336;
// parallel variant cluster.py:647-680): d(i,j) = ||f_i - f_j||_2 = np.linalg.norm(f_i - f_j),
// symmetric, zero diagonal.  numpy's summation order is unspecified, so parity is 1e-9 relative.
//
// FP64 SIMT tile kernel: a CTA (256 threads) owns a 128x128 tile of pairs, every thread an 8x8
// register tile (64 FP64 accumulators); the frequency rows are staged through double-buffered
// shared memory in 16-column slabs, stored [column][row] so that the inner loop reads its operands
// with conflict-free 16-byte LDS (thread (ty,tx) owns rows {2ty,2ty+1}+32j and columns
// {2tx,2tx+1}+32j); global loads are whole 128-byte lines (8 lanes x 16 bytes per row segment).  The
// distance is accumulated in difference form sum((a-b)^2) — one DADD + one
// DFMA per pair-element, FP64-pipe bound — which has no cancellation (the Gram form
// ||a||^2+||b||^2-2ab loses all digits once d^2 << ||a||^2, see DESIGN.md §5.5).  Only tiles on or
// below the diagonal are computed when both row ranges are in the shard; results are mirrored.
#include <math.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "comm.cuh"
#include "common.cuh"

namespace dvs {

constexpr int kEuT = 128;  // tile edge (pairs)
constexpr int kEuK = 16;   // columns per slab
constexpr int kEuPad = 2;  // row padding of the [col][row] slabs (doubles)

// SHARDED: blockIdx.x enumerates this GPU's tiles t = tile_first + tile_step * blockIdx.x of the lower
// triangle (t = ti (ti + 1) / 2 + tj, tj <= ti) of the whole n x n matrix
template <bool SHARDED>
__global__ void __launch_bounds__(256, 1)
k_euclid_tiles(const double* __restrict__ F, uint64_t dim, uint32_t n, uint32_t row_begin, uint32_t row_end,
               const EuOuts outs /* each [(row_end-row_begin)][n] */, uint32_t tile_first, uint32_t tile_step) {
    extern __shared__ double eu_smem[];
    double(*sa)[kEuK][kEuT + kEuPad] = reinterpret_cast<double(*)[kEuK][kEuT + kEuPad]>(eu_smem);
    double(*sb)[kEuK][kEuT + kEuPad] =
        reinterpret_cast<double(*)[kEuK][kEuT + kEuPad]>(eu_smem + 2 * kEuK * (kEuT + kEuPad));
    uint32_t ti = blockIdx.y, tj = blockIdx.x;
    if (SHARDED) {
        const uint64_t t = (uint64_t)tile_first + (uint64_t)tile_step * blockIdx.x;
        ti = (uint32_t)((sqrt(8.0 * (double)t + 1.0) - 1.0) * 0.5);
        while ((uint64_t)ti * (ti + 1) / 2 > t) --ti;
        while ((uint64_t)(ti + 1) * (ti + 2) / 2 <= t) ++ti;
        tj = (uint32_t)(t - (uint64_t)ti * (ti + 1) / 2);
    }
    const uint32_t i0 = row_begin + ti * kEuT, j0 = tj * kEuT;
    if (i0 >= row_end) return;
    // a tile strictly above the diagonal is skipped when its transpose, produced by this launch, mirrors every entry
    // of it: tiles of rows and columns only coincide when row_begin is tile aligned, and the transpose stores rows
    // < row_end only, so all of the tile's columns j0 .. j0+127 must be rows of the call (or lie past n)
    const bool mirror_in_range =
        (row_begin % kEuT == 0) && (j0 >= row_begin) && (j0 + kEuT <= row_end || row_end == n);
    if (mirror_in_range && j0 > i0) return;
    const int t = threadIdx.x, tx = t & 15, ty = t >> 4;
    // loader mapping: a slab row segment is 16 doubles = one 128-byte line; chunk = 16 bytes (2 columns).
    // Thread t moves chunks t, t+256, t+512, t+768 of each operand: 8 consecutive lanes read one whole
    // line of one row (4 lines per warp-wide LDG.128).  (The first version gave each thread 8 consecutive
    // doubles of its own row: 32 rows per warp instruction, 16x the L1 wavefronts, and the kernel sat
    // on long-scoreboard stalls at 60 % FP64-pipe utilisation.)
    const bool vec_ok = (dim % 2 == 0);  // 16-byte alignment of every row
    const int lc2 = t & 7;               // chunk within the row segment -> columns 2*lc2, 2*lc2+1
    const double* parow[4];
    const double* pbrow[4];
    bool varow[4], vbrow[4];
#pragma unroll
    for (int q = 0; q < 4; ++q) {
        const int lr = (t >> 3) + 32 * q;
        const uint32_t ra = i0 + lr, rb = j0 + lr;
        varow[q] = ra < row_end;
        vbrow[q] = rb < n;
        parow[q] = F + (size_t)(varow[q] ? ra : 0) * dim;
        pbrow[q] = F + (size_t)(vbrow[q] ? rb : 0) * dim;
    }

    double acc[8][8];
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) acc[a][b] = 0.0;

    double2 ga[4], gb[4];
    auto gload = [&](uint64_t c0) {
        const uint64_t col = c0 + 2 * lc2;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            if (vec_ok && col + 1 < dim) {
                ga[q] = varow[q] ? *reinterpret_cast<const double2*>(parow[q] + col) : make_double2(0.0, 0.0);
                gb[q] = vbrow[q] ? *reinterpret_cast<const double2*>(pbrow[q] + col) : make_double2(0.0, 0.0);
            } else {
                ga[q].x = (varow[q] && col < dim) ? parow[q][col] : 0.0;
                ga[q].y = (varow[q] && col + 1 < dim) ? parow[q][col + 1] : 0.0;
                gb[q].x = (vbrow[q] && col < dim) ? pbrow[q][col] : 0.0;
                gb[q].y = (vbrow[q] && col + 1 < dim) ? pbrow[q][col + 1] : 0.0;
            }
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const int lr = (t >> 3) + 32 * q;
            sa[buf][2 * lc2][lr] = ga[q].x;
            sa[buf][2 * lc2 + 1][lr] = ga[q].y;
            sb[buf][2 * lc2][lr] = gb[q].x;
            sb[buf][2 * lc2 + 1][lr] = gb[q].y;
        }
    };
    const uint64_t nslab = (dim + kEuK - 1) / kEuK;
    gload(0);
    sstore(0);
    __syncthreads();
    for (uint64_t sl = 0; sl < nslab; ++sl) {
        const int buf = (int)(sl & 1);
        if (sl + 1 < nslab) gload((sl + 1) * kEuK);  // global loads in flight during the FP64 work
#pragma unroll
        for (int c = 0; c < kEuK; ++c) {
            double av[8], bv[8];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const double2 x = *reinterpret_cast<const double2*>(&sa[buf][c][2 * ty + 32 * j]);
                const double2 y = *reinterpret_cast<const double2*>(&sb[buf][c][2 * tx + 32 * j]);
                av[2 * j] = x.x; av[2 * j + 1] = x.y;
                bv[2 * j] = y.x; bv[2 * j + 1] = y.y;
            }
#pragma unroll
            for (int a = 0; a < 8; ++a)
#pragma unroll
                for (int b = 0; b < 8; ++b) {
                    const double d = av[a] - bv[b];
                    acc[a][b] = fma(d, d, acc[a][b]);
                }
        }
        if (sl + 1 < nslab) sstore(buf ^ 1);
        __syncthreads();
    }
#pragma unroll
    for (int a = 0; a < 8; ++a)
#pragma unroll
        for (int b = 0; b < 8; ++b) {
            const uint32_t i = i0 + 2 * ty + 32 * (a >> 1) + (a & 1);
            const uint32_t j = j0 + 2 * tx + 32 * (b >> 1) + (b & 1);
            if (i >= row_end || j >= n) continue;
            const double d = (i == j) ? 0.0 : sqrt(acc[a][b]);
            const bool mirror = mirror_in_range && j >= row_begin && j < row_end && i < n;
            for (int r = 0; r < (SHARDED ? outs.count : 1); ++r) {
                double* out = outs.p[r];
                out[(size_t)(i - row_begin) * n + j] = d;
                if (mirror) out[(size_t)(j - row_begin) * n + i] = d;
            }
        }
}

constexpr size_t kEuSmemBytes = 4ull * kEuK * (kEuT + kEuPad) * sizeof(double);

// ---- Gram form on the FP64 tensor cores --------------------------------------------------------------------
// d^2 = |a|^2 + |b|^2 - 2 a.b needs ONE multiply-add per pair-element where the difference form needs two FP64
// instructions, and DMMA.8x8x4 runs at the full FP64 rate on B200 (37.2 TFLOP/s measured, DFMA 33.8:
// profiles/r2_fp64_bench.txt) while reading its operands 4x less often from shared memory than an 8x8 SIMT
// register tile.  The catch is cancellation: rows of k-mer frequencies are all close to each other
// (d^2 ~ 3 % of |a|^2 for unrelated genomes, 1e-4 and below for relatives, 0 for copies), so the rounding error
// of the long dot product has to stay far below d^2:
//   * the K dimension is cut into SLICES of kEgSlice columns; a slice's 128x128 partial tile is accumulated by
//     DMMA (error <= kEgSlice u a.b, all terms positive) and written to a workspace; the partials are added in
//     a fixed order by the finishing kernel (error <= #slices u a.b).  With 2 a.b <= |a|^2 + |b|^2 the computed
//     d^2 is within  (kEgSlice + #slices + log2 D + 8) u (|a|^2 + |b|^2)  of the true one;
//   * a pair is therefore taken from the Gram form only when d^2 >= kEgTau (|a|^2 + |b|^2), which bounds the
//     relative error of d by 0.5e-9 (half the stated 1e-9); every other pair - near-duplicates, exact copies - is
//     appended to a list and recomputed in difference form (sum (a-b)^2, no cancellation, exact 0 for copies);
//   * if more than an eighth of the pairs end up in the list the whole call falls back to the difference-form
//     tile kernel above (tiny or degenerate inputs).
// A CTA is 16 warps in a 4 x 4 grid, each warp owns a 32 x 32 piece of the tile = 4 x 4 DMMA accumulators
// (64 registers); operands are staged by cp.async in 16-column slabs, 3 stages, rows padded to 20 doubles so
// that the per-lane fragment loads (8 rows x 4 consecutive doubles per half warp) are bank-conflict free.
// Every pair (i > j) is computed by the tile (i / 128, j / 128) of the lower triangle whatever the call's row
// range or GPU, so partial-range calls, single-GPU and sharded calls return identical bits.
constexpr int kEgT = 128, kEgSlab = 16, kEgStride = 20, kEgStages = 3, kEgThreads = 512;
constexpr uint32_t kEgSlice = 2048;
// relative error of a Gram-form d^2 <= (kEgSlice + #slices + log2 D + 8) u / kEgTau, of d half that: 2.3e-10 at
// 32 slices (k=8), 2.9e-10 at 512 (D = 2^20), below 0.5e-9 up to about 2,400 slices (D ~ 4.9 M)
constexpr double kEgTau = 5e-4;
constexpr size_t kEgSmemBytes = (size_t)kEgStages * 2 * kEgT * kEgStride * sizeof(double);

struct EgTile {
    uint32_t ti, tj;  // tile coordinates, tj <= ti
};

__global__ void k_eg_norms(const double* __restrict__ F, uint64_t dim, double* __restrict__ nrm) {
    __shared__ double s_w[8];
    const double* f = F + (size_t)blockIdx.x * dim;
    double acc = 0.0;
    for (uint64_t i = threadIdx.x; i < dim; i += blockDim.x) acc = fma(f[i], f[i], acc);
    for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (unsigned w = 0; w < blockDim.x / 32; ++w) t += s_w[w];
        nrm[blockIdx.x] = t;
    }
}

__device__ __forceinline__ void eg_cp_async16(void* smem_dst, const void* gsrc, int src_bytes) {
    const uint32_t d = (uint32_t)__cvta_generic_to_shared(smem_dst);
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(gsrc), "r"(src_bytes) : "memory");
}

// partial Gram tile of one (tile, slice): P[slice][tile][128][128] = A[i0.., c0..c1) . B[j0.., c0..c1)^T
__global__ void __launch_bounds__(kEgThreads, 1)
k_eg_gram(const double* __restrict__ F, uint64_t dim, uint32_t n, const EgTile* __restrict__ tiles, uint32_t ntiles,
          uint32_t nslices, double* __restrict__ P) {
    extern __shared__ __align__(16) double eg_smem[];
    const uint32_t tile = blockIdx.x % ntiles, slice = blockIdx.x / ntiles;
    const EgTile tt = tiles[tile];
    const uint32_t i0 = tt.ti * kEgT, j0 = tt.tj * kEgT;
    const uint64_t c_begin = (uint64_t)slice * kEgSlice, c_end = min(dim, c_begin + kEgSlice);
    const uint32_t nslab = (uint32_t)((c_end - c_begin + kEgSlab - 1) / kEgSlab);
    const int t = threadIdx.x, lane = t & 31, warp = t >> 5, wi = warp >> 2, wj = warp & 3, g = lane >> 2, tq = lane & 3;
    auto stage_a = [&](int st) { return eg_smem + (size_t)st * 2 * kEgT * kEgStride; };
    auto stage_b = [&](int st) { return eg_smem + (size_t)st * 2 * kEgT * kEgStride + kEgT * kEgStride; };
    // loader: 128 rows x 8 chunks (16 bytes = 2 columns) per operand and slab; thread t moves chunks t and t + 512
    auto load_slab = [&](uint32_t sl, int st) {
        const uint64_t c0 = c_begin + (uint64_t)sl * kEgSlab;
#pragma unroll
        for (int q = 0; q < 2; ++q) {
            const int ch = t + q * kEgThreads, row = ch >> 3, cc = (ch & 7) * 2;
            const uint64_t col = c0 + cc;
            const int bytes = col + 1 < c_end ? 16 : (col < c_end ? 8 : 0);
            const uint32_t ra = i0 + row, rb = j0 + row;
            const double* ga = F + (size_t)min(ra, n - 1) * dim + min(col, dim - 2);
            const double* gb = F + (size_t)min(rb, n - 1) * dim + min(col, dim - 2);
            eg_cp_async16(stage_a(st) + row * kEgStride + cc, ga, ra < n ? bytes : 0);
            eg_cp_async16(stage_b(st) + row * kEgStride + cc, gb, rb < n ? bytes : 0);
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    double c[4][4][2];
#pragma unroll
    for (int m = 0; m < 4; ++m)
#pragma unroll
        for (int q = 0; q < 4; ++q) c[m][q][0] = c[m][q][1] = 0.0;
    for (int st = 0; st < kEgStages - 1; ++st) {
        if ((uint32_t)st < nslab) load_slab(st, st);
        else asm volatile("cp.async.commit_group;" ::: "memory");
    }
    for (uint32_t sl = 0; sl < nslab; ++sl) {
        asm volatile("cp.async.wait_group %0;" ::"n"(kEgStages - 2) : "memory");
        __syncthreads();  // slab sl has landed for everybody; the stage refilled below was consumed in iteration sl - 1
        if (sl + kEgStages - 1 < nslab) load_slab(sl + kEgStages - 1, (sl + kEgStages - 1) % kEgStages);
        else asm volatile("cp.async.commit_group;" ::: "memory");
        const double* As = stage_a(sl % kEgStages) + (wi * 32 + g) * kEgStride + tq;
        const double* Bs = stage_b(sl % kEgStages) + (wj * 32 + g) * kEgStride + tq;
#pragma unroll
        for (int ks = 0; ks < kEgSlab / 4; ++ks) {
            double a[4], b[4];
#pragma unroll
            for (int m = 0; m < 4; ++m) a[m] = As[m * 8 * kEgStride + ks * 4];
#pragma unroll
            for (int q = 0; q < 4; ++q) b[q] = Bs[q * 8 * kEgStride + ks * 4];
#pragma unroll
            for (int m = 0; m < 4; ++m)
#pragma unroll
                for (int q = 0; q < 4; ++q)
                    asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
                                 : "+d"(c[m][q][0]), "+d"(c[m][q][1])
                                 : "d"(a[m]), "d"(b[q]));
        }
    }
    double* out = P + ((size_t)slice * ntiles + tile) * kEgT * kEgT;
#pragma unroll
    for (int m = 0; m < 4; ++m)
#pragma unroll
        for (int q = 0; q < 4; ++q)
            *reinterpret_cast<double2*>(out + (size_t)(wi * 32 + m * 8 + g) * kEgT + wj * 32 + q * 8 + 2 * tq) =
                make_double2(c[m][q][0], c[m][q][1]);
}

// partial tiles -> distances; pairs whose d^2 is too small for the Gram form go to the list.
// A tile is finished in 32 x 32 sub-blocks that pass through shared memory, so that BOTH the (i, j) and the mirrored
// (j, i) stores are 256-byte row segments: with up to 8 destination matrices behind NVLink, element-wise mirrored
// stores (8 bytes each, stride n) made the 8-GPU run slower than one GPU (533 ms against 255 ms).
__global__ void __launch_bounds__(256)
k_eg_finish(const double* __restrict__ P, const double* __restrict__ nrm, const EgTile* __restrict__ tiles, uint32_t ntiles,
            uint32_t nslices, uint32_t n, uint32_t row_begin, uint32_t row_end, const EuOuts outs,
            uint2* __restrict__ flagged, uint32_t flag_cap, uint32_t* __restrict__ flag_count) {
    __shared__ double sd[32][33];  // < 0: nothing to store (outside the matrix / the triangle, or listed)
    const uint32_t tile = blockIdx.x;
    const EgTile tt = tiles[tile];
    const uint32_t i0 = tt.ti * kEgT, j0 = tt.tj * kEgT;
    const uint32_t lane = threadIdx.x & 31u, warp = threadIdx.x >> 5;
    constexpr uint32_t kSub = kEgT / 32;
    for (uint32_t sb = 0; sb < kSub * kSub; ++sb) {
        const uint32_t si = (sb / kSub) * 32, sj = (sb % kSub) * 32;
        if (i0 + si >= n || j0 + sj >= n || j0 + sj > i0 + si + 31) continue;  // (block-uniform)
        for (uint32_t q = 0; q < 4; ++q) {
            const uint32_t r = warp * 4 + q;
            const uint32_t i = i0 + si + r, j = j0 + sj + lane;
            double d = -1.0;
            if (i < n && j < n && j <= i) {
                d = 0.0;
                if (i != j) {
                    const uint32_t e = (si + r) * kEgT + sj + lane;
                    double gsum = 0.0;
                    for (uint32_t sl = 0; sl < nslices; ++sl) gsum += P[((size_t)sl * ntiles + tile) * kEgT * kEgT + e];
                    const double na = nrm[i], nb = nrm[j], d2 = (na + nb) - 2.0 * gsum;
                    if (d2 >= kEgTau * (na + nb)) {
                        d = sqrt(d2);
                    } else {  // written by k_eg_pairs (or by the difference-form kernel if the list overflows)
                        const uint32_t at = atomicAdd(flag_count, 1u);
                        if (at < flag_cap) flagged[at] = make_uint2(i, j);
                        d = -1.0;
                    }
                }
            }
            sd[r][lane] = d;
            if (d >= 0.0 && i >= row_begin && i < row_end)
                for (int o = 0; o < outs.count; ++o) outs.p[o][(size_t)(i - row_begin) * n + j] = d;
        }
        __syncthreads();
        for (uint32_t q = 0; q < 4; ++q) {  // the mirror image: row j of the output, columns i
            const uint32_t c = warp * 4 + q;
            const uint32_t i = i0 + si + lane, j = j0 + sj + c;
            const double d = sd[lane][c];
            if (d >= 0.0 && j >= row_begin && j < row_end)
                for (int o = 0; o < outs.count; ++o) outs.p[o][(size_t)(j - row_begin) * n + i] = d;
        }
        __syncthreads();
    }
}

// difference form for the listed pairs: one warp per pair
__global__ void __launch_bounds__(256)
k_eg_pairs(const double* __restrict__ F, uint64_t dim, uint32_t n, const uint2* __restrict__ flagged,
           const uint32_t* __restrict__ flag_count, uint32_t row_begin, uint32_t row_end, const EuOuts outs) {
    const uint32_t np = *flag_count;
    const uint32_t lane = threadIdx.x & 31;
    for (uint32_t p = blockIdx.x * (blockDim.x / 32) + (threadIdx.x >> 5); p < np; p += gridDim.x * (blockDim.x / 32)) {
        const uint2 ij = flagged[p];
        const double* a = F + (size_t)ij.x * dim;
        const double* b = F + (size_t)ij.y * dim;
        double acc0 = 0.0, acc1 = 0.0;
        if (dim % 2 == 0) {
            for (uint64_t c0 = 2 * lane; c0 < dim; c0 += 64) {
                const double2 x = *reinterpret_cast<const double2*>(a + c0), y = *reinterpret_cast<const double2*>(b + c0);
                const double d0 = x.x - y.x, d1 = x.y - y.y;
                acc0 = fma(d0, d0, acc0);
                acc1 = fma(d1, d1, acc1);
            }
        } else {
            for (uint64_t c0 = lane; c0 < dim; c0 += 32) {
                const double d0 = a[c0] - b[c0];
                acc0 = fma(d0, d0, acc0);
            }
        }
        double acc = acc0 + acc1;
        for (int o = 16; o; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
        if (lane == 0) {
            const double d = sqrt(acc);
            const uint32_t i = ij.x, j = ij.y;
            for (int r = 0; r < outs.count; ++r) {
                if (i >= row_begin && i < row_end) outs.p[r][(size_t)(i - row_begin) * n + j] = d;
                if (j >= row_begin && j < row_end) outs.p[r][(size_t)(j - row_begin) * n + i] = d;
            }
        }
    }
}

// Gram path over a list of lower-triangle tiles; returns 1 in *fell_back when the caller has to run the
// difference-form tile kernel instead (odd row length, most pairs near-duplicate)
static int euclid_gram(dvs_ctx* ctx, const dvs_kfreqs* f, const std::vector<EgTile>& tiles, uint32_t row_begin,
                       uint32_t row_end, const EuOuts& outs, bool* fell_back) {
    *fell_back = true;
    const char* env = getenv("DVS_EUCLID_GRAM");
    const uint64_t dim = f->dim;
    const uint32_t n = f->nrec;
    if ((env && env[0] == '0') || dim % 2 != 0 || dim < 2 || tiles.empty()) return DVS_OK;
    cudaStream_t st = ctx->stream;
    const uint32_t ntiles = (uint32_t)tiles.size();
    const uint32_t nslices = (uint32_t)((dim + kEgSlice - 1) / kEgSlice);
    if ((uint64_t)ntiles * nslices > 0x7FFFFFFFull) return DVS_OK;
    DevBuf<EgTile> d_tiles;
    DevBuf<double> d_nrm, d_P;
    DevBuf<uint2> d_flag;
    DevBuf<uint32_t> d_cnt;
    const uint64_t npairs = (uint64_t)ntiles * kEgT * kEgT;
    const uint32_t flag_cap = (uint32_t)std::min<uint64_t>(std::max<uint64_t>(npairs / 8, 1024), 1u << 26);
    DVS_TRY(d_tiles.alloc(ntiles));
    DVS_TRY(d_nrm.alloc(n));
    if (d_P.alloc((size_t)ntiles * nslices * kEgT * kEgT) != DVS_OK) return DVS_OK;  // no room for the workspace
    DVS_TRY(d_flag.alloc(flag_cap));
    DVS_TRY(d_cnt.alloc(1));
    DVS_CUDA_TRY(cudaMemcpyAsync(d_tiles.p, tiles.data(), ntiles * sizeof(EgTile), cudaMemcpyHostToDevice, st));
    DVS_CUDA_TRY(cudaMemsetAsync(d_cnt.p, 0, sizeof(uint32_t), st));
    DVS_CUDA_TRY(cudaFuncSetAttribute(k_eg_gram, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEgSmemBytes));
    k_eg_norms<<<n, 256, 0, st>>>(f->freqs.p, dim, d_nrm.p);
    DVS_LAUNCHED(ctx);
    k_eg_gram<<<ntiles * nslices, kEgThreads, kEgSmemBytes, st>>>(f->freqs.p, dim, n, d_tiles.p, ntiles, nslices, d_P.p);
    DVS_LAUNCHED(ctx);
    k_eg_finish<<<ntiles, 256, 0, st>>>(d_P.p, d_nrm.p, d_tiles.p, ntiles, nslices, n, row_begin, row_end, outs, d_flag.p,
                                        flag_cap, d_cnt.p);
    DVS_LAUNCHED(ctx);
    uint32_t h_cnt = 0;
    DVS_CUDA_TRY(cudaMemcpyAsync(&h_cnt, d_cnt.p, sizeof(uint32_t), cudaMemcpyDeviceToHost, st));
    DVS_CUDA_TRY(cudaStreamSynchronize(st));
    if (h_cnt > flag_cap) return DVS_OK;  // mostly near-duplicates: the difference-form kernel does everything
    if (h_cnt) {
        k_eg_pairs<<<(unsigned)std::min<uint32_t>((h_cnt + 7) / 8, (uint32_t)ctx->sm_count * 16), 256, 0, st>>>(
            f->freqs.p, dim, n, d_flag.p, d_cnt.p, row_begin, row_end, outs);
        DVS_LAUNCHED(ctx);
    }
    ctx->last_euclid_fallback_pairs = h_cnt;
    *fell_back = false;
    return DVS_OK;
}

// lower-triangle tiles that hold a pair with a row in [row_begin, row_end)
static std::vector<EgTile> eg_tiles_for_rows(uint32_t n, uint32_t row_begin, uint32_t row_end) {
    std::vector<EgTile> tiles;
    if (row_end <= row_begin) return tiles;
    const uint32_t nt = (n + kEgT - 1) / kEgT, t0 = row_begin / kEgT, t1 = (row_end - 1) / kEgT;
    for (uint32_t ti = 0; ti < nt; ++ti)
        for (uint32_t tj = 0; tj <= ti; ++tj)
            if ((ti >= t0 && ti <= t1) || (tj >= t0 && tj <= t1)) tiles.push_back({ti, tj});
    return tiles;
}

}  // namespace dvs

using namespace dvs;

extern "C" uint32_t dvs_euclid_last_fallback_pairs(dvs_ctx* ctx) { return ctx->last_euclid_fallback_pairs; }

extern "C" int dvs_euclid_distances(dvs_ctx* ctx, const dvs_kfreqs* f, uint32_t row_begin, uint32_t row_end,
                                    double* dist) {
    if (!ctx || !f || !dist || row_begin > row_end || row_end > f->nrec) {
        set_error("dvs_euclid_distances: bad argument");
        return DVS_ERR_ARG;
    }
    const size_t nrows = row_end - row_begin, n = f->nrec;
    if (nrows == 0 || n == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    DevBuf<double> d_out;
    DVS_TRY(d_out.alloc(nrows * n));
    EuOuts outs;
    memset(&outs, 0, sizeof outs);
    outs.p[0] = d_out.p;
    outs.count = 1;
    PhaseTimer pt(ctx, DVS_PHASE_EUCLID);
    bool fell_back = true;
    ctx->last_euclid_fallback_pairs = 0;
    DVS_TRY(euclid_gram(ctx, f, eg_tiles_for_rows((uint32_t)n, row_begin, row_end), row_begin, row_end, outs, &fell_back));
    if (fell_back) {
        dim3 grid((unsigned)((n + kEuT - 1) / kEuT), (unsigned)((nrows + kEuT - 1) / kEuT));
        DVS_CUDA_TRY(cudaFuncSetAttribute(k_euclid_tiles<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEuSmemBytes));
        k_euclid_tiles<false><<<grid, 256, kEuSmemBytes, ctx->stream>>>(f->freqs.p, f->dim, (uint32_t)n, row_begin, row_end, outs, 0, 0);
        DVS_LAUNCHED(ctx);
    }
    pt.stop();
    DVS_CUDA_TRY(cudaMemcpyAsync(dist, d_out.p, nrows * n * sizeof(double), cudaMemcpyDefault, ctx->stream));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DVS_OK;
}

// all ranks hold the same rows (dvs_count_kmers_sharded / dvs_kfreqs_allgather); every rank gets the whole matrix
extern "C" int dvs_euclid_distances_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_kfreqs* f_all, double* dist) {
    if (!ctx || !c || !c->connected || !f_all || !dist) {
        set_error("dvs_euclid_distances_sharded: bad argument / communicator not connected");
        return DVS_ERR_ARG;
    }
    const size_t n = f_all->nrec;
    if (n == 0) return DVS_OK;
    DVS_CUDA_TRY(dvs::enter(ctx));
    cudaStream_t st = ctx->stream;
    uint64_t hoff = 0;
    DVS_TRY(comm_heap_alloc(c, n * n * sizeof(double), &hoff));
    int rc = comm_barrier(ctx, c);  // nobody still uses this block of its window
    cudaError_t e = cudaSuccess;
    if (rc == DVS_OK) {
        const uint64_t nt = (n + kEuT - 1) / kEuT, tiles = nt * (nt + 1) / 2;
        const uint64_t mine = tiles > (uint64_t)c->rank ? (tiles - c->rank + c->world - 1) / c->world : 0;
        EuOuts outs;
        memset(&outs, 0, sizeof outs);
        for (int r = 0; r < c->world; ++r) outs.p[r] = reinterpret_cast<double*>(c->peer[(c->rank + r) % c->world] + hoff);
        outs.count = c->world;
        PhaseTimer pt(ctx, DVS_PHASE_EUCLID);
        // Gram form on this GPU's share of the lower-triangle tiles (t = rank, rank + world, ...).  Each rank decides
        // on its own whether to fall back to the difference form: row length and workspace are the same everywhere,
        // but a rank whose list overflows runs the tile kernel over exactly its own tiles while the other ranks keep
        // their Gram results, so the ranks need not agree
        bool fell_back = true;
        {
            std::vector<EgTile> my_tiles;
            uint64_t t = 0;
            for (uint32_t ti = 0; ti < nt; ++ti)
                for (uint32_t tj = 0; tj <= ti; ++tj, ++t)
                    if (t % (uint64_t)c->world == (uint64_t)c->rank) my_tiles.push_back({ti, tj});
            ctx->last_euclid_fallback_pairs = 0;
            rc = euclid_gram(ctx, f_all, my_tiles, 0, (uint32_t)n, outs, &fell_back);
            if (my_tiles.empty()) fell_back = false;
        }
        if (rc == DVS_OK && fell_back)
            e = cudaFuncSetAttribute(k_euclid_tiles<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kEuSmemBytes);
        if (rc == DVS_OK && fell_back && e == cudaSuccess && mine) {
            k_euclid_tiles<true><<<(unsigned)mine, 256, kEuSmemBytes, st>>>(f_all->freqs.p, f_all->dim, (uint32_t)n, 0,
                                                                           (uint32_t)n, outs, (uint32_t)c->rank,
                                                                           (uint32_t)c->world);
            ctx->launches++;
            e = cudaGetLastError();
        }
        pt.stop();
        if (e == cudaSuccess) rc = comm_barrier(ctx, c);  // every GPU's tiles have landed in this window
        if (e == cudaSuccess && rc == DVS_OK)
            e = cudaMemcpyAsync(dist, c->window + hoff, n * n * sizeof(double), cudaMemcpyDefault, st);
        if (e == cudaSuccess && rc == DVS_OK) rc = comm_check_error(ctx, c, "dvs_euclid_distances_sharded");
    }
    comm_heap_free(c, hoff);
    if (e != cudaSuccess) {
        set_error("dvs_euclid_distances_sharded: %s", cudaGetErrorString(e));
        return DVS_ERR_CUDA;
    }
    return rc;
}
