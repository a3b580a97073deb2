// Exact, reference-order Shannon entropy on the device.
//
// The reference's `entropy` (/root/reference/src/record.rs:86-106) is a sequential f64 loop
//     e += -x * log2(x);  t += x;      (skipping x == 0)
// whose result depends on the order of the additions and on libm's log2.  Selection decisions
// (`jsd > total_jsd + EPS`, strict-< argmin; src/records.rs:86-92,246) compare such sums, so to
// make the same decisions the device evaluates the SAME sum:
//   * the per-element terms -x*log2(x) are independent and are produced in parallel by the
//     "producer" warps with dvs_log2 (bit-identical to glibc, log2_glibc.h) and explicit
//     __dmul_rn (no FMA contraction, as in Rust);
//   * the two running sums are inherently serial; lane 0 and lane 1 of warp 0 carry the e-chain
//     and the t-chain side by side in one SIMT instruction stream, reading the terms from a
//     double-buffered shared-memory tile while the producers fill the next tile.
// Latency is therefore ~dim x (dependent DADD latency); throughput comes from running one such
// block per row, many rows per SM.
//
// Skipped elements contribute +0.0 to both chains, which is bit-identical to skipping because
// neither chain can be -0.0 (they start at +0.0 and (+0.0)+(-0.0) = +0.0 in round-to-nearest).
#pragma once
#include "common.cuh"
#include "log2_glibc.h"

namespace dvs {

constexpr int kEntTile = 512;          // elements per shared-memory tile
constexpr int kEntThreads = 128;       // 1 chain warp + 3 producer warps
constexpr size_t kEntSmemBytes = 2 /*buffers*/ * 2 /*term,val*/ * kEntTile * sizeof(double);

struct EntropyResult {
    double e;  // entropy
    double t;  // total frequency (for the reference's sum-to-one check)
};

// reference tolerance check: |t - 1| > len * EPS  -> panic  (src/record.rs:101-104)
__device__ __forceinline__ bool entropy_total_bad(double t, uint64_t len) {
    double tol = __dmul_rn((double)len, kEps);
    return fabs(__dsub_rn(t, 1.0)) > tol;
}

// All kEntThreads threads of the block must call this.  `elem(i)` returns element i of the
// frequency vector (any thread may be asked for any i).  `smem` must hold kEntSmemBytes.
// The result is returned to every thread.
// x / b through a correctly rounded reciprocal and two fused-remainder steps (Markstein): the second
// step starts from a faithful quotient and therefore rounds correctly, i.e. the result equals IEEE
// division (__ddiv_rn) bit for bit — checked on the host for 8.2e7 random numerators x every integer
// divisor <= 4100 and for 1.5e8 count/total pairs incl. all-ones significands, and on the device in
// tests/test_gpu_parity.py — without __ddiv_rn's ~20 instructions and slow-path branch.  Requires a
// normal quotient well above the subnormal range (callers: k-mer frequencies, or guarded by fast_term_ok).
struct FastDiv {
    double b, y;  // divisor and RN(1/b)
};
__device__ __forceinline__ FastDiv make_fast_div(double b) { return FastDiv{b, __drcp_rn(b)}; }
__device__ __forceinline__ double div_exact(double a, const FastDiv& d) {
    double q = __dmul_rn(a, d.y);
    double r = __fma_rn(-q, d.b, a);
    q = __fma_rn(r, d.y, q);
    r = __fma_rn(-q, d.b, a);
    return __fma_rn(r, d.y, q);
}

// Staging hook of a row source (select.cu): called by every thread of the block with the first element of each
// group of kEntStageTiles tiles before the producers read it.  Rows held in memory need none.
constexpr int kEntStageTiles = 8;
struct NoStage {
    __device__ __forceinline__ void operator()(uint64_t) const {}
};

template <class Elem, class Stage = NoStage>
__device__ EntropyResult block_entropy_exact(uint64_t dim, Elem elem, double* smem, Stage stage = Stage()) {
    double* term[2] = {smem, smem + 2 * kEntTile};
    double* val[2] = {smem + kEntTile, smem + 3 * kEntTile};
    __shared__ double s_res[2];
    // log2 goes through the branch-free table path of the restatement (table in shared memory, one
    // lookup per lane) and only falls back to the full dvs_log2 for the inputs that path does not cover
    // (|x - 1| small, subnormal, <= 0, inf, nan): same bits, about a third of the instructions
    __shared__ double2 s_ltab[64];
    dvs_log2_stage_table(s_ltab);
    __syncthreads();
    const int tid = threadIdx.x;
    const int warp = tid >> 5, lane = tid & 31;
    const uint64_t ntiles = (dim + kEntTile - 1) / kEntTile;

    auto produce = [&](uint64_t tile, int first, int step) {
        const uint64_t base = tile * kEntTile;
        const int n = (int)min((uint64_t)kEntTile, dim - base);
        double* tb = term[tile & 1];
        double* vb = val[tile & 1];
        for (int j = first; j < n; j += step) {
            double x = elem(base + j);
            double tm = 0.0, v = 0.0;
            if (!(x == 0.0)) {  // NaN is not skipped, like `*freq == 0.0` in Rust
                int special = 0;
                double l = dvs_log2_main(x, s_ltab, special);
                if (special) l = dvs_log2(x);
                tm = __dmul_rn(-x, l);
                v = x;
            }
            tb[j] = tm;
            vb[j] = v;
        }
    };

    double acc = 0.0;  // lane 0: e-chain, lane 1: t-chain
    if (ntiles > 0) {
        stage(0);
        produce(0, tid, kEntThreads);  // everybody helps with the first tile
    }
    __syncthreads();
    for (uint64_t tile = 0; tile < ntiles; ++tile) {
        if ((tile + 1) % kEntStageTiles == 0 && tile + 1 < ntiles) stage((tile + 1) * kEntTile);
        if (warp == 0) {
            if (lane < 2) {
                const uint64_t base = tile * kEntTile;
                const int n = (int)min((uint64_t)kEntTile, dim - base);
                const double* src = lane == 0 ? term[tile & 1] : val[tile & 1];
                int j = 0;
                // 16-byte loads: with two active lanes every LDS is a whole LSU wavefront, and the chain's
                // loads were the largest share of an LSU pipe that ncu showed 84 % busy in k_freq_entropy
                for (; j + 8 <= n; j += 8) {
                    const double2 p0 = *reinterpret_cast<const double2*>(src + j);
                    const double2 p1 = *reinterpret_cast<const double2*>(src + j + 2);
                    const double2 p2 = *reinterpret_cast<const double2*>(src + j + 4);
                    const double2 p3 = *reinterpret_cast<const double2*>(src + j + 6);
                    acc = __dadd_rn(acc, p0.x);
                    acc = __dadd_rn(acc, p0.y);
                    acc = __dadd_rn(acc, p1.x);
                    acc = __dadd_rn(acc, p1.y);
                    acc = __dadd_rn(acc, p2.x);
                    acc = __dadd_rn(acc, p2.y);
                    acc = __dadd_rn(acc, p3.x);
                    acc = __dadd_rn(acc, p3.y);
                }
                for (; j < n; ++j) acc = __dadd_rn(acc, src[j]);
            }
        } else if (tile + 1 < ntiles) {
            produce(tile + 1, tid - 32, kEntThreads - 32);
        }
        __syncthreads();
    }
    if (tid < 2) s_res[tid] = acc;
    __syncthreads();
    EntropyResult r{s_res[0], s_res[1]};
    __syncthreads();  // s_res may be reused by a following call
    return r;
}

}  // namespace dvs
