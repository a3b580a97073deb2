// Shared plumbing for libdvs_b200: error reporting, context, launch accounting.
#pragma once
#include <cuda_runtime.h>
#include <stdarg.h>
#include <stdint.h>
#include <stdio.h>

#include <string>
#include <vector>

#include "../../include/dvs_b200.h"

namespace dvs {

constexpr double kEps = 2.220446049250313e-16;  // f64::EPSILON

void set_error(const char* fmt, ...);
const char* get_error();

#define DVS_CUDA_TRY(expr)                                                                   \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            ::dvs::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, \
                             __LINE__);                                                      \
            return DVS_ERR_CUDA;                                                             \
        }                                                                                    \
    } while (0)

#define DVS_TRY(expr)            \
    do {                         \
        int _rc = (expr);        \
        if (_rc != DVS_OK) return _rc; \
    } while (0)

// counts a launch and checks the launch error
#define DVS_LAUNCHED(ctx)                                                                   \
    do {                                                                                    \
        (ctx)->launches++;                                                                  \
        cudaError_t _e = cudaGetLastError();                                                \
        if (_e != cudaSuccess) {                                                            \
            ::dvs::set_error("kernel launch failed: %s (%s:%d)", cudaGetErrorString(_e), __FILE__, \
                             __LINE__);                                                     \
            return DVS_ERR_CUDA;                                                            \
        }                                                                                   \
    } while (0)

// Stream used for stream-ordered allocation by the API call running on this thread (set by
// dvs::enter).  Allocations come from the device's default memory pool (cudaMallocAsync) whose
// release threshold is raised at context creation, so the per-call scratch and result buffers of
// repeated calls are recycled instead of paying cudaMalloc/cudaFree (which synchronise the device).
extern thread_local cudaStream_t tl_stream;

// RAII device buffer
template <class T>
struct DevBuf {
    T* p = nullptr;
    size_t n = 0;
    cudaStream_t stream = nullptr;  // stream the block was allocated on (nullptr: plain cudaMalloc)
    bool borrowed = false;          // points into memory owned by somebody else (a peer window)
    DevBuf() = default;
    DevBuf(const DevBuf&) = delete;
    DevBuf& operator=(const DevBuf&) = delete;
    ~DevBuf() { release(); }
    void release() {
        if (p && !borrowed) {
            if (stream) cudaFreeAsync(p, stream); else cudaFree(p);
        }
        p = nullptr;
        n = 0;
        borrowed = false;
    }
    void borrow(T* ptr, size_t count) {
        release();
        p = ptr;
        n = count;
        borrowed = true;
    }
    int alloc(size_t count) {
        release();
        if (count == 0) count = 1;
        stream = tl_stream;
        cudaError_t e = stream ? cudaMallocAsync((void**)&p, count * sizeof(T), stream)
                               : cudaMalloc((void**)&p, count * sizeof(T));
        if (e != cudaSuccess) {
            set_error("device allocation of %zu bytes failed: %s", count * sizeof(T), cudaGetErrorString(e));
            p = nullptr;
            return DVS_ERR_CUDA;
        }
        n = count;
        return DVS_OK;
    }
};

}  // namespace dvs

constexpr int kNumPhases = 13;

struct dvs_ctx {
    int device = 0;
    // optional per-phase CUDA-event timing on the launching stream (dvs_ctx_enable_timing)
    bool timing = false;
    cudaEvent_t ev_start[kNumPhases] = {};
    cudaEvent_t ev_stop[kNumPhases] = {};
    bool ev_valid[kNumPhases] = {};
    int sm_count = 0;
    size_t smem_optin = 0;
    cudaStream_t stream = nullptr;
    cudaStream_t stream2 = nullptr;  // second stream (created on demand): counting of dvs_count_select
    cudaStream_t stream_hi = nullptr;  // high-priority stream: the trailing selection kernel on its own SMs
    cudaEvent_t ev_hi_in = nullptr, ev_hi_out = nullptr;
    cudaEvent_t ev_first = nullptr, ev_count_done = nullptr, ev_fork = nullptr;
    unsigned* d_ready = nullptr;      // trailing selection: positions published so far
    uint64_t launches = 0;
    cudaEvent_t ev_chunk[128] = {};   // per-chunk start/stop of the counting launches (DVS_PHASE_COUNT_LAUNCHES)
    uint32_t n_chunk_ev = 0;          // pairs recorded by the last chunked counting
    uint32_t last_accepts = 0;
    uint32_t last_trail_launches = 0, last_trail_sms = 0;  // trailing kernel launches / fewest distinct SMs one sat on
    uint32_t last_trail_accepts = 0;  // of those, made while the counting was still running (dvs_count_select)
    uint32_t last_exact_evals = 0;  // exact re-evaluations forced by the fast path's error bound
    uint64_t last_upload_wire_bytes = 0;
    uint32_t last_euclid_fallback_pairs = 0;  // pairs the Gram-form Euclid kernel handed to the difference form
    double euclid_rows_ms = -1.0;  // peer row copies of the last dvs_euclid_distances_sparse_sharded (timing on)
    void* upload_stage = nullptr;  // pinned/device staging ring of the packed upload path (upload.cu)
    // pinned scratch for small device->host readbacks
    void* pinned = nullptr;
    size_t pinned_bytes = 0;
};

namespace dvs {
// every API entry: select the device and route this thread's allocations to the ctx stream
inline cudaError_t enter(dvs_ctx* ctx) {
    tl_stream = ctx->stream;
    return cudaSetDevice(ctx->device);
}
}  // namespace dvs

// Records start/stop events for one phase around a scope when timing is enabled.
struct PhaseTimer {
    dvs_ctx* ctx;
    int phase;
    PhaseTimer(dvs_ctx* c, int ph) : ctx(c), phase(ph) {
        if (ctx && ctx->timing) {
            cudaEventRecord(ctx->ev_start[phase], ctx->stream);
            ctx->ev_valid[phase] = false;
        }
    }
    void stop() {
        if (ctx && ctx->timing) {
            cudaEventRecord(ctx->ev_stop[phase], ctx->stream);
            ctx->ev_valid[phase] = true;
        }
        ctx = nullptr;
    }
    ~PhaseTimer() { stop(); }
};

// Front padding (bytes) before the first sequence byte so aligned halo loads at (addr-16) stay in
// the allocation, and tail slack so 16-byte loads covering the last byte do too.
constexpr size_t kSeqFrontPad = 256;
constexpr size_t kSeqTailPad = 256;

struct dvs_seqset {
    int device = 0;
    uint32_t nrec = 0;
    uint64_t total = 0;
    dvs::DevBuf<uint8_t> raw;        // kSeqFrontPad + total + kSeqTailPad
    dvs::DevBuf<uint64_t> offsets;   // nrec+1 (device)
    std::vector<uint64_t> h_offsets;  // nrec+1 (host)
    // counting work list of the last (chunk, nparts) asked for, kept on the device so that repeated
    // counting of one seqset (several k, several passes) does not rebuild and re-send it
    mutable dvs::DevBuf<uint8_t> work_cache;
    mutable uint64_t work_chunk = 0;
    mutable uint32_t work_nparts = 0, work_items = 0;
    mutable std::vector<uint32_t> work_seq;  // the record sequence the cached list follows (empty: 0..nrec-1)
    mutable std::vector<uint32_t> work_item_begin;  // nrec+1: first work item of every record (items are record-major)
    const uint8_t* data() const { return raw.p + kSeqFrontPad; }
    uint8_t* data() { return raw.p + kSeqFrontPad; }
};

struct dvs_kfreqs {
    int device = 0;
    uint32_t nrec = 0;
    uint64_t dim = 0;
    int k = 0, num_states = 0;
    dvs::DevBuf<uint32_t> counts;   // [nrec][dim]  (empty when built from rows)
    dvs::DevBuf<uint64_t> totals;   // [nrec]
    dvs::DevBuf<double> freqs;      // [nrec][dim]
    dvs::DevBuf<double> entropy;    // [nrec]
    dvs::DevBuf<uint8_t> valid;     // [nrec]  1 = has valid k-mers
    dvs::DevBuf<uint8_t> err;       // [nrec]  1 = reference entropy() would panic (sum check)
    dvs::DevBuf<double> err_total;  // [nrec]  the offending total
    bool has_counts = false;
    // rows gathered from all ranks live in the symmetric heap of a peer window (comm.cuh)
    struct dvs_comm* heap = nullptr;
    uint64_t heap_off = 0;
};

struct dvs_sketches {
    int device = 0;
    uint32_t nrec = 0;
    uint32_t stride = 0;
    dvs::DevBuf<uint32_t> data;  // [nrec][stride] ascending
    dvs::DevBuf<uint32_t> lens;  // [nrec]
};
