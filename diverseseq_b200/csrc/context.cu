// Context, error reporting and sequence-set residency for libdvs_b200.
#include <stdlib.h>
#include <string.h>

#include "common.cuh"

namespace dvs {

int upload_packed(dvs_ctx* ctx, const uint8_t* src, uint8_t* d_dst, size_t total);  // upload.cu
void upload_stage_free(void* p);

static thread_local std::string g_error;
thread_local cudaStream_t tl_stream = nullptr;

void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_error = buf;
}

const char* get_error() { return g_error.c_str(); }

__global__ void k_fill_u8(uint8_t* p, size_t n, uint8_t v) {
    size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = v;
}

}  // namespace dvs

using namespace dvs;

extern "C" {

const char* dvs_last_error(void) { return get_error(); }
const char* dvs_version(void) { return "dvs_b200 0.1 (sm_100a)"; }

int dvs_ctx_create(int device, dvs_ctx** out) {
    if (!out) {
        set_error("dvs_ctx_create: out is NULL");
        return DVS_ERR_ARG;
    }
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        set_error("no CUDA device available (%s); libdvs_b200 has no CPU fallback",
                  e == cudaSuccess ? "device count is 0" : cudaGetErrorString(e));
        return DVS_ERR_CUDA;
    }
    if (device < 0 || device >= ndev) {
        set_error("dvs_ctx_create: device %d out of range (have %d)", device, ndev);
        return DVS_ERR_ARG;
    }
    DVS_CUDA_TRY(cudaSetDevice(device));
    auto* ctx = new dvs_ctx();
    ctx->device = device;
    cudaDeviceProp prop;
    DVS_CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    ctx->sm_count = prop.multiProcessorCount;
    ctx->smem_optin = prop.sharedMemPerBlockOptin;
    DVS_CUDA_TRY(cudaStreamCreateWithFlags(&ctx->stream, cudaStreamNonBlocking));
    {
        cudaMemPool_t pool;
        DVS_CUDA_TRY(cudaDeviceGetDefaultMemPool(&pool, device));
        uint64_t keep = ~0ULL;  // never trim: freed blocks stay in the pool for the next call
        DVS_CUDA_TRY(cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &keep));
    }
    ctx->pinned_bytes = 1 << 20;
    DVS_CUDA_TRY(cudaHostAlloc(&ctx->pinned, ctx->pinned_bytes, cudaHostAllocDefault));
    *out = ctx;
    return DVS_OK;
}

void dvs_ctx_destroy(dvs_ctx* ctx) {
    if (!ctx) return;
    dvs::enter(ctx);
    if (ctx->stream) {
        cudaStreamSynchronize(ctx->stream);
        cudaStreamDestroy(ctx->stream);
    }
    if (ctx->stream_hi) {
        cudaStreamSynchronize(ctx->stream_hi);
        cudaStreamDestroy(ctx->stream_hi);
        cudaEventDestroy(ctx->ev_hi_in);
        cudaEventDestroy(ctx->ev_hi_out);
    }
    if (ctx->stream2) {
        cudaStreamSynchronize(ctx->stream2);
        cudaStreamDestroy(ctx->stream2);
        cudaEventDestroy(ctx->ev_first);
        cudaEventDestroy(ctx->ev_count_done);
        cudaEventDestroy(ctx->ev_fork);
        cudaFree(ctx->d_ready);
    }
    for (cudaEvent_t e : ctx->ev_chunk)
        if (e) cudaEventDestroy(e);
    if (ctx->pinned) cudaFreeHost(ctx->pinned);
    upload_stage_free(ctx->upload_stage);
    for (int i = 0; i < kNumPhases; ++i) {
        if (ctx->ev_start[i]) cudaEventDestroy(ctx->ev_start[i]);
        if (ctx->ev_stop[i]) cudaEventDestroy(ctx->ev_stop[i]);
    }
    delete ctx;
}

int dvs_ctx_sync(dvs_ctx* ctx) {
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DVS_OK;
}

uint64_t dvs_ctx_last_upload_wire_bytes(dvs_ctx* ctx) { return ctx->last_upload_wire_bytes; }

int dvs_ctx_enable_timing(dvs_ctx* ctx, int on) {
    DVS_CUDA_TRY(cudaSetDevice(ctx->device));
    if (on && !ctx->ev_start[0])
        for (int i = 0; i < kNumPhases; ++i) {
            DVS_CUDA_TRY(cudaEventCreate(&ctx->ev_start[i]));
            DVS_CUDA_TRY(cudaEventCreate(&ctx->ev_stop[i]));
        }
    ctx->timing = on != 0;
    return DVS_OK;
}

double dvs_ctx_phase_ms(dvs_ctx* ctx, int phase) {
    if (phase == DVS_PHASE_COUNT_LAUNCHES) {  // sum over the chunk launches of the last chunked counting
        if (!ctx->n_chunk_ev) return -1.0;
        double sum = 0.0;
        for (uint32_t c = 0; c < ctx->n_chunk_ev; ++c) {
            float ms = 0.0f;
            if (cudaEventSynchronize(ctx->ev_chunk[2 * c + 1]) != cudaSuccess ||
                cudaEventElapsedTime(&ms, ctx->ev_chunk[2 * c], ctx->ev_chunk[2 * c + 1]) != cudaSuccess)
                return -1.0;
            sum += ms;
        }
        return sum;
    }
    if (phase == DVS_PHASE_EUCLID_SPARSE_ROWS) return ctx->timing ? ctx->euclid_rows_ms : -1.0;  // (a sum)
    if (phase < 0 || phase >= kNumPhases || !ctx->ev_valid[phase]) return -1.0;
    if (cudaEventSynchronize(ctx->ev_stop[phase]) != cudaSuccess) return -1.0;
    float ms = -1.0f;
    if (cudaEventElapsedTime(&ms, ctx->ev_start[phase], ctx->ev_stop[phase]) != cudaSuccess) return -1.0;
    return (double)ms;
}

void* dvs_ctx_stream(dvs_ctx* ctx) { return (void*)ctx->stream; }

// plain device / pinned host buffers for callers that have no other CUDA binding (the Python host code keeps
// distance matrices on the device and stages sequences in pinned memory without importing torch)
int dvs_device_malloc(dvs_ctx* ctx, uint64_t bytes, void** out) {
    if (!ctx || !out) {
        set_error("dvs_device_malloc: NULL argument");
        return DVS_ERR_ARG;
    }
    DVS_CUDA_TRY(dvs::enter(ctx));
    DVS_CUDA_TRY(cudaMalloc(out, bytes ? bytes : 1));
    return DVS_OK;
}
void dvs_device_free(dvs_ctx* ctx, void* p) {
    if (!p) return;
    if (ctx) cudaSetDevice(ctx->device);
    cudaFree(p);
}
int dvs_device_memcpy(dvs_ctx* ctx, void* dst, const void* src, uint64_t bytes) {
    DVS_CUDA_TRY(dvs::enter(ctx));
    if (bytes) DVS_CUDA_TRY(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, ctx->stream));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DVS_OK;
}
int dvs_host_malloc_pinned(uint64_t bytes, void** out) {
    if (!out) {
        set_error("dvs_host_malloc_pinned: NULL argument");
        return DVS_ERR_ARG;
    }
    DVS_CUDA_TRY(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocDefault));
    return DVS_OK;
}
void dvs_host_free_pinned(void* p) {
    if (p) cudaFreeHost(p);
}
uint64_t dvs_ctx_launch_count(dvs_ctx* ctx) { return ctx->launches; }

// ---- sequence sets -----------------------------------------------------------------------

static int seqset_alloc(dvs_ctx* ctx, const uint64_t* offsets, uint32_t nrec, dvs_seqset** out) {
    for (uint32_t r = 0; r < nrec; ++r)
        if (offsets[r + 1] < offsets[r]) {
            set_error("offsets must be non-decreasing (record %u)", r);
            return DVS_ERR_ARG;
        }
    if (offsets[0] != 0) {
        set_error("offsets[0] must be 0");
        return DVS_ERR_ARG;
    }
    DVS_CUDA_TRY(dvs::enter(ctx));
    auto* s = new dvs_seqset();
    s->device = ctx->device;
    s->nrec = nrec;
    s->total = offsets[nrec];
    s->h_offsets.assign(offsets, offsets + nrec + 1);
    int rc = s->raw.alloc(kSeqFrontPad + s->total + kSeqTailPad);
    if (rc == DVS_OK) rc = s->offsets.alloc(nrec + 1);
    if (rc != DVS_OK) {
        delete s;
        return rc;
    }
    // pads hold 0xFF (invalid for every num_states) so halo/tail vector loads never see a base
    cudaMemsetAsync(s->raw.p, 0xFF, kSeqFrontPad, ctx->stream);
    cudaMemsetAsync(s->raw.p + kSeqFrontPad + s->total, 0xFF, kSeqTailPad, ctx->stream);
    cudaError_t e = cudaMemcpyAsync(s->offsets.p, offsets, (nrec + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice,
                                    ctx->stream);
    if (e != cudaSuccess) {
        set_error("offset upload failed: %s", cudaGetErrorString(e));
        delete s;
        return DVS_ERR_CUDA;
    }
    *out = s;
    return DVS_OK;
}

int dvs_seqset_alloc_internal(dvs_ctx* ctx, const uint64_t* offsets, uint32_t nrec, dvs_seqset** out) {
    return seqset_alloc(ctx, offsets, nrec, out);
}

int dvs_seqset_upload(dvs_ctx* ctx, const uint8_t* seqs, const uint64_t* offsets, uint32_t nrec,
                      dvs_seqset** out) {
    if (!ctx || !offsets || !out || (!seqs && offsets[nrec] > 0)) {
        set_error("dvs_seqset_upload: NULL argument");
        return DVS_ERR_ARG;
    }
    dvs_seqset* s = nullptr;
    DVS_TRY(seqset_alloc(ctx, offsets, nrec, &s));
    PhaseTimer pt(ctx, DVS_PHASE_UPLOAD);
    // large uploads go 2-bit packed over PCIe and are unpacked on the device (upload.cu);
    // DVS_UPLOAD_PACKED=0 forces the plain copy, =1 forces packing for any size
    const char* pk = getenv("DVS_UPLOAD_PACKED");
    const bool packed = pk ? (pk[0] == '1') : (s->total >= (64ull << 20));
    ctx->last_upload_wire_bytes = s->total;
    if (s->total && packed) {
        ctx->last_upload_wire_bytes = 0;  // accumulated by upload_packed
        int rc = upload_packed(ctx, seqs, s->data(), s->total);
        if (rc != DVS_OK) {
            delete s;
            return rc;
        }
    } else if (s->total) {
        cudaError_t e = cudaMemcpyAsync(s->data(), seqs, s->total, cudaMemcpyHostToDevice, ctx->stream);
        if (e != cudaSuccess) {
            set_error("sequence upload failed: %s", cudaGetErrorString(e));
            delete s;
            return DVS_ERR_CUDA;
        }
    }
    pt.stop();
    // the host buffers (seqs, offsets) may be pageable and reused by the caller: finish the copies
    cudaError_t e = cudaStreamSynchronize(ctx->stream);
    if (e != cudaSuccess) {
        set_error("sequence upload failed: %s", cudaGetErrorString(e));
        delete s;
        return DVS_ERR_CUDA;
    }
    *out = s;
    return DVS_OK;
}

uint32_t dvs_seqset_nrec(const dvs_seqset* s) { return s->nrec; }
uint64_t dvs_seqset_total_bases(const dvs_seqset* s) { return s->total; }

int dvs_seqset_offsets(const dvs_seqset* s, uint64_t* offsets_out) {
    memcpy(offsets_out, s->h_offsets.data(), (s->nrec + 1) * sizeof(uint64_t));
    return DVS_OK;
}

int dvs_seqset_download(dvs_ctx* ctx, const dvs_seqset* s, uint32_t first, uint32_t count, uint8_t* seqs_out) {
    if (first + (uint64_t)count > s->nrec) {
        set_error("dvs_seqset_download: range out of bounds");
        return DVS_ERR_ARG;
    }
    uint64_t b = s->h_offsets[first], e = s->h_offsets[first + count];
    DVS_CUDA_TRY(dvs::enter(ctx));
    if (e > b) DVS_CUDA_TRY(cudaMemcpyAsync(seqs_out, s->data() + b, e - b, cudaMemcpyDeviceToHost, ctx->stream));
    DVS_CUDA_TRY(cudaStreamSynchronize(ctx->stream));
    return DVS_OK;
}

void dvs_seqset_free(dvs_seqset* s) {
    if (!s) return;
    cudaSetDevice(s->device);
    delete s;
}

}  // extern "C"
