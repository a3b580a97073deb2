// comm.cuh — peer windows over NVLink: the multi-GPU plumbing of libdvs_b200 (no NCCL, no torch).
//
// One process (or host thread) per GPU.  Every rank owns a WINDOW: one cudaMalloc'ed block that every
// peer maps into its own address space (cudaIpcOpenMemHandle across processes, the raw pointer between
// contexts of one process).  The first kCommCtrlBytes of a window are control words (barrier flags,
// arrival flags of pushes, the selection kernels' exchange slots); the rest is a SYMMETRIC HEAP: every rank
// performs the same sequence of allocations, so an object lives at the same offset in every window and a
// peer's copy is addressed as peer_base + offset.  Data moves by copy-engine pushes (cudaMemcpyAsync on
// mapped peer pointers) or by loads/stores from kernels; ordering is by 8-byte flags that travel behind the
// data on the same stream.
#pragma once
#include "common.cuh"

constexpr int kCommMaxWorld = 16;
constexpr size_t kCommCtrlBytes = 64 * 1024;
// control region layout (byte offsets inside a window)
constexpr size_t kCommBarrierOff = 0;          // u64 [kCommMaxWorld]: barrier epoch written by each source rank
constexpr size_t kCommPushOff = 1024;          // u64 [kCommMaxWorld]: "pushes of epoch e from rank s have landed"
constexpr size_t kCommMinOff = 2048;           // u64 [2][kCommMaxWorld]: small all-reduce(min) slots (value<<32|tag)
constexpr size_t kCommSelOff = 4096;           // selection kernels: 16-byte tagged slots [2][kCommMaxWorld]
constexpr size_t kCommSelUpdOff = 8192;        // u32: flag set by the sharded distance kernels of any rank
constexpr size_t kCommErrOff = 16384;          // u32: a device-side wait gave up (watchdog)

struct CommBlock {
    uint64_t off, bytes;
    bool used;
};

struct dvs_comm {
    int device = 0, rank = 0, world = 1;
    uint8_t* window = nullptr;
    uint64_t window_bytes = 0;
    uint8_t* peer[kCommMaxWorld] = {};
    bool ipc_opened[kCommMaxWorld] = {};
    bool connected = false;
    uint64_t epoch = 0;       // barrier epochs
    uint64_t push_epoch = 0;  // push / gather epochs
    uint64_t min_tag = 0;     // small all-reduce exchanges so far
    uint64_t sel_tag_base = 0;  // exchange tags consumed by the selection kernels so far
    uint64_t* d_epoch_src = nullptr;  // device word holding the current push epoch (source of flag copies)
    cudaStream_t side = nullptr;      // pushes run here, behind an event of the main stream
    cudaEvent_t ev_ready = nullptr, ev_pushed = nullptr;
    // one stream per peer for the row pushes of dvs_count_kmers_sharded: the copies to different peers run on
    // different copy engines instead of one after the other (they fork from / join `side`)
    cudaStream_t peer_stream[kCommMaxWorld] = {};
    cudaEvent_t peer_ev[kCommMaxWorld] = {};
    cudaEvent_t ev_fan = nullptr;
    std::vector<CommBlock> blocks;    // symmetric heap (first fit over [kCommCtrlBytes, window_bytes))
    // Host-synchronised mode (dvs_comm_set_host_barrier): for ranks that SHARE one GPU (threads of one process in
    // the tests).  There, a kernel of one rank that spins on a peer can deadlock against a peer's host call that
    // implicitly waits for the whole device (allocation, pool growth), so the waits are taken on the host instead:
    // finish this rank's stream, meet the other ranks in `host_barrier`, carry on.  Ranks on their own GPUs never
    // set it and keep the device-side waits.
    void (*host_barrier)(void*) = nullptr;
    void* host_barrier_arg = nullptr;
    uint8_t* ctrl(int r) const { return peer[r]; }
};

namespace dvs {
// where a distance kernel's results go: one matrix (plain call) or the same place in the matrix of every GPU
// (the *_sharded Euclidean calls: each kernel stores its results straight into every peer's window - compute and
// all-gather in one kernel)
struct EuOuts {
    double* p[kCommMaxWorld];
    int count;
};

// symmetric heap: every rank must call these in the same order with the same sizes
int comm_heap_alloc(dvs_comm* c, uint64_t bytes, uint64_t* off);
void comm_heap_free(dvs_comm* c, uint64_t off);
// all ranks: wait (on ctx->stream, device side) until every rank has arrived
int comm_barrier(dvs_ctx* ctx, dvs_comm* c);
// the flag protocol of pushes: begin -> (copies on c->side) -> commit (flags to every peer) -> wait (main stream)
int comm_push_begin(dvs_ctx* ctx, dvs_comm* c);
int comm_push_commit(dvs_ctx* ctx, dvs_comm* c);
int comm_push_wait(dvs_ctx* ctx, dvs_comm* c);
// all-reduce(min) of one u32 over the ranks, device side, result in *d_out (device) when the stream gets there
int comm_min_u32(dvs_ctx* ctx, dvs_comm* c, const uint32_t* d_in, uint32_t* d_out);
// host-synchronised mode only: every rank's stream is drained and all ranks meet on the host (no-op otherwise);
// called before a kernel that spins on its peers is launched
int comm_host_rendezvous(dvs_ctx* ctx, dvs_comm* c);
int comm_check_error(dvs_ctx* ctx, dvs_comm* c, const char* what);
// the same only when DVS_COMM_CHECK=1 (it waits for the stream): the call in which a device-side wait timed out
// reports it itself (tests); otherwise the next synchronous check does (dvs_select_sharded, distances, barrier)
int comm_check_error_async(dvs_ctx* ctx, dvs_comm* c, const char* what);
}  // namespace dvs
