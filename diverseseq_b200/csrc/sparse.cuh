// Sparse (index, count) k-mer rows of dvs_count_kmers_sparse (sparse.cu), shared with their consumers
// (euclid_sparse.cu).
#pragma once
#include "common.cuh"

namespace dvs {
constexpr int kSpLowBits = 12;
constexpr uint32_t kSpLowBins = 1u << kSpLowBits;  // bins of one bucket: the low 12 bits of the index
}  // namespace dvs

// Record r owns the slots [h_offsets[r], h_offsets[r + 1]) (its byte range: #k-mers <= #bytes).  Its bucket b
// starts at slot h_offsets[r] + bucket_ptr[r][b] and holds bucket_nnz[r][b] entries in ascending index order
// (index >> 12 == b); the other slots of the bucket have count 0 and index 0xFFFFFFFF.
struct dvs_ksparse {
    int device = 0;
    uint32_t nrec = 0, nb = 0;
    int k = 0;
    uint64_t dim = 0, slots = 0;
    bool has_entropy = false;
    std::vector<uint64_t> h_offsets;        // record base (slot index) = byte offset of the record
    dvs::DevBuf<uint64_t> offsets;          // the same on the device
    dvs::DevBuf<uint32_t> idx, cnt;         // [slots] bucket-major, ascending index inside a record, count 0 = no entry
    dvs::DevBuf<uint32_t> bucket_ptr;       // [nrec][nb + 1] first slot of each bucket inside the record's region
    dvs::DevBuf<uint32_t> bucket_nnz;       // [nrec][nb] entries in use
    dvs::DevBuf<uint64_t> totals, nnz;      // [nrec] valid k-mers, distinct k-mers
    dvs::DevBuf<double> entropy, err_total; // [nrec]
    dvs::DevBuf<uint8_t> valid, err;        // [nrec]
};
