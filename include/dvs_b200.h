/* dvs_b200.h — C ABI of libdvs_b200.so: the B200 (sm_100a) implementation of diverse-seq's
 * data-parallel hot path.  This is the drop-in boundary: every entry point replaces one
 * function of the reference's PyO3 module `diverse_seq._dvs` (or the pure-Python pair loops
 * of diverse_seq/distance.py) and is what a reference-side FFI binding would bind; see
 * INTEGRATION.md for the Rust `extern "C"` / ctypes stubs.  File:line citations are into
 * /root/reference.
 *
 * Conventions
 *   - plain pointers + sizes, caller-owned HOST buffers unless a parameter says "device";
 *     the library never frees caller memory; opaque handles are freed by their *_free.
 *   - sequences are the reference's uint8 index arrays (1 byte/base; T,C,A,G = 0..3 for DNA;
 *     any byte >= num_states is invalid and breaks every k-mer that contains it), all records
 *     concatenated in `seqs`, record r = seqs[offsets[r] .. offsets[r+1]).
 *   - k-mer index is positional base-num_states, first base most significant
 *     (src/record.rs:10-29); a count/frequency row has num_states^k entries.
 *   - return 0 on success.  DVS_ERR_VALUE carries a message the reference raises as
 *     ValueError (a Rust panic, src/lib.rs:36-57); DVS_ERR_CUDA is a CUDA runtime failure
 *     (-> RuntimeError); DVS_ERR_ARG is API misuse.  dvs_last_error() returns the text
 *     (thread-local).  There is NO CPU fallback: without a CUDA device dvs_ctx_create fails.
 *   - one dvs_ctx per host thread/process per GPU; calls on one ctx are not re-entrant.
 */
#ifndef DVS_B200_H
#define DVS_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define DVS_OK 0
#define DVS_ERR_VALUE 1
#define DVS_ERR_CUDA 2
#define DVS_ERR_ARG 3

/* selection modes for dvs_select */
#define DVS_MODE_NMOST 0     /* select_nmost_divergent   src/records.rs:311-342 */
#define DVS_MODE_MAX_STDEV 1 /* select_max_divergent, Stat::Std  src/records.rs:390-454 */
#define DVS_MODE_MAX_COV 2   /* select_max_divergent, Stat::Cov */

typedef struct dvs_ctx dvs_ctx;       /* device, streams, scratch */
typedef struct dvs_seqset dvs_seqset; /* device-resident batch of encoded sequences */
typedef struct dvs_kfreqs dvs_kfreqs; /* device-resident [nrec][num_states^k] rows + entropies */
typedef struct dvs_summed dvs_summed; /* device-resident SummedRecords state */
typedef struct dvs_sketches dvs_sketches; /* device-resident bottom-s MinHash sketches */

const char* dvs_last_error(void);
const char* dvs_version(void);

/* ---- context --------------------------------------------------------------------------- */
int dvs_ctx_create(int device, dvs_ctx** out);
void dvs_ctx_destroy(dvs_ctx* ctx);
int dvs_ctx_sync(dvs_ctx* ctx);
/* the CUDA stream (cudaStream_t) every kernel of this ctx is launched on, for event timing */
void* dvs_ctx_stream(dvs_ctx* ctx);
/* plain device / pinned host buffers for host code without another CUDA binding (distance matrices that stay on
 * the device, pinned staging of sequences); dvs_device_memcpy copies in any direction and waits */
int dvs_device_malloc(dvs_ctx* ctx, uint64_t bytes, void** out);
void dvs_device_free(dvs_ctx* ctx, void* p);
int dvs_device_memcpy(dvs_ctx* ctx, void* dst, const void* src, uint64_t bytes);
int dvs_host_malloc_pinned(uint64_t bytes, void** out);
void dvs_host_free_pinned(void* p);
/* number of kernels this ctx has launched so far (bench.py's gpu_launches) */
uint64_t dvs_ctx_launch_count(dvs_ctx* ctx);

/* per-phase device timing with CUDA events recorded on the ctx stream around the named kernels
 * (bench.py's roofline numbers).  dvs_ctx_phase_ms returns the duration of the most recent
 * occurrence of the phase in milliseconds, or a negative value if it has not run. */
#define DVS_PHASE_COUNT_KERNEL 0   /* k_count: the k-mer histogram kernel alone */
#define DVS_PHASE_FREQ_ENTROPY 1   /* k_freq_entropy: rows + exact entropies */
#define DVS_PHASE_SELECT 2         /* all device work of one dvs_select */
#define DVS_PHASE_SKETCH 3         /* all device work of one dvs_mash_sketch */
#define DVS_PHASE_MASH_PAIRS 4     /* k_mash_pairs */
#define DVS_PHASE_EUCLID 5         /* k_euclid_tiles */
#define DVS_PHASE_UPLOAD 6         /* host->device sequence copy of dvs_seqset_upload */
#define DVS_PHASE_CLUSTER 8        /* k_cl_symmetrise + k_cl_nn_chain of one dvs_linkage_average */
#define DVS_PHASE_SPARSE 9         /* the partition passes of one dvs_count_kmers_sparse (without the optional entropies) */
#define DVS_PHASE_COUNT_LAUNCHES 10 /* chunked counting (sharded / dvs_count_select): sum of the counting launches alone */
#define DVS_PHASE_PREP 7           /* all device work of one dvs_prep_fasta (k_prep x2 + k_prep_carry) */
#define DVS_PHASE_EUCLID_SPARSE 11 /* all device work of one dvs_euclid_distances_sparse (without the output copy);
                                      * of dvs_euclid_distances_sparse_sharded: this rank's blocks, row copies included */
#define DVS_PHASE_EUCLID_SPARSE_ROWS 12 /* dvs_euclid_distances_sparse_sharded: the copies of peer rows, summed */
/* bytes that actually crossed PCIe during the last dvs_seqset_upload (2-bit packed + exceptions for
 * large uploads, see csrc/upload.cu; equal to the input size for the plain copy) */
uint64_t dvs_ctx_last_upload_wire_bytes(dvs_ctx* ctx);
int dvs_ctx_enable_timing(dvs_ctx* ctx, int on);
double dvs_ctx_phase_ms(dvs_ctx* ctx, int phase);

/* ---- sequences: what ZarrStore::read_uint8_array hands the hot path (src/zarr_io.rs:309) - */
int dvs_seqset_upload(dvs_ctx* ctx, const uint8_t* seqs, const uint64_t* offsets, uint32_t nrec,
                      dvs_seqset** out);
/* synthetic genomes generated on the device (bench / tests; SURVEY.md §8d): `nfam` family
 * ancestors from order-2 Markov chains, members = ancestor prefix with per-base substitutions,
 * invalid runs at ~1e-4.  Deterministic in (seed, record, position); lengths in
 * [mean_len*0.75, mean_len*1.25].  dvs_synth_host() is the bit-identical host generator. */
int dvs_seqset_synth(dvs_ctx* ctx, uint64_t seed, uint32_t nrec, uint32_t nfam, uint64_t mean_len,
                     dvs_seqset** out);
/* records [first, first + nrec) of the same generator (one set split over several GPUs) */
int dvs_seqset_synth_range(dvs_ctx* ctx, uint64_t seed, uint32_t first, uint32_t nrec, uint32_t nfam, uint64_t mean_len,
                           dvs_seqset** out);
int dvs_synth_host(uint64_t seed, uint32_t nrec, uint32_t nfam, uint64_t mean_len, uint32_t first,
                   uint32_t count, uint8_t* seqs_out, uint64_t* offsets_out);
int dvs_synth_lengths(uint64_t seed, uint32_t nrec, uint64_t mean_len, uint64_t* lens_out);
uint32_t dvs_seqset_nrec(const dvs_seqset* s);
uint64_t dvs_seqset_total_bases(const dvs_seqset* s);
int dvs_seqset_offsets(const dvs_seqset* s, uint64_t* offsets_out /* nrec+1 */);
int dvs_seqset_download(dvs_ctx* ctx, const dvs_seqset* s, uint32_t first, uint32_t count,
                        uint8_t* seqs_out);
void dvs_seqset_free(dvs_seqset* s);

/* ---- `dvs prep` encode: FASTA text -> index-encoded records, one record per FILE -------------
 * Replaces diverse_seq/io.py:30-34 (converter_fasta: a-z -> A-Z, delete "\n\r\t- "), :47-57
 * (cogent3 iter_fasta_records: split at every '>', first line of a piece is the label, a piece
 * without a newline is dropped), :95-104 (dvs_load_seqs: b"-".join(seqs) -> str2arr) and
 * diverse_seq/util.py:32-45 (str2arr = most_degen_alphabet().to_indices: position in the alphabet,
 * bytes outside it keep their own value).  `text` holds the bytes of `nfiles` files back to back,
 * file f = [file_offsets[f], file_offsets[f+1]).  alphabet NULL = DVS_DNA_ALPHABET, delete_chars
 * NULL = "\n\r\t- ", sep_char < 0 = '-'.  text_on_device != 0: `text` is a 4-byte aligned device
 * pointer (readable up to 3 bytes past the end).  Codes 0..3 (T,C,A,G) are what the hot path
 * consumes; every other code is >= 4 = invalid for it. */
#define DVS_DNA_ALPHABET "TCAG-NRYWSKMBDHV?"
int dvs_prep_fasta(dvs_ctx* ctx, const uint8_t* text, const uint64_t* file_offsets, uint32_t nfiles,
                   const char* alphabet, const char* delete_chars, int sep_char, int text_on_device,
                   dvs_seqset** out);

/* ---- k-mer counting + frequencies + entropy -------------------------------------------------
 * SeqRecord::to_kcounts / to_kmerseq / entropy  (src/record.rs:41-84, 124-141, 86-106).
 * Result rows stay in HBM.  A record with no valid k-mer is marked valid=0 (the reference
 * returns Err and callers skip it, src/records.rs:302,333).  Entropy is evaluated in the
 * reference's sequential order with glibc's log2 algorithm, so it is bit-identical.  Bin counters are 32-bit:
 * a record of 2^32 bases or more is refused with DVS_ERR_ARG (the reference counts in usize). */
int dvs_count_kmers(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, dvs_kfreqs** out);
/* rows already computed elsewhere, e.g. SummedRecordsResult.records of per-chunk results fed to
 * final_nmost / final_max (src/records.rs:344-360): entropy is recomputed from the stored
 * frequencies exactly as KmerSeq::new does.  entropies_or_null == NULL -> recompute. */
int dvs_kfreqs_from_rows(dvs_ctx* ctx, const double* rows, const double* entropies_or_null, uint32_t nrec,
                         uint64_t dim, dvs_kfreqs** out);
/* multi-GPU plumbing (SURVEY.md §8e): raw DEVICE pointers of the row matrix [nrec][dim] f64, the
 * entropies [nrec] f64 and the validity flags [nrec] u8, so a collective library (NCCL) can
 * all-gather shards; and the inverse, a kfreqs built by device-to-device copy from gathered
 * device buffers that live on ctx's GPU.  d_entropies == NULL recomputes every entropy from the
 * rows exactly as KmerSeq::new does (src/records.rs:353), d_valid == NULL marks all rows valid. */
int dvs_kfreqs_device_ptrs(const dvs_kfreqs* f, void** freqs, void** entropies, void** valid);
/* a new kfreqs holding rows `rows[0..n)` of f (device gather; entropies / validity carried over):
 * the records of a SummedRecordsResult, ready to be all-gathered for final_nmost / final_max */
int dvs_kfreqs_take_rows(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* rows, uint32_t n, dvs_kfreqs** out);
int dvs_kfreqs_from_device(dvs_ctx* ctx, const void* d_rows, const void* d_entropies, const void* d_valid,
                           uint32_t nrec, uint64_t dim, dvs_kfreqs** out);
uint32_t dvs_kfreqs_nrec(const dvs_kfreqs* f);
uint64_t dvs_kfreqs_dim(const dvs_kfreqs* f);
/* any output may be NULL.  counts: uint64 like Rust usize (LazySeq.get_kcounts, src/record.rs:247);
 * freqs: count/total as f64 (NaN row when total==0, like LazySeq.get_kfreqs src/record.rs:256). */
int dvs_kfreqs_download(dvs_ctx* ctx, const dvs_kfreqs* f, uint32_t first, uint32_t count, uint64_t* counts,
                        double* freqs, double* entropies, uint8_t* valid);
void dvs_kfreqs_free(dvs_kfreqs* f);
/* one-call host->host form (upload, count, download) */
int dvs_count_kmers_host(dvs_ctx* ctx, const uint8_t* seqs, const uint64_t* offsets, uint32_t nrec, int k,
                         int num_states, uint64_t* counts, double* freqs, double* entropies, uint8_t* valid);

/* ---- sparse counting for large k (9 <= k <= 12, num_states 4) ----------------------------------------
 * to_kcounts where the dense vector is out of reach (4^12 bins = 134 MB of f64 per record, src/record.rs:41-84,
 * 124-131): the result of a record is the ascending list of its DISTINCT k-mer indices with their counts, i.e.
 * the non-zero entries of the reference's vector (8 bytes per distinct k-mer; SURVEY.md §8d).  Frequencies are
 * count / total; want_entropy != 0 also evaluates the reference's sequential entropy over the non-zero entries
 * (bit-identical: the reference skips zeros; ~30 ms per 4 Mbp record, records in parallel).
 * dvs_ksparse_stats: per record the number of distinct k-mers, of valid k-mers, the entropy (NULL unless
 * requested at count time) and validity.  dvs_ksparse_download: one record's (index, count) lists; call with
 * idx = cnt = NULL to learn the length first. */
typedef struct dvs_ksparse dvs_ksparse;
int dvs_count_kmers_sparse(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, int want_entropy, dvs_ksparse** out);
uint32_t dvs_ksparse_nrec(const dvs_ksparse* sp);
int dvs_ksparse_stats(dvs_ctx* ctx, const dvs_ksparse* sp, uint64_t* nnz, uint64_t* totals, double* entropy,
                      uint8_t* valid);
int dvs_ksparse_download(dvs_ctx* ctx, const dvs_ksparse* sp, uint32_t rec, uint32_t* idx, uint32_t* cnt, uint64_t cap,
                         uint64_t* nnz_out);
void dvs_ksparse_free(dvs_ksparse* sp);
/* euclidean_distances over the sparse rows: the matrix dvs_euclid_distances gives for the dense rows of the same
 * records (1e-9 relative; NaN for pairs with a record without valid k-mers, zero diagonal), rows
 * [row_begin,row_end) x all columns, `dist` host or device memory; every pair is bit-identical whatever the row
 * range.  A pair costs one product per k-mer both records hold (exact integer Gram form, DESIGN.md §5.11); the
 * pairs that form cannot give to 1e-9 of the reference's rounded frequencies are recomputed in difference form
 * (their number: dvs_euclid_last_fallback_pairs).  A matrix that does not fit the free device memory is refused
 * with DVS_ERR_ARG: ask for fewer rows per call. */
int dvs_euclid_distances_sparse(dvs_ctx* ctx, const dvs_ksparse* sp, uint32_t row_begin, uint32_t row_end, double* dist);

/* ---- nmost / max selection ------------------------------------------------------------------
 * select_nmost_divergent / select_max_divergent and their *_final forms (src/records.rs:311-507)
 * over the rows of `f`, examined in `order` (order[i] = row index at position i; the row index is
 * the record identity, i.e. stands in for seqid).  Single-pass, order-dependent semantics of the
 * reference with numprocs=1.  Outputs, in the reference's final Vec order: sel_idx[size],
 * sel_delta[size] (delta_jsd per record), stats = {total_jsd, mean_delta_jsd, std_delta_jsd,
 * cov_delta_jsd, summed_entropies}.  sel_idx/sel_delta need capacity max(min_size, max_size); in the max modes
 * with max_size < min_size (rejected only by the reference's CLI, cli.py:311) `size == max_size` never holds and the
 * set may grow to `num` records as in records.rs:427-451, so the capacity must then be `num`. */
int dvs_select(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* order, uint32_t num, int mode,
               uint32_t min_size, uint32_t max_size, uint32_t* sel_idx, double* sel_delta, double* stats5,
               uint32_t* size_out);
/* number of candidates that changed the set during the last dvs_select on this ctx */
uint32_t dvs_select_last_accepts(dvs_ctx* ctx);
/* number of exact re-evaluations the bounded-error fast path had to request during the last
 * dvs_select (0 when every decision was far from a tie; environment DVS_SELECT_EXACT_ONLY=1
 * disables the fast path altogether) */
uint32_t dvs_select_last_exact_evals(dvs_ctx* ctx);
/* ... and how many were accepted while the counting of dvs_count_select was still running */
uint32_t dvs_select_last_trail_accepts(dvs_ctx* ctx);
/* launches of the trailing kernel in that call, and the fewest distinct SMs the CTAs of one of them sat on */
uint32_t dvs_select_last_trail_launches(dvs_ctx* ctx);
uint32_t dvs_select_last_trail_sms(dvs_ctx* ctx);

/* SummedRecords::new over the listed rows + delta_jsd queries: make_summed_records and
 * SummedRecordsWrapper (src/records.rs:509-524, src/records_py.rs:90-125) */
int dvs_summed_create(dvs_ctx* ctx, const dvs_kfreqs* f, const uint32_t* members, uint32_t n, dvs_summed** out);
/* delta_jsd of row `q_row` of `q` against the state (src/records.rs:70-84); is_member != 0 means the
 * query's seqid is already in the set -> 0.0 */
int dvs_summed_delta_jsd(dvs_ctx* ctx, dvs_summed* s, const dvs_kfreqs* q, uint32_t q_row, int is_member,
                         double* out);
/* delta_jsd of EVERY row of `q` in one launch (the dvs_delta_jsd app scores many queries against one
 * state, diverse_seq/records.py:377-429).  is_member_or_null[r] != 0 -> 0.0 (seqid already in the set);
 * rows without valid k-mers get NaN (the reference raises ValueError for those). */
int dvs_summed_delta_jsd_batch(dvs_ctx* ctx, dvs_summed* s, const dvs_kfreqs* q, const uint8_t* is_member_or_null,
                               double* out);
int dvs_summed_result(dvs_ctx* ctx, dvs_summed* s, uint32_t* sel_idx, double* sel_delta, double* stats5,
                      uint32_t* size_out, uint32_t* lowest_out);
void dvs_summed_free(dvs_summed* s);

/* ---- MinHash sketches + mash distances ------------------------------------------------------
 * mash_sketch (src/distance.rs:151-182: reference hash src/distance.rs:21-87, distinct hashes,
 * bottom-s ascending) for every record, and mash_distance for all pairs
 * (diverse_seq/distance.py:230-291, matrix conventions :163-175). */
int dvs_mash_sketch(dvs_ctx* ctx, const dvs_seqset* s, int k, uint64_t sketch_size, int num_states,
                    int canonical, dvs_sketches** out);
int dvs_sketches_from_host(dvs_ctx* ctx, const uint32_t* sketches, uint32_t stride, const uint32_t* lens,
                           uint32_t nrec, dvs_sketches** out);
uint32_t dvs_sketches_nrec(const dvs_sketches* sk);
uint32_t dvs_sketches_stride(const dvs_sketches* sk);
int dvs_sketches_download(dvs_ctx* ctx, const dvs_sketches* sk, uint32_t* sketches /* [nrec][stride] */,
                          uint32_t* lens);
void dvs_sketches_free(dvs_sketches* sk);
/* rows [row_begin,row_end) of the symmetric nrec x nrec matrix (2-D sharding hook); outputs are
 * (row_end-row_begin) x nrec, row-major; inter/uni may be NULL.  The output pointers may be host or
 * device memory (unified addressing). */
int dvs_mash_distances(dvs_ctx* ctx, const dvs_sketches* sk, int k, uint64_t sketch_size, uint32_t row_begin,
                       uint32_t row_end, double* dist, uint32_t* inter, uint32_t* uni);
/* host->host single record, mirrors _dvs.mash_sketch(seq_array, k, sketch_size, num_states, canonical) */
int dvs_mash_sketch_host(dvs_ctx* ctx, const uint8_t* seq, uint64_t len, int k, uint64_t sketch_size,
                         int num_states, int canonical, uint32_t* out, uint64_t cap, uint64_t* out_len);

/* ---- Euclidean k-mer distance matrix --------------------------------------------------------
 * euclidean_distances (diverse_seq/distance.py:294-336, cluster.py:647-680): ||f_i - f_j||_2 over
 * frequency rows, rows [row_begin,row_end) x all columns, zero diagonal; `dist` may be host or device memory. */
int dvs_euclid_distances(dvs_ctx* ctx, const dvs_kfreqs* f, uint32_t row_begin, uint32_t row_end, double* dist);
/* pairs that the Gram-form kernel of the last dvs_euclid_distances(_sharded) on this ctx handed to the
 * difference form because |a|^2 + |b|^2 - 2 a.b would have cancelled too many digits (near-duplicate rows);
 * after dvs_euclid_distances_sparse, the pairs it listed for its difference-form kernel (0 after an argument
 * error or an empty range; after a list overflow, the number of pairs that overflowed the list); after
 * dvs_euclid_distances_sparse_sharded, the pairs THIS rank listed over all of its blocks (reset on entry; after a
 * list overflow on this rank, the overflowing count) */
uint32_t dvs_euclid_last_fallback_pairs(dvs_ctx* ctx);

/* ---- `dvs ctree` tail: average-linkage tree of a precomputed distance matrix -----------------
 * Replaces sklearn AgglomerativeClustering(metric="precomputed", linkage="average").fit(D) in
 * make_cluster_tree (diverse_seq/cluster.py:191-237), i.e. scipy's nearest-neighbour-chain linkage on
 * the upper triangle of D followed by its stable sort and relabelling.  dist: n x n row-major f64 on
 * the host OR the device (e.g. straight from dvs_euclid_distances / dvs_mash_distances, which accept
 * device output pointers too).  children: (n-1) x 2, identical to sklearn's children_ (values < n are
 * leaves, n + i is the cluster made by row i); heights / counts (may be NULL): merge distance and
 * cluster size per row. */
int dvs_linkage_average(dvs_ctx* ctx, const double* dist, uint32_t n, int32_t* children, double* heights,
                        uint32_t* counts);

/* ---- multi-GPU: peer windows over NVLink (SURVEY.md §8e) -------------------------------------
 * One process (or host thread) per GPU, no NCCL and no torch in the data path.  Every rank owns a WINDOW (one
 * cudaMalloc'ed block) that all peers map (cudaIpc across processes, the raw pointer inside one process);
 * its head holds control words (barrier / arrival flags, the selection kernels' exchange slots), the rest is
 * a symmetric heap.  Set-up is two steps around ONE host-side exchange of DVS_COMM_HANDLE_BYTES per rank
 * over any transport (diverseseq_b200/shard.py uses a TCP rendezvous on MASTER_ADDR:MASTER_PORT):
 *   dvs_comm_create   allocate this rank's window, describe it in handle_out
 *   dvs_comm_connect  handles = the `world` blobs in rank order; maps every peer
 * All ranks must call the collective entry points (barrier, allgatherv, *_sharded) in the same order.
 * Device-side waits give up after 20 s (a missing rank becomes DVS_ERR_CUDA instead of a hang). */
typedef struct dvs_comm dvs_comm;
#define DVS_COMM_HANDLE_BYTES 128
int dvs_comm_create(dvs_ctx* ctx, int rank, int world, uint64_t window_bytes, dvs_comm** out, void* handle_out);
int dvs_comm_connect(dvs_ctx* ctx, dvs_comm* c, const void* handles /* world x DVS_COMM_HANDLE_BYTES */);
/* Ranks that SHARE one GPU (threads of one process, as in the tests) must take their waits on the host: a kernel
 * that spins on a peer could deadlock against the peer's host calls that implicitly wait for the whole device.
 * `barrier(arg)` must return once every rank has called it (e.g. a thread barrier); all ranks set it or none.
 * Ranks on their own GPUs never call this and keep the device-side flags. */
int dvs_comm_set_host_barrier(dvs_comm* c, void (*barrier)(void*), void* arg);
int dvs_comm_rank(const dvs_comm* c);
int dvs_comm_world(const dvs_comm* c);
int dvs_comm_barrier(dvs_ctx* ctx, dvs_comm* c);
/* all-gather of device buffers of different sizes: rank r contributes bytes_per_rank[r] bytes from d_src;
 * d_dst (device, sum of the sizes) receives them in rank order.  The window must hold the largest piece. */
int dvs_comm_allgatherv(dvs_ctx* ctx, dvs_comm* c, const void* d_src, const uint64_t* bytes_per_rank, void* d_dst);
void dvs_comm_destroy(dvs_comm* c);

/* Rows of ALL ranks in one kfreqs on every rank (rank-major: rank 0's records first), stored in the
 * symmetric heap of the window.  nrec_per_rank[world] = records held by each rank (the host exchanges these
 * counts; they may differ).  dvs_count_kmers_sharded counts this rank's records in chunks and pushes each
 * chunk's rows to the peers over the copy engines while the next chunk is being counted (prep sharded by
 * record, SURVEY.md §8e row 1); dvs_kfreqs_allgather does the same for rows that already exist.  The result
 * carries entropies, validity and the reference's panic flags of every record; it holds no counts.  Free it
 * with dvs_kfreqs_free BEFORE dvs_comm_destroy. */
int dvs_count_kmers_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_seqset* local, int k, int num_states,
                            const uint32_t* nrec_per_rank, dvs_kfreqs** out_all);
int dvs_kfreqs_allgather(dvs_ctx* ctx, dvs_comm* c, const dvs_kfreqs* local, const uint32_t* nrec_per_rank,
                         dvs_kfreqs** out_all);
/* dvs_select over the rows of all ranks with the scan CANDIDATE-SHARDED over the GPUs (SURVEY.md §8e row 2):
 * the single-pass, numprocs=1 semantics of src/records.rs:311-342 / :390-454 - NOT the -np chunk merge.  Every
 * rank passes the same f_all (from dvs_count_kmers_sharded / dvs_kfreqs_allgather), order and arguments and
 * receives the same result.  Each GPU scores the window positions p with p % world == rank; per round the
 * leaders all-reduce(min) {first_true, first_unsure} through 16-byte tagged slots in the peer windows (one
 * NVLink store per peer and round); the state update is replayed identically on every GPU. */
/* ctree on several GPUs (SURVEY.md §8e rows 3-5).  Sketches of all ranks on every rank (stride_all = the largest
 * dvs_sketches_stride of any rank); then the pairs of the lower triangle (mash) / its 128 x 128 tiles (Euclid)
 * are dealt over the GPUs round-robin and every kernel stores its distances straight into the matrix of EVERY
 * GPU through the peer windows (compute and all-gather in one kernel).  dist: n x n f64, host or device; every
 * rank receives the whole matrix (the row order is the rank-major record order). */
int dvs_sketches_allgather(dvs_ctx* ctx, dvs_comm* c, const dvs_sketches* local, const uint32_t* nrec_per_rank,
                           uint32_t stride_all, dvs_sketches** out_all);
int dvs_mash_distances_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_sketches* sk_all, int k, uint64_t sketch_size,
                               double* dist);
int dvs_euclid_distances_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_kfreqs* f_all, double* dist);
/* euclidean_distances over the sparse rows of ALL ranks.  Collective.  Each rank passes ITS OWN
 * dvs_count_kmers_sparse result; the rows never leave their rank except one peer's at a time.
 * nrec_per_rank[world] = records of every rank.  dist: n x n f64 (n = sum), host or device memory.
 * Every rank receives the whole matrix in rank-major record order.  It is bit-identical to
 * dvs_euclid_distances_sparse over the union of the records.
 * Each rank stages its rows in its window and computes the pairs it owns: its own lower triangle, and at step
 * d = 1 .. world/2 the pairs with rank (rank + d) % world, whose rows it copies into device memory of its own (at
 * d = world/2 the two ranks split that block by the lower rank's first ceil(n/2) records); every distance is stored
 * into every rank's matrix.  The window must hold the staged rows of the largest shard and the matrix
 * (shard.window_bytes_for_sparse; a single rank stages nothing).  Every rank returns the same status: a different k
 * on some rank or an nrec_per_rank that disagrees with any rank's records is DVS_ERR_ARG, a difference-form list
 * overflow on any rank (more than 2^24 listed pairs on one rank) DVS_ERR_VALUE; when ranks fail differently, all return
 * the worst class (DVS_ERR_CUDA before DVS_ERR_ARG before DVS_ERR_VALUE). */
int dvs_euclid_distances_sparse_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_ksparse* local,
                                        const uint32_t* nrec_per_rank, double* dist);
int dvs_select_sharded(dvs_ctx* ctx, dvs_comm* c, const dvs_kfreqs* f_all, const uint32_t* order, uint32_t num,
                       int mode, uint32_t min_size, uint32_t max_size, uint32_t* sel_idx, double* sel_delta,
                       double* stats5, uint32_t* size_out);

/* dvs_count_kmers + dvs_select in one call with the two OVERLAPPED on one GPU (the `dvs prep` -> `dvs nmost` flow of
 * BASELINE.json configs[1]; reference: src/lib.rs nmost() over the records src/record.rs KmerSeq::new builds).
 * The records are counted on a second stream in the sequence `order` examines them, `chunks` launches (0 = default:
 * six launches of relative sizes 3,4,4,3,2,1; at most 64); after each launch the number of positions whose rows exist
 * is published in a device word and the nmost rounds - the SM-replicated selection kernel on a high-priority stream,
 * which takes ~36 SMs for itself while the counting keeps the rest - examine only positions below it.
 * Results (rows in *out, selection, stats) are bit-identical to the two separate calls.  Modes other than
 * DVS_MODE_NMOST, k outside 4..6, n > 1024 or min_size larger than the first chunk run the two steps back to back. */
int dvs_count_select(dvs_ctx* ctx, const dvs_seqset* s, int k, int num_states, const uint32_t* order, uint32_t num,
                     int mode, uint32_t min_size, uint32_t max_size, uint32_t chunks, dvs_kfreqs** out,
                     uint32_t* sel_idx, double* sel_delta, double* stats5, uint32_t* size_out);

/* ---- test hooks ---------------------------------------------------------------------------- */
/* host half of the packed upload (transfer encoding, no GPU needed): packs src[0..n) 4 bases per
 * byte (b0 | b1<<2 | b2<<4 | b3<<6), bytes >= 4 become 0 and are listed as (position, value)
 * exceptions; *nexc may exceed cap (overflow: the real path then ships the block unpacked) */
int dvs_debug_pack_host(const uint8_t* src, uint64_t n, uint8_t* packed, uint32_t* exc_pos, uint8_t* exc_val,
                        uint32_t cap, uint32_t* nexc);
/* device evaluation of the glibc-log2 restatement on n doubles */
int dvs_debug_log2(dvs_ctx* ctx, const double* x, double* y, uint64_t n);
/* building blocks of the bounded-error selection kernels: m[i] = a[i] / b[i] by the reciprocal + two
 * fused-remainder steps (must equal IEEE division), l[i] = table path of the glibc log2 restatement,
 * special[i] != 0 where that path does not apply (m near 1, <= 0, subnormal, inf, nan) */
int dvs_debug_fast_terms(dvs_ctx* ctx, const double* a, const double* b, double* m, double* l, int32_t* special,
                         uint64_t n);
/* exact (reference-order) entropy of each host row on the device; err[r]=1 when the reference
 * would panic (sum check, src/record.rs:101-104) */
int dvs_debug_entropy(dvs_ctx* ctx, const double* rows, uint32_t nrec, uint64_t dim, double* out, uint8_t* err);
/* the difference-form kernel of dvs_euclid_distances_sparse on the given pairs (pairs[2 p], pairs[2 p + 1]) of sp's
 * records: out[p] = sum over the union of the two rows of (fl(c_a/T_a) - fl(c_b/T_b))^2, square-rooted */
int dvs_debug_euclid_sparse_pairs(dvs_ctx* ctx, const dvs_ksparse* sp, const uint32_t* pairs, uint32_t n, double* out);

#ifdef __cplusplus
}
#endif
#endif /* DVS_B200_H */
