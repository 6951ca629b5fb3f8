/*
 * innr_cuda.h -- C-ABI of libinnr_cuda.so: the B200 (sm_100a) device path for innr's batch
 * similarity-search hot path. This is the drop-in boundary a Rust shim crate (`innr-cuda`, see
 * INTEGRATION.md) binds with `extern "C"`; every entry point cites the reference interface
 * (/root/reference, innr 0.6.3) it stands behind.
 *
 * Conventions
 *  - Plain pointers and sizes only. Host buffers are caller-owned; the library copies at upload and
 *    never retains a host pointer. `_dev` entry points take device pointers (and a CUDA stream as
 *    `void*`) so that a host runtime which already owns device memory (torch, a sharded driver) can call
 *    the same kernels without a host round trip.
 *  - Every function returns an `int` status (INNR_OK == 0). No C++ exception crosses the boundary.
 *    The reference panics (assert_eq!) on length/dimension mismatches; the shim asserts before the FFI
 *    call so that panic messages stay identical, and the library answers INNR_EINVAL for the same
 *    conditions. `innr_cuda_last_error()` returns a thread-local message.
 *  - There is no CPU fallback: without a CUDA device every compute entry returns INNR_ECUDA.
 *  - Results follow the reference bit for bit on the scan paths (see DESIGN.md): f32 scores of
 *    batch_dot/l2/cosine/norms and batch_knn* (sequential unfused f32 sum over d), Hamming distances,
 *    u8 asymmetric scores (32 virtual FMA chains), and every returned index (ties -> lower index).
 *    MaxSim is within 1e-5 relative (condition-aware) of the reference.
 *  - Indices: `index_base` is added to local row numbers so a row-sharded corpus reports global
 *    indices; global indices must be < 2^32 - 1 (the reference truncates ids to u32 at
 *    src/batch.rs:403).
 *  - Thread safety: a corpus handle is immutable after upload. The host side of every call is serialised per
 *    device by an internal mutex; calls on different devices run concurrently from different threads.
 *  - Stream ordering of `_dev` entries: they enqueue on the CALLER's stream and return while the work is in
 *    flight. Each device has two internal workspaces. The fused k <= 128 scans (`*_keys_dev` without the
 *    tensor-core filter) need only a workspace and may take either, so two such calls on two streams overlap
 *    on the device; every other `_dev` call and every host-facing call uses the first workspace plus the
 *    scratch buffers. The library orders users of the same workspace with events: a call never observes
 *    another call's partial state, whatever streams the caller uses. Inputs and outputs follow the usual
 *    CUDA rule: they belong to the stream they were passed with until that stream has run the call.
 */
#ifndef INNR_CUDA_H
#define INNR_CUDA_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define INNR_OK 0
#define INNR_EINVAL 1       /* dimension / length mismatch, bad argument (reference: panic) */
#define INNR_ECUDA 2        /* CUDA runtime failure or no device */
#define INNR_ENOMEM 3       /* device or host allocation failed */
#define INNR_EUNSUPPORTED 4 /* shape outside what the kernels cover (message says which) */
#define INNR_EBUSY 5        /* both asynchronous slots of the device are in flight: wait for a ticket first */

/* metric selector for the f32 PDX scans */
#define INNR_METRIC_DOT 0    /* batch_dot / batch_knn_dot        src/batch.rs:270, :742 */
#define INNR_METRIC_COSINE 1 /* batch_cosine / batch_knn_cosine  src/batch.rs:690, :777 */
#define INNR_METRIC_L2 2     /* batch_l2_squared / batch_knn     src/batch.rs:236, :385 */

typedef struct innr_cuda_corpus innr_cuda_corpus; /* opaque, device-resident shard */

/* ---- library / device ---------------------------------------------------------------------- */
int innr_cuda_device_count(int* out_count);
/* Binds the calling thread's subsequent calls to `device` and creates its stream/workspace. */
int innr_cuda_init(int device);
int innr_cuda_shutdown(void);
const char* innr_cuda_last_error(void);
/* Display string of the new `Backend::Cuda` variant (src/backend.rs:18-41: `#[non_exhaustive]` enum,
 * Display strings are a stability contract) -> "cuda". */
const char* innr_cuda_backend_name(void);
/* Device-side analogue of backend::dense_backend(len) (src/backend.rs:46): for a device-resident corpus
 * every length answers 1 (= Backend::Cuda); kept as a function so the shim mirrors the predicate shape. */
int innr_cuda_dense_backend(size_t len, int* out_is_cuda);
/* Tuning knobs (process-wide). Names: "knn_tc" (1/0: tensor-core filter path for large dot/cosine query batches),
 * "knn_tc_min_n" (corpus size from which it is used, default 100000), "knn_tc_min_queries" (default 2; 1 sends single queries through the filter too),
 * "maxsim_tc" (1/0: tcgen05 MaxSim when dim <= 128 is a multiple of 4), "u8_scaled_chains" (1/0: PRMT + FFMA2
 * chains scaled by 2^-23 in the u8 scan when the query allows it), "kernel_timing" (1/0, default 0: host-facing calls
 * bracket their kernels with timed CUDA events for innr_cuda_last_kernel_ms). Results never depend on them. */
int innr_cuda_set_option(const char* name, double value);
/* Statistics of the most recent batch_knn call that went through the tensor-core filter (csrc/knn_tc.cu): time of the
 * whole-corpus filter pass and of the whole device-side call (CUDA events), flops issued by that pass, number of
 * (query, vector) pairs re-scored exactly, queries answered by the exact scan instead, filter passes. Any pointer may be
 * NULL. bench.py's tensor roofline reads this. */
int innr_cuda_knn_tc_last_stats(float* out_filter_ms, float* out_total_ms, double* out_filter_flops,
                                uint64_t* out_candidates, uint32_t* out_exact_scan_queries, int* out_passes);
/* Test hook for the filter's error bound: runs the operands + the dense first pass of the filter and returns, for every
 * query and every row < min(n, 4096), the pair's LOWER bound exactly as production computes it (row-major n_queries x
 * *out_rows), eps, and per query 1 when the filter does not answer it (zero / non-finite norm). The tests assert
 * lower <= reference score (in the filter's units) <= lower + 2 * eps * r on adversarial inputs. Needs >= 4096 rows. */
int innr_cuda_knn_tc_debug_bounds(const innr_cuda_corpus* c, int metric, const float* queries, size_t n_queries,
                                  size_t query_len, float* out_lower, size_t* out_rows, float* out_eps,
                                  uint32_t* out_qflags);
/* Test hook for the screened single-query kNN of a split corpus: the interval [lower, upper] the screen gives every row
 * for this query, exactly as production computes it (n floats each). The tests assert lower <= reference score <= upper
 * on adversarial rows. INNR_EUNSUPPORTED when the corpus is not split, has a non-finite row or the query cannot be
 * screened (norm not finite or above 2^100, largest element outside [2^-100, 2^100]; cosine: norm below the
 * reference's epsilon). */
int innr_cuda_knn_screen_debug_bounds(const innr_cuda_corpus* c, int metric, const float* query, size_t query_len,
                                      float* out_lower, float* out_upper);
/* number of kernels the library has launched so far (bench.py's gpu_launches counter) */
int innr_cuda_launch_count(uint64_t* out_count);

/* ---- f32 VerticalBatch (PDX) corpus: src/batch.rs:88-220 ------------------------------------- */
/* Owned corpora of at least f32_split_min_rows rows (innr_cuda_set_option; default 1,000,000) are stored split: the
 * same bytes as two 16-bit planes (high halves, then low halves, same pitch), plus an 8-bit sketch of every element
 * (one byte per element plus 8 bytes per row: +25 % device memory, 7.68 GB for 10M x 768), which lets a single-query
 * kNN read only the sketch before it rescores a few dozen rows exactly. Every entry gives the same bits on either
 * layout; corpus_info's ld and device_bytes (the f32 matrix alone) keep their meaning. Wrapped device memory stays as
 * the caller laid it out. */
/* host_pdx: the buffer VerticalBatch::data() returns (src/batch.rs:212): data[d*n + i]. */
int innr_cuda_upload_f32_pdx(const float* host_pdx, size_t n, size_t d, uint64_t index_base,
                             innr_cuda_corpus** out);
/* host_rows: row-major n x d (VerticalBatch::from_flat input, src/batch.rs:167); transposed on device. */
int innr_cuda_upload_f32_rows(const float* host_rows, size_t n, size_t d, uint64_t index_base,
                              innr_cuda_corpus** out);
/* Non-owning view over device memory already in PDX layout with row pitch `ld` floats
 * (ld >= n, ld % 4 == 0, base 16-byte aligned): dev_pdx[dd*ld + i]. */
int innr_cuda_wrap_f32_pdx_dev(const float* dev_pdx, size_t n, size_t d, size_t ld, uint64_t index_base,
                               innr_cuda_corpus** out);
/* Matryoshka prefix scans (src/dense.rs:436-462 are the pairwise matryoshka_dot / matryoshka_cosine): a zero-copy view of
 * the first min(prefix_dim, d) dimensions of every vector -- in the PDX layout those are simply the first rows. Every
 * f32 entry works on the view and matches the reference's batch function on the truncated vectors. The view does not
 * own device memory: free it before the corpus it was taken from. */
int innr_cuda_prefix_view(const innr_cuda_corpus* c, size_t prefix_dim, innr_cuda_corpus** out);
/* Synthetic corpus generated on the device (SURVEY.md 8d):
 * generator 0 = G-hash: row r, dim j -> splitmix64(salt + r*d + j) (uniform [-1,1), 24-bit);
 * generator 1 = G-ref : row r = generate_embedding(d, seed = salt + r) (examples/batch_demo.rs:233-242).
 * Rows are [first_row, first_row + n). */
int innr_cuda_generate_f32_pdx(int generator, uint64_t salt, uint64_t first_row, size_t n, size_t d,
                               uint64_t index_base, innr_cuda_corpus** out);
int innr_cuda_free(innr_cuda_corpus* c);
/* kind: 0 f32 pdx, 1 binary codes, 2 u8 codes, 3 token matrix */
int innr_cuda_corpus_info(const innr_cuda_corpus* c, int* kind, size_t* n, size_t* d, size_t* ld,
                          uint64_t* index_base, size_t* device_bytes);
/* copies vector i (local index) back to the host: VerticalBatch::extract_vector, src/batch.rs:217 */
int innr_cuda_extract_vector(const innr_cuda_corpus* c, size_t i, float* out_host);

/* ---- full score vectors: batch_dot / batch_l2_squared / batch_norms / batch_cosine --------------- */
/* query: host, query_len must equal d (src/batch.rs:251, :285). out_host: n floats. */
int innr_cuda_batch_dot(const innr_cuda_corpus* c, const float* query, size_t query_len, float* out_host);
int innr_cuda_batch_l2_squared(const innr_cuda_corpus* c, const float* query, size_t query_len,
                               float* out_host);
int innr_cuda_batch_norms(const innr_cuda_corpus* c, float* out_host);
/* norms: caller-supplied, norms_len must equal n (src/batch.rs:711) */
int innr_cuda_batch_cosine(const innr_cuda_corpus* c, const float* query, size_t query_len,
                           const float* norms, size_t norms_len, float* out_host);

/* ---- kNN with fused top-k: batch_knn / batch_knn_dot / batch_knn_cosine -------------------------- */
/* queries: host, n_queries x d row-major. Writes min(k, n) results per query at stride k into out_idx /
 * out_score (row-major n_queries x k) and the per-query count into *out_count. n == 0 or k == 0 -> count 0.
 * Order: dot/cosine descending, L2 ascending; ties -> lower index (stable sort, src/batch.rs:756-758). */
int innr_cuda_batch_knn(const innr_cuda_corpus* c, int metric, const float* queries, size_t n_queries,
                        size_t query_len, size_t k, uint64_t* out_idx, float* out_score, size_t* out_count);
/* batch_knn_filtered (src/batch.rs:820-882). The reference takes a closure `Fn(usize) -> bool`; closures cannot cross
 * the ABI, so the shim evaluates it into a bitmask first (the reference materialises `mask: Vec<bool>` itself, :839):
 * bit i of mask_words[i / 64], LSB first. L2 distances of the passing vectors only (rows of rejected vectors are not
 * read), stable ascending order, k clamped to the number of passing vectors; indices are positions in the batch. */
int innr_cuda_batch_knn_filtered(const innr_cuda_corpus* c, const float* query, size_t query_len, size_t k,
                                 const uint64_t* mask_words, size_t mask_len_words, uint64_t* out_idx,
                                 float* out_score, size_t* out_count);
/* batch_l2_squared_pruning (src/batch.rs:320-365): every vector none of whose partial squared distances (dimension by
 * dimension, as the reference accumulates them) exceeded `threshold`, as (index, full squared distance) pairs in
 * ascending index order. Writes min(*out_count, capacity) pairs; *out_count is the number of survivors. */
int innr_cuda_batch_l2_squared_pruning(const innr_cuda_corpus* c, const float* query, size_t query_len, float threshold,
                                       uint64_t* out_idx, float* out_dist, size_t capacity, size_t* out_count);
/* batch_dimension_variance (src/batch.rs:572-592): out[dd] = variance of dimension row dd over the batch's vectors (mean
 * and sum of squared deviations as the reference's sequential f32 sums, bit for bit); zeros when the batch holds <= 1
 * vector. out_len must equal the batch dimension. Computed once per corpus handle (the corpus is immutable). */
int innr_cuda_batch_dimension_variance(const innr_cuda_corpus* c, float* out, size_t out_len);
/* batch_knn_reordered (src/batch.rs:621-659): exact L2 kNN whose distances are accumulated over the dimensions in
 * decreasing-variance order (variance_order :599-603: stable under f32::total_cmp), then the reference's stable
 * ascending sort -- ties -> lower index; scores bit-identical to the reference's (they differ from batch_knn's in the
 * last bits because the summation order differs). k clamped to N; N == 0 or k == 0 -> empty. */
int innr_cuda_batch_knn_reordered(const innr_cuda_corpus* c, const float* query, size_t query_len, size_t k,
                                  uint64_t* out_idx, float* out_score, size_t* out_count);
/* batch_knn_adaptive (src/batch.rs:441-564): the reference's APPROXIMATE early-termination L2 kNN -- warm-up over the
 * first warmup_dims dimensions, a threshold extrapolated from the k-th partial distance, pruning dimension by
 * dimension (never below k candidates) with the threshold refreshed after every 32nd dimension. Reproduced exactly:
 * the same candidates survive, with their complete distances, in the reference's stable ascending order. Rows of
 * pruned vectors are not read. warmup_dims == 0 -> INNR_EINVAL ("warmup_dims must be > 0", the reference's assert). */
int innr_cuda_batch_knn_adaptive(const innr_cuda_corpus* c, const float* query, size_t query_len, size_t k,
                                 size_t warmup_dims, uint64_t* out_idx, float* out_score, size_t* out_count);
/* Re-rank stage of the reference's documented two-stage retrieval (src/scalar.rs:366-368 "Re-rank top candidates with
 * exact batch_knn_dot", examples/binary_demo.rs:235-237 "binary retrieves top-1000 candidates, then rerank"): the exact
 * batch_knn (L2) / batch_knn_dot / batch_knn_cosine result over the sub-batch formed by `candidates` (distinct global
 * indices), with the original indices reported; scores bit-identical to the full scan's, ties -> lower index. */
int innr_cuda_batch_knn_subset(const innr_cuda_corpus* c, int metric, const float* query, size_t query_len,
                               const uint64_t* candidates, size_t n_candidates, size_t k, uint64_t* out_idx,
                               float* out_score, size_t* out_count);
/* Device-pointer form used for row-sharded corpora: writes the shard's local top-k as sorted 64-bit
 * composite keys (n_queries x k, padded with 0xFFFF...F) into dev_keys on `stream`. Keys from all shards
 * are exchanged by the caller (one allgather) and merged with innr_cuda_merge_keys_dev. */
int innr_cuda_batch_knn_keys_dev(const innr_cuda_corpus* c, int metric, const float* dev_queries,
                                 size_t n_queries, size_t k, uint64_t* dev_keys, void* stream);
/* dev_keys_in: n_lists x n_queries x k sorted key lists. Writes the merged top-k per query as keys
 * (dev_keys_out, may be NULL) and decoded (dev_idx u64, dev_score f32; either may be NULL).
 * metric selects the key decoding (descending for dot/cosine, ascending for L2). */
int innr_cuda_merge_keys_dev(const uint64_t* dev_keys_in, size_t n_lists, size_t n_queries, size_t k,
                             int metric, uint64_t* dev_keys_out, uint64_t* dev_idx, float* dev_score,
                             void* stream);

/* ---- TopK (src/topk.rs:47-187) as one fused selection ------------------------------------------- */
/* Equivalent to inserting (id = i, distances[i]) for i = 0..n-1 and calling into_sorted(): the k smallest
 * by (total_cmp(distance), id). Exact ties at the boundary: see DESIGN.md (row T). */
int innr_cuda_topk_from_distances(const float* distances, size_t n, size_t k, uint32_t* out_id,
                                  float* out_distance, size_t* out_count);

/* ---- packed binary codes: src/binary.rs:37-165 -------------------------------------------------- */
/* words: host, n x ceil(dim_bits/64) u64 (PackedBinary::data(), LSB-first). Padding bits of the last word
 * are masked on upload (PackedBinary::new, src/binary.rs:59-66). */
int innr_cuda_upload_binary(const uint64_t* words, size_t n, size_t dim_bits, uint64_t index_base,
                            innr_cuda_corpus** out);
/* generator: word w of code r = splitmix64(salt + r*words + w) */
int innr_cuda_generate_binary(uint64_t salt, uint64_t first_row, size_t n, size_t dim_bits,
                              uint64_t index_base, innr_cuda_corpus** out);
/* encode_binary (src/binary.rs:133-141: bit = v > threshold) of every vector of a device-resident f32 corpus, without
 * a host round trip; the code set inherits the corpus' index_base (SURVEY 8f row 2: one ingest, several encodings). */
int innr_cuda_binary_from_f32(const innr_cuda_corpus* f32_corpus, float threshold, innr_cuda_corpus** out);
/* binary_hamming (src/binary.rs:154) of the query against every code: out_host n x u32. query_dim_bits
 * must equal the corpus dimension (src/binary.rs:155-159). */
int innr_cuda_hamming_all(const innr_cuda_corpus* c, const uint64_t* query_words, size_t query_dim_bits,
                          uint32_t* out_host);
/* binary_dot (src/binary.rs:178-185: sum of popcount(a & b)) and binary_jaccard (:198-213: intersection as f32 /
 * union as f32, 1.0 for an empty union) of one query code against every code of the corpus. Exact. */
int innr_cuda_binary_dot_all(const innr_cuda_corpus* c, const uint64_t* query_words, size_t query_dim_bits,
                             uint32_t* out_host);
int innr_cuda_binary_jaccard_all(const innr_cuda_corpus* c, const uint64_t* query_words, size_t query_dim_bits,
                                 float* out_host);
/* Top-k by similarity over a code set: op 0 = binary_dot (src/binary.rs:178), 1 = binary_jaccard (:198), descending, ties
 * -> lower index (the caller composition of examples/binary_demo.rs:174-180 applied to the two similarities). Scores as
 * f32 (dot counts are exact). */
int innr_cuda_binary_topk(const innr_cuda_corpus* c, int op, const uint64_t* query_words, size_t query_dim_bits, size_t k,
                          uint64_t* out_idx, float* out_score, size_t* out_count);
/* caller composition examples/binary_demo.rs:174-180: all distances, stable sort_by_key, take(k). */
int innr_cuda_hamming_topk(const innr_cuda_corpus* c, const uint64_t* query_words, size_t n_queries,
                           size_t query_dim_bits, size_t k, uint64_t* out_idx, uint32_t* out_dist,
                           size_t* out_count);
int innr_cuda_hamming_topk_keys_dev(const innr_cuda_corpus* c, const uint64_t* dev_query_words,
                                    size_t n_queries, size_t k, uint64_t* dev_keys, void* stream);
/* encode_binary (src/binary.rs:133-141): bit i = values[i] > threshold; out_words ceil(n/64) u64 */
int innr_cuda_encode_binary(const float* values, size_t n, float threshold, uint64_t* out_words);

/* ---- packed ternary codes: src/ternary.rs (2 bits per value: 01 = +1, 10 = -1; 32 values per u64) -------- */
/* words: host, n x ceil(dimension/32) u64 (PackedTernary::data()); padding pairs of the last word are masked on upload
 * (PackedTernary::new, src/ternary.rs:72-79). */
int innr_cuda_upload_ternary(const uint64_t* words, size_t n, size_t dimension, uint64_t index_base,
                             innr_cuda_corpus** out);
/* encode_ternary (src/ternary.rs:163-173: v > t -> +1, v < -t -> -1) of every vector of a device-resident f32 corpus */
int innr_cuda_ternary_from_f32(const innr_cuda_corpus* f32_corpus, float threshold, innr_cuda_corpus** out);
/* encode_ternary of a flat host array: out_words = ceil(n/32) u64 */
int innr_cuda_encode_ternary(const float* values, size_t n, float threshold, uint64_t* out_words);
/* One query against every code. op 0: ternary_dot (:191, query = packed words, i32 result), 1: ternary_hamming (:301,
 * packed words, u32 result), 2: ternary::asymmetric_dot (:286, query = f32[dimension], sequential unfused f32 sum,
 * bit-exact). query_dim must equal the corpus dimension. Scores are written as f32 (out_f32_host) and / or, for the
 * integer ops, as i32 (out_i32_host); either may be NULL. */
#define INNR_TERNARY_DOT 0
#define INNR_TERNARY_HAMMING 1
#define INNR_TERNARY_ASYMMETRIC_DOT 2
int innr_cuda_ternary_scores_all(const innr_cuda_corpus* c, int op, const void* query, size_t query_dim,
                                 float* out_f32_host, int32_t* out_i32_host);
/* top-k of those scores (dot / asymmetric dot descending, Hamming ascending; ties -> lower index), any k <= n */
int innr_cuda_ternary_topk(const innr_cuda_corpus* c, int op, const void* query, size_t query_dim, size_t k,
                           uint64_t* out_idx, float* out_score, size_t* out_count);

/* ---- scalar-quantised u8 codes: src/scalar.rs:44-393 --------------------------------------------- */
/* rows: host, n x d bytes (each QuantizedU8::data() packed contiguously by the shim). */
int innr_cuda_upload_u8(const uint8_t* rows, size_t n, size_t d, float alpha, float offset,
                        uint64_t index_base, innr_cuda_corpus** out);
/* G-hash f32 rows (salt + r*d + j) quantised on the device with quantize_u8's formula (src/scalar.rs:212-225) */
int innr_cuda_generate_u8(uint64_t salt, uint64_t first_row, size_t n, size_t d, float alpha, float offset,
                          uint64_t index_base, innr_cuda_corpus** out);
/* quantize_u8 (src/scalar.rs:212-225) of every vector of a device-resident f32 corpus, without a host round trip. */
int innr_cuda_u8_from_f32(const innr_cuda_corpus* f32_corpus, float alpha, float offset, innr_cuda_corpus** out);
/* quantize_u8 (src/scalar.rs:212-225) of a host f32 buffer */
int innr_cuda_quantize_u8(const float* values, size_t n, float alpha, float offset, uint8_t* out_codes);
/* mixed_dot_u8_f32 (src/scalar.rs:314) of the query against every row: out_host n floats */
int innr_cuda_mixed_dot_u8_all(const innr_cuda_corpus* c, const float* query, size_t query_len,
                               float* out_host);
/* asymmetric_dot_u8 (src/scalar.rs:261-300) of the query against every row */
int innr_cuda_asymmetric_dot_u8_all(const innr_cuda_corpus* c, const float* query, size_t query_len,
                                    float* out_host);
/* batch_knn_u8 (src/scalar.rs:370-393): descending, ties -> lower index */
int innr_cuda_batch_knn_u8(const innr_cuda_corpus* c, const float* queries, size_t n_queries,
                           size_t query_len, size_t k, uint64_t* out_idx, float* out_score,
                           size_t* out_count);
int innr_cuda_batch_knn_u8_keys_dev(const innr_cuda_corpus* c, const float* dev_queries, size_t n_queries,
                                    size_t k, uint64_t* dev_keys, void* stream);

/* ---- ColBERT MaxSim over a document set: src/maxsim.rs:96-194 ------------------------------------ */
/* tokens: host, total_tokens x dim row-major; doc j owns rows [doc_offsets[j], doc_offsets[j+1]). */
int innr_cuda_upload_tokens(const float* tokens, const uint64_t* doc_offsets, size_t n_docs, size_t dim,
                            uint64_t index_base, innr_cuda_corpus** out);
/* G-hash token rows (salt + row*dim + j), every doc `tokens_per_doc` tokens; docs [first_doc, first_doc+n_docs) */
int innr_cuda_generate_tokens(uint64_t salt, uint64_t first_doc, size_t n_docs, size_t tokens_per_doc,
                              size_t dim, uint64_t index_base, innr_cuda_corpus** out);
/* A batch of queries against the document set (the caller loop of examples/maxsim_colbert.rs:171-174, for several
 * queries): q_tokens is n_queries x n_q x q_dim, out_scores n_queries x n_docs (query-major). Same per-query results
 * as innr_cuda_maxsim; on the tcgen05 path two queries of <= 32 tokens share every pass over the corpus. */
int innr_cuda_maxsim_batch(const innr_cuda_corpus* c, const float* q_tokens, size_t n_queries, size_t n_q, size_t q_dim,
                           int cosine_flag, float* out_scores_host);
int innr_cuda_maxsim_batch_dev(const innr_cuda_corpus* c, const float* dev_q_tokens, size_t n_queries, size_t n_q,
                               int cosine_flag, float* dev_scores, void* stream);
/* maxsim (cosine_flag 0) / maxsim_cosine (1) of the query token set against every doc:
 * out_scores_host n_docs floats. Empty query or empty doc -> 0.0 (src/maxsim.rs:97-99). q_dim must equal dim. */
int innr_cuda_maxsim(const innr_cuda_corpus* c, const float* q_tokens, size_t n_q, size_t q_dim,
                     int cosine_flag, float* out_scores_host);
int innr_cuda_maxsim_dev(const innr_cuda_corpus* c, const float* dev_q_tokens, size_t n_q, int cosine_flag,
                         float* dev_scores, void* stream);

/* ---- cross-GPU exchange of per-shard top-k lists without a collective library (SURVEY 8e; csrc/exchange.cu) ---------
 * Every rank owns a small mailbox in its device memory and maps every peer's (CUDA IPC between processes,
 * peer access inside one process). innr_cuda_exchange_merge_dev is ONE kernel launch: it publishes this rank's sorted
 * key lists into all mailboxes over NVLink, raises a flag, waits for the peers' flags and merges the n_ranks lists --
 * every rank obtains the same merged top-k (what ncclAllGather + innr_cuda_merge_keys_dev produce, in one launch and
 * without NCCL). All ranks must make the same sequence of calls with the same (n_queries, k). k <= 128 and
 * n_queries * k <= slot_keys; larger requests: gather the lists yourself and use innr_cuda_merge_keys_dev. */
typedef struct innr_cuda_exchange innr_cuda_exchange;
/* on the calling thread's device (innr_cuda_init); slot_keys == 0 -> 16384 keys per rank and call */
int innr_cuda_exchange_create(int n_ranks, int rank, size_t slot_keys, innr_cuda_exchange** out);
/* 64-byte cudaIpcMemHandle_t of this rank's mailbox, to be handed to the other processes */
int innr_cuda_exchange_ipc_handle(const innr_cuda_exchange* ex, void* out_handle64);
/* handles: n_ranks x 64 bytes in rank order (the own entry is ignored) */
int innr_cuda_exchange_connect_ipc(innr_cuda_exchange* ex, const void* handles);
/* ranks 0..n_ranks-1 living in THIS process (possibly on different devices): enables peer access and connects them all */
int innr_cuda_exchange_connect_local(innr_cuda_exchange* const* all, int n_ranks);
int innr_cuda_exchange_free(innr_cuda_exchange* ex);
/* a call whose peers do not publish within the timeout (default 10 s) gives up and sets the status to 1 */
int innr_cuda_exchange_set_timeout_ms(innr_cuda_exchange* ex, double ms);
int innr_cuda_exchange_status(innr_cuda_exchange* ex, int* out_status);
/* dev_local_keys: n_queries x k sorted keys of this rank's shard (what the *_keys_dev entries write). Outputs (device,
 * any may be NULL): merged keys, indices (u64), scores decoded for `metric` (f32), key high halves (u32: Hamming
 * distances). publish_only != 0: publish and return without waiting or merging (ranks that do not need the result). */
int innr_cuda_exchange_merge_dev(innr_cuda_exchange* ex, const uint64_t* dev_local_keys, size_t n_queries, size_t k,
                                 int metric, int publish_only, uint64_t* dev_keys_out, uint64_t* dev_idx,
                                 float* dev_score, uint32_t* dev_dist, void* stream);

/* ---- one process, several GPUs (SURVEY 8e) ---------------------------------------------------------------------------
 * Row shards living on different devices (created after innr_cuda_init(device) on the creating thread, each with
 * index_base = its first global row). The call runs one host thread per shard -- calls on different devices do not
 * serialise -- and merges the k keys per shard on the host in the device's own key order, so results equal the
 * unsharded call (lower global index wins across shards). No collective library is involved. */
int innr_cuda_batch_knn_sharded(const innr_cuda_corpus* const* shards, size_t n_shards, int metric, const float* queries,
                                size_t n_queries, size_t query_len, size_t k, uint64_t* out_idx, float* out_score,
                                size_t* out_count);
int innr_cuda_hamming_topk_sharded(const innr_cuda_corpus* const* shards, size_t n_shards, const uint64_t* query_words,
                                   size_t n_queries, size_t query_dim_bits, size_t k, uint64_t* out_idx,
                                   uint32_t* out_dist, size_t* out_count);
int innr_cuda_batch_knn_u8_sharded(const innr_cuda_corpus* const* shards, size_t n_shards, const float* queries,
                                   size_t n_queries, size_t query_len, size_t k, uint64_t* out_idx, float* out_score,
                                   size_t* out_count);
/* ---- asynchronous host-buffer top-k ------------------------------------------------------------------------
 * The entries above synchronise before they return. These queue the same call -- same arguments, same checks, same
 * results -- and hand back a ticket; innr_cuda_ticket_wait blocks until THAT call is complete, writes min(k, N)
 * results per query at row stride k like the synchronous entry (f32 / u8 corpora: out_score, out_dist may be NULL;
 * binary corpora: out_dist, out_score may be NULL) and releases the ticket. The queries are copied before the call
 * returns (the caller may reuse its buffer at once). At most TWO tickets per device may be in flight (a third submit
 * fails with INNR_EBUSY): submit(i + 1) before wait(i) keeps two shard scans overlapping on the device, which is what
 * hides the ramp at both ends of a launch (DESIGN.md section 6). Tickets belong to the library; a ticket is invalid
 * after its wait (and after innr_cuda_shutdown); the corpus must stay alive until the ticket has been waited for. */
typedef struct innr_cuda_ticket innr_cuda_ticket;
int innr_cuda_batch_knn_async(const innr_cuda_corpus* c, int metric, const float* queries, size_t n_queries,
                              size_t query_len, size_t k, innr_cuda_ticket** out_ticket);
int innr_cuda_hamming_topk_async(const innr_cuda_corpus* c, const uint64_t* query_words, size_t n_queries,
                                 size_t query_dim_bits, size_t k, innr_cuda_ticket** out_ticket);
int innr_cuda_batch_knn_u8_async(const innr_cuda_corpus* c, const float* queries, size_t n_queries, size_t query_len,
                                 size_t k, innr_cuda_ticket** out_ticket);
int innr_cuda_ticket_wait(innr_cuda_ticket* t, uint64_t* out_idx, float* out_score, uint32_t* out_dist,
                          size_t* out_count);
/* The same for row shards on pairwise distinct devices (the peer-mapped exchange route of the *_sharded entries):
 * every device queues its shard scan and its part of the exchange without any host synchronisation, the root's merged
 * keys come back through pinned memory, and ONE ticket stands for the whole call. Two calls per device group may be in
 * flight. *out_ticket stays NULL (status INNR_OK) when the result is empty (no rows, k == 0 or no queries).
 * INNR_EUNSUPPORTED where the exchange route does not apply (shards sharing a device, no peer access, k > 128, a batch
 * larger than the mailboxes): use the synchronous entry. While asynchronous sharded calls are in flight the synchronous
 * sharded entries on the same devices return INNR_EBUSY. */
int innr_cuda_batch_knn_sharded_async(const innr_cuda_corpus* const* shards, size_t n_shards, int metric,
                                      const float* queries, size_t n_queries, size_t query_len, size_t k,
                                      innr_cuda_ticket** out_ticket);
int innr_cuda_hamming_topk_sharded_async(const innr_cuda_corpus* const* shards, size_t n_shards,
                                         const uint64_t* query_words, size_t n_queries, size_t query_dim_bits,
                                         size_t k, innr_cuda_ticket** out_ticket);
int innr_cuda_batch_knn_u8_sharded_async(const innr_cuda_corpus* const* shards, size_t n_shards, const float* queries,
                                         size_t n_queries, size_t query_len, size_t k, innr_cuda_ticket** out_ticket);

/* ---- timing hook: device time (ms) of the last host-facing call's kernels, measured with CUDA events on the
 *      launching stream. Off by default (the two timed event records cost a short call ~15 us): enable with
 *      innr_cuda_set_option("kernel_timing", 1); 0 until then. ------------------------------------------------- */
int innr_cuda_last_kernel_ms(float* out_ms);

#ifdef __cplusplus
}
#endif
#endif /* INNR_CUDA_H */
