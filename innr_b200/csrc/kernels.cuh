// kernels.cuh -- launcher prototypes shared between the kernel translation units and the C-ABI (api.cu).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include <atomic>
#include <vector>

namespace innr {

using LaunchCounter = std::atomic<uint64_t>;  // kernels launched so far (all devices, all threads)

// modes of the f32 PDX scan (scan_f32.cu)
enum PdxMode : int {
  PDX_DOT = 0,          // batch_dot_into            src/batch.rs:284-297
  PDX_COSINE_FUSED = 1, // batch_norms + batch_cosine in ONE pass (knn)  src/batch.rs:672-686, 705-728
  PDX_L2 = 2,           // batch_l2_squared_into     src/batch.rs:250-266
  PDX_NORMS = 3,        // batch_norms_into          src/batch.rs:672-686
  PDX_COSINE_NORMS = 4, // batch_cosine_into with caller-supplied norms  src/batch.rs:705-728
  PDX_L2_PRUNE = 5,     // batch_l2_squared_pruning  src/batch.rs:320-365 (scores mode: pruned vectors -> -1.0)
  PDX_L2_PERM = 6,      // batch_knn_reordered  src/batch.rs:621-659 (L2 summed over a permutation of the dimension rows)
};

struct Workspace {
  uint64_t* partials = nullptr;        // per-CTA top-k lists
  size_t partials_cap = 0;             // in u64
  uint64_t* group_partials = nullptr;  // per-group (32 CTAs) merged lists
  size_t group_cap = 0;                // in u64
  unsigned* tickets = nullptr;         // [0] top level, [1+g] group g; zeroed once, self-resetting
  size_t tickets_cap = 0;
  unsigned long long* shared_thr = nullptr;  // launch-wide bound on the k-th key (common.cuh: SharedThreshold); all ones between launches
  int num_sms = 0;
  // screened single-query kNN (launch_pdx_knn_screened): one optimistic bound per row, the candidate list and its
  // ready-made keys, the k keys of the pessimistic bounds, and ctl = {candidate count, "the exact scan answers" flag}
  float* sc_bounds = nullptr;
  size_t sc_bounds_cap = 0;  // in floats
  uint32_t* sc_cand = nullptr;
  uint64_t* sc_keys = nullptr;
  unsigned* sc_ctl = nullptr;
};

// Persistent grids stride tiles by gridDim: pick the largest grid <= max_ctas for which every CTA gets the same
// number of tiles (+-0), so no CTA runs a whole extra tile while the others idle (matters for small shards).
inline unsigned balanced_grid(unsigned n_tiles, unsigned max_ctas) {
  if (n_tiles == 0 || max_ctas == 0) return 1;
  if (n_tiles <= max_ctas) return n_tiles;
  unsigned waves = (n_tiles + max_ctas - 1) / max_ctas;
  return (n_tiles + waves - 1) / waves;
}

// An f32 corpus in the PDX layout (dimension-major, row pitch ld). Kernels read it through pdx.cuh only: plain corpora
// hold data[dd * ld + i]; split corpora (hi != null) hold the high and low 16 bits of that element at hi[dd * ld + i] and
// lo[dd * ld + i], two planes of one allocation of the plain size.
struct PdxView {
  const float* data;
  size_t n, d, ld;
  uint32_t index_base;
  const uint16_t* hi = nullptr;
  const uint16_t* lo = nullptr;
};
// a corpus being written: data for plain, hi / lo for split (same pitch ld)
struct PdxDst {
  float* data;
  uint16_t* hi;
  uint16_t* lo;
  size_t ld;
  PdxDst at_column(size_t i0) const { return PdxDst{data ? data + i0 : nullptr, hi ? hi + i0 : nullptr, lo ? lo + i0 : nullptr, ld}; }
};

// kNN: queries on device (nq x d row-major); writes nq x k sorted keys (sentinel padded) into dev_keys.
// Returns cudaSuccess or the launch error; `launches` is incremented per kernel launched.
// dev_run_flag (optional): the launch does nothing unless *dev_run_flag != 0 when it starts (read on the device)
cudaError_t launch_pdx_knn(const PdxView& v, int mode, const float* dev_queries, size_t nq, size_t k,
                           uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches,
                           const unsigned* dev_run_flag = nullptr);
// The screened kNN's 8-bit sketch of a split corpus, one allocation built with it (layout.cu, addressing in pdx.cuh):
// codes[dd * ld + i] = 128 + round(x / scale[i]) clamped to [1, 255], scale[i] = absmax_i / 127 (0 for a zero row),
// resid[i] >= || x_i - scale[i] (code_i - 128) ||_2 (rounded outward), for the ld columns of the corpus.
struct PdxSketch {
  uint8_t* codes;
  float* scale;
  float* resid;
};
// Screened single-query kNN of a split corpus (scan_f32.cu): the sketch alone gives every row an interval that holds its
// exact score, the rows whose interval reaches the k-th best pessimistic bound are rescored exactly from both planes.
// Same keys as launch_pdx_knn. Needs the corpus' sidecar (dev_norms and the sketch, all finite), k <= 128,
// d <= SCREEN_MAX_D and ws.sc_* sized for v.ld rows. More than SCREEN_CAP candidates, or a query the screen cannot take
// (norm not finite, largest element outside [2^-100, 2^100], cosine: norm below the reference's epsilon), hand the
// query to the full-read scan, queued behind on the device.
constexpr size_t SCREEN_CAP = 4096;
constexpr size_t SCREEN_MAX_D = 4096;
cudaError_t launch_pdx_knn_screened(const PdxView& v, int mode, const float* dev_norms, const PdxSketch& sk,
                                    const float* dev_query, size_t k, uint64_t* dev_keys, Workspace& ws, cudaStream_t s,
                                    LaunchCounter* launches);
// test hook: the screen's interval [lower, upper] for every row (host arrays of n floats); returns cudaErrorNotSupported
// when the query cannot be screened
cudaError_t launch_pdx_screen_debug_bounds(const PdxView& v, int mode, const float* dev_norms, const PdxSketch& sk,
                                           const float* dev_query, float* host_lower, float* host_upper, Workspace& ws,
                                           cudaStream_t s, LaunchCounter* launches);
// batch_knn_filtered (src/batch.rs:820-882): L2, one query; dev_mask = one bit per local vector (LSB-first u32 words,
// zero padded to ld/32 + 1 words); vectors whose bit is clear are neither read nor offered.
cudaError_t launch_pdx_knn_filtered(const PdxView& v, const float* dev_query, const uint32_t* dev_mask, size_t k,
                                    uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches);
// full score vectors: out[q * ld + i] (device). dev_norms only for PDX_COSINE_NORMS; threshold only for PDX_L2_PRUNE.
cudaError_t launch_pdx_scores(const PdxView& v, int mode, const float* dev_query, const float* dev_norms,
                              float* dev_out, Workspace& ws, cudaStream_t s, LaunchCounter* launches, float threshold = 0.0f,
                              const uint32_t* dev_perm = nullptr);
// batch_knn_reordered (src/batch.rs:621-659): L2 distances accumulated over the dimension rows in the order dev_perm[0..d)
// (a permutation of 0..d, device), ascending keys with ties -> lower index (the reference's stable sort); k <= 128.
cudaError_t launch_pdx_knn_reordered(const PdxView& v, const float* dev_query, const uint32_t* dev_perm, size_t k,
                                     uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches);
// batch_dimension_variance (src/batch.rs:572-592): out[dd] = variance of dimension row dd over the n vectors, each row's
// two sums in the reference's sequential order (one warp per row; the chain of n dependent adds bounds it).
cudaError_t launch_dimension_variance(const PdxView& v, float* dev_out, cudaStream_t s, LaunchCounter* launches);
// stream compaction of a pruned distance vector (entries == -1.0 are dropped): ascending index order.
// Pass 1 (count) fills dev_block_offsets[n_blocks + 1] (exclusive prefix, last = total); pass 2 scatters.
size_t compact_blocks(size_t n);
cudaError_t launch_compact_count(const float* dev_dist, size_t n, unsigned* dev_block_offsets, cudaStream_t s,
                                 LaunchCounter* launches);
cudaError_t launch_compact_scatter(const float* dev_dist, size_t n, uint64_t index_base, const unsigned* dev_block_offsets,
                                   uint64_t* dev_idx, float* dev_out, cudaStream_t s, LaunchCounter* launches);
// merge n_lists x nq x k sorted key lists -> nq x k; optional decode (idx u64, f32 score bits by `descending`)
cudaError_t launch_merge_keys(const uint64_t* dev_in, size_t n_lists, size_t nq, size_t k, int descending,
                              uint64_t* dev_keys_out, uint64_t* dev_idx, float* dev_score, cudaStream_t s,
                              LaunchCounter* launches);
// k smallest keys of a device score vector for ANY k (rounds of <= 128): kind 0 f32 ascending, 1 f32 descending,
// 2 u32 ascending, 3 ready-made keys, 4 u32 descending; ids = index_base + i. Used by every top-k entry when k > 128. dev_mask (one bit per entry, LSB-first
// u32 words) restricts the selection to the entries whose bit is set (batch_knn_filtered with k > 128).
cudaError_t launch_topk_from_scores(const void* dev_scores, int kind, size_t n, uint32_t index_base, size_t k,
                                    uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches,
                                    const uint32_t* dev_ids = nullptr, const uint32_t* dev_mask = nullptr, unsigned seg_len = 1,
                                    unsigned seg_stride = 1);
// the merge for k > 128 (any k): dev_keys_out (nq x k) is required
cudaError_t launch_merge_keys_big(const uint64_t* dev_in, size_t n_lists, size_t nq, size_t k, int descending,
                                  uint64_t* dev_keys_out, uint64_t* dev_idx, float* dev_score, Workspace& ws, cudaStream_t s,
                                  LaunchCounter* launches);
// batch_knn_adaptive (src/batch.rs:441-564), orchestrated by api.cu: see scan_f32.cu
cudaError_t launch_adaptive_threshold(const uint64_t* dev_key, float scale, float* dev_thr, cudaStream_t s,
                                      LaunchCounter* launches);
cudaError_t launch_adaptive_mark(const PdxView& v, const float* dev_dist, float ratio, const float* dev_thr,
                                 uint32_t* dev_mask_out, unsigned* dev_pruned, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_adaptive_epoch(const PdxView& v, const float* dev_query, size_t d0, size_t d1, float* dev_dist,
                                  const uint32_t* dev_mask_in, uint32_t* dev_mask_out, const float* dev_thr, uint32_t* dev_ev,
                                  unsigned* dev_pruned, int no_prune, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_adaptive_event_keys(const uint32_t* dev_before, const uint32_t* dev_after, const uint32_t* dev_ev, size_t n,
                                       uint64_t* dev_keys, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_adaptive_revive(const uint64_t* dev_keys, size_t m, uint32_t* dev_mask, cudaStream_t s,
                                   LaunchCounter* launches);
// exact scores (mode = PDX_DOT / PDX_L2 / PDX_COSINE_FUSED) of m candidate vectors given by GLOBAL id
cudaError_t launch_subset_scores(const PdxView& v, int mode, const float* dev_query, const uint32_t* dev_cand, size_t m,
                                 float* dev_out, cudaStream_t s, LaunchCounter* launches);
// cross-GPU exchange + merge of per-shard top-k lists through peer-mapped mailboxes (exchange.cu)
constexpr int EX_MAX_CTAS = 64;
constexpr int EX_THREADS = 256;
struct ExchangeView {
  uint64_t* mailbox;                 // this rank's mailbox (device memory of this rank)
  uint64_t* const* dev_peer_table;   // device array [n_ranks]: every rank's mailbox as mapped in this process
  int n_ranks, rank;
  size_t slot_keys;                  // capacity of one (parity, rank) slot, in keys
  unsigned* dev_status;              // set to 1 by a call whose peers did not publish within timeout_ns
  uint64_t timeout_ns;
};
size_t exchange_mailbox_bytes(int n_ranks, size_t slot_keys);
// dev_local_keys: nq x k sorted keys (k <= 128, nq * k <= slot_keys). `call` numbers the calls 1, 2, ... identically on
// every rank. Outputs (any may be null): merged keys, indices, f32 scores (decoded by `descending`), u32 high halves.
cudaError_t launch_exchange_merge(const ExchangeView& x, const uint64_t* dev_local_keys, size_t nq, size_t k, uint64_t call,
                                  int publish_only, int descending, uint64_t* dev_keys_out, uint64_t* dev_idx,
                                  float* dev_score, uint32_t* dev_dist, cudaStream_t s, LaunchCounter* launches);
// keys from a plain f32 array (TopK analogue): ascending, id = i
cudaError_t launch_topk_from_distances(const float* dev_dist, size_t n, size_t k, uint64_t* dev_keys,
                                       Workspace& ws, cudaStream_t s, LaunchCounter* launches);

// tensor-core filter path for large query batches (knn_tc.cu): dot / cosine, k <= 32, exact results
struct KnnTcStats {
  float filter_ms = 0, total_ms = 0;   // final (whole-corpus) filter pass; whole device-side call
  double filter_flops = 0;             // flops issued by the final filter pass (2 * rows * padded d * padded queries)
  unsigned long long candidates = 0;   // pairs re-scored exactly
  unsigned overflowed = 0;             // queries answered by the exact scan instead
  int passes = 0;
};
bool knn_tc_supported(const PdxView& v, int mode, size_t nq, size_t k);
size_t knn_tc_dpad(size_t d);  // row pitch (elements) of the f16 operand copy
float knn_tc_eps(size_t d);    // the filter's bound on |S - cosine|
// test hook: lower bounds of the dense first pass (rows < min(n, 4096)) for every query; see knn_tc.cu
cudaError_t launch_knn_tc_debug_bounds(const PdxView& v, const CUtensorMap& tm_xh, const float* dev_norms, int mode,
                                       const float* dev_queries, size_t nq, void* workspace, float* host_lower,
                                       size_t* out_rows, float* out_eps, unsigned* host_qflags, int num_sms, cudaStream_t s,
                                       LaunchCounter* launches);
size_t knn_tc_workspace_bytes(size_t n, size_t d, size_t nq, size_t k);
// once per corpus: dev_xh (n x knn_tc_dpad(d) f16) = unit vectors, from the PDX corpus and its exact norms
cudaError_t launch_knn_tc_build(const PdxView& v, const float* dev_norms, void* dev_xh, unsigned* dev_scratch_u32,
                                CUtensorMap* tm_xh, unsigned* host_nonfinite, cudaStream_t s, LaunchCounter* launches);
// host_counts: pinned buffer of nq unsigned; overflow_queries receives the queries the filter could not answer
// (the caller re-runs them on the exact scan). Synchronises the stream once at the end.
cudaError_t launch_pdx_knn_tc(const PdxView& v, const CUtensorMap& tm_xh, const float* dev_norms, int mode,
                              const float* dev_queries, size_t nq, size_t k, uint64_t* dev_keys, void* workspace,
                              unsigned* host_counts, Workspace& ws, cudaStream_t s, LaunchCounter* launches,
                              std::vector<unsigned>* overflow_queries, KnnTcStats* stats);

// layout / generator kernels (layout.cu)
// n rows (row-major, device) -> columns [0, cols) of dst (cols >= n; columns past n are zero-filled)
cudaError_t launch_transpose_rows_to_pdx(const float* dev_rows, size_t n, size_t d, const PdxDst& dst, size_t cols,
                                         cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_generate_f32_pdx(int generator, uint64_t salt, uint64_t first_row, size_t n, size_t d,
                                    const PdxDst& dst, cudaStream_t s, LaunchCounter* launches);
// `rows` dimension rows of a plain PDX block (row pitch n, device) -> dimension rows [0, rows) of dst (columns past n
// zero-filled up to dst.ld)
cudaError_t launch_pdx_rows_to_dst(const float* dev_src, size_t rows, size_t n, const PdxDst& dst, cudaStream_t s,
                                   LaunchCounter* launches);
// the sketch of a split corpus (PdxSketch) from the corpus and its reference norms (dev_norms, PDX_NORMS bits);
// *dev_nonfinite != 0 when some row's norm, scale or residual bound is not finite
cudaError_t launch_pdx_sketch(const PdxView& v, const float* dev_norms, const PdxSketch& sk, unsigned* dev_nonfinite,
                              cudaStream_t s, LaunchCounter* launches);

// binary codes (hamming.cu): chunk-major layout codes[c * ld + i] (uint4 = 128 bits), chunks = ceil(words/2)
struct BinView {
  const uint4* data;
  size_t n, ld, words, chunks, dim_bits;
  uint32_t index_base;
};
cudaError_t launch_binary_pack(const uint64_t* dev_words_rowmajor, size_t n, size_t words, size_t dim_bits,
                               uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_generate_binary(uint64_t salt, uint64_t first_row, size_t n, size_t words, size_t dim_bits,
                                   uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_hamming_all(const BinView& v, const uint64_t* dev_query_words, uint32_t* dev_out,
                               cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_binary_dot_all(const BinView& v, const uint64_t* dev_query_words, uint32_t* dev_out,
                                  cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_binary_jaccard_all(const BinView& v, const uint64_t* dev_query_words, float* dev_out,
                                      cudaStream_t s, LaunchCounter* launches);
// fused single-pass top-k (k <= 128) by binary_dot (jaccard = 0) / binary_jaccard (1): descending, ties -> lower index
cudaError_t launch_binary_setops_topk(const BinView& v, int jaccard, const uint64_t* dev_query_words, size_t k, uint64_t* dev_keys,
                                      Workspace& ws, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_hamming_topk(const BinView& v, const uint64_t* dev_query_words, size_t nq, size_t k,
                                uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_encode_binary(const float* dev_values, size_t n, float threshold, uint64_t* dev_words,
                                 cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_binary_from_pdx(const PdxView& v, float threshold,
                                   uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches);

// ternary codes (ternary.cu): chunk-major layout codes[c * ld + i] (uint4 = 64 two-bit values), chunks = ceil(dim/64)
struct TerView {
  const uint4* data;
  size_t n, ld, words, chunks, dim;
  uint32_t index_base;
};
cudaError_t launch_ternary_pack(const uint64_t* dev_words_rowmajor, size_t n, size_t words, size_t dim, uint4* dev_codes,
                                size_t ld, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_ternary_from_pdx(const PdxView& v, float threshold, uint4* dev_codes,
                                    size_t ld, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_encode_ternary(const float* dev_values, size_t n, float threshold, uint64_t* dev_words, cudaStream_t s,
                                  LaunchCounter* launches);
// op 0 ternary_dot, 1 ternary_hamming (query = packed words), 2 asymmetric_dot (query = f32); scores as f32 and/or i32
cudaError_t launch_ternary_scores(const TerView& v, int op, const uint64_t* dev_query_words, const float* dev_query,
                                  float* dev_out_f32, int32_t* dev_out_i32, cudaStream_t s, LaunchCounter* launches);

// u8 codes (u8.cu): chunk-major layout codes[c * ld + i] (uint4 = 16 dims), chunks = ceil(d/16)
struct U8View {
  const uint4* data;
  size_t n, d, ld, chunks;
  float alpha, offset;
  uint32_t index_base;
};
cudaError_t launch_u8_pack(const uint8_t* dev_rows, size_t n, size_t d, uint4* dev_codes, size_t ld,
                           cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_generate_u8(uint64_t salt, uint64_t first_row, size_t n, size_t d, float alpha, float offset,
                               uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_quantize_u8(const float* dev_values, size_t n, float alpha, float offset, uint8_t* dev_out,
                               cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_u8_from_pdx(const PdxView& v, float alpha, float offset,
                               uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches);
// mode 0: raw mixed dot, 1: asymmetric score
cudaError_t launch_u8_scores(const U8View& v, int mode, const float* dev_query, float* dev_out,
                             cudaStream_t s, LaunchCounter* launches);
// fused single-pass top-k (k <= 128) of the ternary scores (dot / asymmetric dot descending, Hamming ascending)
cudaError_t launch_ternary_topk(const TerView& v, int op, const uint64_t* dev_query_words, const float* dev_query, size_t k,
                                uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches);
void u8_set_scaled_chains(bool on);  // off = always the de-biasing path (tests compare both)
cudaError_t launch_u8_knn(const U8View& v, const float* dev_queries, size_t nq, size_t k, uint64_t* dev_keys,
                          Workspace& ws, cudaStream_t s, LaunchCounter* launches);

// MaxSim (maxsim.cu)
struct TokView {
  const float* tokens;          // total_tokens x dim row-major
  const uint64_t* doc_offsets;  // n_docs + 1 (device)
  size_t n_docs, dim, total_tokens;
  size_t uniform_tokens;        // > 0 when every doc has exactly this many tokens
  CUtensorMap tmap;             // TMA map over the token matrix (box 32 floats x 32 rows, SWIZZLE_128B)
  bool tmap_valid;
  const float* inv_norms;       // per token 1/||x|| (0 when ||x||^2 <= 1e-18), computed once at upload; may be null
};
// tcgen05 path (maxsim_tc.cu): dim in {32, 64, 96, 128}, 1 <= n_q <= 256 (one corpus pass per 32 query tokens)
bool maxsim_tc_supported(const TokView& v, size_t n_q);
cudaError_t launch_maxsim_tc(const TokView& v, const float* dev_q, size_t n_q, int cosine, float* dev_scores,
                             int num_sms, cudaStream_t s, LaunchCounter* launches);
// batch of n_queries queries of n_q <= 32 tokens each; scores n_queries x n_docs; two queries per corpus pass
cudaError_t launch_maxsim_tc_batch(const TokView& v, const float* dev_q, size_t n_queries, size_t n_q, int cosine,
                                   float* dev_scores, int num_sms, cudaStream_t s, LaunchCounter* launches);
bool make_token_tmap(CUtensorMap* m, const float* dev_tokens, size_t total_tokens, size_t dim);
cudaError_t launch_token_inv_norms(const float* dev_tokens, size_t total_tokens, size_t dim, float* dev_inv,
                                   cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_generate_tokens(uint64_t salt, uint64_t first_row, size_t n_rows, size_t dim, float* dev_tokens,
                                   cudaStream_t s, LaunchCounter* launches);
cudaError_t launch_maxsim(const TokView& v, const float* dev_q, size_t n_q, int cosine, float* dev_scores,
                          cudaStream_t s, LaunchCounter* launches);

}  // namespace innr
