// hamming.cu -- HBM-bound popcount scan over packed binary codes with fused top-k.
//
// Replaces (reference, innr 0.6.3):
//   binary_hamming            src/binary.rs:154-165   (sum of (a ^ b).count_ones() over u64 words)
//   PackedBinary::new masking src/binary.rs:59-66
//   encode_binary             src/binary.rs:133-141   (bit = v > threshold, LSB-first)
//   caller's top-k            examples/binary_demo.rs:174-180 (all distances, stable sort_by_key, take k)
//
// Device layout ("PDX for codes"): 128-bit chunks, chunk-major: codes[c * ld + i] holds words 2c, 2c+1 of
// code i. One thread owns one code; consecutive threads read consecutive 16-byte chunks, so every warp load is
// 512 contiguous bytes and no cross-lane reduction is needed. Integer arithmetic: results are exact.
// Key = (distance << 32) | global index: ascending distance, ties -> lower index == stable sort_by_key.
#include <cstdlib>

#include "common.cuh"
#include "kernels.cuh"
#include "pdx.cuh"

namespace innr {

namespace {

constexpr int HAM_THREADS = 256;

__device__ __forceinline__ unsigned popc_u4(uint4 a, uint4 b) {
  return __popc(a.x ^ b.x) + __popc(a.y ^ b.y) + __popc(a.z ^ b.z) + __popc(a.w ^ b.w);
}

// CHUNKS_CT > 0: compile-time chunk count (fully unrolled, all loads in flight); 0: runtime loop
template <int CHUNKS_CT>
__device__ __forceinline__ unsigned code_distance(const uint4* __restrict__ p, size_t ld, unsigned chunks,
                                                  const uint4* __restrict__ sq) {
  unsigned dist = 0;
  if (CHUNKS_CT > 0) {
    uint4 v[CHUNKS_CT > 0 ? CHUNKS_CT : 1];
#pragma unroll
    for (int c = 0; c < CHUNKS_CT; ++c) v[c] = ldg_stream_u4(p + (size_t)c * ld);
#pragma unroll
    for (int c = 0; c < CHUNKS_CT; ++c) dist += popc_u4(v[c], sq[c]);
  } else {
    unsigned c = 0;
    for (; c + 4 <= chunks; c += 4) {
      uint4 v[4];
#pragma unroll
      for (int u = 0; u < 4; ++u) v[u] = ldg_stream_u4(p + (size_t)(c + u) * ld);
#pragma unroll
      for (int u = 0; u < 4; ++u) dist += popc_u4(v[u], sq[c + u]);
    }
    for (; c < chunks; ++c) dist += popc_u4(ldg_stream_u4(p + (size_t)c * ld), sq[c]);
  }
  return dist;
}

// popcount of 32 words through a Harley-Seal carry-save adder tree: 30 full adders (2 LOP3 each) leave 6 POPCs
// instead of 32. POPC issues at a quarter of the LOP3 rate (16 / clk / SM measured through the 4-query kernel), and the
// batched kernels are bound by exactly that pipe.
__device__ __forceinline__ void csa(unsigned& h, unsigned& l, unsigned a, unsigned b, unsigned c) {
  l = a ^ b ^ c;                       // LOP3 0x96
  h = (a & b) | (a & c) | (b & c);     // LOP3 0xE8
}
__device__ __forceinline__ unsigned popc32words_hs(const unsigned (&w)[32]) {
  unsigned ones = 0, twos = 0, fours = 0, eights = 0, total16 = 0;
#pragma unroll
  for (int blk = 0; blk < 2; ++blk) {
    const unsigned* x = w + 16 * blk;
    unsigned twosA, twosB, foursA, foursB, eightsA, eightsB, sixteens;
    csa(twosA, ones, ones, x[0], x[1]);
    csa(twosB, ones, ones, x[2], x[3]);
    csa(foursA, twos, twos, twosA, twosB);
    csa(twosA, ones, ones, x[4], x[5]);
    csa(twosB, ones, ones, x[6], x[7]);
    csa(foursB, twos, twos, twosA, twosB);
    csa(eightsA, fours, fours, foursA, foursB);
    csa(twosA, ones, ones, x[8], x[9]);
    csa(twosB, ones, ones, x[10], x[11]);
    csa(foursA, twos, twos, twosA, twosB);
    csa(twosA, ones, ones, x[12], x[13]);
    csa(twosB, ones, ones, x[14], x[15]);
    csa(foursB, twos, twos, twosA, twosB);
    csa(eightsB, fours, fours, foursA, foursB);
    csa(sixteens, eights, eights, eightsA, eightsB);
    total16 += __popc(sixteens);
  }
  return 16u * total16 + 8u * __popc(eights) + 4u * __popc(fours) + 2u * __popc(twos) + __popc(ones);
}

// the same code against QB queries: the chunks are loaded once (CHUNKS_CT > 0: all in registers)
template <int CHUNKS_CT, int QB>
__device__ __forceinline__ void code_distance_multi(const uint4* __restrict__ p, size_t ld, unsigned chunks,
                                                    const uint4* __restrict__ sq, unsigned (&dist)[QB]) {
#pragma unroll
  for (int q = 0; q < QB; ++q) dist[q] = 0;
  if (CHUNKS_CT > 0) {
    uint4 v[CHUNKS_CT > 0 ? CHUNKS_CT : 1];
#pragma unroll
    for (int c = 0; c < CHUNKS_CT; ++c) v[c] = ldg_stream_u4(p + (size_t)c * ld);
    if (CHUNKS_CT == 8 && QB >= 4) {  // 1024-bit codes, POPC-bound batch: 32 words per code -> carry-save tree
#pragma unroll
      for (int q = 0; q < QB; ++q) {
        unsigned x[32];
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          const uint4 qv = sq[q * 8 + c];
          x[4 * c + 0] = v[c].x ^ qv.x;
          x[4 * c + 1] = v[c].y ^ qv.y;
          x[4 * c + 2] = v[c].z ^ qv.z;
          x[4 * c + 3] = v[c].w ^ qv.w;
        }
        dist[q] = popc32words_hs(x);
      }
    } else {
#pragma unroll
      for (int q = 0; q < QB; ++q)
#pragma unroll
        for (int c = 0; c < CHUNKS_CT; ++c) dist[q] += popc_u4(v[c], sq[q * CHUNKS_CT + c]);
    }
  } else {
    for (unsigned c = 0; c < chunks; ++c) {
      const uint4 v = ldg_stream_u4(p + (size_t)c * ld);
#pragma unroll
      for (int q = 0; q < QB; ++q) dist[q] += popc_u4(v, sq[q * chunks + c]);
    }
  }
}

struct HamArgs {
  const uint4* data;
  unsigned long long ld;
  unsigned n, chunks, n_tiles, index_base;
  const uint64_t* query_words;  // device: 2*chunks words per query (zero padded)
  int nq_valid;                 // multi-query kernel: queries in this launch (<= QB)
  int k;
  uint64_t* partials;
  uint64_t* out_keys;
  uint64_t* group_partials;
  unsigned* tickets;
  unsigned long long* shared_thr;  // single-query top-k launches: launch-wide bound on the k-th key (may be null)
  uint32_t* dist_out;
};

template <int CHUNKS_CT, int R, bool TOPK>
__global__ void __launch_bounds__(HAM_THREADS) hamming_kernel(const HamArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* sq = reinterpret_cast<uint4*>(smem_raw);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(sq + a.chunks);
  const int lane = threadIdx.x & 31;
  for (unsigned c = threadIdx.x; c < a.chunks; c += blockDim.x) {
    uint64_t w0 = a.query_words[2 * c], w1 = a.query_words[2 * c + 1];
    sq[c] = make_uint4((unsigned)w0, (unsigned)(w0 >> 32), (unsigned)w1, (unsigned)(w1 >> 32));
  }
  __shared__ unsigned long long s_thr[2];
  SharedThreshold sh;
  sh.init(TOPK ? a.shared_thr : nullptr, &s_thr[0], &s_thr[1]);
  __syncthreads();

  WarpList<R> lists[1];
  uint64_t thrs[1];
  lists[0].init();
  thrs[0] = KEY_SENTINEL;

  unsigned it = 0;
  for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x, ++it) {
    const unsigned i = tile * HAM_THREADS + threadIdx.x;
    const bool valid = i < a.n;
    const uint64_t cap = TOPK ? sh.read(it) : KEY_SENTINEL;
    unsigned dist = 0;
    if (valid) dist = code_distance<CHUNKS_CT>(a.data + i, a.ld, a.chunks, sq);
    if (TOPK) {
      lists[0].offer(make_key_u32(dist, a.index_base + i), valid, thrs[0], a.k, lane, cap);
      sh.publish(thrs[0], cap, lane);
    } else if (valid) {
      a.dist_out[i] = dist;
    }
  }
  if (TOPK) block_finish<R, 1>(lists, 1, a.k, smem_keys, a.partials, a.group_partials, a.out_keys, a.tickets, a.shared_thr);
}

// QB queries share one pass over the codes (top-k only): the scan is HBM-bound for one query with the ALU pipe a third
// busy, so up to ~3 queries ride along for free and a batch of 4 costs about 1.5 passes
template <int CHUNKS_CT, int R, int QB>
__global__ void __launch_bounds__(HAM_THREADS) hamming_multi_kernel(const HamArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* sq = reinterpret_cast<uint4*>(smem_raw);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(sq + (size_t)QB * a.chunks);
  const int lane = threadIdx.x & 31;
  for (unsigned t = threadIdx.x; t < QB * a.chunks; t += blockDim.x) {
    const unsigned q = t / a.chunks, c = t % a.chunks;
    uint64_t w0 = 0, w1 = 0;
    if ((int)q < a.nq_valid) {
      w0 = a.query_words[(size_t)q * 2 * a.chunks + 2 * c];
      w1 = a.query_words[(size_t)q * 2 * a.chunks + 2 * c + 1];
    }
    sq[t] = make_uint4((unsigned)w0, (unsigned)(w0 >> 32), (unsigned)w1, (unsigned)(w1 >> 32));
  }
  __syncthreads();
  WarpList<R> lists[QB];
  uint64_t thrs[QB];
#pragma unroll
  for (int q = 0; q < QB; ++q) {
    lists[q].init();
    thrs[q] = KEY_SENTINEL;
  }
  for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const unsigned i = tile * HAM_THREADS + threadIdx.x;
    const bool valid = i < a.n;
    unsigned dist[QB];
#pragma unroll
    for (int q = 0; q < QB; ++q) dist[q] = 0;
    if (valid) code_distance_multi<CHUNKS_CT, QB>(a.data + i, a.ld, a.chunks, sq, dist);
#pragma unroll
    for (int q = 0; q < QB; ++q)
      if (q < a.nq_valid) lists[q].offer(make_key_u32(dist[q], a.index_base + i), valid, thrs[q], a.k, lane);
  }
  block_finish<R, QB>(lists, a.nq_valid, a.k, smem_keys, a.partials, a.group_partials, a.out_keys, a.tickets);
}

// row-major words [n][words] -> chunk-major uint4, masking padding bits (PackedBinary::new)
__global__ void binary_pack_kernel(const uint64_t* __restrict__ words_rm, unsigned n, unsigned words,
                                   unsigned dim_bits, uint4* __restrict__ codes, size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  const unsigned rem = dim_bits % 64;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    uint64_t w[2] = {0, 0};
    if (i < n) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        unsigned wi = 2 * c + h;
        if (wi < words) {
          uint64_t x = words_rm[i * words + wi];
          if (wi == words - 1 && rem != 0) x &= (1ull << rem) - 1;
          w[h] = x;
        }
      }
    }
    codes[t] = make_uint4((unsigned)w[0], (unsigned)(w[0] >> 32), (unsigned)w[1], (unsigned)(w[1] >> 32));
  }
}

__global__ void generate_binary_kernel(uint64_t salt, uint64_t first_row, unsigned n, unsigned words,
                                       unsigned dim_bits, uint4* __restrict__ codes, size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  const unsigned rem = dim_bits % 64;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    uint64_t w[2] = {0, 0};
    if (i < n) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        unsigned wi = 2 * c + h;
        if (wi < words) {
          uint64_t x = splitmix64(salt + (first_row + i) * words + wi);
          if (wi == words - 1 && rem != 0) x &= (1ull << rem) - 1;
          w[h] = x;
        }
      }
    }
    codes[t] = make_uint4((unsigned)w[0], (unsigned)(w[0] >> 32), (unsigned)w[1], (unsigned)(w[1] >> 32));
  }
}

// encode_binary (src/binary.rs:133-141) of every vector of a device-resident PDX f32 corpus straight into the
// chunk-major code layout: thread (chunk c, vector i) reads 128 dimension rows (coalesced along i), bit = v > threshold
__global__ void binary_from_pdx_kernel(const PdxView pdx, unsigned n, unsigned d,
                                       float threshold, uint4* __restrict__ codes, size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    unsigned w[4] = {0, 0, 0, 0};
    if (i < n) {
#pragma unroll 8
      for (int b = 0; b < 128; ++b) {
        const unsigned dd = 128 * c + b;
        if (dd < d && pdx_load1(pdx, (size_t)dd * pdx.ld + i) > threshold) w[b >> 5] |= 1u << (b & 31);
      }
    }
    codes[t] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// encode_binary: one warp per output u64 word (two ballots)
__global__ void encode_binary_kernel(const float* __restrict__ values, size_t n, float threshold,
                                     uint64_t* __restrict__ words, size_t n_words) {
  const int lane = threadIdx.x & 31;
  const size_t warp = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
  for (size_t w = warp; w < n_words; w += n_warps) {
    size_t i0 = w * 64 + lane, i1 = i0 + 32;
    unsigned lo = __ballot_sync(FULL_MASK, i0 < n && values[i0] > threshold);
    unsigned hi = __ballot_sync(FULL_MASK, i1 < n && values[i1] > threshold);
    if (lane == 0) words[w] = ((uint64_t)hi << 32) | lo;
  }
}

// intersection (and, for JACCARD, union) popcounts of one code against the query
template <bool JACCARD>
__device__ __forceinline__ void setop_counts(const HamArgs& a, const uint4* __restrict__ p, const uint4* __restrict__ sq,
                                             unsigned& inter, unsigned& uni) {
  inter = 0;
  uni = 0;
  unsigned c = 0;
  for (; c + 4 <= a.chunks; c += 4) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = ldg_stream_u4(p + (size_t)(c + u) * a.ld);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint4 q = sq[c + u];
      inter += __popc(v[u].x & q.x) + __popc(v[u].y & q.y) + __popc(v[u].z & q.z) + __popc(v[u].w & q.w);
      if (JACCARD) uni += __popc(v[u].x | q.x) + __popc(v[u].y | q.y) + __popc(v[u].z | q.z) + __popc(v[u].w | q.w);
    }
  }
  for (; c < a.chunks; ++c) {
    const uint4 v = ldg_stream_u4(p + (size_t)c * a.ld), q = sq[c];
    inter += __popc(v.x & q.x) + __popc(v.y & q.y) + __popc(v.z & q.z) + __popc(v.w & q.w);
    if (JACCARD) uni += __popc(v.x | q.x) + __popc(v.y | q.y) + __popc(v.z | q.z) + __popc(v.w | q.w);
  }
}

// Top-k by binary_dot / binary_jaccard with the selection fused into the scan (one pass, nothing of size n written):
// descending similarity, ties -> lower index. Keys as launch_topk_from_scores builds them from the score vectors:
// dot (~count << 32) | index, Jaccard make_key_desc(intersection as f32 / union as f32, index).
template <bool JACCARD, int R>
__global__ void __launch_bounds__(HAM_THREADS) binary_setops_topk_kernel(const HamArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* sq = reinterpret_cast<uint4*>(smem_raw);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(sq + a.chunks);
  const int lane = threadIdx.x & 31;
  for (unsigned c = threadIdx.x; c < a.chunks; c += blockDim.x) {
    uint64_t w0 = a.query_words[2 * c], w1 = a.query_words[2 * c + 1];
    sq[c] = make_uint4((unsigned)w0, (unsigned)(w0 >> 32), (unsigned)w1, (unsigned)(w1 >> 32));
  }
  __syncthreads();
  WarpList<R> lists[1];
  uint64_t thrs[1];
  lists[0].init();
  thrs[0] = KEY_SENTINEL;
  for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const unsigned i = tile * HAM_THREADS + threadIdx.x;
    const bool valid = i < a.n;
    uint64_t key = KEY_SENTINEL;
    if (valid) {
      unsigned inter, uni;
      setop_counts<JACCARD>(a, a.data + i, sq, inter, uni);
      if (JACCARD) key = make_key_desc(uni == 0 ? 1.0f : __fdiv_rn(__uint2float_rn(inter), __uint2float_rn(uni)), a.index_base + i);
      else key = make_key_u32(~inter, a.index_base + i);
    }
    lists[0].offer(key, valid, thrs[0], a.k, lane);
  }
  block_finish<R, 1>(lists, 1, a.k, smem_keys, a.partials, a.group_partials, a.out_keys, a.tickets);
}

// binary_dot (src/binary.rs:178-185) and binary_jaccard (:198-213) of one query against every code: same scan shape,
// AND / OR instead of XOR. JACCARD: intersection as f32 / union as f32, 1.0 when the union is empty.
template <bool JACCARD>
__global__ void __launch_bounds__(HAM_THREADS) binary_setops_kernel(const HamArgs a, float* __restrict__ jaccard_out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* sq = reinterpret_cast<uint4*>(smem_raw);
  for (unsigned c = threadIdx.x; c < a.chunks; c += blockDim.x) {
    uint64_t w0 = a.query_words[2 * c], w1 = a.query_words[2 * c + 1];
    sq[c] = make_uint4((unsigned)w0, (unsigned)(w0 >> 32), (unsigned)w1, (unsigned)(w1 >> 32));
  }
  __syncthreads();
  const unsigned i = blockIdx.x * HAM_THREADS + threadIdx.x;
  if (i >= a.n) return;
  const uint4* p = a.data + i;
  unsigned inter = 0, uni = 0;
  unsigned c = 0;
  for (; c + 4 <= a.chunks; c += 4) {
    uint4 v[4];
#pragma unroll
    for (int u = 0; u < 4; ++u) v[u] = ldg_stream_u4(p + (size_t)(c + u) * a.ld);
#pragma unroll
    for (int u = 0; u < 4; ++u) {
      const uint4 q = sq[c + u];
      inter += __popc(v[u].x & q.x) + __popc(v[u].y & q.y) + __popc(v[u].z & q.z) + __popc(v[u].w & q.w);
      if (JACCARD) uni += __popc(v[u].x | q.x) + __popc(v[u].y | q.y) + __popc(v[u].z | q.z) + __popc(v[u].w | q.w);
    }
  }
  for (; c < a.chunks; ++c) {
    const uint4 v = ldg_stream_u4(p + (size_t)c * a.ld), q = sq[c];
    inter += __popc(v.x & q.x) + __popc(v.y & q.y) + __popc(v.z & q.z) + __popc(v.w & q.w);
    if (JACCARD) uni += __popc(v.x | q.x) + __popc(v.y | q.y) + __popc(v.z | q.z) + __popc(v.w | q.w);
  }
  if (JACCARD) jaccard_out[i] = uni == 0 ? 1.0f : __fdiv_rn(__uint2float_rn(inter), __uint2float_rn(uni));
  else a.dist_out[i] = inter;
}

template <int CHUNKS_CT, int R, bool TOPK>
cudaError_t launch_ham(const HamArgs& a, size_t smem, int num_sms, cudaStream_t s) {
  auto kern = hamming_kernel<CHUNKS_CT, R, TOPK>;
  int occ = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, HAM_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  unsigned grid = TOPK ? balanced_grid(a.n_tiles, (unsigned)occ * (unsigned)num_sms) : (a.n_tiles ? a.n_tiles : 1);
  kern<<<grid, HAM_THREADS, smem, s>>>(a);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_binary_pack(const uint64_t* dev_words_rowmajor, size_t n, size_t words, size_t dim_bits,
                               uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches) {
  if (n == 0 || words == 0) return cudaSuccess;
  unsigned chunks = (unsigned)((words + 1) / 2);
  binary_pack_kernel<<<148 * 8, 256, 0, s>>>(dev_words_rowmajor, (unsigned)n, (unsigned)words, (unsigned)dim_bits,
                                             dev_codes, ld, chunks);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_generate_binary(uint64_t salt, uint64_t first_row, size_t n, size_t words, size_t dim_bits,
                                   uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches) {
  if (n == 0 || words == 0) return cudaSuccess;
  unsigned chunks = (unsigned)((words + 1) / 2);
  generate_binary_kernel<<<148 * 16, 256, 0, s>>>(salt, first_row, (unsigned)n, (unsigned)words, (unsigned)dim_bits,
                                                  dev_codes, ld, chunks);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_binary_from_pdx(const PdxView& v, float threshold,
                                   uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0 || v.d == 0) return cudaSuccess;
  binary_from_pdx_kernel<<<148 * 16, 256, 0, s>>>(v, (unsigned)v.n, (unsigned)v.d, threshold, dev_codes, ld,
                                                  (unsigned)((v.d + 127) / 128));
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_encode_binary(const float* dev_values, size_t n, float threshold, uint64_t* dev_words,
                                 cudaStream_t s, LaunchCounter* launches) {
  size_t n_words = (n + 63) / 64;
  if (n_words == 0) return cudaSuccess;
  unsigned grid = (unsigned)((n_words * 32 + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  encode_binary_kernel<<<grid, 256, 0, s>>>(dev_values, n, threshold, dev_words, n_words);
  ++*launches;
  return cudaGetLastError();
}

static HamArgs make_args(const BinView& v, const uint64_t* q) {
  HamArgs a{};
  a.data = v.data;
  a.ld = v.ld;
  a.n = (unsigned)v.n;
  a.chunks = (unsigned)v.chunks;
  a.n_tiles = (unsigned)((v.n + HAM_THREADS - 1) / HAM_THREADS);
  a.index_base = v.index_base;
  a.query_words = q;
  return a;
}

cudaError_t launch_hamming_all(const BinView& v, const uint64_t* dev_query_words, uint32_t* dev_out,
                               cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0) return cudaSuccess;
  HamArgs a = make_args(v, dev_query_words);
  a.dist_out = dev_out;
  size_t smem = v.chunks * sizeof(uint4);
  cudaError_t e = (v.chunks == 8) ? launch_ham<8, 1, false>(a, smem, 148, s) : launch_ham<0, 1, false>(a, smem, 148, s);
  if (e == cudaSuccess) ++*launches;
  return e;
}

cudaError_t launch_binary_dot_all(const BinView& v, const uint64_t* dev_query_words, uint32_t* dev_out,
                                  cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0) return cudaSuccess;
  HamArgs a = make_args(v, dev_query_words);
  a.dist_out = dev_out;
  binary_setops_kernel<false><<<a.n_tiles, HAM_THREADS, v.chunks * sizeof(uint4), s>>>(a, nullptr);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_binary_jaccard_all(const BinView& v, const uint64_t* dev_query_words, float* dev_out,
                                      cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0) return cudaSuccess;
  HamArgs a = make_args(v, dev_query_words);
  binary_setops_kernel<true><<<a.n_tiles, HAM_THREADS, v.chunks * sizeof(uint4), s>>>(a, dev_out);
  ++*launches;
  return cudaGetLastError();
}

namespace {
template <bool JACCARD, int R>
cudaError_t launch_setops_topk(const HamArgs& a, size_t smem, int num_sms, cudaStream_t s) {
  auto kern = binary_setops_topk_kernel<JACCARD, R>;
  int occ = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, HAM_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  kern<<<balanced_grid(a.n_tiles, (unsigned)occ * (unsigned)num_sms), HAM_THREADS, smem, s>>>(a);
  return cudaGetLastError();
}
}  // namespace

// fused single-pass top-k (k <= 128) by binary_dot (jaccard = 0) or binary_jaccard (1)
cudaError_t launch_binary_setops_topk(const BinView& v, int jaccard, const uint64_t* dev_query_words, size_t k, uint64_t* dev_keys,
                                      Workspace& ws, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0 || k == 0 || k > 128) return cudaErrorInvalidValue;
  HamArgs a = make_args(v, dev_query_words);
  a.k = (int)k;
  a.partials = ws.partials;
  a.group_partials = ws.group_partials;
  a.tickets = ws.tickets;
  a.out_keys = dev_keys;
  const size_t smem = v.chunks * sizeof(uint4) + (size_t)(HAM_THREADS / 32) * k * sizeof(uint64_t);
  if (smem > 48 * 1024) return cudaErrorInvalidValue;
  cudaError_t e;
  if (k <= 32) e = jaccard ? launch_setops_topk<true, 1>(a, smem, ws.num_sms, s) : launch_setops_topk<false, 1>(a, smem, ws.num_sms, s);
  else e = jaccard ? launch_setops_topk<true, 4>(a, smem, ws.num_sms, s) : launch_setops_topk<false, 4>(a, smem, ws.num_sms, s);
  if (e == cudaSuccess) ++*launches;
  return e;
}

namespace {
// queries per pass: the 128-slot lists of k > 32 cost 8 registers per query and lane, and registers decide how many
// bytes the CTAs of an SM keep in flight -- 4 queries per pass with 32-slot lists, 2 with 128-slot lists
template <int R> constexpr int ham_qb() { return R == 1 ? 4 : 2; }
template <int CHUNKS_CT, int R>
cudaError_t launch_ham_multi(const HamArgs& a, size_t smem, int num_sms, cudaStream_t s) {
  auto kern = hamming_multi_kernel<CHUNKS_CT, R, ham_qb<R>()>;
  int occ = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, HAM_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  kern<<<balanced_grid(a.n_tiles, (unsigned)occ * (unsigned)num_sms), HAM_THREADS, smem, s>>>(a);
  return cudaGetLastError();
}
}  // namespace

cudaError_t launch_hamming_topk(const BinView& v, const uint64_t* dev_query_words, size_t nq, size_t k,
                                uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches) {
  if (k > 128) return cudaErrorInvalidValue;
  size_t q0 = 0;
  // batches: groups of 4 queries share one pass over the codes
  const size_t qb = k <= 32 ? ham_qb<1>() : ham_qb<4>();
  const size_t multi_smem = qb * v.chunks * sizeof(uint4) + qb * (size_t)(HAM_THREADS / 32) * k * sizeof(uint64_t);
  while (nq - q0 >= 2 && multi_smem <= 48 * 1024) {
    const size_t take = nq - q0 < qb ? nq - q0 : qb;
    HamArgs a = make_args(v, dev_query_words + q0 * 2 * v.chunks);
    a.nq_valid = (int)take;
    a.k = (int)k;
    a.partials = ws.partials;
    a.group_partials = ws.group_partials;
    a.tickets = ws.tickets;
    a.out_keys = dev_keys + q0 * k;
    cudaError_t e;
    if (v.chunks == 8)
      e = (k <= 32) ? launch_ham_multi<8, 1>(a, multi_smem, ws.num_sms, s) : launch_ham_multi<8, 4>(a, multi_smem, ws.num_sms, s);
    else
      e = (k <= 32) ? launch_ham_multi<0, 1>(a, multi_smem, ws.num_sms, s) : launch_ham_multi<0, 4>(a, multi_smem, ws.num_sms, s);
    if (e != cudaSuccess) return e;
    ++*launches;
    q0 += take;
  }
  for (size_t q = q0; q < nq; ++q) {
    HamArgs a = make_args(v, dev_query_words + q * 2 * v.chunks);
    a.k = (int)k;
    a.partials = ws.partials;
    a.group_partials = ws.group_partials;
    a.tickets = ws.tickets;
    static const bool shared_off = getenv("INNR_SHARED_THR") && atoi(getenv("INNR_SHARED_THR")) == 0;  // A/B switch
    a.shared_thr = shared_off ? nullptr : ws.shared_thr;
    a.out_keys = dev_keys + q * k;
    size_t smem = v.chunks * sizeof(uint4) + (size_t)(HAM_THREADS / 32) * k * sizeof(uint64_t);
    cudaError_t e;
    if (v.chunks == 8)
      e = (k <= 32) ? launch_ham<8, 1, true>(a, smem, ws.num_sms, s) : launch_ham<8, 4, true>(a, smem, ws.num_sms, s);
    else
      e = (k <= 32) ? launch_ham<0, 1, true>(a, smem, ws.num_sms, s) : launch_ham<0, 4, true>(a, smem, ws.num_sms, s);
    if (e != cudaSuccess) return e;
    ++*launches;
  }
  return cudaSuccess;
}

namespace {
// Queries the tensor-core filter (bin_tc.cu) flagged on the device: grid (FLAGGED_CTAS, nq), CTA (x, q) returns at once
// unless counts[q] > cap. Otherwise the FLAGGED_CTAS CTAs of query q split the rows, each merges its warps' lists into
// partials[q][x], and the last of them to finish (ticket tickets[q], zero on entry, reset on exit) merges the
// FLAGGED_CTAS lists into out_keys[q]. The keys are those of the single-query kernels above.
template <int OP, int R>
__global__ void __launch_bounds__(HAM_THREADS) binary_flagged_topk_kernel(const HamArgs a, const unsigned* __restrict__ counts,
                                                                          unsigned cap) {
  const unsigned q = blockIdx.y;
  if (counts[q] <= cap) return;
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* sq = reinterpret_cast<uint4*>(smem_raw);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(sq + a.chunks);
  __shared__ unsigned s_last;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  const uint64_t* qw = a.query_words + (size_t)q * 2 * a.chunks;
  for (unsigned c = threadIdx.x; c < a.chunks; c += blockDim.x) {
    const uint64_t w0 = qw[2 * c], w1 = qw[2 * c + 1];
    sq[c] = make_uint4((unsigned)w0, (unsigned)(w0 >> 32), (unsigned)w1, (unsigned)(w1 >> 32));
  }
  __syncthreads();
  WarpList<R> list;
  list.init();
  uint64_t thr = KEY_SENTINEL;
  for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const unsigned i = tile * HAM_THREADS + threadIdx.x;
    const bool valid = i < a.n;
    uint64_t key = KEY_SENTINEL;
    if (valid) {
      if (OP == 0) {
        key = make_key_u32(code_distance<0>(a.data + i, a.ld, a.chunks, sq), a.index_base + i);
      } else {
        unsigned inter, uni;
        setop_counts<OP == 2>(a, a.data + i, sq, inter, uni);
        if (OP == 2) key = make_key_desc(uni == 0 ? 1.0f : __fdiv_rn(__uint2float_rn(inter), __uint2float_rn(uni)), a.index_base + i);
        else key = make_key_u32(~inter, a.index_base + i);
      }
    }
    list.offer(key, valid, thr, a.k, lane);
  }
  block_tree_merge<R>(list, a.k, smem_keys);
  uint64_t* mine = a.partials + ((size_t)q * gridDim.x + blockIdx.x) * a.k;
  if (warp == 0) list.store(mine, a.k, lane);
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_last = (atomicAdd(&a.tickets[q], 1u) == gridDim.x - 1) ? 1u : 0u;
  __syncthreads();
  if (!s_last) return;
  __threadfence();
  WarpList<R> acc;
  acc.init();
  warp_merge_lists<R, true>(acc, a.partials + (size_t)q * gridDim.x * a.k, warp, n_warps, (int)gridDim.x, (size_t)a.k, a.k,
                            lane);
  block_tree_merge<R>(acc, a.k, smem_keys);
  if (warp == 0) acc.store(a.out_keys + (size_t)q * a.k, a.k, lane);
  if (threadIdx.x == 0) a.tickets[q] = 0u;
}

template <int OP, int R>
cudaError_t launch_flagged(const HamArgs& a, size_t nq, const unsigned* counts, unsigned cap, size_t smem, cudaStream_t s) {
  binary_flagged_topk_kernel<OP, R><<<dim3(BIN_FLAGGED_CTAS, (unsigned)nq), HAM_THREADS, smem, s>>>(a, counts, cap);
  return cudaGetLastError();
}
template <int R>
cudaError_t launch_flagged_op(int op, const HamArgs& a, size_t nq, const unsigned* counts, unsigned cap, size_t smem,
                              cudaStream_t s) {
  if (op == 0) return launch_flagged<0, R>(a, nq, counts, cap, smem, s);
  if (op == 1) return launch_flagged<1, R>(a, nq, counts, cap, smem, s);
  return launch_flagged<2, R>(a, nq, counts, cap, smem, s);
}
}  // namespace

cudaError_t launch_binary_flagged_topk(const BinView& v, int op, const uint64_t* dev_query_words, size_t nq, size_t k,
                                       const unsigned* dev_counts, unsigned cap, uint64_t* partials, unsigned* tickets,
                                       uint64_t* dev_keys, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0 || nq == 0 || k == 0 || k > 128 || op < 0 || op > 2) return cudaErrorInvalidValue;
  HamArgs a = make_args(v, dev_query_words);
  a.k = (int)k;
  a.partials = partials;
  a.tickets = tickets;
  a.out_keys = dev_keys;
  const size_t smem = v.chunks * sizeof(uint4) + (size_t)(HAM_THREADS / 32) * k * sizeof(uint64_t);
  if (smem > 48 * 1024) return cudaErrorInvalidValue;
  const cudaError_t e = k <= 32 ? launch_flagged_op<1>(op, a, nq, dev_counts, cap, smem, s)
                                : launch_flagged_op<4>(op, a, nq, dev_counts, cap, smem, s);
  if (e == cudaSuccess) ++*launches;
  return e;
}

}  // namespace innr
