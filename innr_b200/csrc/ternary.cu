// ternary.cu -- scans over packed ternary codes (2 bits per value: 01 = +1, 10 = -1, 32 values per u64).
//
// Replaces (reference, innr 0.6.3, src/ternary.rs; SURVEY.md 8f row 4 "same scan shape, other codecs"):
//   PackedTernary::new masking   :63-82      encode_ternary        :163-173
//   ternary_dot                  :191-281    (popcount of same-sign minus different-sign positions; popcnt == portable)
//   ternary::asymmetric_dot      :286-296    (f32 query: sequential sum += q * t, unfused)
//   ternary_hamming              :301-324
//
// Device layout: the binary layout with twice the bits -- 128-bit chunks (64 values), chunk-major: codes[c * ld + i].
// One thread owns one code; consecutive threads read consecutive 16-byte chunks. Integer results are exact; the
// asymmetric dot reproduces the reference's sequential unfused f32 sum bit for bit (a 0 value still multiplies:
// q * 0.0 is -0.0 or NaN for negative / non-finite q, exactly as on the CPU).
#include "common.cuh"
#include "kernels.cuh"
#include "pdx.cuh"

namespace innr {

namespace {

constexpr int TER_THREADS = 256;
constexpr unsigned T_ODD = 0x55555555u, T_EVEN = 0xAAAAAAAAu;

struct TerArgs {
  const uint4* data;
  unsigned long long ld;
  unsigned n, chunks, dim;
  const uint64_t* query_words;  // TER_DOT / TER_HAMMING: 2 * chunks words (zero padded)
  const float* query;           // TER_ASYM: dim floats
  float* out_f32;               // scores as f32 (exact for the integer ops while |score| < 2^24)
  int32_t* out_i32;             // optional raw integer scores
};

__device__ __forceinline__ void dot32(unsigned wa, unsigned wb, unsigned& same, unsigned& diff) {
  const unsigned pos_a = wa & ~((wa & T_EVEN) >> 1) & T_ODD, pos_b = wb & ~((wb & T_EVEN) >> 1) & T_ODD;
  const unsigned neg_a = ~wa & ((wa & T_EVEN) >> 1) & T_ODD, neg_b = ~wb & ((wb & T_EVEN) >> 1) & T_ODD;
  same += __popc((pos_a & pos_b) | (neg_a & neg_b));
  diff += __popc((pos_a & neg_b) | (neg_a & pos_b));
}
__device__ __forceinline__ unsigned ham32(unsigned wa, unsigned wb) {
  const unsigned nz_a = (wa & T_ODD) | ((wa & T_EVEN) >> 1), nz_b = (wb & T_ODD) | ((wb & T_EVEN) >> 1);
  const unsigned x = wa ^ wb;
  const unsigned df = (x & T_ODD) | ((x & T_EVEN) >> 1);
  return __popc(df & nz_a & nz_b);
}

// score of one code (its first chunk at p): f32 value (what the scores kernel writes), and for the integer ops the raw i32
template <int OP>
__device__ __forceinline__ float ternary_score(const TerArgs& a, const uint4* __restrict__ p, const uint4* __restrict__ sqw,
                                               const float* __restrict__ sqf, int32_t& si) {
  if (OP == 2) {
    float sum = 0.0f;
    unsigned k = 0;
    for (unsigned c = 0; c < a.chunks; ++c) {
      const uint4 v = ldg_stream_u4(p + (size_t)c * a.ld);
      const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
      for (int h = 0; h < 4; ++h) {
#pragma unroll
        for (int j = 0; j < 16; ++j, ++k) {
          if (k < a.dim) {  // the reference loops over query.iter(): exactly `dimension` terms
            const unsigned bits = (w[h] >> (2 * j)) & 3u;
            const float tv = bits == 1u ? 1.0f : (bits == 2u ? -1.0f : 0.0f);  // ternary.get(i) as f32
            sum = __fadd_rn(sum, __fmul_rn(sqf[k], tv));                       // sum += q * t
          }
        }
      }
    }
    si = 0;
    return sum;
  }
  unsigned same = 0, diff = 0, ham = 0;
  for (unsigned c = 0; c < a.chunks; ++c) {
    const uint4 v = ldg_stream_u4(p + (size_t)c * a.ld), q = sqw[c];
    if (OP == 0) {
      dot32(v.x, q.x, same, diff);
      dot32(v.y, q.y, same, diff);
      dot32(v.z, q.z, same, diff);
      dot32(v.w, q.w, same, diff);
    } else {
      ham += ham32(v.x, q.x) + ham32(v.y, q.y) + ham32(v.z, q.z) + ham32(v.w, q.w);
    }
  }
  si = OP == 0 ? (int32_t)same - (int32_t)diff : (int32_t)ham;
  return (float)si;
}

// OP 0: ternary_dot, 1: ternary_hamming, 2: asymmetric_dot
template <int OP>
__global__ void __launch_bounds__(TER_THREADS) ternary_scores_kernel(const TerArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* sqw = reinterpret_cast<uint4*>(smem_raw);
  float* sqf = reinterpret_cast<float*>(smem_raw);
  if (OP == 2) {
    for (unsigned k = threadIdx.x; k < a.chunks * 64; k += blockDim.x) sqf[k] = k < a.dim ? a.query[k] : 0.0f;
  } else {
    for (unsigned c = threadIdx.x; c < a.chunks; c += blockDim.x) {
      const uint64_t w0 = a.query_words[2 * c], w1 = a.query_words[2 * c + 1];
      sqw[c] = make_uint4((unsigned)w0, (unsigned)(w0 >> 32), (unsigned)w1, (unsigned)(w1 >> 32));
    }
  }
  __syncthreads();
  const unsigned i = blockIdx.x * TER_THREADS + threadIdx.x;
  if (i >= a.n) return;
  int32_t si = 0;
  const float sc = ternary_score<OP>(a, a.data + i, sqw, sqf, si);
  if (OP != 2 && a.out_i32) a.out_i32[i] = si;
  if (a.out_f32) a.out_f32[i] = sc;
}

// The same scan with the top-k fused in (one pass, nothing of size n written): dot / asymmetric dot descending, Hamming
// ascending, ties -> lower index -- the keys launch_topk_from_scores builds from the f32 score vector.
template <int OP, int R>
__global__ void __launch_bounds__(TER_THREADS) ternary_topk_kernel(const TerArgs a, int k, unsigned index_base, unsigned n_tiles,
                                                                  uint64_t* partials, uint64_t* group_partials,
                                                                  uint64_t* out_keys, unsigned* tickets) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint4* sqw = reinterpret_cast<uint4*>(smem_raw);
  float* sqf = reinterpret_cast<float*>(smem_raw);
  const size_t q_bytes = OP == 2 ? (size_t)a.chunks * 64 * sizeof(float) : (size_t)a.chunks * sizeof(uint4);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(smem_raw + q_bytes);
  if (OP == 2) {
    for (unsigned kk = threadIdx.x; kk < a.chunks * 64; kk += blockDim.x) sqf[kk] = kk < a.dim ? a.query[kk] : 0.0f;
  } else {
    for (unsigned c = threadIdx.x; c < a.chunks; c += blockDim.x) {
      const uint64_t w0 = a.query_words[2 * c], w1 = a.query_words[2 * c + 1];
      sqw[c] = make_uint4((unsigned)w0, (unsigned)(w0 >> 32), (unsigned)w1, (unsigned)(w1 >> 32));
    }
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  WarpList<R> lists[1];
  uint64_t thrs[1];
  lists[0].init();
  thrs[0] = KEY_SENTINEL;
  for (unsigned tile = blockIdx.x; tile < n_tiles; tile += gridDim.x) {
    const unsigned i = tile * TER_THREADS + threadIdx.x;
    const bool valid = i < a.n;
    uint64_t key = KEY_SENTINEL;
    if (valid) {
      int32_t si;
      const float sc = ternary_score<OP>(a, a.data + i, sqw, sqf, si);
      key = OP == 1 ? make_key_asc(sc, index_base + i) : make_key_desc(sc, index_base + i);
    }
    lists[0].offer(key, valid, thrs[0], k, lane);
  }
  block_finish<R, 1>(lists, 1, k, smem_keys, partials, group_partials, out_keys, tickets);
}

// row-major words [n][words] -> chunk-major uint4, masking the padding pairs of the last word (PackedTernary::new)
__global__ void ternary_pack_kernel(const uint64_t* __restrict__ words_rm, unsigned n, unsigned words, unsigned dim,
                                    uint4* __restrict__ codes, size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  const unsigned rem = dim % 32;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    uint64_t w[2] = {0, 0};
    if (i < n) {
#pragma unroll
      for (int h = 0; h < 2; ++h) {
        const unsigned wi = 2 * c + h;
        if (wi < words) {
          uint64_t x = words_rm[i * words + wi];
          if (wi == words - 1 && rem != 0) x &= (1ull << (rem * 2)) - 1;
          w[h] = x;
        }
      }
    }
    codes[t] = make_uint4((unsigned)w[0], (unsigned)(w[0] >> 32), (unsigned)w[1], (unsigned)(w[1] >> 32));
  }
}

// encode_ternary of every vector of a device-resident PDX f32 corpus: thread (chunk c, vector i) reads 64 dimension rows
__global__ void ternary_from_pdx_kernel(const PdxView pdx, unsigned n, unsigned d, float threshold,
                                        uint4* __restrict__ codes, size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    unsigned w[4] = {0, 0, 0, 0};
    if (i < n) {
#pragma unroll 8
      for (int b = 0; b < 64; ++b) {
        const unsigned dd = 64 * c + b;
        if (dd < d) {
          const float v = pdx_load1(pdx, (size_t)dd * pdx.ld + i);
          const unsigned bits = v > threshold ? 1u : (v < -threshold ? 2u : 0u);
          w[b >> 4] |= bits << (2 * (b & 15));
        }
      }
    }
    codes[t] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// encode_ternary of a flat f32 array: one thread per output u64 word
__global__ void encode_ternary_kernel(const float* __restrict__ values, size_t n, float threshold,
                                      uint64_t* __restrict__ words, size_t n_words) {
  for (size_t w = (size_t)blockIdx.x * blockDim.x + threadIdx.x; w < n_words; w += (size_t)gridDim.x * blockDim.x) {
    uint64_t x = 0;
    for (int j = 0; j < 32; ++j) {
      const size_t i = w * 32 + j;
      if (i < n) {
        const float v = values[i];
        const uint64_t bits = v > threshold ? 1u : (v < -threshold ? 2u : 0u);
        x |= bits << (2 * j);
      }
    }
    words[w] = x;
  }
}

}  // namespace

cudaError_t launch_ternary_pack(const uint64_t* dev_words_rowmajor, size_t n, size_t words, size_t dim, uint4* dev_codes,
                                size_t ld, cudaStream_t s, LaunchCounter* launches) {
  if (n == 0 || words == 0) return cudaSuccess;
  ternary_pack_kernel<<<148 * 8, 256, 0, s>>>(dev_words_rowmajor, (unsigned)n, (unsigned)words, (unsigned)dim, dev_codes, ld,
                                              (unsigned)((words + 1) / 2));
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_ternary_from_pdx(const PdxView& v, float threshold, uint4* dev_codes,
                                    size_t ld, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0 || v.d == 0) return cudaSuccess;
  ternary_from_pdx_kernel<<<148 * 16, 256, 0, s>>>(v, (unsigned)v.n, (unsigned)v.d, threshold, dev_codes, ld,
                                                   (unsigned)((v.d + 63) / 64));
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_encode_ternary(const float* dev_values, size_t n, float threshold, uint64_t* dev_words, cudaStream_t s,
                                  LaunchCounter* launches) {
  const size_t n_words = (n + 31) / 32;
  if (n_words == 0) return cudaSuccess;
  unsigned grid = (unsigned)((n_words + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  encode_ternary_kernel<<<grid, 256, 0, s>>>(dev_values, n, threshold, dev_words, n_words);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_ternary_scores(const TerView& v, int op, const uint64_t* dev_query_words, const float* dev_query,
                                  float* dev_out_f32, int32_t* dev_out_i32, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0) return cudaSuccess;
  TerArgs a{};
  a.data = v.data;
  a.ld = v.ld;
  a.n = (unsigned)v.n;
  a.chunks = (unsigned)v.chunks;
  a.dim = (unsigned)v.dim;
  a.query_words = dev_query_words;
  a.query = dev_query;
  a.out_f32 = dev_out_f32;
  a.out_i32 = dev_out_i32;
  const unsigned grid = (unsigned)((v.n + TER_THREADS - 1) / TER_THREADS);
  const size_t smem = op == 2 ? v.chunks * 64 * sizeof(float) : v.chunks * sizeof(uint4);
  if (smem > 227 * 1024 || op < 0 || op > 2) return cudaErrorInvalidValue;
  if (smem > 48 * 1024) {  // wide codes (> 12288 dimensions for the f32 query): opt in to the large carve-out
    cudaError_t e = op == 0   ? cudaFuncSetAttribute(ternary_scores_kernel<0>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                    : op == 1 ? cudaFuncSetAttribute(ternary_scores_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)
                              : cudaFuncSetAttribute(ternary_scores_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  if (op == 0) ternary_scores_kernel<0><<<grid, TER_THREADS, smem, s>>>(a);
  else if (op == 1) ternary_scores_kernel<1><<<grid, TER_THREADS, smem, s>>>(a);
  else ternary_scores_kernel<2><<<grid, TER_THREADS, smem, s>>>(a);
  ++*launches;
  return cudaGetLastError();
}

namespace {
template <int OP, int R>
cudaError_t launch_ter_topk(const TerArgs& a, size_t k, uint32_t index_base, uint64_t* dev_keys, Workspace& ws, cudaStream_t s) {
  auto kern = ternary_topk_kernel<OP, R>;
  const size_t q_bytes = OP == 2 ? (size_t)a.chunks * 64 * sizeof(float) : (size_t)a.chunks * sizeof(uint4);
  const size_t smem = q_bytes + (size_t)(TER_THREADS / 32) * k * sizeof(uint64_t);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  cudaError_t e;
  if (smem > 48 * 1024 && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem)) != cudaSuccess) return e;
  int occ = 0;
  if ((e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, TER_THREADS, smem)) != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  const unsigned n_tiles = (a.n + TER_THREADS - 1) / TER_THREADS;
  kern<<<balanced_grid(n_tiles, (unsigned)occ * (unsigned)ws.num_sms), TER_THREADS, smem, s>>>(a, (int)k, index_base, n_tiles, ws.partials,
                                                                                             ws.group_partials, dev_keys, ws.tickets);
  return cudaGetLastError();
}
}  // namespace

// fused single-pass top-k (k <= 128) of the ternary scores: the keys of launch_topk_from_scores over the f32 score vector
cudaError_t launch_ternary_topk(const TerView& v, int op, const uint64_t* dev_query_words, const float* dev_query, size_t k,
                                uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0 || k == 0 || k > 128 || op < 0 || op > 2) return cudaErrorInvalidValue;
  TerArgs a{};
  a.data = v.data;
  a.ld = v.ld;
  a.n = (unsigned)v.n;
  a.chunks = (unsigned)v.chunks;
  a.dim = (unsigned)v.dim;
  a.query_words = dev_query_words;
  a.query = dev_query;
  cudaError_t e;
  if (k <= 32) e = op == 0 ? launch_ter_topk<0, 1>(a, k, v.index_base, dev_keys, ws, s) : op == 1 ? launch_ter_topk<1, 1>(a, k, v.index_base, dev_keys, ws, s) : launch_ter_topk<2, 1>(a, k, v.index_base, dev_keys, ws, s);
  else e = op == 0 ? launch_ter_topk<0, 4>(a, k, v.index_base, dev_keys, ws, s) : op == 1 ? launch_ter_topk<1, 4>(a, k, v.index_base, dev_keys, ws, s) : launch_ter_topk<2, 4>(a, k, v.index_base, dev_keys, ws, s);
  if (e == cudaSuccess) ++*launches;
  return e;
}

}  // namespace innr
