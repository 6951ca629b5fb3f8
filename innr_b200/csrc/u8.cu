// u8.cu -- HBM-bound asymmetric f32 x u8 scan with fused top-k (bit-exact with the reference's AVX2 kernel).
//
// Replaces (reference, innr 0.6.3):
//   dot_u8_f32_avx2                  src/arch/x86_64.rs:928-1020 (reached via src/scalar.rs:327-349 for n >= 16,
//                                    on AVX-512 hosts too -- no AVX-512 variant exists)
//   mixed_dot_u8_f32_portable        src/scalar.rs:353-358 (n < 16)
//   asymmetric_dot_u8[_precomputed]  src/scalar.rs:261-300:  (alpha/255)*mixed + offset*query_sum, unfused
//   query_context                    src/scalar.rs:236-240
//   quantize_u8                      src/scalar.rs:212-225
//   batch_knn_u8                     src/scalar.rs:370-393 (stable descending sort, truncate)
//
// Bit-exact recipe (SURVEY.md 8a, verified against the intrinsics in tests/test_oracle_simd.py): the AVX2 kernel
// is 32 independent FMA chains -- chain c accumulates elements idx == c (mod 32), ascending, with fused
// multiply-add; the four 8-lane accumulators combine as (a0+a1)+(a2+a3), then lanes j+(j+4), (0+2),(1+3), and
// the sum of those two. Then an 8-wide remainder (own 8 chains, same horizontal sum, added), then a scalar tail
// with separately rounded multiply and add. fmaf on the GPU is IEEE-exact, so one thread holding the 32 chains
// of one vector reproduces the CPU result bit for bit.
//
// Device layout: 16-byte chunks (16 dimensions), chunk-major: codes[c * ld + i]. One thread owns one vector.
// The chunk rows of a 256-vector tile (4 KB each, contiguous) are staged through a shared-memory ring by a producer
// warp with cp.async.bulk + mbarriers (16 KB stages, 6 deep), so the bytes in flight towards HBM do not depend on
// registers; consumers read their 16 bytes per chunk with one conflict-free LDS.128.
// u8 -> f32 is exact via the 2^23 magic number (PRMT + FADD, no I2F); the subtraction and the FMA chains run as
// packed FADD2 / FFMA2 (two IEEE-exact f32 operations per instruction: 2.3 instructions per byte instead of 3.3).
#include <type_traits>

#include "common.cuh"
#include "kernels.cuh"
#include "pdx.cuh"
#include "tc_common.cuh"

namespace innr {

namespace {

constexpr int U8_THREADS = 256;            // consumer threads = vectors per tile
constexpr int U8_CTA = U8_THREADS + 32;     // + one producer warp
constexpr int U8_STAGE_CHUNKS = 4;          // chunk rows per stage (even: chunk parity selects the accumulator half)
constexpr int U8_STAGES = 6;
constexpr int U8_ROW_BYTES = U8_THREADS * 16;
constexpr int U8_STAGE_BYTES = U8_STAGE_CHUNKS * U8_ROW_BYTES;  // 16 KB

// The 2^23 magic constant is kept in a register the compiler cannot see through, so that PRMT takes the byte
// selector as its immediate operand (with a literal constant the selector is re-materialised by a MOV per byte).
// (An asm mov is folded by ptxas too, so the value travels as a kernel argument: U8Args::magic.)
__device__ __forceinline__ float byte_to_f32_biased(unsigned word, int k, unsigned magic) {
  // bytes: [b_k, 0x00, 0x00, 0x4B] = 2^23 + b_k as f32
  return __uint_as_float(__byte_perm(word, magic, 0x7440u | (unsigned)k));
}
__device__ __forceinline__ float byte_to_f32(unsigned word, int k, unsigned magic) {
  return __fsub_rn(byte_to_f32_biased(word, k, magic), 8388608.0f);  // subtracting 2^23 is exact
}

// packed f32x2 (sm_100): two independent IEEE round-to-nearest operations per instruction
__device__ __forceinline__ void add2(float& x0, float& x1, float c) {
  uint64_t x, y;
  asm("mov.b64 %0, {%1, %2};" : "=l"(x) : "f"(x0), "f"(x1));
  asm("mov.b64 %0, {%1, %1};" : "=l"(y) : "f"(c));
  asm("add.rn.f32x2 %0, %0, %1;" : "+l"(x) : "l"(y));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(x0), "=f"(x1) : "l"(x));
}
__device__ __forceinline__ void fma2(float& d0, float& d1, float a0, float a1, float b0, float b1) {
  uint64_t d, a, b;
  asm("mov.b64 %0, {%1, %2};" : "=l"(a) : "f"(a0), "f"(a1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(b) : "f"(b0), "f"(b1));
  asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "f"(d0), "f"(d1));
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
  asm("mov.b64 {%0, %1}, %2;" : "=f"(d0), "=f"(d1) : "l"(d));
}

// 16 FMA chains advance by one element each: acc[j] = fma(q[j], float(byte j of v), acc[j]).
// SCALED: the byte enters as the f32 whose BITS are the byte (= b * 2^-149, exact) and the query was pre-multiplied by
// 2^126, so the whole chain runs scaled by 2^-23 and needs no de-biasing FADD: PRMT + FFMA2 only (1.75 instructions
// per byte instead of 2.3). Rounding commutes with the power-of-two scale as long as no intermediate leaves the
// normal range, which the kernel guarantees by taking this path only when every query element is 0 or in
// [2^-80, 4): all partial sums are then multiples of 2^-103, i.e. normal (>= 2^-126) after scaling, or zero.
template <bool SCALED>
__device__ __forceinline__ void fma16(const uint4 v, const float* __restrict__ q, float* acc, unsigned magic) {
  const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    const float4 qv = *reinterpret_cast<const float4*>(q + 4 * g);  // 16-byte aligned by construction
    float x0, x1, x2, x3;
    if (SCALED) {
      x0 = __uint_as_float(__byte_perm(w[g], 0u, 0x4440u));
      x1 = __uint_as_float(__byte_perm(w[g], 0u, 0x4441u));
      x2 = __uint_as_float(__byte_perm(w[g], 0u, 0x4442u));
      x3 = __uint_as_float(__byte_perm(w[g], 0u, 0x4443u));
    } else {
      x0 = byte_to_f32_biased(w[g], 0, magic), x1 = byte_to_f32_biased(w[g], 1, magic);
      x2 = byte_to_f32_biased(w[g], 2, magic), x3 = byte_to_f32_biased(w[g], 3, magic);
      add2(x0, x1, -8388608.0f);
      add2(x2, x3, -8388608.0f);
    }
    fma2(acc[4 * g + 0], acc[4 * g + 1], qv.x, qv.y, x0, x1);
    fma2(acc[4 * g + 2], acc[4 * g + 3], qv.z, qv.w, x2, x3);
  }
}

// the same 16 bytes against TWO queries: the byte -> f32 conversion (the PRMTs) is shared
template <bool SCALED>
__device__ __forceinline__ void fma16_pair(const uint4 v, const float* __restrict__ qa, const float* __restrict__ qb,
                                           float* acc_a, float* acc_b, unsigned magic) {
  const unsigned w[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
  for (int g = 0; g < 4; ++g) {
    float x0, x1, x2, x3;
    if (SCALED) {
      x0 = __uint_as_float(__byte_perm(w[g], 0u, 0x4440u));
      x1 = __uint_as_float(__byte_perm(w[g], 0u, 0x4441u));
      x2 = __uint_as_float(__byte_perm(w[g], 0u, 0x4442u));
      x3 = __uint_as_float(__byte_perm(w[g], 0u, 0x4443u));
    } else {
      x0 = byte_to_f32_biased(w[g], 0, magic), x1 = byte_to_f32_biased(w[g], 1, magic);
      x2 = byte_to_f32_biased(w[g], 2, magic), x3 = byte_to_f32_biased(w[g], 3, magic);
      add2(x0, x1, -8388608.0f);
      add2(x2, x3, -8388608.0f);
    }
    const float4 a4 = *reinterpret_cast<const float4*>(qa + 4 * g);
    fma2(acc_a[4 * g + 0], acc_a[4 * g + 1], a4.x, a4.y, x0, x1);
    fma2(acc_a[4 * g + 2], acc_a[4 * g + 3], a4.z, a4.w, x2, x3);
    const float4 b4 = *reinterpret_cast<const float4*>(qb + 4 * g);
    fma2(acc_b[4 * g + 0], acc_b[4 * g + 1], b4.x, b4.y, x0, x1);
    fma2(acc_b[4 * g + 2], acc_b[4 * g + 3], b4.z, b4.w, x2, x3);
  }
}

__device__ __forceinline__ float hsum8(const float* v) {  // src/arch/x86_64.rs:982-987
  float s0 = __fadd_rn(v[0], v[4]), s1 = __fadd_rn(v[1], v[5]);
  float s2 = __fadd_rn(v[2], v[6]), s3 = __fadd_rn(v[3], v[7]);
  return __fadd_rn(__fadd_rn(s0, s2), __fadd_rn(s1, s3));
}

// Everything after the 32-wide main loop: combine the 32 chains, 8-wide remainder chains, scalar tail; or the
// portable sequential sum when d < 16. w = the (up to) two chunks after the main loop, zero padded.
__device__ __forceinline__ float mixed_dot_finish(const float* acc, const unsigned* w, unsigned d,
                                                  const float* __restrict__ sq, const unsigned magic,
                                                  const float unscale = 1.0f) {
  if (d == 0) return 0.0f;
  if (d < 16) {  // portable path: sequential unfused sum (src/scalar.rs:353-358)
    float s = 0.0f;
#pragma unroll
    for (int e = 0; e < 16; ++e)
      if ((unsigned)e < d) s = __fadd_rn(s, __fmul_rn(sq[e], byte_to_f32(w[e >> 2], e & 3, magic)));
    return s;
  }
  float all[8];
#pragma unroll
  for (int j = 0; j < 8; ++j)
    all[j] = __fadd_rn(__fadd_rn(acc[j], acc[8 + j]), __fadd_rn(acc[16 + j], acc[24 + j]));
  float result = __fmul_rn(hsum8(all), unscale);  // 2^23 on the scaled path (exact), else 1
  const unsigned rs = (d / 32) * 32, remaining = d - rs, n8 = (remaining / 8) * 8;
  if (remaining == 0) return __fadd_rn(result, 0.0f);  // the empty 8-wide accumulator is still added (x86_64.rs:1004-1009)
  float rem[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) rem[j] = 0.0f;
#pragma unroll
  for (int e = 0; e < 24; ++e)  // 8-wide chunks (at most 3)
    if ((unsigned)e < n8) rem[e & 7] = fmaf(sq[rs + e], byte_to_f32(w[e >> 2], e & 3, magic), rem[e & 7]);
  result = __fadd_rn(result, hsum8(rem));  // always added, even when empty (src/arch/x86_64.rs:1004-1009)
#pragma unroll
  for (int e = 0; e < 31; ++e)  // scalar tail, unfused (src/arch/x86_64.rs:1013-1017)
    if ((unsigned)e >= n8 && (unsigned)e < remaining)
      result = __fadd_rn(result, __fmul_rn(sq[rs + e], byte_to_f32(w[e >> 2], e & 3, magic)));
  return result;
}

struct U8Args {
  const uint4* data;
  unsigned long long ld;
  unsigned n, d, chunks, n_tiles, index_base;
  float alpha, offset;
  unsigned magic;      // 0x4B000000 (2^23 as f32 bits), see byte_to_f32
  int allow_scaled;    // option "u8_scaled_chains" (default 1): PRMT + FFMA2 chains when the query allows it
  const float* query;  // device, d floats
  const float* query_b;  // pair kernel: the second query
  int k, mode;         // mode (scores kernel): 0 raw mixed dot, 1 asymmetric score
  uint64_t* partials;
  uint64_t* out_keys;
  uint64_t* group_partials;
  unsigned* tickets;
  float* scores_out;
};

int g_u8_allow_scaled = 1;

struct U8Shared {
  uint64_t full[U8_STAGES], empty[U8_STAGES];
};
// pair kernel: 64 accumulators per thread leave room for one CTA per SM only, so its ring is twice as deep
constexpr int U8_PAIR_STAGES = 12;
struct U8PairShared {
  uint64_t full[U8_PAIR_STAGES], empty[U8_PAIR_STAGES];
};

// bulk copy global -> shared, completion on an mbarrier (complete_tx::bytes); 16-byte aligned, size % 16 == 0
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(tc::smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(tc::smem_u32(bar))
               : "memory");
}

template <int R, bool KNN>
__global__ void __launch_bounds__(U8_CTA, 2) u8_scan_kernel(const U8Args a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  // [ring: U8_STAGES x 16 KB][query d_pad floats][misc 4 floats][barriers][keys]
  unsigned char* ring = smem_raw;
  const unsigned d_pad = (a.d + 31) / 32 * 32 + 32;
  float* sq = reinterpret_cast<float*>(smem_raw + U8_STAGES * U8_STAGE_BYTES);
  float* s_misc = sq + d_pad;  // [0] = query_sum
  U8Shared* st = reinterpret_cast<U8Shared*>(s_misc + 4);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(st + 1);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool producer = warp == U8_THREADS / 32;
  // Scaled chains (see fma16) need every query element of the 32-wide main loop to be 0 or in [2^-80, 4)
  const unsigned main_elems = (a.d >= 16) ? (a.d / 32) * 32 : 0;
  bool q_ok = true;
  for (unsigned i = threadIdx.x; i < d_pad; i += blockDim.x) {
    const float v = i < a.d ? a.query[i] : 0.0f;
    sq[i] = v;
    if (i < main_elems) q_ok &= (v == 0.0f) || (fabsf(v) >= 0x1p-80f && fabsf(v) < 4.0f);  // NaN fails both
  }
  if (threadIdx.x == 0) {
    for (int sg = 0; sg < U8_STAGES; ++sg) {
      tc::mbar_init(&st->full[sg], 1);
      tc::mbar_init(&st->empty[sg], U8_THREADS / 32);
    }
    tc::fence_barrier_init();
  }
  const bool scaled = __syncthreads_and(q_ok) && a.allow_scaled;
  if (threadIdx.x == 32) {  // query_context: query.iter().sum() sequential (src/scalar.rs:236-240), from the shared copy
    float s = 0.0f;         // (a dependent chain of global loads would delay every CTA by several microseconds)
    for (unsigned i = 0; i < a.d; ++i) s = __fadd_rn(s, sq[i]);
    s_misc[0] = s;
  }
  __syncthreads();
  if (scaled) {  // only the main-loop part; the remainder / portable paths read the query as given
    for (unsigned i = threadIdx.x; i < main_elems; i += blockDim.x) sq[i] *= 0x1p126f;  // exact: |q| < 4
    __syncthreads();
  }
  const float scale = __fdiv_rn(a.alpha, 255.0f);             // params.alpha / 255.0
  const float bias = __fmul_rn(a.offset, s_misc[0]);          // params.offset * ctx.query_sum
  const unsigned stages_per_tile = (a.chunks + U8_STAGE_CHUNKS - 1) / U8_STAGE_CHUNKS;
  const unsigned main_chunks = (a.d >= 16) ? (a.d / 32) * 2 : 0;  // chunks consumed by the 32-wide loop

  WarpList<R> lists[1];
  uint64_t thrs[1];
  lists[0].init();
  thrs[0] = KEY_SENTINEL;

  if (producer) {
    if (lane == 0) {
      unsigned slot = 0, phase = 1;  // the first pass over the ring finds every slot free
      for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const unsigned long long col = (unsigned long long)tile * U8_THREADS;
        const unsigned long long left = a.ld - col;  // vectors of this tile inside the row pitch (multiple of 16)
        const unsigned row_bytes = (unsigned)(left < U8_THREADS ? left : U8_THREADS) * 16u;
        for (unsigned sgi = 0; sgi < stages_per_tile; ++sgi) {
          const unsigned c0 = sgi * U8_STAGE_CHUNKS;
          const unsigned rows = min((unsigned)U8_STAGE_CHUNKS, a.chunks - c0);
          while (!tc::mbar_try_wait(&st->empty[slot], phase)) __nanosleep(64);  // do not steal issue slots while full
          tc::mbar_arrive_expect_tx(&st->full[slot], rows * row_bytes);
          for (unsigned r = 0; r < rows; ++r)
            bulk_load(ring + slot * U8_STAGE_BYTES + r * U8_ROW_BYTES, a.data + (size_t)(c0 + r) * a.ld + col, row_bytes,
                      &st->full[slot]);
          if (++slot == U8_STAGES) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else {
   auto consume = [&](auto scaled_tag) {
    constexpr bool SCALED = decltype(scaled_tag)::value;
    const unsigned full_stages = main_chunks / U8_STAGE_CHUNKS;  // stages made of main-loop chunks only
    unsigned slot = 0, phase = 0;
    const uint4* const ring_v = reinterpret_cast<const uint4*>(ring) + threadIdx.x;
    for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
      const unsigned i = tile * U8_THREADS + threadIdx.x;
      const bool valid = i < a.n;
      float acc[32];
#pragma unroll
      for (int c = 0; c < 32; ++c) acc[c] = 0.0f;
      unsigned w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      unsigned sgi = 0;
      const float* qp = sq;
      for (; sgi < full_stages; ++sgi, qp += 16 * U8_STAGE_CHUNKS) {
        tc::mbar_wait(&st->full[slot], phase);
        const uint4* sv = ring_v + slot * (U8_STAGE_BYTES / 16);
        uint4 v[U8_STAGE_CHUNKS];
#pragma unroll
        for (int g = 0; g < U8_STAGE_CHUNKS; ++g) v[g] = sv[g * U8_THREADS];
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&st->empty[slot]);  // the slot is in registers: the producer may refill it
        if (++slot == U8_STAGES) { slot = 0; phase ^= 1; }
#pragma unroll
        for (int g = 0; g < U8_STAGE_CHUNKS; ++g) fma16<SCALED>(v[g], qp + 16 * g, acc + 16 * (g & 1), a.magic);
      }
      for (; sgi < stages_per_tile; ++sgi) {  // last stage(s): remainder chunks (d % 64 != 0), or everything when d < 16
        const unsigned c0 = sgi * U8_STAGE_CHUNKS;
        tc::mbar_wait(&st->full[slot], phase);
        const uint4* sv = ring_v + slot * (U8_STAGE_BYTES / 16);
        uint4 v[U8_STAGE_CHUNKS];
#pragma unroll
        for (int g = 0; g < U8_STAGE_CHUNKS; ++g) v[g] = sv[g * U8_THREADS];  // rows past `chunks`: stale, unused
        __syncwarp();
        if (lane == 0) tc::mbar_arrive(&st->empty[slot]);
        if (++slot == U8_STAGES) { slot = 0; phase ^= 1; }
#pragma unroll
        for (int g = 0; g < U8_STAGE_CHUNKS; ++g) {
          const unsigned c = c0 + g;
          if (c < main_chunks) {
            fma16<SCALED>(v[g], sq + 16 * c, acc + 16 * (g & 1), a.magic);
          } else if (c < a.chunks) {  // the (up to) two chunks of the remainder / of the d < 16 path
            if (c == main_chunks) { w[0] = v[g].x; w[1] = v[g].y; w[2] = v[g].z; w[3] = v[g].w; }
            else { w[4] = v[g].x; w[5] = v[g].y; w[6] = v[g].z; w[7] = v[g].w; }
          }
        }
      }
      const float mixed = mixed_dot_finish(acc, w, a.d, sq, a.magic, SCALED ? 0x1p23f : 1.0f);
      const float score = (KNN || a.mode == 1) ? __fadd_rn(__fmul_rn(scale, mixed), bias) : mixed;  // src/scalar.rs:299
      if (KNN) lists[0].offer(make_key_desc(score, a.index_base + i), valid, thrs[0], a.k, lane);
      else if (valid) a.scores_out[i] = score;
    }
   };
   if (scaled) consume(std::true_type{}); else consume(std::false_type{});
  }
  // the producer warp takes part in the CTA-wide merge with an empty list
  if (KNN) block_finish<R, 1>(lists, 1, a.k, smem_keys, a.partials, a.group_partials, a.out_keys, a.tickets);
}

// Two queries per pass (top-k only): the scan is instruction-bound under the power cap and the byte -> f32 conversion is
// more than half of its instructions, so a second query rides along for ~40 % more work instead of 100 %.
// a.query = query A, a.query_b = query B; keys to a.out_keys (A) and a.out_keys + k (B).
template <int R>
__global__ void __launch_bounds__(U8_CTA, 1) u8_scan_pair_kernel(const U8Args a) {
  extern __shared__ __align__(1024) unsigned char smem_raw[];
  unsigned char* ring = smem_raw;
  const unsigned d_pad = (a.d + 31) / 32 * 32 + 32;
  float* sqa = reinterpret_cast<float*>(smem_raw + U8_PAIR_STAGES * U8_STAGE_BYTES);
  float* sqb = sqa + d_pad;
  float* s_misc = sqb + d_pad;  // [0], [1] = query sums
  U8PairShared* st = reinterpret_cast<U8PairShared*>(s_misc + 4);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(st + 1);
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const bool producer = warp == U8_THREADS / 32;
  const unsigned main_elems = (a.d >= 16) ? (a.d / 32) * 32 : 0;
  bool q_ok = true;
  for (unsigned i = threadIdx.x; i < d_pad; i += blockDim.x) {
    const float va = i < a.d ? a.query[i] : 0.0f, vb = i < a.d ? a.query_b[i] : 0.0f;
    sqa[i] = va;
    sqb[i] = vb;
    if (i < main_elems)
      q_ok &= ((va == 0.0f) || (fabsf(va) >= 0x1p-80f && fabsf(va) < 4.0f)) &&
              ((vb == 0.0f) || (fabsf(vb) >= 0x1p-80f && fabsf(vb) < 4.0f));
  }
  if (threadIdx.x == 0) {
    for (int sg = 0; sg < U8_PAIR_STAGES; ++sg) {
      tc::mbar_init(&st->full[sg], 1);
      tc::mbar_init(&st->empty[sg], U8_THREADS / 32);
    }
    tc::fence_barrier_init();
  }
  const bool scaled = __syncthreads_and(q_ok) && a.allow_scaled;
  if (threadIdx.x == 32 || threadIdx.x == 64) {  // query_context of each query: sequential sum (src/scalar.rs:236-240)
    const float* qp = threadIdx.x == 64 ? sqb : sqa;
    float sum = 0.0f;
    for (unsigned i = 0; i < a.d; ++i) sum = __fadd_rn(sum, qp[i]);
    s_misc[threadIdx.x == 64 ? 1 : 0] = sum;
  }
  __syncthreads();
  if (scaled) {
    for (unsigned i = threadIdx.x; i < main_elems; i += blockDim.x) {
      sqa[i] *= 0x1p126f;
      sqb[i] *= 0x1p126f;
    }
    __syncthreads();
  }
  const float scale = __fdiv_rn(a.alpha, 255.0f);
  const float bias_a = __fmul_rn(a.offset, s_misc[0]), bias_b = __fmul_rn(a.offset, s_misc[1]);
  const unsigned stages_per_tile = (a.chunks + U8_STAGE_CHUNKS - 1) / U8_STAGE_CHUNKS;
  const unsigned main_chunks = (a.d >= 16) ? (a.d / 32) * 2 : 0;

  WarpList<R> lists[2];
  uint64_t thrs[2];
  lists[0].init();
  lists[1].init();
  thrs[0] = thrs[1] = KEY_SENTINEL;

  if (producer) {
    if (lane == 0) {
      unsigned slot = 0, phase = 1;
      for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const unsigned long long col = (unsigned long long)tile * U8_THREADS;
        const unsigned long long left = a.ld - col;
        const unsigned row_bytes = (unsigned)(left < U8_THREADS ? left : U8_THREADS) * 16u;
        for (unsigned sgi = 0; sgi < stages_per_tile; ++sgi) {
          const unsigned c0 = sgi * U8_STAGE_CHUNKS;
          const unsigned rows = min((unsigned)U8_STAGE_CHUNKS, a.chunks - c0);
          while (!tc::mbar_try_wait(&st->empty[slot], phase)) __nanosleep(64);
          tc::mbar_arrive_expect_tx(&st->full[slot], rows * row_bytes);
          for (unsigned r = 0; r < rows; ++r)
            bulk_load(ring + slot * U8_STAGE_BYTES + r * U8_ROW_BYTES, a.data + (size_t)(c0 + r) * a.ld + col, row_bytes,
                      &st->full[slot]);
          if (++slot == U8_PAIR_STAGES) { slot = 0; phase ^= 1; }
        }
      }
    }
  } else {
    auto consume = [&](auto scaled_tag) {
      constexpr bool SCALED = decltype(scaled_tag)::value;
      unsigned slot = 0, phase = 0;
      const uint4* const ring_v = reinterpret_cast<const uint4*>(ring) + threadIdx.x;
      for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
        const unsigned i = tile * U8_THREADS + threadIdx.x;
        const bool valid = i < a.n;
        float acc_a[32], acc_b[32];
#pragma unroll
        for (int c = 0; c < 32; ++c) acc_a[c] = acc_b[c] = 0.0f;
        unsigned w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (unsigned sgi = 0; sgi < stages_per_tile; ++sgi) {
          const unsigned c0 = sgi * U8_STAGE_CHUNKS;
          tc::mbar_wait(&st->full[slot], phase);
          const uint4* sv = ring_v + slot * (U8_STAGE_BYTES / 16);
          uint4 v[U8_STAGE_CHUNKS];
#pragma unroll
          for (int g = 0; g < U8_STAGE_CHUNKS; ++g) v[g] = sv[g * U8_THREADS];  // rows past `chunks`: stale, unused
          __syncwarp();
          if (lane == 0) tc::mbar_arrive(&st->empty[slot]);
          if (++slot == U8_PAIR_STAGES) { slot = 0; phase ^= 1; }
#pragma unroll
          for (int g = 0; g < U8_STAGE_CHUNKS; ++g) {
            const unsigned c = c0 + g;
            if (c < main_chunks) {
              fma16_pair<SCALED>(v[g], sqa + 16 * c, sqb + 16 * c, acc_a + 16 * (g & 1), acc_b + 16 * (g & 1), a.magic);
            } else if (c < a.chunks) {
              if (c == main_chunks) { w[0] = v[g].x; w[1] = v[g].y; w[2] = v[g].z; w[3] = v[g].w; }
              else { w[4] = v[g].x; w[5] = v[g].y; w[6] = v[g].z; w[7] = v[g].w; }
            }
          }
        }
        const float unscale = SCALED ? 0x1p23f : 1.0f;
        const float ma = mixed_dot_finish(acc_a, w, a.d, sqa, a.magic, unscale);
        const float mb = mixed_dot_finish(acc_b, w, a.d, sqb, a.magic, unscale);
        lists[0].offer(make_key_desc(__fadd_rn(__fmul_rn(scale, ma), bias_a), a.index_base + i), valid, thrs[0], a.k, lane);
        lists[1].offer(make_key_desc(__fadd_rn(__fmul_rn(scale, mb), bias_b), a.index_base + i), valid, thrs[1], a.k, lane);
      }
    };
    if (scaled) consume(std::true_type{}); else consume(std::false_type{});
  }
  block_finish<R, 2>(lists, 2, a.k, smem_keys, a.partials, a.group_partials, a.out_keys, a.tickets);
}

__global__ void u8_pack_kernel(const uint8_t* __restrict__ rows, unsigned n, unsigned d, uint4* __restrict__ codes,
                               size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    unsigned w[4] = {0, 0, 0, 0};
    if (i < n) {
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        unsigned dd = 16 * c + e;
        if (dd < d) w[e >> 2] |= (unsigned)rows[i * d + dd] << (8 * (e & 3));
      }
    }
    codes[t] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__device__ __forceinline__ unsigned quantize_one(float v, float offset, float inv_alpha) {
  // let normalized = (v - params.offset) * inv_alpha; normalized.round().clamp(0.0, 255.0) as u8
  float r = roundf(__fmul_rn(__fsub_rn(v, offset), inv_alpha));  // f32::round: half away from zero
  if (r != r) return 0u;                                         // NaN as u8 == 0
  r = fminf(fmaxf(r, 0.0f), 255.0f);
  return (unsigned)r;
}

__global__ void generate_u8_kernel(uint64_t salt, uint64_t first_row, unsigned n, unsigned d, float alpha,
                                   float offset, uint4* __restrict__ codes, size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  const float inv_alpha = __fdiv_rn(255.0f, alpha);
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    unsigned w[4] = {0, 0, 0, 0};
    if (i < n) {
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        unsigned dd = 16 * c + e;
        if (dd < d) {
          float v = ghash_value(salt, (first_row + i) * d + dd);
          w[e >> 2] |= quantize_one(v, offset, inv_alpha) << (8 * (e & 3));
        }
      }
    }
    codes[t] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

// quantize_u8 (src/scalar.rs:212-225) of a device-resident PDX f32 corpus straight into the chunk-major u8 layout:
// thread (chunk c, vector i) reads 16 dimension rows (coalesced along i) and writes one uint4
__global__ void u8_from_pdx_kernel(const PdxView pdx, unsigned n, unsigned d, float alpha,
                                   float offset, uint4* __restrict__ codes, size_t ld, unsigned chunks) {
  const size_t total = (size_t)chunks * ld;
  const float inv_alpha = __fdiv_rn(255.0f, alpha);
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned c = (unsigned)(t / ld);
    const size_t i = t % ld;
    unsigned w[4] = {0, 0, 0, 0};
    if (i < n) {
#pragma unroll
      for (int e = 0; e < 16; ++e) {
        const unsigned dd = 16 * c + e;
        if (dd < d) w[e >> 2] |= quantize_one(pdx_load1(pdx, (size_t)dd * pdx.ld + i), offset, inv_alpha) << (8 * (e & 3));
      }
    }
    codes[t] = make_uint4(w[0], w[1], w[2], w[3]);
  }
}

__global__ void quantize_u8_kernel(const float* __restrict__ values, size_t n, float alpha, float offset,
                                   uint8_t* __restrict__ out) {
  const float inv_alpha = __fdiv_rn(255.0f, alpha);
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < n; t += (size_t)gridDim.x * blockDim.x)
    out[t] = (uint8_t)quantize_one(values[t], offset, inv_alpha);
}

size_t u8_smem(size_t d, size_t k, bool knn) {
  size_t d_pad = (d + 31) / 32 * 32 + 32;
  return (size_t)U8_STAGES * U8_STAGE_BYTES + (d_pad + 4) * sizeof(float) + sizeof(U8Shared) +
         (knn ? (size_t)(U8_CTA / 32) * k * sizeof(uint64_t) : 0);
}

template <int R, bool KNN>
cudaError_t launch_u8(const U8Args& a, size_t smem, int num_sms, cudaStream_t s) {
  auto kern = u8_scan_kernel<R, KNN>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
  }
  int occ = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, U8_CTA, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  unsigned grid = balanced_grid(a.n_tiles, (unsigned)occ * (unsigned)num_sms);  // persistent: the ring stays warm
  kern<<<grid, U8_CTA, smem, s>>>(a);
  return cudaGetLastError();
}

U8Args make_args(const U8View& v, const float* q) {
  U8Args a{};
  a.data = v.data;
  a.ld = v.ld;
  a.n = (unsigned)v.n;
  a.d = (unsigned)v.d;
  a.chunks = (unsigned)v.chunks;
  a.n_tiles = (unsigned)((v.n + U8_THREADS - 1) / U8_THREADS);
  a.index_base = v.index_base;
  a.alpha = v.alpha;
  a.offset = v.offset;
  a.magic = 0x4B000000u;
  a.allow_scaled = g_u8_allow_scaled;
  a.query = q;
  return a;
}

}  // namespace

void u8_set_scaled_chains(bool on) { g_u8_allow_scaled = on ? 1 : 0; }

cudaError_t launch_u8_pack(const uint8_t* dev_rows, size_t n, size_t d, uint4* dev_codes, size_t ld,
                           cudaStream_t s, LaunchCounter* launches) {
  if (n == 0 || d == 0) return cudaSuccess;
  u8_pack_kernel<<<148 * 8, 256, 0, s>>>(dev_rows, (unsigned)n, (unsigned)d, dev_codes, ld, (unsigned)((d + 15) / 16));
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_generate_u8(uint64_t salt, uint64_t first_row, size_t n, size_t d, float alpha, float offset,
                               uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches) {
  if (n == 0 || d == 0) return cudaSuccess;
  generate_u8_kernel<<<148 * 16, 256, 0, s>>>(salt, first_row, (unsigned)n, (unsigned)d, alpha, offset, dev_codes, ld,
                                              (unsigned)((d + 15) / 16));
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_u8_from_pdx(const PdxView& v, float alpha, float offset,
                               uint4* dev_codes, size_t ld, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0 || v.d == 0) return cudaSuccess;
  u8_from_pdx_kernel<<<148 * 16, 256, 0, s>>>(v, (unsigned)v.n, (unsigned)v.d, alpha, offset, dev_codes, ld,
                                              (unsigned)((v.d + 15) / 16));
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_quantize_u8(const float* dev_values, size_t n, float alpha, float offset, uint8_t* dev_out,
                               cudaStream_t s, LaunchCounter* launches) {
  if (n == 0) return cudaSuccess;
  unsigned grid = (unsigned)((n + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  quantize_u8_kernel<<<grid, 256, 0, s>>>(dev_values, n, alpha, offset, dev_out);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_u8_scores(const U8View& v, int mode, const float* dev_query, float* dev_out,
                             cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0) return cudaSuccess;
  U8Args a = make_args(v, dev_query);
  a.mode = mode;
  a.scores_out = dev_out;
  size_t smem = u8_smem(v.d, 0, false);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  cudaError_t e = launch_u8<1, false>(a, smem, 148, s);
  if (e == cudaSuccess) ++*launches;
  return e;
}

namespace {
template <int R>
cudaError_t launch_u8_pair(const U8Args& a, size_t smem, int num_sms, cudaStream_t s) {
  auto kern = u8_scan_pair_kernel<R>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
  if (e != cudaSuccess) return e;
  int occ = 0;
  e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, U8_CTA, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  kern<<<balanced_grid(a.n_tiles, (unsigned)occ * (unsigned)num_sms), U8_CTA, smem, s>>>(a);
  return cudaGetLastError();
}
}  // namespace

cudaError_t launch_u8_knn(const U8View& v, const float* dev_queries, size_t nq, size_t k, uint64_t* dev_keys,
                          Workspace& ws, cudaStream_t s, LaunchCounter* launches) {
  if (k > 128) return cudaErrorInvalidValue;
  size_t smem = u8_smem(v.d, k, true);
  if (smem > 227 * 1024) return cudaErrorInvalidValue;
  size_t q0 = 0;
  // query batches: two queries per pass
  const size_t d_pad = (v.d + 31) / 32 * 32 + 32;
  const size_t pair_smem = (size_t)U8_PAIR_STAGES * U8_STAGE_BYTES + (2 * d_pad + 4) * sizeof(float) + sizeof(U8PairShared) +
                           2 * (size_t)(U8_CTA / 32) * k * sizeof(uint64_t);
  for (; nq - q0 >= 2 && pair_smem <= 227 * 1024; q0 += 2) {
    U8Args a = make_args(v, dev_queries + q0 * v.d);
    a.query_b = dev_queries + (q0 + 1) * v.d;
    a.k = (int)k;
    a.partials = ws.partials;
    a.group_partials = ws.group_partials;
    a.tickets = ws.tickets;
    a.out_keys = dev_keys + q0 * k;
    cudaError_t e = (k <= 32) ? launch_u8_pair<1>(a, pair_smem, ws.num_sms, s) : launch_u8_pair<4>(a, pair_smem, ws.num_sms, s);
    if (e != cudaSuccess) return e;
    ++*launches;
  }
  for (size_t q = q0; q < nq; ++q) {
    U8Args a = make_args(v, dev_queries + q * v.d);
    a.k = (int)k;
    a.partials = ws.partials;
    a.group_partials = ws.group_partials;
    a.tickets = ws.tickets;
    a.out_keys = dev_keys + q * k;
    cudaError_t e = (k <= 32) ? launch_u8<1, true>(a, smem, ws.num_sms, s) : launch_u8<4, true>(a, smem, ws.num_sms, s);
    if (e != cudaSuccess) return e;
    ++*launches;
  }
  return cudaSuccess;
}

}  // namespace innr
