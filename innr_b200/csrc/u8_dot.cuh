// u8_dot.cuh -- the per-vector arithmetic of the bit-exact f32 x u8 mixed dot product (u8.cu header), shared by the scan
// kernels (u8.cu) and the exact rescoring of the tensor-core filter (u8_tc.cu), so both produce the same bits.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace innr {
namespace {

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

}  // namespace
}  // namespace innr
