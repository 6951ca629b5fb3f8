// pdx.cuh -- the one place that knows how an f32 PDX corpus is stored on the device.
//
// Plain: data[dd * ld + i] (f32). Split (owned corpora of at least f32_split_min_rows rows): the same bytes as two u16
// planes of the same pitch, hi[dd * ld + i] = the high 16 bits of the f32 (sign, exponent, 7 mantissa bits) and
// lo[dd * ld + i] = its low 16 bits. Joining the halves gives back the f32 bit for bit, so every reader computes what it
// computes on a plain corpus. The layout is the same for every thread of a launch, so the branch below is uniform.
// A split corpus also has an 8-bit sketch (PdxSketch, built in layout.cu, read by the screened single-query kNN in
// scan_f32.cu) in the same dimension-major order and pitch: pdx_sketch_off.
#pragma once
#include "common.cuh"
#include "kernels.cuh"

namespace innr {

__device__ __forceinline__ uint2 ldg_stream_u2(const uint16_t* p) {
  uint2 r;
  asm volatile("ld.global.nc.L1::no_allocate.v2.u32 {%0, %1}, [%2];" : "=r"(r.x), "=r"(r.y) : "l"(p));
  return r;
}

// elements off .. off + 3 of the corpus (off = dd * ld + i, i % 4 == 0): one 16 B load plain, two 8 B loads split.
// pdx_load4_as<SPLIT> is for loops that branch on the layout once, outside the loop.
template <bool SPLIT>
__device__ __forceinline__ float4 pdx_load4_as(const PdxView& v, size_t off) {
  if (SPLIT) {
    const uint2 h = ldg_stream_u2(v.hi + off), l = ldg_stream_u2(v.lo + off);
    return make_float4(__uint_as_float(__byte_perm(l.x, h.x, 0x5410)), __uint_as_float(__byte_perm(l.x, h.x, 0x7632)),
                       __uint_as_float(__byte_perm(l.y, h.y, 0x5410)), __uint_as_float(__byte_perm(l.y, h.y, 0x7632)));
  }
  return ldg_stream_f4(v.data + off);
}
__device__ __forceinline__ float4 pdx_load4(const PdxView& v, size_t off) {
  return v.hi ? pdx_load4_as<true>(v, off) : pdx_load4_as<false>(v, off);
}

// one element (gathers, tails)
__device__ __forceinline__ float pdx_load1(const PdxView& v, size_t off) {
  if (v.hi) return __uint_as_float(((uint32_t)__ldg(v.hi + off) << 16) | (uint32_t)__ldg(v.lo + off));
  return __ldg(v.data + off);
}

// writers: element `off` of a corpus being built (dst_f for plain, dst_hi / dst_lo for split)
__device__ __forceinline__ void pdx_store1(float* dst_f, uint16_t* dst_hi, uint16_t* dst_lo, size_t off, float x) {
  if (dst_hi) {
    const uint32_t b = __float_as_uint(x);
    dst_hi[off] = (uint16_t)(b >> 16);
    dst_lo[off] = (uint16_t)b;
  } else {
    dst_f[off] = x;
  }
}

// the sketch code of element dd of row i: one byte per element, so one 16 B load holds 16 consecutive rows of one
// dimension and the next dimension is ld bytes further on
__device__ __forceinline__ size_t pdx_sketch_off(size_t ld, size_t dd, size_t i) { return dd * ld + i; }

}  // namespace innr
