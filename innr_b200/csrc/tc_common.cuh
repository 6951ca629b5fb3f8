// tc_common.cuh -- minimal sm_100a building blocks written as inline PTX: mbarrier, TMA (cp.async.bulk.tensor),
// tcgen05 (alloc / mma kind::tf32 / commit / ld / fences), UMMA shared-memory + instruction descriptors.
// Bit layouts follow the PTX ISA as mirrored by CuTe's cute/arch/mma_sm100_desc.hpp (read for layouts only).
#pragma once
#include <cuda.h>
#include <cuda_runtime.h>
#include <stdint.h>

namespace innr {
namespace tc {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier -------------------------------------------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  while (!mbar_try_wait(bar, parity)) {
  }
}

// ---- TMA ------------------------------------------------------------------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const CUtensorMap* m) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(m) : "memory");
}
// 2D tile load global -> shared, completion on an mbarrier (complete_tx::bytes)
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
      ::"r"(smem_u32(smem_dst)), "l"(m), "r"(smem_u32(bar)), "r"(c0), "r"(c1)
      : "memory");
}
// generic-proxy writes to shared memory -> visible to the async proxy (TMA / tcgen05.mma operand reads)
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}

// ---- tcgen05 ----------------------------------------------------------------------------------------------------
template <int NCOLS>
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst) {  // one full warp
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "n"(NCOLS)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
template <int NCOLS>
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr) {  // the same warp that allocated
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "n"(NCOLS) : "memory");
}
__device__ __forceinline__ void tc_fence_before_sync() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after_sync() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem] * B[smem], kind::tf32, issued by ONE thread
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                          uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// all previously issued MMAs of this thread -> arrive(1) on the mbarrier when they complete
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar))
               : "memory");
}
// TMEM -> registers: lane l of the warp reads TMEM lane (taddr.lane + l), 32 consecutive 32-bit columns
__device__ __forceinline__ void tmem_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]), "=r"(r[16]),
        "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]),
        "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
// registers -> TMEM: lane l of the warp writes TMEM lane (taddr.lane + l), 32 consecutive 32-bit columns
__device__ __forceinline__ void tmem_st_32x32b_x32(uint32_t taddr, const uint32_t (&r)[32]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_32x32b_x1(uint32_t taddr, uint32_t v) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x1.b32 [%0], {%1};" ::"r"(taddr), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t tmem_ld_32x32b_x1(uint32_t taddr) {
  uint32_t v;
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x1.b32 {%0}, [%1];" : "=r"(v) : "r"(taddr) : "memory");
  return v;
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
// D[tmem] (+)= A[tmem] * B[smem]: A is M lanes x K 32-bit columns in tensor memory
__device__ __forceinline__ void umma_tf32_ts(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc,
                                             uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
// compile-time accumulate flag (the predicate folds to PT / !PT: no SETP, no register) for fully unrolled K loops
template <bool ACC>
__device__ __forceinline__ void umma_tf32_c(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "n"(ACC ? 1 : 0)
      : "memory");
}
template <bool ACC>
__device__ __forceinline__ void umma_tf32_ts_c(uint32_t d_tmem, uint32_t a_tmem, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n\t}"
      ::"r"(d_tmem), "r"(a_tmem), "l"(b_desc), "r"(idesc), "n"(ACC ? 1 : 0)
      : "memory");
}
// one lane of a converged warp (the warp runs the surrounding control flow uniformly, so descriptors and addresses
// stay in uniform registers; only the tcgen05 issue itself is single-lane)
__device__ __forceinline__ bool elect_one_sync() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "elect.sync _|p, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, p;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
// descriptor of the same operand `bytes` further on (the start-address field counts 16-byte units; no carry out of it
// for offsets inside one buffer)
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (uint64_t)(bytes >> 4); }
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// ---- integer MMAs on K-major byte operands (u8_tc.cu, bin_tc.cu) ----------------------------------------------------
// one contiguous global -> shared bulk copy (no tensor map), completion on an mbarrier (complete_tx::bytes)
__device__ __forceinline__ void bulk_load(void* smem_dst, const void* gsrc, unsigned bytes, uint64_t* bar) {
  asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
               ::"r"(smem_u32(smem_dst)), "l"(gsrc), "r"(bytes), "r"(smem_u32(bar))
               : "memory");
}
template <bool ACC>
__device__ __forceinline__ void umma_i8_c(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::i8 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "n"(ACC ? 1 : 0)
      : "memory");
}
// kind::i8: D = S32 (c_format 2), A = UINT8 (a_format 0), B = INT8 (b_format 1), both K-major
__device__ __forceinline__ uint32_t make_idesc_u8s8(int M, int N) {
  return (2u << 4) | (0u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}
// K-major operand without swizzle: 8-row x 16-byte core matrices (128 contiguous bytes); SBO = byte stride between
// core matrices along M / N (8 rows), LBO = byte stride between them along K (one chunk to the next)
__device__ __forceinline__ uint64_t make_smem_desc_kmajor_noswizzle(uint32_t smem_addr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;  // version; layout type 0 = SWIZZLE_NONE
  return d;
}

// ---- descriptors ----------------------------------------------------------------------------------------------------
// K-major operand panel stored as [rows][128 bytes] with the 128-byte swizzle (what TMA SWIZZLE_128B writes):
// canonical layout ((8,n),2):((8,SBO),1) in 16-byte units -> SBO = 8 rows * 128 B = 1024 B, LBO unused (1).
// bits: [0,14) start>>4 | [16,30) LBO>>4 | [32,46) SBO>>4 | [46,48) version=1 | [49,52) base_offset | [61,64) layout
__device__ __forceinline__ uint64_t make_smem_desc_kmajor_sw128(uint32_t smem_addr) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)1 << 16;
  d |= (uint64_t)(1024 >> 4) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;  // SWIZZLE_128B
  return d;
}
// MN-major operand (contiguous along M/N, e.g. a PDX corpus tile [k][vector]) stored as TMA SWIZZLE_128B boxes of
// [k rows][32 floats]: canonical layout ((8,n),(8,k)):((1,LBO),(8,SBO)) in 16-byte units -> LBO = byte stride between
// 32-element MN atoms (the box stride), SBO = byte stride between 8-row K atoms (1024 B inside a box).
// For 32-bit (tf32) MN-major operands the only legal shared-memory layout is SWIZZLE_128B_BASE32B (layout type 1):
// 128-byte rows, 32-byte chunks XOR-ed with (row % 4) -- what TMA writes with CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
// the K atom is 4 rows (512 B).
__device__ __forceinline__ uint64_t make_smem_desc_mnmajor_sw128_32b(uint32_t smem_addr, uint32_t lbo_bytes,
                                                                     uint32_t sbo_bytes) {
  uint64_t d = 0;
  d |= (uint64_t)((smem_addr >> 4) & 0x3FFF);
  d |= (uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16;
  d |= (uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)1 << 61;  // SWIZZLE_128B_BASE32B
  return d;
}
// kind::tf32, F32 accumulate, A and B K-major: c_format[4,6)=1, a_format[7,10)=2, b_format[10,13)=2,
// n_dim[17,23)=N>>3, m_dim[24,29)=M>>4
__host__ __device__ constexpr uint32_t make_idesc_tf32(int M, int N, bool a_mn_major = false) {
  return (1u << 4) | (2u << 7) | (2u << 10) | (a_mn_major ? (1u << 15) : 0u) | ((uint32_t)(N >> 3) << 17) |
         ((uint32_t)(M >> 4) << 24);
}

}  // namespace tc

// ---- host: tensor map for a row-major f32 matrix [rows][cols], box = 32 floats x box_rows, 128B swizzle ----
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

// pitch_floats: row pitch of the matrix in floats (>= cols; 0 = dense)
inline bool make_tmap_f32_rows(CUtensorMap* m, const float* base, uint64_t rows, uint64_t cols, uint32_t box_rows,
                               uint64_t pitch_floats = 0, bool atom32 = false) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return false;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {(pitch_floats ? pitch_floats : cols) * sizeof(float)};
  cuuint32_t box[2] = {32, box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, (void*)base, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
             atom32 ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B,
             CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

}  // namespace innr
