// u8_tc.cu -- batch_knn_u8 for query batches with the tensor cores as an exact-result FILTER (DESIGN.md section 3.10).
//
// The reference scores a pair as f(mixed) = RN(RN(c * mixed) + RN(offset * query_sum)), c = RN(alpha / 255)
// (src/scalar.rs:299), where mixed is the 32-chain FMA sum of q_j * b_j (u8.cu header). For c > 0, f is monotone
// non-decreasing, so an interval [L, U] around the reference's `mixed` gives f(L) <= score <= f(U), computed with the
// reference's own two operations. The tensor cores deliver the integer part of that interval:
//
//   0. once per corpus  r_i = ||b_i - 128||_2 over the real d, rounded up (4 B per row)
//   1. per call         query -> qi_j = rint(q_j 2^p) in [-127, 127] (2^p: the power of two with max|q| 2^p in
//                       [63.5, 127)), e_j = q_j - 2^-p qi_j (exact), the s8 operand in the corpus' chunk-major layout
//   2. filter passes    A_i = sum_j qi_j b_j on tcgen05 (kind::i8, u8 codes as A, s8 queries as B, s32 in TMEM). Then
//                         sum_j q_j b_j = 2^-p A_i + 128 sum_j e_j + sum_j e_j (b_j - 128)
//                       and the last term is within +-||e||_2 r_i (Cauchy-Schwarz); the reference's own rounding adds
//                       +-G = gamma_(d+16) 255 sum|q_j| + (2d + 64) 2^-149. Every constant is rounded outwards, the
//                       interval ends are evaluated with directed rounding, and the s32 -> f32 conversion rounds down /
//                       up (exact below 2^24). The passes follow tc_filter.cuh: prefixes of the corpus, the k-th lower
//                       bound of one pass is the threshold of the next.
//   3. rescore          the final candidates are re-scored with the scan's own per-vector code (u8_dot.cuh) and selected
//                       on the scan's keys -> indices and scores bit-identical to the u8 scan. A query whose list
//                       overflows, or that the filter does not answer (non-finite or all-zero elements, max|q| outside
//                       [2^-100, 2^100], non-finite offset * query_sum), is re-run on the exact scan by the caller.
//
// Filter kernel: persistent, one CTA per SM, 192 threads: 4 epilogue warps, bulk-copy producer warp, MMA issuer warp.
// Work unit = 128 rows x 256 queries, query group fastest (the row tile of consecutive units comes from L2), K loop over
// blocks of 8 chunks (128 dimensions): A = 8 x 2 KB chunk rows of the corpus as stored (each 128-row chunk is one
// contiguous 2 KB run of codes[c * ld + i], a column of 16 canonical 8 x 16-byte core matrices), B = 8 x 4 KB of the
// query operand; 4 stages of 48 KB, 4 MMAs (M128 N256 K32) per block, two 256-column accumulators in TMEM.
// The epilogue is the expected limiter: per (row, query) it makes one integer compare of A_i against a per-query
// threshold on A valid for every row radius of the warp; only pairs that pass evaluate the exact interval.
#include <cfloat>
#include <climits>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "kernels.cuh"
#include "tc_common.cuh"
#include "tc_filter.cuh"
#include "u8_dot.cuh"

namespace innr {

namespace {

using namespace tc;
using tcf::CAND_CAP;

constexpr int UT_THREADS = 192;
constexpr int VT = 128;       // rows per work unit (UMMA M)
constexpr int QT = 256;       // queries per work unit (UMMA N, up to)
constexpr int KC = 8;         // chunks (16 dimensions each) per K block
constexpr int STAGES = 4;
constexpr int A_CHUNK_BYTES = VT * 16;      // 2 KB: one chunk of a 128-row tile
constexpr int B_CHUNK_BYTES = QT * 16;      // 4 KB: one chunk of a 256-query group
constexpr int A_BYTES = KC * A_CHUNK_BYTES;  // 16 KB
constexpr int B_BYTES = KC * B_CHUNK_BYTES;  // 32 KB
constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
constexpr int QAUX = 7;       // per-query constants, [QAUX][nq_pad]: see enum below
enum { QA_INV, QA_E1LO, QA_E1HI, QA_EN, QA_G, QA_BIAS, QA_ENP };
// |A| <= 127 * 255 * d stays below 2^31 up to d = 66,311; the rescoring kernel keeps the query in 48 KB of shared memory
constexpr unsigned MAX_D = 8192;

constexpr unsigned MAX_NQ = 1024;  // queries per filter launch: their per-query values stay in shared memory

struct UtShared {
  uint64_t full[STAGES], empty[STAGES], acc_full[2], acc_empty[2];
  alignas(16) double t0[MAX_NQ];  // threshold on A before the row-radius term
  alignas(16) float thr[MAX_NQ];
  alignas(16) float enp[MAX_NQ];  // ||e||_2 2^p
  alignas(16) int tq[4][QT];      // per warp: integer threshold on A of the current unit
  uint32_t tmem_base;
};

struct UtArgs {
  const uint8_t* codes;  // chunk-major corpus bytes: chunk c of row i at (c * ld + i) * 16
  const uint8_t* qop;    // s8 query operand, the same layout with pitch nq_pad, kblocks * KC chunk rows (zero padded)
  unsigned long long ld;
  unsigned n_rows, n_qgroups, kblocks, nq_pad, chunks;
  int dense;             // first pass: every pair kept, slot = row, no counters
  float c;               // RN(alpha / 255) > 0
  double amax;           // 127 * 255 * d >= |A|
  const float* radius;   // r_i rounded up
  const float* qaux;     // QAUX x nq_pad
  const unsigned* qflag;
  const float* thr;      // nq_pad thresholds (score domain)
  unsigned* cand_count;
  unsigned* cand_idx;
  float* cand_lb;
  float* cand_ub;        // test hook only (dense pass): upper bounds, else null
};

// the pair's score interval from its integer product A and the row radius (directed rounding throughout)
struct PairBound {
  float lo, hi;
};
__device__ __forceinline__ PairBound pair_bound(int A, float rad, const float* qaux, unsigned nq_pad, unsigned q, float c) {
  const float inv = qaux[QA_INV * nq_pad + q], en = qaux[QA_EN * nq_pad + q], g = qaux[QA_G * nq_pad + q];
  const float bias = qaux[QA_BIAS * nq_pad + q];
  const float mhi = __fadd_ru(__fmaf_ru(en, rad, __fmaf_ru(inv, __int2float_ru(A), qaux[QA_E1HI * nq_pad + q])), g);
  const float mlo = __fadd_rd(__fmaf_rd(-en, rad, __fmaf_rd(inv, __int2float_rd(A), qaux[QA_E1LO * nq_pad + q])), -g);
  return PairBound{__fadd_rn(__fmul_rn(c, mlo), bias), __fadd_rn(__fmul_rn(c, mhi), bias)};
}

// A threshold T0 on A (before the row term) such that f(mhi) >= thr implies A >= T0 - ||e|| 2^p r_i:
//   RN(y) >= t  implies  y >= t - (|t| 2^-22 + 2^-148), applied to both roundings of f, then divided by c > 0, gives the
//   least `mixed` that can reach thr; the directed operations of pair_bound() add at most 2^-21 relative, covered by the
//   2^-18 margin together with the double rounding of this computation.
__device__ __forceinline__ double a_threshold(float thr, unsigned flagged, const float* qaux, unsigned nq_pad, unsigned q,
                                              float c, double amax) {
  if (flagged) return 1e300;      // never a candidate
  if (!(fabsf(thr) < INFINITY)) return -1e300;  // -inf (keep everything) or +inf: the exact test decides
  const double t = thr, bias = qaux[QA_BIAS * nq_pad + q];
  const double sc = 1.0 / (double)qaux[QA_INV * nq_pad + q];  // 2^p, exact
  const double t1 = t - (fabs(t) * 0x1p-22 + 0x1p-148);
  const double t2 = t1 - bias;
  const double t3 = t2 - (fabs(t2) * 0x1p-22 + 0x1p-148);
  const double e1 = (double)qaux[QA_E1HI * nq_pad + q] * sc, g = (double)qaux[QA_G * nq_pad + q] * sc;
  const double need = (t3 / (double)c) * sc - e1 - g;
  return need - (0x1p-18 * (amax + fabs(need) + fabs(e1) + g) + 4.0);
}

__global__ void __launch_bounds__(UT_THREADS, 1) u8_tc_filter_kernel(const UtArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  UtShared* st = reinterpret_cast<UtShared*>(smem + STAGES * STAGE_BYTES);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // contiguous range of (row tile, query group) units for this CTA, query group fastest
  const unsigned n_vtiles = (a.n_rows + VT - 1) / VT;
  const unsigned long long total_units = (unsigned long long)n_vtiles * a.n_qgroups;
  const unsigned u_lo = (unsigned)(total_units * blockIdx.x / gridDim.x);
  const unsigned u_hi = (unsigned)(total_units * (blockIdx.x + 1) / gridDim.x);
  const unsigned n_units = u_hi - u_lo;
  const unsigned n_iters = n_units * a.kblocks;

  if (threadIdx.x == 0) {
    for (int s = 0; s < STAGES; ++s) {
      mbar_init(&st->full[s], 1);
      mbar_init(&st->empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&st->acc_full[b], 1);
      mbar_init(&st->acc_empty[b], 4);
    }
    fence_barrier_init();
  }
  if (warp == 5) tmem_alloc<512>(&st->tmem_base);
  // the per-query values of the pass, once: every unit's epilogue reads them from shared memory
  for (unsigned q = threadIdx.x; q < a.nq_pad; q += 128) {
    if (threadIdx.x >= 128) break;
    const float t = a.thr[q];
    st->thr[q] = t;
    st->t0[q] = a_threshold(t, a.qflag[q], a.qaux, a.nq_pad, q, a.c, a.amax);
    st->enp[q] = a.qaux[QA_ENP * a.nq_pad + q];
  }
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = st->tmem_base;

  if (warp == 4) {
    // =========================== bulk-copy producer ===========================
    if (lane == 0) {
      for (unsigned it = 0; it < n_iters; ++it) {
        const unsigned unit = u_lo + it / a.kblocks, kb = it % a.kblocks;
        const unsigned vt = unit / a.n_qgroups, qg = unit % a.n_qgroups;
        const unsigned qt_u = min((unsigned)QT, a.nq_pad - qg * QT);
        const unsigned long long row0 = (unsigned long long)vt * VT;
        const unsigned rows = (unsigned)min((unsigned long long)VT, a.ld - row0);  // rows inside the pitch (x16)
        const unsigned c0 = kb * KC, nca = min((unsigned)KC, a.chunks - c0);      // chunks past d: B is zero there
        const int s = it % STAGES;
        mbar_wait(&st->empty[s], ((it / STAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(&st->full[s], nca * rows * 16 + KC * qt_u * 16);
        uint8_t* sa = smem + s * STAGE_BYTES;
        uint8_t* sb = sa + A_BYTES;
        for (unsigned c = 0; c < nca; ++c)
          bulk_load(sa + c * A_CHUNK_BYTES, a.codes + ((unsigned long long)(c0 + c) * a.ld + row0) * 16, rows * 16, &st->full[s]);
        for (unsigned c = 0; c < (unsigned)KC; ++c)
          bulk_load(sb + c * B_CHUNK_BYTES, a.qop + ((unsigned long long)(c0 + c) * a.nq_pad + qg * QT) * 16, qt_u * 16,
                    &st->full[s]);
      }
    }
  } else if (warp == 5) {
    // =========================== MMA issuer ===========================
    const uint64_t a_desc0 = make_smem_desc_kmajor_noswizzle(smem_u32(smem), A_CHUNK_BYTES, 128);
    const uint64_t b_desc0 = make_smem_desc_kmajor_noswizzle(smem_u32(smem + A_BYTES), B_CHUNK_BYTES, 128);
    unsigned it = 0;
    for (unsigned ul = 0; ul < n_units; ++ul) {
      const unsigned qg = (u_lo + ul) % a.n_qgroups;
      const unsigned qt_u = min((unsigned)QT, a.nq_pad - qg * QT);
      const uint32_t idesc = make_idesc_u8s8(VT, (int)qt_u);
      const uint32_t acc = tmem + (ul & 1) * QT;
      mbar_wait(&st->acc_empty[ul & 1], ((ul >> 1) & 1) ^ 1);
      for (unsigned kb = 0; kb < a.kblocks; ++kb, ++it) {
        const int s = it % STAGES;
        mbar_wait(&st->full[s], (it / STAGES) & 1);
        tc_fence_after_sync();
        if (elect_one_sync()) {
          const uint64_t ad = desc_advance(a_desc0, (uint32_t)s * STAGE_BYTES);
          const uint64_t bd = desc_advance(b_desc0, (uint32_t)s * STAGE_BYTES);
          if (kb == 0) umma_i8_c<false>(acc, ad, bd, idesc);
          else umma_i8_c<true>(acc, ad, bd, idesc);
#pragma unroll
          for (int ks = 1; ks < KC / 2; ++ks)  // K = 32 bytes = two chunks per MMA
            umma_i8_c<true>(acc, desc_advance(ad, ks * 2 * A_CHUNK_BYTES), desc_advance(bd, ks * 2 * B_CHUNK_BYTES), idesc);
          umma_commit(&st->empty[s]);
          if (kb == a.kblocks - 1) umma_commit(&st->acc_full[ul & 1]);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== epilogue: integer test, exact interval, append ===========================
    auto row_of = [&](unsigned ul) { return (u_lo + ul) / a.n_qgroups * VT + warp * 32 + lane; };
    float rad_next = (n_units && row_of(0) < a.n_rows) ? a.radius[row_of(0)] : 0.0f;
    for (unsigned ul = 0; ul < n_units; ++ul) {
      const unsigned unit = u_lo + ul;
      const unsigned vt = unit / a.n_qgroups, qg = unit % a.n_qgroups;
      const unsigned qt_u = min((unsigned)QT, a.nq_pad - qg * QT);
      const int ab = ul & 1;
      const unsigned v = vt * VT + warp * 32 + lane;
      const bool vvalid = v < a.n_rows;
      const float rad = rad_next;
      if (ul + 1 < n_units) rad_next = row_of(ul + 1) < a.n_rows ? a.radius[row_of(ul + 1)] : 0.0f;  // in flight meanwhile
      float rmax = rad;
#pragma unroll
      for (int o = 16; o > 0; o >>= 1) rmax = fmaxf(rmax, __shfl_xor_sync(0xffffffffu, rmax, o));
      __syncwarp();  // (the warp's last unit has read tq[warp] already)
#pragma unroll
      for (int j = 0; j < QT / 32; ++j) {
        const unsigned c = lane + 32 * j;
        double tw = 2147483647.0;  // columns past the group: never
        if (c < qt_u) {
          tw = floor(st->t0[qg * QT + c] - (double)st->enp[qg * QT + c] * (double)rmax * (1.0 + 0x1p-18));
          tw = fmin(fmax(tw, (double)INT_MIN), (double)INT_MAX);
        }
        st->tq[warp][c] = (int)tw;
      }
      __syncwarp();
      mbar_wait(&st->acc_full[ab], (ul >> 1) & 1);
      tc_fence_after_sync();
      const uint32_t taddr = tmem + ((uint32_t)(warp * 32) << 16) + ab * QT;
#pragma unroll 1
      for (unsigned c0 = 0; c0 < qt_u; c0 += 32) {
        uint32_t r[32];
        tmem_ld_32x32b_x32(taddr + c0, r);
        tmem_ld_wait();
        if (c0 + 32 >= qt_u) {
          tc_fence_before_sync();
          if (lane == 0) mbar_arrive(&st->acc_empty[ab]);
        }
        if (a.dense) {  // every pair is kept: bounds to slot v of its query, no atomics (the counters are preset)
          if (vvalid) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c0 + j < qt_u) {
                const unsigned q = qg * QT + c0 + j;
                const PairBound b = pair_bound((int)r[j], rad, a.qaux, a.nq_pad, q, a.c);
                const size_t o = (size_t)q * CAND_CAP + v;
                a.cand_idx[o] = v;
                a.cand_lb[o] = b.lo;
                if (a.cand_ub) a.cand_ub[o] = b.hi;
              }
          }
          continue;
        }
        const int4* t4 = reinterpret_cast<const int4*>(&st->tq[warp][c0]);
        bool any = false;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const int4 t = t4[j4];
          any |= (int)r[4 * j4 + 0] >= t.x;
          any |= (int)r[4 * j4 + 1] >= t.y;
          any |= (int)r[4 * j4 + 2] >= t.z;
          any |= (int)r[4 * j4 + 3] >= t.w;
        }
        if (any && vvalid) {  // rare outside the dense pass: the exact interval of every pair that passed
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (c0 + j >= qt_u || (int)r[j] < st->tq[warp][c0 + j]) continue;
            const unsigned q = qg * QT + c0 + j;
            const PairBound b = pair_bound((int)r[j], rad, a.qaux, a.nq_pad, q, a.c);
            if (b.hi < st->thr[q]) continue;  // a NaN bound stays a candidate
            const unsigned pos = atomicAdd(&a.cand_count[q], 1u);
            if (pos < CAND_CAP) {
              const size_t o = (size_t)q * CAND_CAP + pos;
              a.cand_idx[o] = v;
              a.cand_lb[o] = b.lo;
            }
          }
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 5) tmem_dealloc<512>(tmem);
}

// ---- once per corpus: r_i = ||b_i - 128||_2 over the real d, rounded up ------------------------------------------------
__global__ void u8_tc_radius_kernel(const uint4* __restrict__ codes, size_t ld, unsigned n, unsigned d, unsigned chunks,
                                    float* __restrict__ radius) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    unsigned ss = 0;  // <= 128^2 * MAX_D
    for (unsigned c = 0; c < chunks; ++c) {
      const uint4 w4 = codes[(size_t)c * ld + i];
      const unsigned w[4] = {w4.x, w4.y, w4.z, w4.w};
#pragma unroll
      for (int e = 0; e < 16; ++e)
        if (16 * c + e < d) {
          const int b = (int)((w[e >> 2] >> (8 * (e & 3))) & 0xFFu) - 128;
          ss += (unsigned)(b * b);
        }
    }
    radius[i] = __fsqrt_ru(__uint2float_ru(ss));
  }
}

// ---- per call: the s8 operand, the per-query constants of the bound, first-pass thresholds and counters -------------
// one 128-thread block per (padded) query
__global__ void u8_tc_prep_kernel(const float* __restrict__ q, unsigned nq, unsigned d, unsigned nq_pad, unsigned chunks_pad,
                                  float offset, int8_t* __restrict__ qop, unsigned* __restrict__ qflag,
                                  float* __restrict__ thr, unsigned* __restrict__ cand_count, float* __restrict__ qaux,
                                  unsigned first_pass_rows) {
  const unsigned row = blockIdx.x;
  __shared__ float s_scale;
  __shared__ unsigned s_bad;
  if (threadIdx.x == 0) {
    unsigned bad = 1;
    float scale = 0.0f;
    if (row < nq) {
      const float* x = q + (size_t)row * d;
      float mx = 0.0f, qsum = 0.0f;
      bool finite = true;
      for (unsigned j = 0; j < d; ++j) {
        const float v = x[j];
        finite = finite && fabsf(v) < INFINITY;  // NaN fails too
        mx = fmaxf(mx, fabsf(v));
        qsum = __fadd_rn(qsum, v);  // query_context: sequential sum (src/scalar.rs:236-240)
      }
      const float bias = __fmul_rn(offset, qsum);
      bad = (!finite || !(mx >= 0x1p-100f) || mx > 0x1p100f || !(fabsf(bias) < INFINITY)) ? 1u : 0u;
      float e1lo = 0.0f, e1hi = 0.0f, e2 = 0.0f, sabs = 0.0f, inv = 0.0f;
      if (!bad) {
        int ex;
        frexpf(mx, &ex);  // mx in [2^(ex-1), 2^ex)
        int p = 7 - ex;   // mx 2^p in [64, 128)
        if (__fmul_rn(mx, ldexpf(1.0f, p)) >= 127.0f) --p;
        scale = ldexpf(1.0f, p);
        inv = ldexpf(1.0f, -p);
        for (unsigned j = 0; j < d; ++j) {
          const float v = x[j];
          const float qi = rintf(__fmul_rn(v, scale));
          const float e = __fsub_rn(v, __fmul_rn(qi, inv));  // exact (Sterbenz, or qi = 0)
          e1lo = __fadd_rd(e1lo, e);
          e1hi = __fadd_ru(e1hi, e);
          e2 = __fmaf_ru(e, e, e2);
          sabs = __fadd_ru(sabs, fabsf(v));
        }
      }
      const float en = __fsqrt_ru(e2);
      // the reference's rounding: every product passes through at most d + 16 roundings (32 FMA chains of d/32, their
      // combination, the 8-wide remainder, the scalar tail; the sequential sum when d < 16), each of relative error
      // <= 2^-24, plus an absolute 2^-150 per rounding that underflows
      const double gam = (double)(d + 16) * 0x1p-24 / (1.0 - (double)(d + 16) * 0x1p-24);
      const float g = __fmaf_ru(__double2float_ru(gam * 255.0), sabs, __double2float_ru((2.0 * d + 64.0) * 0x1p-149));
      qaux[QA_INV * nq_pad + row] = inv;
      qaux[QA_E1LO * nq_pad + row] = __fmul_rd(e1lo, 128.0f);
      qaux[QA_E1HI * nq_pad + row] = __fmul_ru(e1hi, 128.0f);
      qaux[QA_EN * nq_pad + row] = en;
      qaux[QA_G * nq_pad + row] = g;
      qaux[QA_BIAS * nq_pad + row] = bias;
      qaux[QA_ENP * nq_pad + row] = __fmul_ru(en, scale);
    } else {
      for (int i = 0; i < QAUX; ++i) qaux[i * nq_pad + row] = 0.0f;
    }
    s_scale = scale;
    s_bad = bad;
    qflag[row] = bad;
    thr[row] = INFINITY;                // queries the filter does not answer keep +inf in every pass
    cand_count[row] = first_pass_rows;  // the dense first pass stores the pair (q, row v) in slot v
  }
  __syncthreads();
  const float scale = s_scale;
  const bool bad = s_bad != 0;
  for (unsigned t = threadIdx.x; t < chunks_pad * 16; t += blockDim.x) {
    const unsigned c = t / 16, e = t % 16, j = t;
    int8_t qi = 0;
    if (!bad && j < d) qi = (int8_t)__float2int_rn(__fmul_rn(q[(size_t)row * d + j], scale));
    qop[((size_t)c * nq_pad + row) * 16 + e] = qi;
  }
}

// ---- exact rescoring + selection: one CTA per query, the scan's per-vector arithmetic (u8_dot.cuh) -------------------
constexpr int RS_THREADS = 256;

template <int R>
__global__ void __launch_bounds__(RS_THREADS) u8_tc_rescore_kernel(const uint4* __restrict__ codes, size_t ld, unsigned d,
                                                                   unsigned chunks, unsigned index_base, float alpha,
                                                                   const float* __restrict__ queries, unsigned nq_pad,
                                                                   const float* __restrict__ qaux,
                                                                   const unsigned* __restrict__ qflag,
                                                                   unsigned* __restrict__ cand_count,
                                                                   const unsigned* __restrict__ cand, int k, unsigned magic,
                                                                   uint64_t* __restrict__ out_keys) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned sq_len = chunks * 16 + 32;
  float* sq = reinterpret_cast<float*>(smem_raw);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(sq + sq_len);
  const unsigned q = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  unsigned cnt = cand_count[q];
  if (qflag[q] || cnt > CAND_CAP) {  // not filtered / overflowed: the caller runs the exact scan for it
    if (threadIdx.x == 0) cand_count[q] = 0xFFFFFFFFu;
    return;
  }
  for (unsigned i = threadIdx.x; i < sq_len; i += blockDim.x) sq[i] = i < d ? queries[(size_t)q * d + i] : 0.0f;
  __syncthreads();
  const float scale = __fdiv_rn(alpha, 255.0f), bias = qaux[QA_BIAS * nq_pad + q];
  const unsigned main_chunks = (d >= 16) ? (d / 32) * 2 : 0;
  const unsigned cnt_round = (cnt + 31u) / 32u * 32u;
  WarpList<R> list;
  list.init();
  uint64_t thr = KEY_SENTINEL;
  for (unsigned c = threadIdx.x; c < cnt_round; c += blockDim.x) {
    const bool valid = c < cnt;
    uint64_t key = KEY_SENTINEL;
    if (valid) {
      const unsigned i = cand[(size_t)q * CAND_CAP + c];
      float acc[32];
#pragma unroll
      for (int j = 0; j < 32; ++j) acc[j] = 0.0f;
      unsigned w[8] = {0, 0, 0, 0, 0, 0, 0, 0};
      unsigned ch = 0;
      for (; ch + 2 <= main_chunks; ch += 2) {  // chunk parity selects the accumulator half, as in the scan
        const uint4 v0 = codes[(size_t)ch * ld + i], v1 = codes[(size_t)(ch + 1) * ld + i];
        fma16<false>(v0, sq + 16 * ch, acc, magic);
        fma16<false>(v1, sq + 16 * (ch + 1), acc + 16, magic);
      }
      if (ch < chunks) {
        const uint4 v = codes[(size_t)ch * ld + i];
        w[0] = v.x; w[1] = v.y; w[2] = v.z; w[3] = v.w;
      }
      if (ch + 1 < chunks) {
        const uint4 v = codes[(size_t)(ch + 1) * ld + i];
        w[4] = v.x; w[5] = v.y; w[6] = v.z; w[7] = v.w;
      }
      const float mixed = mixed_dot_finish(acc, w, d, sq, magic, 1.0f);
      key = make_key_desc(__fadd_rn(__fmul_rn(scale, mixed), bias), index_base + i);  // src/scalar.rs:299
    }
    list.offer(key, valid, thr, k, lane);
  }
  block_tree_merge<R>(list, k, smem_keys);
  if (warp == 0) list.store(out_keys + (size_t)q * k, k, lane);
}

// workspace layout ------------------------------------------------------------------------------------------------------
struct U8TcPlan {
  unsigned nq_pad, kblocks;
  size_t off_qop, off_qflag, off_thr, off_cnt, off_qaux, off_idx, off_lb, off_ub, total;
};

U8TcPlan make_plan(size_t d, size_t nq, bool with_ub) {
  U8TcPlan p{};
  p.nq_pad = (unsigned)((nq + 15) / 16 * 16);
  p.kblocks = (unsigned)((d + KC * 16 - 1) / (KC * 16));
  tcf::WsCursor w;
  p.off_qop = w.take((size_t)p.kblocks * KC * p.nq_pad * 16);
  p.off_qflag = w.take((size_t)p.nq_pad * 4);
  p.off_thr = w.take((size_t)p.nq_pad * 4);
  p.off_cnt = w.take((size_t)p.nq_pad * 4);
  p.off_qaux = w.take((size_t)p.nq_pad * QAUX * 4);
  p.off_idx = w.take((size_t)p.nq_pad * CAND_CAP * 4);
  p.off_lb = w.take((size_t)p.nq_pad * CAND_CAP * 4);
  p.off_ub = with_ub ? w.take((size_t)p.nq_pad * CAND_CAP * 4) : 0;
  p.total = w.o;
  return p;
}

struct Bufs {
  int8_t* qop;
  unsigned *qflag, *cnt, *idx;
  float *thr, *qaux, *lb, *ub;
};
Bufs bufs(const U8TcPlan& p, void* workspace, bool with_ub) {
  uint8_t* w = (uint8_t*)workspace;
  return Bufs{(int8_t*)(w + p.off_qop), (unsigned*)(w + p.off_qflag), (unsigned*)(w + p.off_cnt), (unsigned*)(w + p.off_idx),
              (float*)(w + p.off_thr), (float*)(w + p.off_qaux), (float*)(w + p.off_lb),
              with_ub ? (float*)(w + p.off_ub) : nullptr};
}

constexpr size_t FILTER_SMEM = (size_t)STAGES * STAGE_BYTES + sizeof(UtShared);

cudaError_t set_filter_smem() {
  static bool done_dev[16] = {};
  bool& done = done_dev[current_device_slot()];
  if (done) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(u8_tc_filter_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FILTER_SMEM);
  if (e == cudaSuccess) done = true;
  return e;
}

UtArgs base_args(const U8View& v, const float* dev_radius, const U8TcPlan& p, const Bufs& b) {
  UtArgs a{};
  a.codes = (const uint8_t*)v.data;
  a.qop = (const uint8_t*)b.qop;
  a.ld = v.ld;
  a.n_qgroups = (p.nq_pad + QT - 1) / QT;
  a.kblocks = p.kblocks;
  a.nq_pad = p.nq_pad;
  a.chunks = (unsigned)v.chunks;
  a.c = v.alpha / 255.0f;
  a.amax = 127.0 * 255.0 * (double)v.d;
  a.radius = dev_radius;
  a.qaux = b.qaux;
  a.qflag = b.qflag;
  a.thr = b.thr;
  a.cand_count = b.cnt;
  a.cand_idx = b.idx;
  a.cand_lb = b.lb;
  return a;
}

cudaError_t launch_filter(const UtArgs& a, int num_sms, cudaStream_t s) {
  const unsigned long long units = (unsigned long long)((a.n_rows + VT - 1) / VT) * a.n_qgroups;
  unsigned grid = (unsigned)num_sms;
  if (grid > units) grid = (unsigned)units;
  u8_tc_filter_kernel<<<grid, UT_THREADS, FILTER_SMEM, s>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_prep(const U8View& v, const float* dev_queries, size_t nq, const U8TcPlan& p, const Bufs& b, size_t first_rows,
                        cudaStream_t s) {
  u8_tc_prep_kernel<<<p.nq_pad, 128, 0, s>>>(dev_queries, (unsigned)nq, (unsigned)v.d, p.nq_pad, p.kblocks * KC, v.offset,
                                             b.qop, b.qflag, b.thr, b.cnt, b.qaux, (unsigned)first_rows);
  return cudaGetLastError();
}

}  // namespace

bool u8_tc_supported(const U8View& v, size_t nq, size_t k) {
  const float c = v.alpha / 255.0f;  // the reference's RN(alpha / 255): f is monotone only for c > 0
  return nq >= 1 && k >= 1 && k <= 128 && v.n >= 1 && v.n < 0x7FFFFF00ull && v.d >= 1 && v.d <= MAX_D && c > 0.0f &&
         c < INFINITY;
}

size_t u8_tc_workspace_bytes(size_t d, size_t nq, bool debug) { return make_plan(d, nq < MAX_NQ ? nq : MAX_NQ, debug).total; }

cudaError_t launch_u8_tc_radius(const U8View& v, float* dev_radius, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0) return cudaSuccess;
  unsigned grid = (unsigned)((v.n + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  u8_tc_radius_kernel<<<grid, 256, 0, s>>>(v.data, v.ld, (unsigned)v.n, (unsigned)v.d, (unsigned)v.chunks, dev_radius);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_u8_tc_debug_bounds(const U8View& v, const float* dev_radius, const float* dev_queries, size_t nq,
                                      void* workspace, float* host_lower, float* host_upper, size_t* out_rows,
                                      unsigned* host_qflags, int num_sms, cudaStream_t s, LaunchCounter* launches) {
  if (nq > MAX_NQ) return cudaErrorInvalidValue;
  const U8TcPlan p = make_plan(v.d, nq, true);
  const Bufs b = bufs(p, workspace, true);
  const size_t rows = v.n < CAND_CAP ? v.n : CAND_CAP;
  cudaError_t e = launch_prep(v, dev_queries, nq, p, b, rows, s);
  ++*launches;
  if (e != cudaSuccess) return e;
  if ((e = set_filter_smem()) != cudaSuccess) return e;
  UtArgs a = base_args(v, dev_radius, p, b);
  a.n_rows = (unsigned)rows;
  a.dense = 1;
  a.cand_ub = b.ub;
  if ((e = launch_filter(a, num_sms, s)) != cudaSuccess) return e;
  ++*launches;
  if ((e = cudaMemcpy2DAsync(host_lower, rows * sizeof(float), b.lb, CAND_CAP * sizeof(float), rows * sizeof(float), nq,
                             cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaMemcpy2DAsync(host_upper, rows * sizeof(float), b.ub, CAND_CAP * sizeof(float), rows * sizeof(float), nq,
                             cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaMemcpyAsync(host_qflags, b.qflag, nq * sizeof(unsigned), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
  *out_rows = rows;
  return cudaSuccess;
}

namespace {
// one launch sequence for up to MAX_NQ queries: prep, passes, rescore; appends the unanswered queries (offset by q0)
cudaError_t knn_tc_chunk(const U8View& v, const float* dev_radius, const float* dev_queries, size_t nq, size_t q0, size_t k,
                         uint64_t* dev_keys, void* workspace, unsigned* host_counts, Workspace& ws, cudaStream_t s,
                         LaunchCounter* launches, std::vector<unsigned>* overflow_queries, KnnTcStats* stats) {
  const U8TcPlan p = make_plan(v.d, nq, false);
  const Bufs b = bufs(p, workspace, false);
  cudaError_t e;
  static cudaEvent_t ev_dev[16][2] = {};  // per device: final pass begin / end
  cudaEvent_t(&ev)[2] = ev_dev[current_device_slot()];
  if (!ev[0])
    for (auto& x : ev)
      if ((e = cudaEventCreate(&x)) != cudaSuccess) return e;

  // 1. operands, first-pass thresholds, counters preset for the dense pass
  const size_t first_rows = tcf::first_rows(v.n, k, 0);
  if ((e = launch_prep(v, dev_queries, nq, p, b, first_rows, s)) != cudaSuccess) return e;
  ++*launches;
  if ((e = set_filter_smem()) != cudaSuccess) return e;

  // 2. filter passes over growing prefixes (tc_filter.cuh)
  size_t levels[6];
  const int n_levels = tcf::levels(v.n, k, first_rows, 0, levels);
  UtArgs a = base_args(v, dev_radius, p, b);
  for (int l = 0; l < n_levels; ++l) {
    const bool last = l == n_levels - 1;
    a.n_rows = (unsigned)levels[l];
    a.dense = l == 0;
    if (last) cudaEventRecord(ev[0], s);
    if ((e = launch_filter(a, ws.num_sms, s)) != cudaSuccess) return e;
    ++*launches;
    if (last) {
      cudaEventRecord(ev[1], s);
    } else {
      tcf::launch_select(nq, k, b.qflag, b.cnt, b.lb, b.thr, s);
      ++*launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
  }
  // 3. exact rescoring + selection
  const size_t rs_smem = (v.chunks * 16 + 32) * sizeof(float) + (size_t)(RS_THREADS / 32) * k * 8;
  if (k <= 32)
    u8_tc_rescore_kernel<1><<<(unsigned)nq, RS_THREADS, rs_smem, s>>>(v.data, v.ld, (unsigned)v.d, (unsigned)v.chunks,
                                                                      v.index_base, v.alpha, dev_queries, p.nq_pad, b.qaux,
                                                                      b.qflag, b.cnt, b.idx, (int)k, 0x4B000000u, dev_keys);
  else
    u8_tc_rescore_kernel<4><<<(unsigned)nq, RS_THREADS, rs_smem, s>>>(v.data, v.ld, (unsigned)v.d, (unsigned)v.chunks,
                                                                      v.index_base, v.alpha, dev_queries, p.nq_pad, b.qaux,
                                                                      b.qflag, b.cnt, b.idx, (int)k, 0x4B000000u, dev_keys);
  ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  // 4. overflowed / unfiltered queries -> the caller re-runs them on the exact scan
  if ((e = cudaMemcpyAsync(host_counts, b.cnt, nq * 4, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
  for (size_t q = 0; q < nq; ++q) {
    if (host_counts[q] > CAND_CAP) overflow_queries->push_back((unsigned)(q0 + q));
    else stats->candidates += host_counts[q];
  }
  float ms = 0.0f;
  cudaEventElapsedTime(&ms, ev[0], ev[1]);
  stats->filter_ms += ms;
  stats->filter_flops += 2.0 * (double)((v.n + VT - 1) / VT * VT) * (double)(p.kblocks * KC * 16) * (double)p.nq_pad;
  stats->passes = n_levels;
  return cudaSuccess;
}
}  // namespace

cudaError_t launch_u8_knn_tc(const U8View& v, const float* dev_radius, const float* dev_queries, size_t nq, size_t k,
                             uint64_t* dev_keys, void* workspace, unsigned* host_counts, Workspace& ws, cudaStream_t s,
                             LaunchCounter* launches, std::vector<unsigned>* overflow_queries, KnnTcStats* stats) {
  cudaError_t e;
  static cudaEvent_t ev_dev[16][2] = {};  // per device: call begin / end
  cudaEvent_t(&ev)[2] = ev_dev[current_device_slot()];
  if (!ev[0])
    for (auto& x : ev)
      if ((e = cudaEventCreate(&x)) != cudaSuccess) return e;
  cudaEventRecord(ev[0], s);
  overflow_queries->clear();
  KnnTcStats st;
  for (size_t q0 = 0; q0 < nq; q0 += MAX_NQ) {  // batches of MAX_NQ queries, one after the other
    const size_t m = nq - q0 < MAX_NQ ? nq - q0 : MAX_NQ;
    if ((e = knn_tc_chunk(v, dev_radius, dev_queries + q0 * v.d, m, q0, k, dev_keys + q0 * k, workspace, host_counts, ws, s,
                          launches, overflow_queries, &st)) != cudaSuccess)
      return e;
  }
  cudaEventRecord(ev[1], s);
  if ((e = cudaEventSynchronize(ev[1])) != cudaSuccess) return e;
  cudaEventElapsedTime(&st.total_ms, ev[0], ev[1]);
  st.overflowed = (unsigned)overflow_queries->size();
  if (stats) *stats = st;
  return cudaSuccess;
}

}  // namespace innr
