// knn_tc.cu -- multi-query batch_knn (L2) / batch_knn_dot / batch_knn_cosine with the tensor cores as an exact-result
// FILTER.
//
// For large query batches (BASELINE C2b: 1024 queries over 10M x 768) scoring is a dense contraction. The reference
// (src/batch.rs:742-800) scores every (query, vector) pair in f32 and fully sorts; results must stay bit-exact with
// it, which no tensor-core contraction delivers directly. So the tensor cores only *prune*, with a rigorous bound:
//
//   0. once per corpus  exact norms (the bit-exact scan) and Xh = f16(x / ||x||), row-major [n][d] (K-major operand);
//   1. per call         Qh = f16(q / ||q||), row-major [nq][d];
//   2. filter passes    S = Xh * Qh^T on tcgen05 (kind::f16, f32 accumulate in TMEM) ~ cosine(q, x), |S - cos| <= eps.
//                       With r = ||x|| (dot) or [||x|| > 1e-9] (cosine), every pair has the interval
//                       [S*r - eps*r, S*r + eps*r] around the reference's score (in units of score/||q|| for dot).
//                       A pass over rows [0, n_i) appends (index, lower bound) of every pair whose UPPER bound reaches
//                       the query's threshold; the k-th largest LOWER bound of the appended pairs is a valid lower
//                       bound of the reference's k-th best score and becomes the threshold of the next, larger pass
//                       (n_0 = 4096 rows, every pair kept, then n/128, n/16, n). No exact sample scan is needed.
//   3. rescore          the final candidates (~20 k per query) are re-scored with the reference's exact sequential
//                       f32 arithmetic and selected on the same 64-bit keys as the scan kernel -> indices and scores
//                       bit-identical to batch_knn_dot / batch_knn_cosine. A query whose final list overflows, or
//                       whose norm is zero / non-finite, is re-run on the exact scan by the caller.
//
// eps = 1.05e-3 + 3.5e-7*d bounds: f16 rounding of both unit vectors (2*2^-11 of sum|q'x'| <= 1, plus the subnormal
// floor), the f32 accumulation of d exact products in the tensor core (d*2^-23, truncation), and the distance of the
// reference's own sequential f32 score from the real-valued one (2*d*2^-24). Corpora with a non-finite norm never
// take this path.
//
// Filter kernel: persistent, one CTA per SM, 192 threads: 4 epilogue warps (TMEM -> registers, bound test, append),
// TMA producer warp, MMA issuer warp. Work unit = 128 vectors x 256 queries, K loop over 64-dimension blocks through a
// 4-stage shared-memory ring (X 16 KB + Q 32 KB per stage), 4 MMAs (M128 N256 K16) per block, two 256-column
// accumulators in TMEM so the epilogue of one unit overlaps the MMAs of the next.
#include <cuda_fp16.h>

#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <vector>

#include "common.cuh"
#include "kernels.cuh"
#include "pdx.cuh"
#include "tc_common.cuh"
#include "tc_filter.cuh"

namespace innr {

namespace {

using namespace tc;

constexpr int KT_THREADS = 192;
constexpr int VT = 128;    // vectors per work unit (UMMA M)
constexpr int QT = 256;    // queries per work unit (UMMA N, up to)
constexpr int KB = 64;     // dimensions per K block (128 bytes of f16 = one swizzle row)
constexpr int KSTAGES = 4;
constexpr int X_BYTES = VT * KB * 2;   // 16 KB
constexpr int Q_BYTES = QT * KB * 2;   // 32 KB
constexpr int KSTAGE_BYTES = X_BYTES + Q_BYTES;
// Q-resident variant (<= 64 queries, <= 12 K blocks): the whole f16 query operand stays in shared memory (one 8 KB box of
// 64 rows per K block) and the ring carries X only, twice as deep -- with few queries the pass is a pure HBM stream of
// Xh and the 4 x 16 KB of X the streaming variant keeps in flight per SM are far too little (5.7 ms instead of 2.2)
constexpr int QR_ROWS = 64;
constexpr int QR_BOX_BYTES = QR_ROWS * KB * 2;   // 8 KB
constexpr int QR_MAX_KBLOCKS = 12;
constexpr int QR_STAGES = 7;    // 7 x 16 KB ring + 96 KB of Q + barriers and per-column arrays = 217 KB
constexpr int KT_MAX_STAGES = 8;
constexpr float COS_NORM_EPS = 1e-9f;   // src/batch.rs:721-727
constexpr float TINY_NORM = 1e-30f;     // below this a vector / query is not normalised (handled by the exact path)
using tcf::CAND_CAP;

struct KtShared {
  uint64_t full[KT_MAX_STAGES], empty[KT_MAX_STAGES], acc_full[2], acc_empty[2], q_full;
  alignas(16) float thr[2][QT];  // read as float4; L2: threshold minus the query's constant slack
  alignas(16) float hlo[2][QT];  // L2: 1/(2||q||) * (1 - delta), per query column
  alignas(16) float hhi[2][QT];  // L2: 1/(2||q||) * (1 + delta)
  alignas(16) float cq[2][QT];   // L2: per-query constant slack (the reference's own rounding, relative to ||q||)
  uint32_t tmem_base;
};

struct KtArgs {
  unsigned n_rows;          // rows [0, n_rows) of the corpus are filtered by this pass
  unsigned n_qgroups, kblocks, nq_pad;
  int cosine;
  int l2;                   // squared-L2 metric: u = ||x|| S - ||x||^2 / (2||q||) ranks like -distance (see header)
  const float* qaux;        // l2: 3 x nq_pad floats: hlo, hhi, cq
  int dense;                // first pass (threshold -inf, n_rows <= CAND_CAP): slot = row, no counters
  float eps;
  const float* norms;       // exact ||x|| per vector
  const float* thr;         // nq_pad thresholds (+inf: accept nothing)
  unsigned* cand_count;     // nq_pad counters
  unsigned* cand_idx;       // nq_pad x CAND_CAP local vector indices
  float* cand_lb;           // nq_pad x CAND_CAP lower bounds
};

__device__ __forceinline__ void umma_f16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc,
                                         uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
template <bool ACC>
__device__ __forceinline__ void umma_f16_c(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(d_tmem), "l"(a_desc), "l"(b_desc), "r"(idesc), "n"(ACC ? 1 : 0)
      : "memory");
}
// kind::f16, A = B = F16 (format 0), K-major, F32 accumulate
__device__ __forceinline__ uint32_t make_idesc_f16(int M, int N) {
  return (1u << 4) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

template <bool QRES>
__global__ void __launch_bounds__(KT_THREADS, 1) knn_tc_filter_kernel(const __grid_constant__ CUtensorMap tm_x,
                                                                       const __grid_constant__ CUtensorMap tm_q,
                                                                       const KtArgs a) {
  constexpr int NST = QRES ? QR_STAGES : KSTAGES;
  constexpr int ST_BYTES = QRES ? X_BYTES : KSTAGE_BYTES;
  constexpr int RING_BYTES = NST * ST_BYTES;
  extern __shared__ __align__(1024) uint8_t smem[];
  uint8_t* s_qres = smem + RING_BYTES;  // QRES: kblocks x 8 KB
  KtShared* st = reinterpret_cast<KtShared*>(smem + RING_BYTES + (QRES ? QR_MAX_KBLOCKS * QR_BOX_BYTES : 0));
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  // contiguous range of (vector tile, query group) units for this CTA, query group fastest: the X tile of consecutive
  // units is the same and is re-read from L2, not from HBM
  const unsigned n_vtiles = (a.n_rows + VT - 1) / VT;
  const unsigned long long total_units = (unsigned long long)n_vtiles * a.n_qgroups;
  const unsigned u_lo = (unsigned)(total_units * blockIdx.x / gridDim.x);
  const unsigned u_hi = (unsigned)(total_units * (blockIdx.x + 1) / gridDim.x);
  const unsigned n_units = u_hi - u_lo;
  const unsigned n_iters = n_units * a.kblocks;

  if (threadIdx.x == 0) {
    for (int s = 0; s < NST; ++s) {
      mbar_init(&st->full[s], 1);
      mbar_init(&st->empty[s], 1);
    }
    mbar_init(&st->q_full, 1);
    for (int b = 0; b < 2; ++b) {
      mbar_init(&st->acc_full[b], 1);
      mbar_init(&st->acc_empty[b], 4);
    }
    fence_barrier_init();
    tma_prefetch_desc(&tm_x);
    tma_prefetch_desc(&tm_q);
  }
  if (warp == 5) tmem_alloc<512>(&st->tmem_base);
  tc_fence_before_sync();
  __syncthreads();
  tc_fence_after_sync();
  const uint32_t tmem = st->tmem_base;

  if (warp == 4) {
    // =========================== TMA producer ===========================
    if (lane == 0) {
      if (QRES && n_iters) {  // the whole query operand once (one group: n_qgroups == 1)
        mbar_arrive_expect_tx(&st->q_full, a.kblocks * QR_BOX_BYTES);
        for (unsigned kb = 0; kb < a.kblocks; ++kb) tma_load_2d(s_qres + kb * QR_BOX_BYTES, &tm_q, &st->q_full, (int)(kb * KB), 0);
      }
      for (unsigned it = 0; it < n_iters; ++it) {
        const unsigned unit = u_lo + it / a.kblocks, kb = it % a.kblocks;
        const unsigned vt = unit / a.n_qgroups, qg = unit % a.n_qgroups;
        const int s = it % NST;
        mbar_wait(&st->empty[s], ((it / NST) & 1) ^ 1);
        mbar_arrive_expect_tx(&st->full[s], ST_BYTES);
        uint8_t* sb = smem + s * ST_BYTES;
        tma_load_2d(sb, &tm_x, &st->full[s], (int)(kb * KB), (int)(vt * VT));
        if (!QRES) tma_load_2d(sb + X_BYTES, &tm_q, &st->full[s], (int)(kb * KB), (int)(qg * QT));
      }
    }
  } else if (warp == 5) {
    // =========================== MMA issuer ===========================
    // the whole warp runs the loop (warp-uniform addresses and descriptors), one elected lane issues
    const uint64_t x_desc0 = make_smem_desc_kmajor_sw128(smem_u32(smem));
    const uint64_t q_desc0 = make_smem_desc_kmajor_sw128(smem_u32(QRES ? s_qres : smem + X_BYTES));
    unsigned it = 0;
    if (QRES && n_units) mbar_wait(&st->q_full, 0);
    for (unsigned ul = 0; ul < n_units; ++ul) {
      const unsigned qg = (u_lo + ul) % a.n_qgroups;
      const unsigned qt_u = min((unsigned)QT, a.nq_pad - qg * QT);
      const uint32_t idesc = make_idesc_f16(VT, (int)qt_u);
      const uint32_t acc = tmem + (ul & 1) * QT;
      mbar_wait(&st->acc_empty[ul & 1], ((ul >> 1) & 1) ^ 1);
      for (unsigned kb = 0; kb < a.kblocks; ++kb, ++it) {
        const int s = it % NST;
        mbar_wait(&st->full[s], (it / NST) & 1);
        tc_fence_after_sync();
        if (elect_one_sync()) {
          const uint64_t xd = desc_advance(x_desc0, (uint32_t)s * ST_BYTES);
          const uint64_t qd = desc_advance(q_desc0, QRES ? kb * QR_BOX_BYTES : (uint32_t)s * ST_BYTES);
          if (kb == 0) umma_f16_c<false>(acc, xd, qd, idesc);
          else umma_f16_c<true>(acc, xd, qd, idesc);
#pragma unroll
          for (int ks = 1; ks < KB / 16; ++ks) umma_f16_c<true>(acc, desc_advance(xd, ks * 32), desc_advance(qd, ks * 32), idesc);
          umma_commit(&st->empty[s]);  // the stage is no longer read by the tensor core
          if (kb == a.kblocks - 1) umma_commit(&st->acc_full[ul & 1]);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== epilogue: bound test + append ===========================
    for (unsigned ul = 0; ul < n_units; ++ul) {
      const unsigned unit = u_lo + ul;
      const unsigned vt = unit / a.n_qgroups, qg = unit % a.n_qgroups;
      const unsigned qt_u = min((unsigned)QT, a.nq_pad - qg * QT);
      const int ab = ul & 1;
      const unsigned v = vt * VT + warp * 32 + lane;  // local vector index of this lane
      for (unsigned c = threadIdx.x; c < QT; c += 128) {
        const bool cv = c < qt_u;
        float cq = 0.0f;
        if (a.l2) {
          st->hlo[ab][c] = cv ? a.qaux[qg * QT + c] : 0.0f;
          st->hhi[ab][c] = cv ? a.qaux[a.nq_pad + qg * QT + c] : 0.0f;
          cq = cv ? a.qaux[2 * a.nq_pad + qg * QT + c] : 0.0f;
          st->cq[ab][c] = cq;
        }
        st->thr[ab][c] = cv ? a.thr[qg * QT + c] - cq : INFINITY;
      }
      float rn = 0.0f, e = 0.0f, xx = 0.0f;
      const bool vvalid = v < a.n_rows;
      if (vvalid) {
        const float nv = a.norms[v];
        if (a.cosine) {
          rn = nv > COS_NORM_EPS ? 1.0f : 0.0f;
          e = a.eps * rn;
        } else {
          rn = nv >= TINY_NORM ? nv : 0.0f;
          e = a.eps * rn + 1e-18f;
          if (a.l2) xx = nv * nv;
        }
      }
      asm volatile("bar.sync 1, 128;" ::: "memory");  // thresholds of this unit visible to the 4 epilogue warps
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
        // upper / lower bound of the pair's rank value: S*r +- e, for L2 minus ||x||^2 * 1/(2||q||) (widened by delta)
        // and minus the query's constant slack on the lower side (the thresholds in shared memory carry it already)
        auto upper = [&](int j) {
          float u = fmaf(__uint_as_float(r[j]), rn, e);
          if (a.l2) u = fmaf(-xx, st->hlo[ab][c0 + j], u);
          return u;
        };
        auto lower = [&](int j) {
          float l = fmaf(__uint_as_float(r[j]), rn, -e);
          if (a.l2) l = fmaf(-xx, st->hhi[ab][c0 + j], l) - st->cq[ab][c0 + j];
          return l;
        };
        if (a.dense) {  // every pair is kept: lower bound to slot v of its query, no atomics (the counters are preset)
          if (vvalid) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c0 + j < qt_u) {
                const size_t o = (size_t)(qg * QT + c0 + j) * CAND_CAP + v;
                a.cand_idx[o] = v;
                a.cand_lb[o] = lower(j);
              }
          }
          continue;
        }
        const float4* t4 = reinterpret_cast<const float4*>(&st->thr[ab][c0]);
        bool any = false;
        if (a.l2) {
          const float4* h4 = reinterpret_cast<const float4*>(&st->hlo[ab][c0]);
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 t = t4[j4], h = h4[j4];
            any |= fmaf(-xx, h.x, fmaf(__uint_as_float(r[4 * j4 + 0]), rn, e)) >= t.x;
            any |= fmaf(-xx, h.y, fmaf(__uint_as_float(r[4 * j4 + 1]), rn, e)) >= t.y;
            any |= fmaf(-xx, h.z, fmaf(__uint_as_float(r[4 * j4 + 2]), rn, e)) >= t.z;
            any |= fmaf(-xx, h.w, fmaf(__uint_as_float(r[4 * j4 + 3]), rn, e)) >= t.w;
          }
        } else {
#pragma unroll
          for (int j4 = 0; j4 < 8; ++j4) {
            const float4 t = t4[j4];
            any |= fmaf(__uint_as_float(r[4 * j4 + 0]), rn, e) >= t.x;
            any |= fmaf(__uint_as_float(r[4 * j4 + 1]), rn, e) >= t.y;
            any |= fmaf(__uint_as_float(r[4 * j4 + 2]), rn, e) >= t.z;
            any |= fmaf(__uint_as_float(r[4 * j4 + 3]), rn, e) >= t.w;
          }
        }
        if (any && vvalid) {  // rare except in the first, dense pass. All atomics of the lane are issued before any
                              // of their results is used, so their round trips overlap.
          unsigned pos[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            const bool hit = (c0 + j < qt_u) && upper(j) >= st->thr[ab][c0 + j];
            pos[j] = hit ? atomicAdd(&a.cand_count[qg * QT + c0 + j], 1u) : 0xFFFFFFFFu;
          }
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (pos[j] < CAND_CAP) {
              const size_t o = (size_t)(qg * QT + c0 + j) * CAND_CAP + pos[j];
              a.cand_idx[o] = v;
              a.cand_lb[o] = lower(j);
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

// ---- once per corpus: Xh[i][k] = f16(x[k][i] / ||x_i||) from the PDX corpus and its exact norms ----------------------
__global__ void knn_tc_build_xh_kernel(const PdxView pdx, unsigned n, unsigned d, unsigned d_pad,
                                       const float* __restrict__ norms, __half* __restrict__ xh,
                                       unsigned* __restrict__ nonfinite) {
  __shared__ float tile[32][33];
  const unsigned i0 = blockIdx.x * 32;
  const unsigned tx = threadIdx.x, ty = threadIdx.y;  // 32 x 8
  float inv[4];
#pragma unroll
  for (int r = 0; r < 4; ++r) {
    const unsigned i = i0 + ty * 4 + r;
    float nv = i < n ? norms[i] : 0.0f;
    const bool finite = nv == nv && nv < INFINITY;
    if (i < n && !finite && tx == 0) atomicAdd(nonfinite, 1u);
    inv[r] = (finite && nv >= TINY_NORM) ? 1.0f / nv : 0.0f;
  }
  for (unsigned d0 = 0; d0 < d_pad; d0 += 32) {
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const unsigned dd = d0 + ty * 4 + r, i = i0 + tx;
      tile[ty * 4 + r][tx] = (dd < d && i < n) ? pdx_load1(pdx, (size_t)dd * pdx.ld + i) : 0.0f;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < 4; ++r) {
      const unsigned i = i0 + ty * 4 + r, dd = d0 + tx;
      if (i < n && dd < d_pad) xh[(size_t)i * d_pad + dd] = __float2half_rn(tile[tx][ty * 4 + r] * inv[r]);
    }
  }
}

// ---- squared L2 through the same filter ------------------------------------------------------------------------
// d(q,x) = ||q||^2 + ||x||^2 - 2 q.x, so u = (||q||^2 - d) / (2||q||) = ||x|| cos(q,x) - ||x||^2 / (2||q||) ranks like
// -distance within a query, and ||x|| S +- ||x|| eps brackets its first term exactly as for the dot product. Slack
// for everything else, relative to the two positive terms d <= 2(||q||^2 + ||x||^2) is made of:
//   * the reference's own f32 result (sequential sum of d terms, 3 roundings each): |d_ref - d| <= (d+2) 2^-24 d
//     -> (d+2) 2^-24 (||q|| + ||x||^2/||q||) in units of u: a per-query constant l2_cq and 2(d+2) 2^-24 on the second term;
//   * ||x|| as stored (sqrt of the sequential f32 sum), its square, 1/(2||q||), the fmas of the bound itself:
//     <= (2d + 16) 2^-24 relative on the second term.
__host__ __device__ __forceinline__ float l2_delta(unsigned d) { return (4.0f * (float)d + 32.0f) * 5.9604645e-8f; }
__host__ __device__ __forceinline__ float l2_cq(unsigned d, float qn) { return 2.0f * ((float)d + 2.0f) * 5.9604645e-8f * qn; }

// ---- per call: Qh row = f16(q / ||q||); ||q|| is the sequential f32 sum of batch_cosine_into (src/batch.rs:714) ------
__global__ void knn_tc_prep_queries_kernel(const float* __restrict__ q, unsigned nq, unsigned d, unsigned nq_pad,
                                           unsigned d_pad, int cosine, int l2, __half* __restrict__ qh,
                                           unsigned* __restrict__ qflag, float* __restrict__ thr,
                                           unsigned* __restrict__ cand_count, float* __restrict__ qaux,
                                           unsigned first_pass_rows) {
  const unsigned row = blockIdx.x;
  __shared__ float s_inv;
  __shared__ unsigned s_bad;
  if (threadIdx.x == 0) {
    float inv = 0.0f;
    unsigned bad = 0;
    if (row < nq) {
      float ss = 0.0f;
      for (unsigned k = 0; k < d; ++k) ss = __fadd_rn(ss, __fmul_rn(q[(size_t)row * d + k], q[(size_t)row * d + k]));
      const float qn = __fsqrt_rn(ss);
      const bool finite = qn == qn && qn < INFINITY;
      // zero / denormal / non-finite norms, and cosine queries below the reference's 1e-9 guard (all scores 0.0):
      // answered by the exact scan
      bad = (!finite || qn < TINY_NORM || (cosine && qn < COS_NORM_EPS)) ? 1u : 0u;
      inv = bad ? 0.0f : 1.0f / qn;
      if (l2) {  // see l2_slack(): h = 1/(2||q||) widened by delta, constant slack gamma * ||q||
        const float h = bad ? 0.0f : 0.5f * inv;
        qaux[row] = h * (1.0f - l2_delta(d));
        qaux[nq_pad + row] = h * (1.0f + l2_delta(d));
        qaux[2 * nq_pad + row] = bad ? 0.0f : l2_cq(d, qn);
      }
    } else if (l2) {
      qaux[row] = qaux[nq_pad + row] = qaux[2 * nq_pad + row] = 0.0f;
    }
    s_inv = inv;
    s_bad = bad;
    qflag[row] = bad;
    thr[row] = INFINITY;                // queries the filter does not answer keep +inf (accept nothing) in every pass
    cand_count[row] = first_pass_rows;  // the dense first pass stores the pair (q, row v) in slot v
  }
  __syncthreads();
  const float inv = s_inv;
  for (unsigned k = threadIdx.x; k < d_pad; k += blockDim.x) {
    const float v = (row < nq && k < d) ? q[(size_t)row * d + k] * inv : 0.0f;
    qh[(size_t)row * d_pad + k] = __float2half_rn(v);
  }
}

// ---- exact rescoring + selection: one CTA per query -------------------------------------------------------------------
constexpr int RS_THREADS = 256;

template <int R>
__global__ void __launch_bounds__(RS_THREADS) knn_tc_rescore_kernel(const PdxView data, unsigned n,
                                                                    unsigned d, unsigned index_base,
                                                                    const float* __restrict__ queries, int cosine,
                                                                    int l2, float eps, const float* __restrict__ norms,
                                                                    const unsigned* __restrict__ qflag,
                                                                    unsigned* __restrict__ cand_count,
                                                                    const unsigned* __restrict__ cand,
                                                                    const float* __restrict__ cand_lb, int k,
                                                                    uint64_t* __restrict__ out_keys) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sq = reinterpret_cast<float*>(smem_raw);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(sq + ((d + 3) & ~3u));
  __shared__ float s_qn, s_bound;
  const unsigned q = blockIdx.x;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (qflag[q]) {  // not filtered: reported as overflowed so that the caller runs the exact scan for it
    if (threadIdx.x == 0) cand_count[q] = 0xFFFFFFFFu;
    return;
  }
  for (unsigned i = threadIdx.x; i < d; i += blockDim.x) sq[i] = queries[(size_t)q * d + i];
  if (threadIdx.x == 0) {
    float ss = 0.0f;
    for (unsigned i = 0; i < d; ++i) ss = __fadd_rn(ss, __fmul_rn(queries[(size_t)q * d + i], queries[(size_t)q * d + i]));
    s_qn = __fsqrt_rn(ss);
  }
  unsigned cnt = cand_count[q];
  if (cnt > CAND_CAP) cnt = CAND_CAP;
  const unsigned cnt_round = (cnt + 31u) / 32u * 32u;
  // 1. the k-th largest lower bound of the final candidates bounds the k-th best score from below: only candidates
  //    whose upper bound reaches it can be in the result (typically 10-20 of a few hundred)
  {
    WarpList<R> lbs;
    lbs.init();
    uint64_t t = KEY_SENTINEL;
    for (unsigned c = threadIdx.x; c < cnt_round; c += blockDim.x) {
      const bool valid = c < cnt;
      const float lb = valid ? cand_lb[(size_t)q * CAND_CAP + c] : 0.0f;
      lbs.offer(make_key_desc(lb, c), valid, t, k, lane);
    }
    block_tree_merge<R>(lbs, k, smem_keys);
    if (warp == 0) {
      const uint64_t kth = lbs.at(k - 1);
      if (lane == 0)
        s_bound = (kth == KEY_SENTINEL) ? -INFINITY : __uint_as_float(order_bits_to_f32_bits(~(uint32_t)(kth >> 32)));
    }
  }
  __syncthreads();
  const float qn = s_qn, bound = s_bound;
  // 2. exact scores of the survivors, selection on the scan kernel's keys
  WarpList<R> list;
  list.init();
  uint64_t thr = KEY_SENTINEL;
  for (unsigned c = threadIdx.x; c < cnt_round; c += blockDim.x) {
    bool valid = c < cnt;
    uint64_t key = KEY_SENTINEL;
    unsigned i = 0;
    if (valid) {
      i = cand[(size_t)q * CAND_CAP + c];
      const float lb = cand_lb[(size_t)q * CAND_CAP + c];
      const float nv = norms[i];
      const float e = cosine ? (nv > COS_NORM_EPS ? eps : 0.0f) : (eps * (nv >= TINY_NORM ? nv : 0.0f) + 1e-18f);
      float ub = fmaf(2.0f, e, lb) + 1e-6f * (fabsf(lb) + e);  // the filter's upper bound, rounding included
      if (l2) {  // + the widening of the ||x||^2 / (2||q||) term and twice the query's constant slack
        const float t = nv * nv * (0.5f / qn);
        ub += 2.0f * l2_delta(d) * t + 2.0f * l2_cq(d, qn) + 1e-6f * t;
      }
      valid = ub >= bound;
    }
    if (valid) {
      const size_t p = i, ld = data.ld;
      float acc = 0.0f, ss = 0.0f;
      unsigned dd = 0;
      // the reference's sequential unfused sums (src/batch.rs:257-265, 290-296, 676-681), 8 rows in flight per thread
      // (32 in flight measured slower: 1.0 ms instead of 0.6 for 1024 queries -- every row of a candidate is its own
      // 32-byte sector 4 ld bytes from the last one, and the deeper queue only thrashes the TLB)
      for (; dd + 8 <= d; dd += 8) {
        float v[8];
#pragma unroll
        for (int u = 0; u < 8; ++u) v[u] = pdx_load1(data, p + (size_t)(dd + u) * ld);
#pragma unroll
        for (int u = 0; u < 8; ++u) {
          if (l2) {
            const float diff = __fsub_rn(sq[dd + u], v[u]);
            acc = __fadd_rn(acc, __fmul_rn(diff, diff));
          } else {
            acc = __fadd_rn(acc, __fmul_rn(sq[dd + u], v[u]));
            ss = __fadd_rn(ss, __fmul_rn(v[u], v[u]));
          }
        }
      }
      for (; dd < d; ++dd) {
        const float v = pdx_load1(data, p + (size_t)dd * ld);
        if (l2) {
          const float diff = __fsub_rn(sq[dd], v);
          acc = __fadd_rn(acc, __fmul_rn(diff, diff));
        } else {
          acc = __fadd_rn(acc, __fmul_rn(sq[dd], v));
          ss = __fadd_rn(ss, __fmul_rn(v, v));
        }
      }
      float s = acc;
      if (cosine) {
        const float nrm = __fsqrt_rn(ss);
        s = (!(qn < COS_NORM_EPS) && nrm > COS_NORM_EPS) ? __fdiv_rn(acc, __fmul_rn(qn, nrm)) : 0.0f;
      }
      key = l2 ? make_key_asc(s, index_base + i) : make_key_desc(s, index_base + i);
    }
    list.offer(key, valid, thr, k, lane);
  }
  block_tree_merge<R>(list, k, smem_keys);
  if (warp == 0) list.store(out_keys + (size_t)q * k, k, lane);
}

// tensor map over a row-major f16 matrix [rows][pitch] (pitch in elements, multiple of 8): box = 64 x box_rows, SW128
bool make_tmap_f16_rows(CUtensorMap* m, const void* base, uint64_t rows, uint64_t cols, uint64_t pitch, uint32_t box_rows) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc || rows == 0 || cols == 0) return false;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {pitch * 2};
  cuuint32_t box[2] = {KB, box_rows};
  cuuint32_t estr[2] = {1, 1};
  return enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<void*>(base), gdim, gstride, box, estr,
             CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
             CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// workspace layout ------------------------------------------------------------------------------------------------------
struct KnnTcPlan {
  unsigned nq_pad, d_pad;
  size_t off_qh, off_qflag, off_thr, off_cnt, off_qaux, off_idx, off_lb, total;
};

KnnTcPlan make_plan(size_t d, size_t nq) {
  KnnTcPlan p{};
  p.nq_pad = (unsigned)((nq + 15) / 16 * 16);
  p.d_pad = (unsigned)knn_tc_dpad(d);
  tcf::WsCursor w;
  p.off_qh = w.take((size_t)p.nq_pad * p.d_pad * 2);
  p.off_qflag = w.take((size_t)p.nq_pad * 4);
  p.off_thr = w.take((size_t)p.nq_pad * 4);
  p.off_cnt = w.take((size_t)p.nq_pad * 4);
  p.off_qaux = w.take((size_t)p.nq_pad * 3 * 4);
  p.off_idx = w.take((size_t)p.nq_pad * CAND_CAP * 4);
  p.off_lb = w.take((size_t)p.nq_pad * CAND_CAP * 4);
  p.total = w.o;
  return p;
}

}  // namespace

size_t knn_tc_dpad(size_t d) { return (d + 7) / 8 * 8; }
// |S - cos| <= eps (header of this file): f16 rounding of both unit vectors, f32 accumulation in the tensor core, and the
// distance of the reference's own sequential f32 score from the real-valued one
float knn_tc_eps(size_t d) { return 1.05e-3f + 3.5e-7f * (float)d; }

size_t knn_tc_workspace_bytes(size_t n, size_t d, size_t nq, size_t k) {
  (void)n;
  (void)k;
  return make_plan(d, nq).total;
}

bool knn_tc_supported(const PdxView& v, int mode, size_t nq, size_t k) {
  return (mode == PDX_DOT || mode == PDX_COSINE_FUSED || mode == PDX_L2) && nq >= 1 && k >= 1 && k <= 128 && v.d >= 1 && v.n >= 4096 &&
         v.n < 0x7FFFFF00ull;
}

// Xh + its tensor map from the PDX corpus and its exact norms; *host_nonfinite = vectors with a NaN / inf norm (the
// caller disables the path for the corpus when it is not 0). Synchronises the stream.
cudaError_t launch_knn_tc_build(const PdxView& v, const float* dev_norms, void* dev_xh, unsigned* dev_scratch_u32,
                                CUtensorMap* tm_xh, unsigned* host_nonfinite, cudaStream_t s, LaunchCounter* launches) {
  const unsigned d_pad = (unsigned)knn_tc_dpad(v.d);
  cudaError_t e = cudaMemsetAsync(dev_scratch_u32, 0, 4, s);
  if (e != cudaSuccess) return e;
  knn_tc_build_xh_kernel<<<(unsigned)((v.n + 31) / 32), dim3(32, 8), 0, s>>>(v, (unsigned)v.n, (unsigned)v.d, d_pad,
                                                                             dev_norms, (__half*)dev_xh, dev_scratch_u32);
  ++*launches;
  e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  e = cudaMemcpyAsync(host_nonfinite, dev_scratch_u32, 4, cudaMemcpyDeviceToHost, s);
  if (e != cudaSuccess) return e;
  e = cudaStreamSynchronize(s);
  if (e != cudaSuccess) return e;
  if (!make_tmap_f16_rows(tm_xh, dev_xh, v.n, d_pad, d_pad, VT)) return cudaErrorInvalidValue;
  return cudaSuccess;
}

// Test hook (innr_cuda_knn_tc_debug_bounds): the operands and the DENSE first pass of the filter only -- for every query
// q and every row v < min(n, CAND_CAP) the pair's lower bound lands in cand_lb[q * CAND_CAP + v] exactly as the
// production passes compute it. Copies them to host_lower (nq x rows) and reports eps; synchronises the stream.
cudaError_t launch_knn_tc_debug_bounds(const PdxView& v, const CUtensorMap& tm_xh, const float* dev_norms, int mode,
                                       const float* dev_queries, size_t nq, void* workspace, float* host_lower,
                                       size_t* out_rows, float* out_eps, unsigned* host_qflags, int num_sms, cudaStream_t s,
                                       LaunchCounter* launches) {
  const int cosine = mode == PDX_COSINE_FUSED, l2 = mode == PDX_L2;
  const KnnTcPlan p = make_plan(v.d, nq);
  uint8_t* w = (uint8_t*)workspace;
  __half* qh = (__half*)(w + p.off_qh);
  unsigned* qflag = (unsigned*)(w + p.off_qflag);
  float* thr = (float*)(w + p.off_thr);
  unsigned* cnt = (unsigned*)(w + p.off_cnt);
  float* qaux = (float*)(w + p.off_qaux);
  const unsigned rows = (unsigned)(CAND_CAP < v.n ? CAND_CAP : v.n);
  knn_tc_prep_queries_kernel<<<p.nq_pad, 128, 0, s>>>(dev_queries, (unsigned)nq, (unsigned)v.d, p.nq_pad, p.d_pad, cosine, l2, qh,
                                                      qflag, thr, cnt, qaux, rows);
  ++*launches;
  const bool qres = p.nq_pad <= QR_ROWS && (p.d_pad + KB - 1) / KB <= QR_MAX_KBLOCKS;
  CUtensorMap tm_q;
  if (!make_tmap_f16_rows(&tm_q, qh, p.nq_pad, p.d_pad, p.d_pad, qres ? QR_ROWS : QT)) return cudaErrorInvalidValue;
  const size_t smem_stream = (size_t)KSTAGES * KSTAGE_BYTES + sizeof(KtShared);
  const size_t smem_qres = (size_t)QR_STAGES * X_BYTES + (size_t)QR_MAX_KBLOCKS * QR_BOX_BYTES + sizeof(KtShared);
  cudaError_t e = cudaFuncSetAttribute(knn_tc_filter_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_stream);
  if (e != cudaSuccess) return e;
  e = cudaFuncSetAttribute(knn_tc_filter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_qres);
  if (e != cudaSuccess) return e;
  KtArgs a{};
  a.n_qgroups = (p.nq_pad + QT - 1) / QT;
  a.kblocks = (p.d_pad + KB - 1) / KB;
  a.nq_pad = p.nq_pad;
  a.cosine = cosine;
  a.l2 = l2;
  a.qaux = qaux;
  a.eps = knn_tc_eps(v.d);
  a.norms = dev_norms;
  a.thr = thr;
  a.cand_count = cnt;
  a.cand_idx = (unsigned*)(w + p.off_idx);
  a.cand_lb = (float*)(w + p.off_lb);
  a.n_rows = rows;
  a.dense = 1;
  const unsigned long long units = (unsigned long long)((rows + VT - 1) / VT) * a.n_qgroups;
  unsigned grid = (unsigned)num_sms;
  if (grid > units) grid = (unsigned)units;
  if (qres) knn_tc_filter_kernel<true><<<grid, KT_THREADS, smem_qres, s>>>(tm_xh, tm_q, a);
  else knn_tc_filter_kernel<false><<<grid, KT_THREADS, smem_stream, s>>>(tm_xh, tm_q, a);
  ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = cudaMemcpy2DAsync(host_lower, rows * sizeof(float), a.cand_lb, CAND_CAP * sizeof(float), rows * sizeof(float), nq,
                             cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaMemcpyAsync(host_qflags, qflag, nq * sizeof(unsigned), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
  *out_rows = rows;
  *out_eps = a.eps;
  return cudaSuccess;
}

cudaError_t launch_pdx_knn_tc(const PdxView& v, const CUtensorMap& tm_xh, const float* dev_norms, int mode,
                              const float* dev_queries, size_t nq, size_t k, uint64_t* dev_keys, void* workspace,
                              unsigned* host_counts, Workspace& ws, cudaStream_t s, LaunchCounter* launches,
                              std::vector<unsigned>* overflow_queries, KnnTcStats* stats) {
  const int cosine = mode == PDX_COSINE_FUSED, l2 = mode == PDX_L2;
  const KnnTcPlan p = make_plan(v.d, nq);
  uint8_t* w = (uint8_t*)workspace;
  __half* qh = (__half*)(w + p.off_qh);
  unsigned* qflag = (unsigned*)(w + p.off_qflag);
  float* thr = (float*)(w + p.off_thr);
  unsigned* cnt = (unsigned*)(w + p.off_cnt);
  float* qaux = (float*)(w + p.off_qaux);
  unsigned* cand_idx = (unsigned*)(w + p.off_idx);
  float* cand_lb = (float*)(w + p.off_lb);
  cudaError_t e;
  static const bool trace = getenv("INNR_KNN_TC_TRACE") != nullptr;
  static cudaEvent_t ev_dev[16][4] = {};  // per device: call begin, final pass begin / end, call end
  cudaEvent_t(&ev)[4] = ev_dev[current_device_slot()];
  if (!ev[0])
    for (auto& x : ev)
      if ((e = cudaEventCreate(&x)) != cudaSuccess) return e;
  cudaEventRecord(ev[0], s);
  cudaEvent_t tev[12];
  int n_tev = 0;
  auto tmark = [&]() {
    if (trace && n_tev < 12) {
      cudaEventCreate(&tev[n_tev]);
      cudaEventRecord(tev[n_tev++], s);
    }
  };
  tmark();

  // 1. operands, first-pass thresholds, zeroed counters
  // the dense first pass keeps every pair of its rows (tc_filter.cuh)
  static const int first_env = getenv("INNR_KNN_TC_FIRST") ? atoi(getenv("INNR_KNN_TC_FIRST")) : 0;
  const size_t first_rows = tcf::first_rows(v.n, k, first_env);
  knn_tc_prep_queries_kernel<<<p.nq_pad, 128, 0, s>>>(dev_queries, (unsigned)nq, (unsigned)v.d, p.nq_pad, p.d_pad, cosine, l2, qh,
                                                      qflag, thr, cnt, qaux, (unsigned)first_rows);
  ++*launches;
  const bool qres = p.nq_pad <= QR_ROWS && (p.d_pad + KB - 1) / KB <= QR_MAX_KBLOCKS;
  CUtensorMap tm_q;
  if (!make_tmap_f16_rows(&tm_q, qh, p.nq_pad, p.d_pad, p.d_pad, qres ? QR_ROWS : QT)) return cudaErrorInvalidValue;
  tmark();

  // 2. filter passes over growing prefixes
  static bool attr_set_dev[16] = {};
  bool& attr_set = attr_set_dev[current_device_slot()];
  const size_t smem_stream = (size_t)KSTAGES * KSTAGE_BYTES + sizeof(KtShared);
  const size_t smem_qres = (size_t)QR_STAGES * X_BYTES + (size_t)QR_MAX_KBLOCKS * QR_BOX_BYTES + sizeof(KtShared);
  if (!attr_set) {
    e = cudaFuncSetAttribute(knn_tc_filter_kernel<false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_stream);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(knn_tc_filter_kernel<true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_qres);
    if (e != cudaSuccess) return e;
    attr_set = true;
  }
  size_t levels[6];
  static const int sched = getenv("INNR_KNN_TC_SCHED") ? atoi(getenv("INNR_KNN_TC_SCHED")) : 0;
  const int n_levels = tcf::levels(v.n, k, first_rows, sched, levels);
  KtArgs a{};
  a.n_qgroups = (p.nq_pad + QT - 1) / QT;
  a.kblocks = (p.d_pad + KB - 1) / KB;
  a.nq_pad = p.nq_pad;
  a.cosine = cosine;
  a.l2 = l2;
  a.qaux = qaux;
  a.eps = knn_tc_eps(v.d);
  a.norms = dev_norms;
  a.thr = thr;
  a.cand_count = cnt;
  a.cand_idx = cand_idx;
  a.cand_lb = cand_lb;
  for (int l = 0; l < n_levels; ++l) {
    const bool last = l == n_levels - 1;
    a.n_rows = (unsigned)levels[l];
    a.dense = l == 0;
    const unsigned long long units = (unsigned long long)((a.n_rows + VT - 1) / VT) * a.n_qgroups;
    unsigned grid = (unsigned)ws.num_sms;
    if (grid > units) grid = (unsigned)units;
    if (last) cudaEventRecord(ev[1], s);
    if (qres) knn_tc_filter_kernel<true><<<grid, KT_THREADS, smem_qres, s>>>(tm_xh, tm_q, a);
    else knn_tc_filter_kernel<false><<<grid, KT_THREADS, smem_stream, s>>>(tm_xh, tm_q, a);
    ++*launches;
    if ((e = cudaGetLastError()) != cudaSuccess) return e;
    if (last) {
      cudaEventRecord(ev[2], s);
    } else {
      tcf::launch_select(nq, k, qflag, cnt, cand_lb, thr, s);
      ++*launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
    tmark();
  }
  // 3. exact rescoring + selection
  const size_t rs_smem = ((v.d + 3) & ~(size_t)3) * 4 + (size_t)(RS_THREADS / 32) * k * 8;
  if (k <= 32)
    knn_tc_rescore_kernel<1><<<(unsigned)nq, RS_THREADS, rs_smem, s>>>(v, (unsigned)v.n, (unsigned)v.d, v.index_base,
                                                                       dev_queries, cosine, l2, a.eps, dev_norms, qflag, cnt, cand_idx,
                                                                       cand_lb, (int)k, dev_keys);
  else
    knn_tc_rescore_kernel<4><<<(unsigned)nq, RS_THREADS, rs_smem, s>>>(v, (unsigned)v.n, (unsigned)v.d, v.index_base,
                                                                       dev_queries, cosine, l2, a.eps, dev_norms, qflag, cnt, cand_idx,
                                                                       cand_lb, (int)k, dev_keys);
  ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  cudaEventRecord(ev[3], s);
  tmark();
  // 4. overflowed / unfiltered queries -> the caller re-runs them on the exact scan
  if ((e = cudaMemcpyAsync(host_counts, cnt, nq * 4, cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
  overflow_queries->clear();
  unsigned long long tot = 0, mx = 0;
  for (size_t q = 0; q < nq; ++q) {
    if (host_counts[q] > CAND_CAP) {
      overflow_queries->push_back((unsigned)q);
    } else {
      tot += host_counts[q];
      if (host_counts[q] > mx) mx = host_counts[q];
    }
  }
  if (stats) {
    cudaEventElapsedTime(&stats->filter_ms, ev[1], ev[2]);
    cudaEventElapsedTime(&stats->total_ms, ev[0], ev[3]);
    stats->filter_flops = 2.0 * (double)((v.n + VT - 1) / VT * VT) * (double)(a.kblocks * KB) * (double)p.nq_pad;
    stats->candidates = tot;
    stats->overflowed = (unsigned)overflow_queries->size();
    stats->passes = n_levels;
    if (trace) {
      fprintf(stderr, "[knn_tc] passes %d | final filter %.3f ms | whole call %.3f ms | candidates total %llu max %llu | exact-scan queries %zu | phases (prep, passes.., rescore):",
              n_levels, stats->filter_ms, stats->total_ms, tot, mx, overflow_queries->size());
      for (int i = 0; i + 1 < n_tev; ++i) {
        float t = 0;
        cudaEventElapsedTime(&t, tev[i], tev[i + 1]);
        fprintf(stderr, " %.3f", t);
      }
      fprintf(stderr, "\n");
    }
  }
  for (int i = 0; i < n_tev; ++i) cudaEventDestroy(tev[i]);
  return cudaSuccess;
}

}  // namespace innr
