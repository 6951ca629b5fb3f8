// scan_f32.cu -- HBM-bound scan of a device-resident VerticalBatch (PDX layout) with fused exact top-k.
//
// Replaces (reference, innr 0.6.3):
//   batch_dot_into          src/batch.rs:284-297      batch_l2_squared_into  src/batch.rs:250-266
//   batch_norms_into        src/batch.rs:672-686      batch_cosine_into      src/batch.rs:705-728
//   batch_knn (L2 + TopK)   src/batch.rs:385-411      batch_knn_dot          src/batch.rs:742-764
//   batch_knn_cosine        src/batch.rs:777-800      TopK::insert           src/topk.rs:96-121
//
// Bit-exactness (SURVEY.md F4/F5): the reference's batch loops are `acc[i] += q[d] * v[d][i]` with d
// ascending and NO fused multiply-add, so one thread owning vector i and computing
// __fadd_rn(acc, __fmul_rn(q, v)) for d = 0..D-1 reproduces every score bit for bit. The PDX layout makes that
// mapping perfectly coalesced: a thread owns 4 consecutive vectors (one 128-bit load per dimension row), a warp
// reads 512 contiguous bytes per row, a CTA tile covers TILE = 4 * blockDim vectors.
//
// batch_knn_cosine recomputes all corpus norms on every call (src/batch.rs:788); here sum(v*v) is accumulated
// in the same pass over the same registers (same sequential order => same bits) at zero extra HBM bytes.
//
// Selection never materialises N scores: scores become 64-bit composite keys (common.cuh) and flow into a
// per-warp register list, a CTA merge and a last-CTA merge -- one launch per query group.
#include <algorithm>
#include <cmath>
#include <type_traits>

#include "common.cuh"
#include "kernels.cuh"
#include "pdx.cuh"

namespace innr {

namespace {

constexpr int SCAN_THREADS = 256;
constexpr int VPT = 4;                        // vectors per thread (one float4)
constexpr int TILE = SCAN_THREADS * VPT;      // vectors per CTA tile
constexpr float NORM_EPS = 1e-9f;             // crate::NORM_EPSILON, src/lib.rs:178

struct PdxArgs {
  PdxView v;
  unsigned long long ld;
  unsigned n, d, ld4;     // ld4 = ld (u32 copy for bounds checks; ld < 2^32)
  unsigned n_tiles;
  unsigned index_base;
  const float* queries;   // nq_total x d (device); blockIdx.y selects the group of QB queries
  int nq_valid;           // queries in this launch (all y groups together)
  int k;
  uint64_t* partials;
  uint64_t* out_keys;
  uint64_t* group_partials;
  unsigned* tickets;
  float* scores_out;      // scores mode: out[q * ld + i]
  const float* norms_in;  // PDX_COSINE_NORMS
  const uint32_t* mask;   // MASKED: bit i set = vector i passes the predicate (batch_knn_filtered)
  const uint32_t* perm;   // PDX_L2_PERM: the order in which the dimension rows are accumulated (batch_knn_reordered)
  float threshold;        // PDX_L2_PRUNE
  float one;              // 1.0f, opaque to the compiler (see add2_unfusable)
  const unsigned* run_flag;  // non-null: the launch returns at once unless *run_flag != 0
};

template <int MODE>
__device__ __forceinline__ void accumulate(float q, float v, float& acc) {
  if (MODE == PDX_L2 || MODE == PDX_L2_PRUNE || MODE == PDX_L2_PERM) {
    float diff = __fsub_rn(q, v);                 // let diff = q_d - v_d;
    acc = __fadd_rn(acc, __fmul_rn(diff, diff));  // *dist += diff * diff;
  } else {
    acc = __fadd_rn(acc, __fmul_rn(q, v));        // *prod += q_d * v_d;
  }
}

// the same for two vectors at once (acc, v: packed pairs; q2 = {q, q}): unfused mul + add per lane, bit-identical
template <int MODE>
__device__ __forceinline__ void accumulate2(uint64_t q2, uint64_t v2, uint64_t& acc2, uint64_t one2) {
  if (MODE == PDX_L2 || MODE == PDX_L2_PRUNE || MODE == PDX_L2_PERM) {
    const uint64_t diff = sub2_rn(q2, v2);
    acc2 = add2_unfusable(mul2_rn(diff, diff), acc2, one2);
  } else {
    acc2 = add2_unfusable(mul2_rn(q2, v2), acc2, one2);
  }
}

template <int MODE, int QB, int R, bool KNN, bool MASKED = false, int UX = 0>
__global__ void __launch_bounds__(SCAN_THREADS) pdx_scan_kernel(const PdxArgs a_in) {
  static_assert(MODE != PDX_L2_PRUNE || (QB == 1 && !KNN), "pruning is a single-query scores scan");
  static_assert(MODE != PDX_L2_PERM || (QB == 1 && !MASKED), "the reordered scan is a single-query scan");
  constexpr bool PERM = (MODE == PDX_L2_PERM);
  constexpr bool NEED_SS = (MODE == PDX_COSINE_FUSED || MODE == PDX_NORMS);
  constexpr bool NEED_DOT = (MODE != PDX_NORMS);
  // dimension rows in flight per thread. The sum over d is sequential by contract, so a thread makes D / U round trips
  // to memory: 8 (4 with eight queries' accumulators) saturate HBM when every SM holds several CTAs; launches with at
  // most a couple of CTAs per SM (small corpora, small shards, C1) are bound by that latency chain instead and use the
  // deep variants (UX = 32 / 16).
  constexpr int U = UX ? UX : ((QB == 1) ? 8 : 4);

  extern __shared__ __align__(16) unsigned char smem_raw[];
  // [d][QB] interleaved queries (padded so the d-loop can read whole float4 groups), then qnorm[QB], then keys
  const unsigned d_pad = (a_in.d + 31u) / 32u * 32u;  // same for every U (scan_smem_bytes)
  float* sq = reinterpret_cast<float*>(smem_raw);
  float* s_qn = sq + (size_t)d_pad * QB;
  unsigned* s_perm = reinterpret_cast<unsigned*>(s_qn + ((QB + 3) & ~3));  // PERM: d_pad row indices (d_pad % 8 == 0)
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(s_perm + (PERM ? d_pad : 0u));

  const int lane = threadIdx.x & 31;
  if (a_in.run_flag && *a_in.run_flag == 0) return;  // the whole grid leaves: no ticket is taken

  // query group of this CTA (grid.y): shifts the query, output and merge-workspace pointers
  PdxArgs a = a_in;
  {
    const unsigned y = blockIdx.y;
    const unsigned n_groups = (gridDim.x + FINISH_GROUP - 1) / FINISH_GROUP;
    a.queries += (size_t)y * QB * a.d;
    a.nq_valid = min(QB, a_in.nq_valid - (int)(y * QB));
    a.out_keys += (size_t)y * QB * a.k;
    a.partials += (size_t)y * gridDim.x * QB * a.k;
    a.group_partials += (size_t)y * n_groups * QB * a.k;
    a.tickets += (size_t)y * (1 + n_groups);
  }

  if (NEED_DOT) {
    for (unsigned idx = threadIdx.x; idx < d_pad * QB; idx += blockDim.x) {
      unsigned dd = idx / QB, q = idx % QB;
      if (PERM) {  // step j of the reordered scan pairs query[order[j]] with row order[j]
        const unsigned row = dd < a.d ? a.perm[dd] : 0u;
        s_perm[dd] = row;
        sq[idx] = dd < a.d ? a.queries[row] : 0.0f;
      } else {
        sq[idx] = (dd < a.d && (int)q < a.nq_valid) ? a.queries[(size_t)q * a.d + dd] : 0.0f;
      }
    }
  }
  __syncthreads();
  constexpr bool NEED_QN = NEED_DOT && (MODE == PDX_COSINE_FUSED || MODE == PDX_COSINE_NORMS);
  if (NEED_QN) {
    // query_norm = query.iter().map(|x| x * x).sum::<f32>().sqrt()   (src/batch.rs:714) -- sequential, so one thread per
    // query; read from the shared-memory copy (a dependent chain of global loads cost ~20 us per launch). The chain is
    // d dependent multiply-adds (~3 us at d = 768) and its result is only needed in the first tile's epilogue, so the
    // CTA does NOT wait for it here: the last warp computes it and joins the scan late, the other warps start streaming
    // at once, and the barrier in front of the first epilogue (below) finds it long finished.
    if (threadIdx.x >= SCAN_THREADS - 32 && threadIdx.x - (SCAN_THREADS - 32) < QB) {
      const unsigned q = threadIdx.x - (SCAN_THREADS - 32);
      float ss = 0.0f;
      if ((int)q < a.nq_valid) {
        for (unsigned dd = 0; dd < a.d; ++dd) {
          const float x = sq[(size_t)dd * QB + q];
          ss = __fadd_rn(ss, __fmul_rn(x, x));
        }
      }
      s_qn[q] = __fsqrt_rn(ss);
    }
  }
  bool qn_visible = !NEED_QN;

  WarpList<R> lists[QB];
  uint64_t thrs[QB];
  if (KNN) {
#pragma unroll
    for (int q = 0; q < QB; ++q) {
      lists[q].init();
      thrs[q] = KEY_SENTINEL;
    }
  }

  for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const unsigned i0 = tile * TILE + threadIdx.x * VPT;
    bool active = i0 < a.ld4;  // ld is a multiple of 4: the whole float4 is in bounds
    unsigned nib = 0xFu;       // MASKED: predicate bits of this thread's four vectors (i0 % 4 == 0: one word)
    if (MASKED) {
      nib = active ? (a.mask[i0 >> 5] >> (i0 & 31)) & 0xFu : 0u;
      active = nib != 0;       // predicate pushdown: rows of rejected vectors are not even read
    }
    // accumulators as packed pairs (vectors 0,1 and 2,3 of this thread): the unfused multiply and add of the reference
    // run as FMUL2 / FADD2 -- two IEEE operations per instruction, same bits, half the FP32 issue slots (what bounds
    // the multi-query kernel)
    uint64_t acc2[QB][2];
    uint64_t ss2[2];
    float mx[VPT];   // PDX_L2_PRUNE: running max of the non-NaN partial distances
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      ss2[h] = 0ull;  // {+0.0f, +0.0f}
#pragma unroll
      for (int q = 0; q < QB; ++q) acc2[q][h] = 0ull;
    }
#pragma unroll
    for (int j = 0; j < VPT; ++j) mx[j] = -INFINITY;  // the initial 0.0 is not a partial the reference tests
    const unsigned amask = (MODE == PDX_L2_PRUNE) ? __ballot_sync(FULL_MASK, active) : 0u;
    const uint64_t one2 = pack2(a.one, a.one);
    auto step = [&](const float4& v, unsigned dq) {
      const uint64_t v01 = pack2(v.x, v.y), v23 = pack2(v.z, v.w);
      if (NEED_SS) {
        ss2[0] = add2_unfusable(mul2_rn(v01, v01), ss2[0], one2);
        ss2[1] = add2_unfusable(mul2_rn(v23, v23), ss2[1], one2);
      }
      if (NEED_DOT) {
#pragma unroll
        for (int q = 0; q < QB; ++q) {
          const float qv = sq[(size_t)dq * QB + q];
          const uint64_t q2 = pack2(qv, qv);
          accumulate2<MODE>(q2, v01, acc2[q][0], one2);
          accumulate2<MODE>(q2, v23, acc2[q][1], one2);
        }
      }
      if (MODE == PDX_L2_PRUNE) {
        // the reference prunes vector i at the first dimension whose partial distance exceeds the threshold
        // (src/batch.rs:347-351). Partial sums of squares never decrease until one becomes NaN (a NaN compares
        // false and stays alive), so "some partial > threshold" == "max of the non-NaN partials > threshold".
        float p0, p1, p2, p3;
        unpack2(acc2[0][0], p0, p1);
        unpack2(acc2[0][1], p2, p3);
        mx[0] = fmaxf(mx[0], p0);
        mx[1] = fmaxf(mx[1], p1);
        mx[2] = fmaxf(mx[2], p2);
        mx[3] = fmaxf(mx[3], p3);
      }
    };
    // the layout branch is taken once per tile, so each loop below holds loads of one kind only
    auto rows = [&](auto split) {
      constexpr bool SPLIT = decltype(split)::value;
      size_t p = i0;
      unsigned dd = 0;
      for (; dd + U <= a.d; dd += U) {
        float4 v[U];
#pragma unroll
        for (int u = 0; u < U; ++u) v[u] = pdx_load4_as<SPLIT>(a.v, PERM ? i0 + (size_t)s_perm[dd + u] * a.ld : p + (size_t)u * a.ld);
        if (!PERM) p += (size_t)U * a.ld;
#pragma unroll
        for (int u = 0; u < U; ++u) step(v[u], dd + u);
        if (MODE == PDX_L2_PRUNE) {  // every vector this warp owns in the tile is pruned: stop reading its rows
          const bool dead = mx[0] > a.threshold && mx[1] > a.threshold && mx[2] > a.threshold && mx[3] > a.threshold;
          if (__all_sync(amask, dead)) { dd = a.d; break; }
        }
      }
      for (; dd < a.d; ++dd) {  // D % U tail
        const float4 v = pdx_load4_as<SPLIT>(a.v, PERM ? i0 + (size_t)s_perm[dd] * a.ld : p);
        if (!PERM) p += a.ld;
        step(v, dd);
      }
    };
    if (active) {
      if (a.v.hi) rows(std::true_type{});
      else rows(std::false_type{});
    }
    float acc[QB][VPT];
    float ss[VPT];
    unpack2(ss2[0], ss[0], ss[1]);
    unpack2(ss2[1], ss[2], ss[3]);
#pragma unroll
    for (int q = 0; q < QB; ++q) {
      unpack2(acc2[q][0], acc[q][0], acc[q][1]);
      unpack2(acc2[q][1], acc[q][2], acc[q][3]);
    }
    if (MODE == PDX_L2_PRUNE) {
#pragma unroll
      for (int j = 0; j < VPT; ++j) ss[j] = mx[j];
    }

    // epilogue: scores (and keys)
    if (!qn_visible) {  // first tile of this CTA: the query norm written by the last warp (CTA-uniform branch)
      __syncthreads();
      qn_visible = true;
    }
    float nrm[VPT];
    if (MODE == PDX_COSINE_FUSED || MODE == PDX_NORMS) {
#pragma unroll
      for (int j = 0; j < VPT; ++j) nrm[j] = __fsqrt_rn(ss[j]);  // *norm = norm.sqrt()  (src/batch.rs:683-685)
    }
    if (MODE == PDX_COSINE_NORMS) {
#pragma unroll
      for (int j = 0; j < VPT; ++j) nrm[j] = (active && i0 + j < a.n) ? a.norms_in[i0 + j] : 0.0f;
    }
    auto score = [&](int q, int j) -> float {
      if (MODE == PDX_COSINE_FUSED || MODE == PDX_COSINE_NORMS) {
        const float qn = s_qn[q];
        // src/batch.rs:716-727: qn < eps -> 0 for all; norm > eps ? dot / (qn * norm) : 0
        float c = 0.0f;
        if (!(qn < NORM_EPS) && nrm[j] > NORM_EPS) c = __fdiv_rn(acc[q][j], __fmul_rn(qn, nrm[j]));
        return c;
      } else if (MODE == PDX_NORMS) {
        return nrm[j];
      } else if (MODE == PDX_L2_PRUNE) {
        return ss[j] > a.threshold ? -1.0f : acc[q][j];  // distances are never negative: -1.0 marks "pruned"
      }
      return acc[q][j];
    };
    auto make_key = [&](float sc, unsigned i) -> uint64_t {
      return (MODE == PDX_L2 || MODE == PDX_L2_PERM) ? make_key_asc(sc, a.index_base + i) : make_key_desc(sc, a.index_base + i);
    };
    if (KNN && QB > 1) {
      // vector j of this thread against all QB queries at once: the QB lists are updated in lock step (offer_multi)
#pragma unroll
      for (int j = 0; j < VPT; ++j) {
        const unsigned i = i0 + j;
        uint64_t key[QB];
#pragma unroll
        for (int q = 0; q < QB; ++q) key[q] = make_key(score(q, j), i);
        offer_multi<R, QB>(lists, key, active && i < a.n && (!MASKED || ((nib >> j) & 1u)), thrs, a.nq_valid, a.k, lane);
      }
    } else {
#pragma unroll
      for (int q = 0; q < QB; ++q) {
        if (KNN) {
          if (q < a.nq_valid) {
#pragma unroll
            for (int j = 0; j < VPT; ++j) {
              const unsigned i = i0 + j;
              lists[q].offer(make_key(score(q, j), i), active && i < a.n && (!MASKED || ((nib >> j) & 1u)), thrs[q], a.k, lane);
            }
          }
        } else if (active && q < a.nq_valid) {
          *reinterpret_cast<float4*>(a.scores_out + (size_t)q * a.ld + i0) =
              make_float4(score(q, 0), score(q, 1), score(q, 2), score(q, 3));
        }
      }
    }
  }

  if (KNN) block_finish<R, QB>(lists, a.nq_valid, a.k, smem_keys, a.partials, a.group_partials, a.out_keys, a.tickets);
}

template <int MODE, int QB, int R, bool KNN, bool MASKED = false, int UX = 0>
cudaError_t launch_one(const PdxArgs& a, size_t smem, int ny, int num_sms, cudaStream_t s) {
  auto kern = pdx_scan_kernel<MODE, QB, R, KNN, MASKED, UX>;
  static size_t smem_set_dev[16] = {};
  size_t& smem_set = smem_set_dev[current_device_slot()];
  if (smem > 48 * 1024 && smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    smem_set = smem;
  }
  int occ = 0;
  cudaError_t eo = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, SCAN_THREADS, smem);
  if (eo != cudaSuccess) return eo;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  unsigned grid = balanced_grid(a.n_tiles, (unsigned)occ * (unsigned)num_sms);
  if (!KNN) grid = a.n_tiles ? a.n_tiles : 1;  // no cross-tile state: one CTA per tile, hardware scheduler balances
  kern<<<dim3(grid, ny > 0 ? ny : 1), SCAN_THREADS, smem, s>>>(a);
  return cudaGetLastError();
}

// grid.x the KNN launch will use (needed to size the merge workspace per query group)
template <int MODE, int QB, int R, int UX = 0>
unsigned knn_grid_x(unsigned n_tiles, size_t smem, int num_sms) {
  int occ = 0;
  if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pdx_scan_kernel<MODE, QB, R, true, false, UX>, SCAN_THREADS, smem) != cudaSuccess || occ < 1) occ = 1;
  return balanced_grid(n_tiles, (unsigned)occ * (unsigned)num_sms);
}

size_t scan_smem_bytes(size_t d, int qb, int k, bool knn, bool perm = false) {
  size_t d_pad = (d + 31) / 32 * 32;
  size_t b = d_pad * qb * sizeof(float) + ((qb + 3) & ~3) * sizeof(float);
  if (perm) b += d_pad * sizeof(unsigned);
  if (knn) b += (size_t)(SCAN_THREADS / 32) * k * sizeof(uint64_t) * qb;  // QB > 1: every warp parks QB lists (block_finish)
  return b;
}

}  // namespace

unsigned pdx_max_grid(int num_sms) { return (unsigned)num_sms * 8u; }

namespace {
// the arguments every scan launch shares. Columns actually scanned: n rounded up to a whole float4 (the row pitch is a
// multiple of 4, so the last float4 is in bounds); a prefix view (n << ld) scans only its own columns.
PdxArgs base_args(const PdxView& v, const Workspace& ws, size_t k) {
  PdxArgs a{};
  a.v = v;
  a.ld = v.ld;
  a.ld4 = (unsigned)std::min<size_t>(v.ld, (v.n + 3) / 4 * 4);
  a.n = (unsigned)v.n;
  a.d = (unsigned)v.d;
  a.n_tiles = (unsigned)(((size_t)a.ld4 + TILE - 1) / TILE);
  a.index_base = v.index_base;
  a.one = 1.0f;
  a.k = (int)k;
  a.partials = ws.partials;
  a.group_partials = ws.group_partials;
  a.tickets = ws.tickets;
  a.nq_valid = 1;
  return a;
}
}  // namespace

cudaError_t launch_pdx_knn(const PdxView& v, int mode, const float* dev_queries, size_t nq, size_t k,
                           uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches,
                           const unsigned* dev_run_flag) {
  PdxArgs a = base_args(v, ws, k);
  a.run_flag = dev_run_flag;
  const bool big_k = k > 32;
  // query blocking: 8 queries share one pass over the corpus when their lists fit in registers; several groups of 8
  // run as grid.y of ONE launch as long as their merge workspaces fit (small corpora / many queries: C1, sample pass)
  size_t done = 0;
  while (done < nq) {
    int qb = (nq - done >= 2 && !big_k) ? 8 : 1;
    size_t smem = scan_smem_bytes(v.d, qb, (int)k, true);
    if (smem > 200 * 1024 && qb == 8) {
      qb = 1;
      smem = scan_smem_bytes(v.d, 1, (int)k, true);
    }
    if (smem > 227 * 1024) return cudaErrorInvalidValue;
    int ny = 1;
    // at most ~2 CTAs per SM in the whole launch: the per-thread latency chain binds, use the deep-prefetch variants
    const size_t groups_left8 = (nq - done + 7) / 8;
    const bool deep = !big_k && (size_t)a.n_tiles * (qb == 8 ? groups_left8 : 1) <= 2 * (size_t)ws.num_sms;
    // not even one CTA per SM with eight queries per CTA (C1): four per CTA = twice the warps to hide latency with
    if (qb == 8 && deep && (size_t)a.n_tiles * groups_left8 <= (size_t)ws.num_sms) {
      qb = 4;
      smem = scan_smem_bytes(v.d, 4, (int)k, true);
    }
    if (qb > 1) {
      unsigned gx = 1;
      if (qb == 4) {
        if (mode == PDX_DOT) gx = knn_grid_x<PDX_DOT, 4, 1, 16>(a.n_tiles, smem, ws.num_sms);
        else if (mode == PDX_L2) gx = knn_grid_x<PDX_L2, 4, 1, 16>(a.n_tiles, smem, ws.num_sms);
        else gx = knn_grid_x<PDX_COSINE_FUSED, 4, 1, 16>(a.n_tiles, smem, ws.num_sms);
      } else if (deep) {
        if (mode == PDX_DOT) gx = knn_grid_x<PDX_DOT, 8, 1, 16>(a.n_tiles, smem, ws.num_sms);
        else if (mode == PDX_L2) gx = knn_grid_x<PDX_L2, 8, 1, 16>(a.n_tiles, smem, ws.num_sms);
        else gx = knn_grid_x<PDX_COSINE_FUSED, 8, 1, 16>(a.n_tiles, smem, ws.num_sms);
      } else if (mode == PDX_DOT) gx = knn_grid_x<PDX_DOT, 8, 1>(a.n_tiles, smem, ws.num_sms);
      else if (mode == PDX_L2) gx = knn_grid_x<PDX_L2, 8, 1>(a.n_tiles, smem, ws.num_sms);
      else gx = knn_grid_x<PDX_COSINE_FUSED, 8, 1>(a.n_tiles, smem, ws.num_sms);
      const size_t n_groups = (gx + FINISH_GROUP - 1) / FINISH_GROUP;
      size_t fit = ws.partials_cap / ((size_t)gx * qb * k);
      fit = std::min(fit, ws.group_cap / (n_groups * qb * k));
      fit = std::min(fit, ws.tickets_cap / (1 + n_groups));
      const size_t groups_left = (nq - done + qb - 1) / qb;
      ny = (int)std::max<size_t>(1, std::min<size_t>(std::min<size_t>(fit, groups_left), 65535));
    }
    const size_t nq_launch = std::min<size_t>(nq - done, (size_t)ny * qb);
    a.queries = dev_queries + done * v.d;
    a.nq_valid = (int)nq_launch;
    a.out_keys = dev_keys + done * k;
    cudaError_t e;
#define INNR_DISPATCH(MODE)                                                                          \
  if (qb == 4) e = launch_one<MODE, 4, 1, true, false, 16>(a, smem, ny, ws.num_sms, s);              \
  else if (qb == 8 && deep) e = launch_one<MODE, 8, 1, true, false, 16>(a, smem, ny, ws.num_sms, s); \
  else if (qb == 8) e = launch_one<MODE, 8, 1, true>(a, smem, ny, ws.num_sms, s);                    \
  else if (deep) e = launch_one<MODE, 1, 1, true, false, 32>(a, smem, 1, ws.num_sms, s);             \
  else if (!big_k) e = launch_one<MODE, 1, 1, true>(a, smem, 1, ws.num_sms, s);                      \
  else e = launch_one<MODE, 1, 4, true>(a, smem, 1, ws.num_sms, s);
    if (mode == PDX_DOT) { INNR_DISPATCH(PDX_DOT) }
    else if (mode == PDX_L2) { INNR_DISPATCH(PDX_L2) }
    else if (mode == PDX_COSINE_FUSED) { INNR_DISPATCH(PDX_COSINE_FUSED) }
    else return cudaErrorInvalidValue;
#undef INNR_DISPATCH
    if (e != cudaSuccess) return e;
    ++*launches;
    done += nq_launch;
  }
  return cudaSuccess;
}

cudaError_t launch_pdx_knn_filtered(const PdxView& v, const float* dev_query, const uint32_t* dev_mask, size_t k,
                                    uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches) {
  PdxArgs a = base_args(v, ws, k);
  a.queries = dev_query;
  a.out_keys = dev_keys;
  a.mask = dev_mask;
  const size_t smem = scan_smem_bytes(v.d, 1, (int)k, true);
  if (smem > 227 * 1024 || k > 128) return cudaErrorInvalidValue;
  cudaError_t e = (k <= 32) ? launch_one<PDX_L2, 1, 1, true, true>(a, smem, 1, ws.num_sms, s)
                            : launch_one<PDX_L2, 1, 4, true, true>(a, smem, 1, ws.num_sms, s);
  if (e == cudaSuccess) ++*launches;
  return e;
}

cudaError_t launch_pdx_knn_reordered(const PdxView& v, const float* dev_query, const uint32_t* dev_perm, size_t k,
                                     uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches) {
  PdxArgs a = base_args(v, ws, k);
  a.queries = dev_query;
  a.out_keys = dev_keys;
  a.perm = dev_perm;
  const size_t smem = scan_smem_bytes(v.d, 1, (int)k, true, true);
  if (smem > 227 * 1024 || k > 128 || !dev_perm) return cudaErrorInvalidValue;
  cudaError_t e = (k <= 32) ? launch_one<PDX_L2_PERM, 1, 1, true>(a, smem, 1, ws.num_sms, s)
                            : launch_one<PDX_L2_PERM, 1, 4, true>(a, smem, 1, ws.num_sms, s);
  if (e == cudaSuccess) ++*launches;
  return e;
}

// ---------------------------------------------------------------------------------------------------------
// batch_dimension_variance (src/batch.rs:572-592). Both sums of a dimension row are sequential f32 sums over all n
// vectors, so a row is one chain of n dependent adds whatever the hardware: one warp per row, rows in parallel (d warps);
// the chain, not HBM, bounds it (~4 cycles per vector per pass).
// ---------------------------------------------------------------------------------------------------------
namespace {

constexpr int VAR_WARPS = 4;

constexpr int VAR_UV = 4;  // 128-value groups per step (512 values: 2 KB of shared memory per warp)

// One sequential f32 sum over a dimension row: sum of x (CENTERED = false) or of (x - mean) * (x - mean), unfused.
// The warp loads 512 consecutive values per step (the next step's loads are issued before this step's chain runs),
// parks them in shared memory, and every lane replays the chain from broadcast 128-bit reads.
template <bool CENTERED>
__device__ __forceinline__ float row_chain(const PdxView& v, size_t row, unsigned n, float mean, int lane, float4* buf) {
  float acc = 0.0f;
  constexpr unsigned STEP = 128u * VAR_UV;
  const unsigned n_steps = n / STEP;
  float4 cur[VAR_UV], nxt[VAR_UV];
  if (n_steps) {
#pragma unroll
    for (int u = 0; u < VAR_UV; ++u) cur[u] = pdx_load4(v, row + 128u * u + 4u * lane);
  }
  for (unsigned st = 0; st < n_steps; ++st) {
    if (st + 1 < n_steps) {
      const size_t p = row + (size_t)(st + 1) * STEP + 4u * lane;
#pragma unroll
      for (int u = 0; u < VAR_UV; ++u) nxt[u] = pdx_load4(v, p + 128u * u);
    }
#pragma unroll
    for (int u = 0; u < VAR_UV; ++u) {
      float4 x = cur[u];
      if (CENTERED) {  // computed once per value by the lane that loaded it
        x.x = __fsub_rn(x.x, mean); x.y = __fsub_rn(x.y, mean); x.z = __fsub_rn(x.z, mean); x.w = __fsub_rn(x.w, mean);
        x.x = __fmul_rn(x.x, x.x); x.y = __fmul_rn(x.y, x.y); x.z = __fmul_rn(x.z, x.z); x.w = __fmul_rn(x.w, x.w);
      }
      buf[u * 32 + lane] = x;
    }
    __syncwarp();
#pragma unroll 16
    for (int j = 0; j < VAR_UV * 32; ++j) {
      const float4 x = buf[j];
      acc = __fadd_rn(acc, x.x);
      acc = __fadd_rn(acc, x.y);
      acc = __fadd_rn(acc, x.z);
      acc = __fadd_rn(acc, x.w);
    }
    __syncwarp();
#pragma unroll
    for (int u = 0; u < VAR_UV; ++u) cur[u] = nxt[u];
  }
#pragma unroll 8
  for (unsigned i = n_steps * STEP; i < n; ++i) {  // tail (< 512 values): every lane reads the same value
    float x = pdx_load1(v, row + i);
    if (CENTERED) { x = __fsub_rn(x, mean); x = __fmul_rn(x, x); }
    acc = __fadd_rn(acc, x);
  }
  return acc;
}

__global__ void __launch_bounds__(VAR_WARPS * 32) dimension_variance_kernel(const PdxView v, unsigned n, unsigned d,
                                                                            float* __restrict__ out) {
  __shared__ float4 s_buf[VAR_WARPS][VAR_UV * 32];
  const unsigned dd = blockIdx.x * VAR_WARPS + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (dd >= d) return;
  float4* buf = s_buf[threadIdx.x >> 5];
  const size_t row = (size_t)dd * v.ld;
  const float nf = (float)n;                                     // let n = batch.num_vectors as f32;
  const float mean = __fdiv_rn(row_chain<false>(v, row, n, 0.0f, lane, buf), nf);
  const float var = __fdiv_rn(row_chain<true>(v, row, n, mean, lane, buf), nf);
  if (lane == 0) out[dd] = var;
}

}  // namespace

cudaError_t launch_dimension_variance(const PdxView& v, float* dev_out, cudaStream_t s, LaunchCounter* launches) {
  if (v.d == 0) return cudaSuccess;
  if (v.n <= 1) return cudaMemsetAsync(dev_out, 0, v.d * sizeof(float), s);  // src/batch.rs:573-575
  dimension_variance_kernel<<<(unsigned)((v.d + VAR_WARPS - 1) / VAR_WARPS), VAR_WARPS * 32, 0, s>>>(v, (unsigned)v.n, (unsigned)v.d,
                                                                                                  dev_out);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_pdx_scores(const PdxView& v, int mode, const float* dev_query, const float* dev_norms,
                              float* dev_out, Workspace& ws, cudaStream_t s, LaunchCounter* launches, float threshold,
                              const uint32_t* dev_perm) {
  PdxArgs a = base_args(v, ws, 0);
  a.perm = dev_perm;
  a.queries = dev_query;
  a.scores_out = dev_out;
  a.norms_in = dev_norms;
  a.threshold = threshold;
  size_t smem = scan_smem_bytes(v.d, 1, 0, false, mode == PDX_L2_PERM);
  if (smem > 227 * 1024 || (mode == PDX_L2_PERM && !dev_perm)) return cudaErrorInvalidValue;
  cudaError_t e;
  // few tiles (<= 2 per SM): the D / U round trips of each thread bind, not HBM -> deep-prefetch instantiations
  const bool deep = (size_t)a.n_tiles <= 2 * (size_t)ws.num_sms;
  if (deep && (mode == PDX_DOT || mode == PDX_L2 || mode == PDX_NORMS || mode == PDX_COSINE_NORMS || mode == PDX_COSINE_FUSED)) {
    switch (mode) {
      case PDX_DOT: e = launch_one<PDX_DOT, 1, 1, false, false, 32>(a, smem, 1, ws.num_sms, s); break;
      case PDX_L2: e = launch_one<PDX_L2, 1, 1, false, false, 32>(a, smem, 1, ws.num_sms, s); break;
      case PDX_NORMS: e = launch_one<PDX_NORMS, 1, 1, false, false, 32>(a, smem, 1, ws.num_sms, s); break;
      case PDX_COSINE_NORMS: e = launch_one<PDX_COSINE_NORMS, 1, 1, false, false, 32>(a, smem, 1, ws.num_sms, s); break;
      default: e = launch_one<PDX_COSINE_FUSED, 1, 1, false, false, 32>(a, smem, 1, ws.num_sms, s); break;
    }
    if (e == cudaSuccess) ++*launches;
    return e;
  }
  switch (mode) {
    case PDX_L2_PERM: e = launch_one<PDX_L2_PERM, 1, 1, false>(a, smem, 1, ws.num_sms, s); break;
    case PDX_DOT: e = launch_one<PDX_DOT, 1, 1, false>(a, smem, 1, ws.num_sms, s); break;
    case PDX_L2: e = launch_one<PDX_L2, 1, 1, false>(a, smem, 1, ws.num_sms, s); break;
    case PDX_NORMS: e = launch_one<PDX_NORMS, 1, 1, false>(a, smem, 1, ws.num_sms, s); break;
    case PDX_COSINE_NORMS: e = launch_one<PDX_COSINE_NORMS, 1, 1, false>(a, smem, 1, ws.num_sms, s); break;
    case PDX_L2_PRUNE: e = launch_one<PDX_L2_PRUNE, 1, 1, false>(a, smem, 1, ws.num_sms, s); break;
    case PDX_COSINE_FUSED: e = launch_one<PDX_COSINE_FUSED, 1, 1, false>(a, smem, 1, ws.num_sms, s); break;
    default: return cudaErrorInvalidValue;
  }
  if (e == cudaSuccess) ++*launches;
  return e;
}

// ---------------------------------------------------------------------------------------------------------
// merge of key lists (K10: after the allgather of per-shard top-k) and the TopK analogue
// ---------------------------------------------------------------------------------------------------------
namespace {

template <int R>
__global__ void __launch_bounds__(32) merge_keys_kernel(const uint64_t* in, int n_lists, int nq, int k,
                                                        int descending, uint64_t* keys_out, uint64_t* idx_out,
                                                        float* score_out) {
  const int q = blockIdx.x, lane = threadIdx.x;
  WarpList<R> list;
  list.init();
  warp_merge_lists<R, true>(list, in + (size_t)q * k, 0, 1, n_lists, (size_t)nq * k, k, lane);
#pragma unroll
  for (int r = 0; r < R; ++r) {
    int p = r * 32 + lane;
    if (p < k) {
      uint64_t key = list.v[r];
      if (keys_out) keys_out[(size_t)q * k + p] = key;
      if (idx_out) idx_out[(size_t)q * k + p] = key & 0xFFFFFFFFull;
      if (score_out) {
        uint32_t hi = (uint32_t)(key >> 32);
        if (descending) hi = ~hi;
        score_out[(size_t)q * k + p] = __uint_as_float(order_bits_to_f32_bits(hi));
      }
    }
  }
}

// Selection over a device score vector. KIND 0: f32 ascending (TopK analogue / L2), 1: f32 descending (dot, cosine,
// u8), 2: u32 ascending (Hamming). Keys carry index_base + i. `floor_key` (device, may be null) makes the launch one
// ROUND of a larger selection: only keys strictly greater than *floor_key take part, so consecutive rounds of <= 128
// keys each, every one starting above the last key of the round before, enumerate the k smallest keys for any k
// (keys are unique: the index is their low half).
template <int R, int KIND>
__global__ void __launch_bounds__(SCAN_THREADS) topk_scores_kernel(const void* scores, unsigned n, unsigned index_base,
                                                                  const uint32_t* ids,  // null: id = index_base + i
                                                                  const uint32_t* mask, // non-null: only entries whose bit is set
                                                                  unsigned seg_len, unsigned seg_stride,  // KIND 3 (see below)
                                                                  int k, const uint64_t* floor_key, uint64_t* partials,
                                                                  uint64_t* group_partials, uint64_t* out_keys,
                                                                  unsigned* tickets) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(smem_raw);
  const int lane = threadIdx.x & 31;
  WarpList<R> lists[1];
  uint64_t thrs[1];
  lists[0].init();
  thrs[0] = KEY_SENTINEL;
  const bool has_floor = floor_key != nullptr;
  const uint64_t floor = has_floor ? *floor_key : 0ull;
  // grid-stride over whole warps so every lane reaches the ballots together
  const unsigned stride = gridDim.x * blockDim.x;
  const unsigned n_round = (n + 31u) / 32u * 32u;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += stride) {
    bool valid = i < n && (!mask || ((mask[i >> 5] >> (i & 31)) & 1u));
    uint64_t key = KEY_SENTINEL;
    if (valid) {
      const unsigned id = ids ? ids[i] : index_base + i;
      if (KIND == 3) key = static_cast<const uint64_t*>(scores)[(size_t)(i / seg_len) * seg_stride + (i % seg_len)];
      else if (KIND == 4) key = make_key_u32(~static_cast<const uint32_t*>(scores)[i], id);
      else if (KIND == 2) key = make_key_u32(static_cast<const uint32_t*>(scores)[i], id);
      else if (KIND == 1) key = make_key_desc(static_cast<const float*>(scores)[i], id);
      else key = make_key_asc(static_cast<const float*>(scores)[i], id);
      valid = (KIND != 3 || key != KEY_SENTINEL) && (!has_floor || (key > floor && floor != KEY_SENTINEL));
    }
    lists[0].offer(key, valid, thrs[0], k, lane);
  }
  block_finish<R, 1>(lists, 1, k, smem_keys, partials, group_partials, out_keys, tickets);
}

}  // namespace

// ---------------------------------------------------------------------------------------------------------
// compaction of a pruned distance vector: survivors (entries != -1.0) in ascending index order, the order of the
// reference's `alive.iter().enumerate().filter(..).collect()` (src/batch.rs:358-364)
// ---------------------------------------------------------------------------------------------------------
namespace {
constexpr int CP_THREADS = 256, CP_ITEMS = 4, CP_BLOCK = CP_THREADS * CP_ITEMS;

__device__ __forceinline__ bool survivor(float d) { return !(d == -1.0f); }  // NaN distances survive (never pruned)

__global__ void __launch_bounds__(CP_THREADS) compact_count_kernel(const float* __restrict__ dist, unsigned n,
                                                                   unsigned* __restrict__ block_counts) {
  const unsigned base = blockIdx.x * CP_BLOCK;
  unsigned c = 0;
#pragma unroll
  for (int it = 0; it < CP_ITEMS; ++it) {
    const unsigned i = base + it * CP_THREADS + threadIdx.x;
    c += __popc(__ballot_sync(FULL_MASK, i < n && survivor(dist[i])));
  }
  __shared__ unsigned s_c[CP_THREADS / 32];
  if ((threadIdx.x & 31) == 0) s_c[threadIdx.x >> 5] = c;  // every lane of the warp holds the warp total
  __syncthreads();
  if (threadIdx.x == 0) {
    unsigned t = 0;
    for (int w = 0; w < CP_THREADS / 32; ++w) t += s_c[w];
    block_counts[blockIdx.x] = t;
  }
}

// in place: counts -> exclusive prefix; offsets[n_blocks] = total. One CTA (n_blocks <= 2^32 / 1024).
__global__ void __launch_bounds__(1024) compact_scan_kernel(unsigned* __restrict__ offsets, unsigned n_blocks) {
  __shared__ unsigned s_w[32];
  __shared__ unsigned s_carry;
  if (threadIdx.x == 0) s_carry = 0;
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  for (unsigned b0 = 0; b0 < n_blocks; b0 += 1024) {
    const unsigned b = b0 + threadIdx.x;
    const unsigned v = b < n_blocks ? offsets[b] : 0u;
    unsigned x = v;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const unsigned y = __shfl_up_sync(FULL_MASK, x, o);
      if (lane >= o) x += y;
    }
    if (lane == 31) s_w[warp] = x;
    __syncthreads();
    if (warp == 0) {
      unsigned w = s_w[lane];
#pragma unroll
      for (int o = 1; o < 32; o <<= 1) {
        const unsigned y = __shfl_up_sync(FULL_MASK, w, o);
        if (lane >= o) w += y;
      }
      s_w[lane] = w;  // inclusive over warps
    }
    __syncthreads();
    const unsigned carry = s_carry;
    const unsigned incl = carry + (warp ? s_w[warp - 1] : 0u) + x;
    if (b < n_blocks) offsets[b] = incl - v;
    __syncthreads();
    if (threadIdx.x == 1023) s_carry = incl;
    __syncthreads();
  }
  if (threadIdx.x == 0) offsets[n_blocks] = s_carry;
}

__global__ void __launch_bounds__(CP_THREADS) compact_scatter_kernel(const float* __restrict__ dist, unsigned n,
                                                                     unsigned long long index_base,
                                                                     const unsigned* __restrict__ block_offsets,
                                                                     uint64_t* __restrict__ out_idx,
                                                                     float* __restrict__ out_dist) {
  const unsigned base = blockIdx.x * CP_BLOCK;
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  __shared__ unsigned s_c[CP_ITEMS][CP_THREADS / 32];
  float d[CP_ITEMS];
  unsigned bal[CP_ITEMS];
#pragma unroll
  for (int it = 0; it < CP_ITEMS; ++it) {
    const unsigned i = base + it * CP_THREADS + threadIdx.x;
    d[it] = i < n ? dist[i] : -1.0f;
    bal[it] = __ballot_sync(FULL_MASK, survivor(d[it]));
    if (lane == 0) s_c[it][warp] = __popc(bal[it]);
  }
  __syncthreads();
  // position of (it, warp) inside the block: items are laid out it-major (index = base + it*256 + tid)
  unsigned before = block_offsets[blockIdx.x];
#pragma unroll
  for (int it = 0; it < CP_ITEMS; ++it) {
    unsigned pre = 0;
    for (int w = 0; w < warp; ++w) pre += s_c[it][w];
    if (survivor(d[it])) {
      const unsigned pos = before + pre + __popc(bal[it] & ((1u << lane) - 1u));
      out_idx[pos] = index_base + base + it * CP_THREADS + threadIdx.x;
      out_dist[pos] = d[it];
    }
    unsigned tot = 0;
    for (int w = 0; w < CP_THREADS / 32; ++w) tot += s_c[it][w];
    before += tot;
  }
}
}  // namespace

size_t compact_blocks(size_t n) { return (n + CP_BLOCK - 1) / CP_BLOCK; }

cudaError_t launch_compact_count(const float* dev_dist, size_t n, unsigned* dev_block_offsets, cudaStream_t s,
                                 LaunchCounter* launches) {
  const unsigned nb = (unsigned)compact_blocks(n);
  if (nb == 0) return cudaMemsetAsync(dev_block_offsets, 0, sizeof(unsigned), s);
  compact_count_kernel<<<nb, CP_THREADS, 0, s>>>(dev_dist, (unsigned)n, dev_block_offsets);
  compact_scan_kernel<<<1, 1024, 0, s>>>(dev_block_offsets, nb);
  *launches += 2;
  return cudaGetLastError();
}

cudaError_t launch_compact_scatter(const float* dev_dist, size_t n, uint64_t index_base, const unsigned* dev_block_offsets,
                                   uint64_t* dev_idx, float* dev_out, cudaStream_t s, LaunchCounter* launches) {
  const unsigned nb = (unsigned)compact_blocks(n);
  if (nb == 0) return cudaSuccess;
  compact_scatter_kernel<<<nb, CP_THREADS, 0, s>>>(dev_dist, (unsigned)n, index_base, dev_block_offsets, dev_idx, dev_out);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_merge_keys(const uint64_t* dev_in, size_t n_lists, size_t nq, size_t k, int descending,
                              uint64_t* dev_keys_out, uint64_t* dev_idx, float* dev_score, cudaStream_t s,
                              LaunchCounter* launches) {
  if (k > 128) return cudaErrorInvalidValue;
  if (k <= 32)
    merge_keys_kernel<1><<<(unsigned)nq, 32, 0, s>>>(dev_in, (int)n_lists, (int)nq, (int)k, descending,
                                                      dev_keys_out, dev_idx, dev_score);
  else
    merge_keys_kernel<4><<<(unsigned)nq, 32, 0, s>>>(dev_in, (int)n_lists, (int)nq, (int)k, descending,
                                                      dev_keys_out, dev_idx, dev_score);
  ++*launches;
  return cudaGetLastError();
}

namespace {
// Exact scores of a SUBSET of the corpus (re-rank stage of a two-stage search: binary / u8 first pass -> exact f32,
// src/scalar.rs:366-368, examples/binary_demo.rs:235-237). One thread per candidate, the reference's sequential unfused
// arithmetic (same bits as the full scan); out-of-range candidates score the metric's worst value.
template <int MODE>
__global__ void __launch_bounds__(SCAN_THREADS) subset_scores_kernel(const PdxView v, unsigned n,
                                                                    unsigned d, unsigned index_base,
                                                                    const float* __restrict__ query,
                                                                    const uint32_t* __restrict__ cand, unsigned m,
                                                                    float* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sq = reinterpret_cast<float*>(smem_raw);
  __shared__ float s_qn;
  for (unsigned i = threadIdx.x; i < d; i += blockDim.x) sq[i] = query[i];
  if (threadIdx.x == 0) {
    float ss = 0.0f;
    for (unsigned i = 0; i < d; ++i) ss = __fadd_rn(ss, __fmul_rn(query[i], query[i]));
    s_qn = __fsqrt_rn(ss);
  }
  __syncthreads();
  const unsigned j = blockIdx.x * blockDim.x + threadIdx.x;
  if (j >= m) return;
  const unsigned gid = cand[j];
  const unsigned i = gid - index_base;  // candidates carry global ids
  if (gid < index_base || i >= n) {
    out[j] = MODE == PDX_L2 ? __int_as_float(0x7FC00000) : __int_as_float(0xFFC00000);  // sorts last under total_cmp
    return;
  }
  float acc = 0.0f, ss = 0.0f;
  for (unsigned dd = 0; dd < d; ++dd) {
    const float x = pdx_load1(v, (size_t)dd * v.ld + i);
    accumulate<MODE == PDX_COSINE_FUSED ? PDX_DOT : MODE>(sq[dd], x, acc);
    if (MODE == PDX_COSINE_FUSED) ss = __fadd_rn(ss, __fmul_rn(x, x));
  }
  float sc = acc;
  if (MODE == PDX_COSINE_FUSED) {
    const float nrm = __fsqrt_rn(ss), qn = s_qn;
    sc = (!(qn < NORM_EPS) && nrm > NORM_EPS) ? __fdiv_rn(acc, __fmul_rn(qn, nrm)) : 0.0f;
  }
  out[j] = sc;
}
}  // namespace

cudaError_t launch_subset_scores(const PdxView& v, int mode, const float* dev_query, const uint32_t* dev_cand, size_t m,
                                 float* dev_out, cudaStream_t s, LaunchCounter* launches) {
  if (m == 0) return cudaSuccess;
  const unsigned grid = (unsigned)((m + SCAN_THREADS - 1) / SCAN_THREADS);
  const size_t smem = ((v.d + 3) & ~(size_t)3) * sizeof(float);
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
#define INNR_SUBSET(MODE)                                                                                           \
  {                                                                                                                 \
    auto kern = subset_scores_kernel<MODE>;                                                                         \
    if (smem > 48 * 1024) {                                                                                         \
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);           \
      if (e != cudaSuccess) return e;                                                                               \
    }                                                                                                               \
    kern<<<grid, SCAN_THREADS, smem, s>>>(v, (unsigned)v.n, (unsigned)v.d, v.index_base, dev_query,                 \
                                          dev_cand, (unsigned)m, dev_out);                                          \
  }
  if (mode == PDX_DOT) INNR_SUBSET(PDX_DOT)
  else if (mode == PDX_L2) INNR_SUBSET(PDX_L2)
  else if (mode == PDX_COSINE_FUSED) INNR_SUBSET(PDX_COSINE_FUSED)
  else return cudaErrorInvalidValue;
#undef INNR_SUBSET
  ++*launches;
  return cudaGetLastError();
}

// k keys of a score vector, any k: rounds of <= 128 keys, each bounded below by the last key of the round before
// (read on the device: no host synchronisation between rounds)
cudaError_t launch_topk_from_scores(const void* dev_scores, int kind, size_t n, uint32_t index_base, size_t k,
                                    uint64_t* dev_keys, Workspace& ws, cudaStream_t s, LaunchCounter* launches,
                                    const uint32_t* dev_ids, const uint32_t* dev_mask, unsigned seg_len, unsigned seg_stride) {
  unsigned grid = (unsigned)((n + SCAN_THREADS - 1) / SCAN_THREADS);
  unsigned cap = (unsigned)ws.num_sms * 4u;
  if (grid > cap) grid = cap;
  if (grid == 0) grid = 1;
  for (size_t done = 0; done < k; done += 128) {
    const int kr = (int)std::min<size_t>(128, k - done);
    const uint64_t* floor = done ? dev_keys + done - 1 : nullptr;
    uint64_t* out = dev_keys + done;
    const size_t smem = (size_t)(SCAN_THREADS / 32) * kr * sizeof(uint64_t);
#define INNR_TOPK_LAUNCH(R, KIND)                                                                                   \
  topk_scores_kernel<R, KIND><<<grid, SCAN_THREADS, smem, s>>>(dev_scores, (unsigned)n, index_base, dev_ids, dev_mask, seg_len, seg_stride, kr, floor, \
                                                               ws.partials, ws.group_partials, out, ws.tickets)
    if (kr <= 32) {
      if (kind == 0) INNR_TOPK_LAUNCH(1, 0); else if (kind == 1) INNR_TOPK_LAUNCH(1, 1);
      else if (kind == 2) INNR_TOPK_LAUNCH(1, 2); else if (kind == 3) INNR_TOPK_LAUNCH(1, 3); else INNR_TOPK_LAUNCH(1, 4);
    } else {
      if (kind == 0) INNR_TOPK_LAUNCH(4, 0); else if (kind == 1) INNR_TOPK_LAUNCH(4, 1);
      else if (kind == 2) INNR_TOPK_LAUNCH(4, 2); else if (kind == 3) INNR_TOPK_LAUNCH(4, 3); else INNR_TOPK_LAUNCH(4, 4);
    }
#undef INNR_TOPK_LAUNCH
    ++*launches;
    cudaError_t e = cudaGetLastError();
    if (e != cudaSuccess) return e;
  }
  return cudaSuccess;
}

namespace {
__global__ void decode_keys_kernel(const uint64_t* __restrict__ keys, size_t total, int descending, uint64_t* __restrict__ idx,
                                   float* __restrict__ score) {
  const size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= total) return;
  const uint64_t key = keys[t];
  if (idx) idx[t] = key & 0xFFFFFFFFull;
  if (score) {
    uint32_t hi = (uint32_t)(key >> 32);
    if (descending) hi = ~hi;
    score[t] = __uint_as_float(order_bits_to_f32_bits(hi));
  }
}
}  // namespace

// merge for k > 128: per query, selection rounds of <= 128 over the n_lists * k gathered keys, then one decode launch
cudaError_t launch_merge_keys_big(const uint64_t* dev_in, size_t n_lists, size_t nq, size_t k, int descending,
                                  uint64_t* dev_keys_out, uint64_t* dev_idx, float* dev_score, Workspace& ws, cudaStream_t s,
                                  LaunchCounter* launches) {
  for (size_t q = 0; q < nq; ++q) {
    cudaError_t e = launch_topk_from_scores(dev_in + q * k, 3, n_lists * k, 0, k, dev_keys_out + q * k, ws, s, launches, nullptr,
                                            nullptr, (unsigned)k, (unsigned)(nq * k));
    if (e != cudaSuccess) return e;
  }
  if (dev_idx || dev_score) {
    const size_t total = nq * k;
    decode_keys_kernel<<<(unsigned)((total + 255) / 256), 256, 0, s>>>(dev_keys_out, total, descending, dev_idx, dev_score);
    ++*launches;
  }
  return cudaGetLastError();
}

// ---------------------------------------------------------------------------------------------------------
// batch_knn_adaptive (src/batch.rs:441-564). The reference walks the dimensions one by one and, inside a dimension, the
// vectors in index order, pruning a candidate when its partial distance exceeds a threshold that is refreshed after
// every dimension d with d % 32 == 0 -- and never pruning once only k candidates are left. Between two refreshes the
// threshold is constant, so an "epoch" (the dimensions up to and including the next refresh point) is one pass: every
// live vector continues its sequential sum and notes the first dimension at which it exceeded the threshold. Unless
// fewer than k candidates would remain, all of those are pruned, in any order; otherwise the host resolves the
// reference's (dimension, index) order from the noted dimensions (api.cu). Rows of dead vectors are not read.
// ---------------------------------------------------------------------------------------------------------
namespace {

struct AdaptArgs {
  PdxView v;
  unsigned long long ld;
  unsigned ld4;
  const float* query;
  unsigned d0, d1;          // dimensions [d0, d1) of this epoch
  float* dist;              // partial distances (in/out)
  const uint32_t* mask_in;  // bit i: vector i is a live candidate
  uint32_t* mask_out;
  const float* thr;         // thr[0]: the epoch's threshold (device)
  uint32_t* ev;             // ev[i]: first dimension at which vector i exceeded the threshold (written when it did)
  unsigned* pruned;         // += number of vectors that exceeded it
  int no_prune;             // only k candidates left: accumulate, never prune (src/batch.rs:520 `alive_count > k`)
};

__global__ void __launch_bounds__(SCAN_THREADS) adaptive_epoch_kernel(const AdaptArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  float* sq = reinterpret_cast<float*>(smem_raw);
  const unsigned nd = a.d1 - a.d0;
  for (unsigned j = threadIdx.x; j < nd; j += blockDim.x) sq[j] = a.query[a.d0 + j];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const unsigned i0 = (blockIdx.x * SCAN_THREADS + threadIdx.x) * VPT;
  const bool in = i0 < a.ld4;
  unsigned nib = in ? (a.mask_in[i0 >> 5] >> (i0 & 31)) & 0xFu : 0u;
  unsigned n_dead = 0;
  if (nib) {
    float4 acc = *reinterpret_cast<const float4*>(a.dist + i0);
    const float T = a.thr[0];
    unsigned ex = 0, e0 = 0, e1 = 0, e2 = 0, e3 = 0;
    size_t p = (size_t)a.d0 * a.ld + i0;
    auto step = [&](const float4& v, unsigned j) {
      const float q = sq[j];
      float df;
      df = __fsub_rn(q, v.x); acc.x = __fadd_rn(acc.x, __fmul_rn(df, df));
      df = __fsub_rn(q, v.y); acc.y = __fadd_rn(acc.y, __fmul_rn(df, df));
      df = __fsub_rn(q, v.z); acc.z = __fadd_rn(acc.z, __fmul_rn(df, df));
      df = __fsub_rn(q, v.w); acc.w = __fadd_rn(acc.w, __fmul_rn(df, df));
      if (!(ex & 1u) && acc.x > T) { ex |= 1u; e0 = a.d0 + j; }   // *dist > threshold  (src/batch.rs:520)
      if (!(ex & 2u) && acc.y > T) { ex |= 2u; e1 = a.d0 + j; }
      if (!(ex & 4u) && acc.z > T) { ex |= 4u; e2 = a.d0 + j; }
      if (!(ex & 8u) && acc.w > T) { ex |= 8u; e3 = a.d0 + j; }
    };
    constexpr int U = 8;
    unsigned j = 0;
    for (; j + U <= nd; j += U) {
      float4 v[U];
#pragma unroll
      for (int u = 0; u < U; ++u) v[u] = pdx_load4(a.v, p + (size_t)u * a.ld);
      p += (size_t)U * a.ld;
#pragma unroll
      for (int u = 0; u < U; ++u) step(v[u], j + u);
    }
    for (; j < nd; ++j) {
      const float4 v = pdx_load4(a.v, p);
      p += a.ld;
      step(v, j);
    }
    *reinterpret_cast<float4*>(a.dist + i0) = acc;
    if (!a.no_prune) {
      const unsigned dead = ex & nib;
      if (dead & 1u) a.ev[i0] = e0;
      if (dead & 2u) a.ev[i0 + 1] = e1;
      if (dead & 4u) a.ev[i0 + 2] = e2;
      if (dead & 8u) a.ev[i0 + 3] = e3;
      nib &= ~dead;
      n_dead = __popc(dead);
    }
  }
  // eight lanes hold the 32 bits of one mask word
  unsigned w = nib << (4 * (lane & 7));
  w |= __shfl_xor_sync(FULL_MASK, w, 1);
  w |= __shfl_xor_sync(FULL_MASK, w, 2);
  w |= __shfl_xor_sync(FULL_MASK, w, 4);
  if (in && (lane & 7) == 0) a.mask_out[i0 >> 5] = w;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) n_dead += __shfl_xor_sync(FULL_MASK, n_dead, o);
  if (lane == 0 && n_dead) atomicAdd(a.pruned, n_dead);
}

// thr[0] = (score of *key) * scale, thr[1] = thr[0] * 1.5  (src/batch.rs:486-487, :496, :546)
__global__ void adaptive_threshold_kernel(const uint64_t* key, float scale, float* thr) {
  const float t = __fmul_rn(__uint_as_float(order_bits_to_f32_bits((uint32_t)(*key >> 32))), scale);
  thr[0] = t;
  thr[1] = __fmul_rn(t, 1.5f);
}

// first pruning round (src/batch.rs:493-501): candidate i dies when dist[i] * ratio > threshold * 1.5
__global__ void __launch_bounds__(SCAN_THREADS) adaptive_mark_kernel(const float* __restrict__ dist, unsigned n, unsigned ld4,
                                                                    float ratio, const float* __restrict__ thr,
                                                                    uint32_t* __restrict__ mask_out, unsigned* pruned) {
  const int lane = threadIdx.x & 31;
  const unsigned i = blockIdx.x * SCAN_THREADS + threadIdx.x;
  const unsigned words32 = (ld4 + 31u) / 32u * 32u;
  bool alive = false, dead = false;
  if (i < n) {
    dead = __fmul_rn(dist[i], ratio) > thr[1];
    alive = !dead;
  }
  const unsigned w = __ballot_sync(FULL_MASK, alive);
  const unsigned nd = __popc(__ballot_sync(FULL_MASK, dead));
  if (lane == 0) {
    if (i < words32) mask_out[i >> 5] = w;
    if (nd) atomicAdd(pruned, nd);
  }
}

// vectors that were live before the epoch and are not after it, as keys ordered by DEcreasing (dimension, index)
__global__ void __launch_bounds__(SCAN_THREADS) adaptive_event_keys_kernel(const uint32_t* __restrict__ before,
                                                                          const uint32_t* __restrict__ after,
                                                                          const uint32_t* __restrict__ ev, unsigned n,
                                                                          uint64_t* __restrict__ keys) {
  const unsigned i = blockIdx.x * SCAN_THREADS + threadIdx.x;
  if (i >= n) return;
  const bool event = ((before[i >> 5] & ~after[i >> 5]) >> (i & 31)) & 1u;
  keys[i] = event ? ~(((uint64_t)ev[i] << 32) | i) : KEY_SENTINEL;
}

__global__ void adaptive_revive_kernel(const uint64_t* __restrict__ keys, unsigned m, uint32_t* mask) {
  const unsigned t = blockIdx.x * blockDim.x + threadIdx.x;
  if (t >= m) return;
  const unsigned i = (unsigned)(~keys[t] & 0xFFFFFFFFull);
  atomicOr(mask + (i >> 5), 1u << (i & 31));
}

}  // namespace

cudaError_t launch_adaptive_threshold(const uint64_t* dev_key, float scale, float* dev_thr, cudaStream_t s,
                                      LaunchCounter* launches) {
  adaptive_threshold_kernel<<<1, 1, 0, s>>>(dev_key, scale, dev_thr);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_adaptive_mark(const PdxView& v, const float* dev_dist, float ratio, const float* dev_thr,
                                 uint32_t* dev_mask_out, unsigned* dev_pruned, cudaStream_t s, LaunchCounter* launches) {
  const unsigned ld4 = (unsigned)std::min<size_t>(v.ld, (v.n + 3) / 4 * 4);
  const unsigned span = (ld4 + 31u) / 32u * 32u;
  adaptive_mark_kernel<<<(span + SCAN_THREADS - 1) / SCAN_THREADS, SCAN_THREADS, 0, s>>>(dev_dist, (unsigned)v.n, ld4, ratio,
                                                                                      dev_thr, dev_mask_out, dev_pruned);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_adaptive_epoch(const PdxView& v, const float* dev_query, size_t d0, size_t d1, float* dev_dist,
                                  const uint32_t* dev_mask_in, uint32_t* dev_mask_out, const float* dev_thr, uint32_t* dev_ev,
                                  unsigned* dev_pruned, int no_prune, cudaStream_t s, LaunchCounter* launches) {
  AdaptArgs a{};
  a.v = v;
  a.ld = v.ld;
  a.ld4 = (unsigned)std::min<size_t>(v.ld, (v.n + 3) / 4 * 4);
  a.query = dev_query;
  a.d0 = (unsigned)d0;
  a.d1 = (unsigned)d1;
  a.dist = dev_dist;
  a.mask_in = dev_mask_in;
  a.mask_out = dev_mask_out;
  a.thr = dev_thr;
  a.ev = dev_ev;
  a.pruned = dev_pruned;
  a.no_prune = no_prune;
  const unsigned span = (a.ld4 + 31u) / 32u * 32u;  // whole mask words: every word of the output mask is written
  const unsigned grid = (span / VPT + SCAN_THREADS - 1) / SCAN_THREADS;
  adaptive_epoch_kernel<<<grid, SCAN_THREADS, (d1 - d0) * sizeof(float), s>>>(a);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_adaptive_event_keys(const uint32_t* dev_before, const uint32_t* dev_after, const uint32_t* dev_ev, size_t n,
                                       uint64_t* dev_keys, cudaStream_t s, LaunchCounter* launches) {
  adaptive_event_keys_kernel<<<(unsigned)((n + SCAN_THREADS - 1) / SCAN_THREADS), SCAN_THREADS, 0, s>>>(dev_before, dev_after,
                                                                                                     dev_ev, (unsigned)n, dev_keys);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_adaptive_revive(const uint64_t* dev_keys, size_t m, uint32_t* dev_mask, cudaStream_t s,
                                   LaunchCounter* launches) {
  if (m == 0) return cudaSuccess;
  adaptive_revive_kernel<<<(unsigned)((m + 255) / 256), 256, 0, s>>>(dev_keys, (unsigned)m, dev_mask);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_topk_from_distances(const float* dev_dist, size_t n, size_t k, uint64_t* dev_keys,
                                       Workspace& ws, cudaStream_t s, LaunchCounter* launches) {
  return launch_topk_from_scores(dev_dist, 0, n, 0, k, dev_keys, ws, s, launches, nullptr, nullptr, 1, 1);
}

// ---------------------------------------------------------------------------------------------------------
// Screened single-query kNN of a split corpus (DESIGN.md section 3.1). Three steps, all on the device:
//  1. screen: stream the 8-bit sketch only; for each row an interval [lower, upper] that holds the reference's score.
//     Selection on the pessimistic bound (lower for dot / cosine, upper for L2) gives T, its k-th best value; every row
//     gets its optimistic bound written to ws.sc_bounds.
//  2. compaction: the rows whose optimistic bound reaches T. At least k rows have a score at least as good as T, so
//     every row of the top k (ties on the k-th score included) is among them.
//  3. rescoring from both planes with the reference's sequential unfused arithmetic, selection on the scan's keys.
// The bound (u = 2^-24, g = gamma of the launch >= (d + 2) u / (1 - (d + 2) u); row v = s (b - 128) + e with the sketch's
// scale s, codes b in [1, 255] and |e| <= r):
//  S = the screen's sum of q * b (fused, any order, scaled by a power of two): |S - sum q b| <= 255 g sum|q| + d 2^-p;
//  Q = the sequential sum of q: |Q - sum q| <= g sum|q|; so q.v lies in s [S - 128 Q -+ E1] -+ |q| r with
//  E1 = 383 g sum|q| + d 2^-p.
//  dot:    + the reference's own rounding g |q| |v| + eta, |v| <= (nrm (1 + 2u) + nu) (1 + g), nu = sqrt(d 2^-149);
//  cosine: ref = RN(dot / P) with P = RN(qn * nrm) computed here with the reference's bits; RN(x / P) is monotone in x.
//  L2:     |q|^2 - 2 q.v + |v|^2 with |v|^2 >= ((nrm (1 - 2u))^2 - eta)(1 - g), the reference's within (1 +- g) plus eta.
// Every step rounds outward (RD / RU); a bound that is not finite, or a product |q| |v| past 2^100, makes the row a
// candidate whatever T is.
// ---------------------------------------------------------------------------------------------------------
namespace {

constexpr int SC_VPT = 16;                      // rows per thread: one 16 B load of the sketch
constexpr int SC_TILE = SCAN_THREADS * SC_VPT;  // rows per CTA tile
constexpr int SC_U = 8;                         // sketch loads in flight per thread
constexpr int RS_WARPS = 4;                     // rescoring: warps per CTA, one candidate per warp

struct ScreenArgs {
  PdxSketch sk;
  unsigned long long ld;
  unsigned n, d, ld16, n_tiles, index_base;
  int k;
  const float* query;
  const float* norms;    // the reference's norm of each row
  float gamma, eta, nu;
  uint64_t* partials;
  uint64_t* group_partials;
  unsigned* tickets;
  uint64_t* tkeys;       // out: the k keys of the pessimistic bounds
  float* opt;            // out: optimistic bound of every row
  float* pess;           // out (test hook only, may be null): pessimistic bound of every row
  unsigned* ctl;         // ctl[1] = 1: the query cannot be screened
};

// the query's side of the bound, in shared memory (written by one thread while the others stream)
struct alignas(16) ScreenQuery {
  float qn_ref, qn_up;  // the reference's |q| bits, an upper bound on |q|
  float qq_lo, qq_hi;   // bounds on |q|^2
  float q128;           // 128 Q
  float e1;             // E1
  float gq;             // an upper bound on g |q|
  float unscale;        // 2^(149 - p): the screen's sums are q * b scaled by 2^(p - 149)
  unsigned wmax[SCAN_THREADS / 32];  // per warp: the bits of max |q_j|
};

template <int MODE>
__device__ __forceinline__ void screen_bounds(float acc, float s, float r, float nv, const ScreenQuery& c,
                                              const ScreenArgs& a, float& lower, float& upper) {
  const float g = a.gamma;
  const float v_up = __fmul_ru(__fadd_ru(__fmul_ru(nv, 1.0f + 0x1p-23f), a.nu), __fadd_ru(1.0f, g));
  if (!(__fmul_ru(c.qn_up, v_up) <= 0x1p100f)) {
    lower = -INFINITY;
    upper = INFINITY;
    return;
  }
  const float m_lo = __fsub_rd(__fsub_rd(__fmul_rd(acc, c.unscale), c.q128), c.e1);
  const float m_hi = __fadd_ru(__fsub_ru(__fmul_ru(acc, c.unscale), c.q128), c.e1);
  const float qr = __fmul_ru(c.qn_up, r);
  const float x_lo = __fsub_rd(__fmul_rd(s, m_lo), qr);  // the exact q.v lies in [x_lo, x_hi]
  const float x_hi = __fadd_ru(__fmul_ru(s, m_hi), qr);
  if (MODE == PDX_L2) {
    const float n_lo = __fmul_rd(nv, 1.0f - 0x1p-23f);
    const float vv_lo = fmaxf(0.0f, __fmul_rd(__fsub_rd(__fmul_rd(n_lo, n_lo), a.eta), __fsub_rd(1.0f, g)));
    const float l_lo = fmaxf(0.0f, __fadd_rd(__fsub_rd(c.qq_lo, 2.0f * x_hi), vv_lo));
    const float l_hi = __fadd_ru(__fsub_ru(c.qq_hi, 2.0f * x_lo), __fmul_ru(v_up, v_up));
    lower = fmaxf(0.0f, __fsub_rd(__fmul_rd(l_lo, __fsub_rd(1.0f, g)), a.eta));
    upper = __fadd_ru(__fmul_ru(l_hi, __fadd_ru(1.0f, g)), a.eta);
    if (!(upper <= 3.0e38f)) { lower = -INFINITY; upper = INFINITY; }
    return;
  }
  const float e = __fmaf_ru(c.gq, v_up, a.eta);
  lower = __fsub_rd(x_lo, e);
  upper = __fadd_ru(x_hi, e);
  if (MODE == PDX_COSINE_FUSED) {
    if (!(nv > NORM_EPS)) {  // the reference's score is exactly 0 (src/batch.rs:716-727)
      lower = upper = 0.0f;
      return;
    }
    const float p = __fmul_rn(c.qn_ref, nv);
    lower = __fdiv_rd(lower, p);
    upper = __fdiv_ru(upper, p);
  }
}

// The query is pre-scaled by 2^p so that max |q_j| 2^p lies in [2^126, 2^127), and each code enters as the f32 whose
// bits are the byte (b 2^-149, exact): PRMT + FFMA2 per byte pair, no conversion. The scaled products stay below 2^-14
// and their sums below 2^-2 (d <= 4096), so nothing overflows; an operation whose result falls below 2^-126 errs by at
// most 2^-150 absolutely, d 2^-149 in all, d 2^-p once unscaled. Scaling q up by powers of two is exact; queries with
// max |q_j| outside [2^-100, 2^100] (NaN included) are not screened.
template <int MODE, int R>
__global__ void __launch_bounds__(SCAN_THREADS) pdx_screen_kernel(const ScreenArgs a) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned d_pad = (a.d + 31u) / 32u * 32u;
  float* sq = reinterpret_cast<float*>(smem_raw);  // the query as given
  float* sqs = sq + d_pad;                          // pre-scaled by 2^p
  ScreenQuery* sc = reinterpret_cast<ScreenQuery*>(sqs + d_pad);
  uint64_t* smem_keys = reinterpret_cast<uint64_t*>(sc + 1);
  const int lane = threadIdx.x & 31;
  unsigned mb = 0;
  for (unsigned dd = threadIdx.x; dd < d_pad; dd += blockDim.x) {
    const float x = dd < a.d ? a.query[dd] : 0.0f;
    sq[dd] = x;
    mb = max(mb, __float_as_uint(x) & 0x7FFFFFFFu);
  }
  mb = __reduce_max_sync(FULL_MASK, mb);
  if (lane == 0) sc->wmax[threadIdx.x >> 5] = mb;
  __syncthreads();
#pragma unroll
  for (int w = 0; w < SCAN_THREADS / 32; ++w) mb = max(mb, sc->wmax[w]);
  // a query that cannot be pre-scaled: every CTA sees the same and leaves before taking a ticket
  if (!(mb >= 0x0D800000u && mb <= 0x71800000u)) {  // 2^-100, 2^100
    if (threadIdx.x == 0) a.ctl[1] = 1u;
    return;
  }
  const int p = 253 - (int)(mb >> 23);  // 126 - the exponent of max |q_j|: 26 .. 226
  const float f1 = __uint_as_float((unsigned)(p / 2 + 127) << 23), f2 = __uint_as_float((unsigned)(p - p / 2 + 127) << 23);
  for (unsigned dd = threadIdx.x; dd < d_pad; dd += blockDim.x) sqs[dd] = __fmul_rn(__fmul_rn(sq[dd], f1), f2);
  __syncthreads();
  // the query's d-long chains: the last thread computes them while the others stream (read after the first tile)
  if (threadIdx.x == SCAN_THREADS - 1) {
    float ss = 0.0f, su = 0.0f, sl = 0.0f, qs = 0.0f, sa = 0.0f;
    for (unsigned dd = 0; dd < a.d; ++dd) {
      const float x = sq[dd];
      ss = __fadd_rn(ss, __fmul_rn(x, x));
      su = __fmaf_ru(x, x, su);
      sl = __fmaf_rd(x, x, sl);
      qs = __fadd_rn(qs, x);
      sa = __fadd_ru(sa, fabsf(x));
    }
    const float us = __uint_as_float((unsigned)(276 - p) << 23);
    sc->qn_ref = __fsqrt_rn(ss);
    sc->qn_up = __fsqrt_ru(su);
    sc->qq_lo = sl;
    sc->qq_hi = su;
    sc->q128 = 128.0f * qs;  // exact: |qs| <= sum|q| <= 2^112
    sc->e1 = __fadd_ru(__fmul_ru(a.gamma, __fmul_ru(383.0f, sa)), __fmul_ru(__uint_as_float(a.d), us));  // d 2^-149 us
    sc->gq = __fmul_ru(a.gamma, sc->qn_up);
    sc->unscale = us;
  }
  bool qn_visible = false;
  WarpList<R> lists[1];
  lists[0].init();
  uint64_t thr = KEY_SENTINEL;

  for (unsigned tile = blockIdx.x; tile < a.n_tiles; tile += gridDim.x) {
    const unsigned i0 = tile * SC_TILE + threadIdx.x * SC_VPT;
    const bool active = i0 < a.ld16;
    uint64_t acc[SC_VPT / 2];  // rows (2j, 2j + 1)
#pragma unroll
    for (int j = 0; j < SC_VPT / 2; ++j) acc[j] = 0;
    auto step = [&](const uint4& w, float q) {
      const uint64_t q2 = pack2(q, q);
      const unsigned x[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int t = 0; t < 4; ++t) {
        const float b0 = __uint_as_float(__byte_perm(x[t], 0u, 0x4440u)), b1 = __uint_as_float(__byte_perm(x[t], 0u, 0x4441u));
        const float b2 = __uint_as_float(__byte_perm(x[t], 0u, 0x4442u)), b3 = __uint_as_float(__byte_perm(x[t], 0u, 0x4443u));
        acc[2 * t] = fma2_rn(q2, pack2(b0, b1), acc[2 * t]);
        acc[2 * t + 1] = fma2_rn(q2, pack2(b2, b3), acc[2 * t + 1]);
      }
    };
    if (active) {
      const uint8_t* p = a.sk.codes + pdx_sketch_off(a.ld, 0, i0);
      const size_t next = pdx_sketch_off(a.ld, 1, 0);  // one dimension on
      unsigned dd = 0;
      for (; dd + SC_U <= a.d; dd += SC_U) {
        uint4 w[SC_U];
#pragma unroll
        for (int u = 0; u < SC_U; ++u) w[u] = ldg_stream_u4(reinterpret_cast<const uint4*>(p + u * next));
        p += SC_U * next;
#pragma unroll
        for (int u = 0; u < SC_U; ++u) step(w[u], sqs[dd + u]);
      }
      for (; dd < a.d; ++dd, p += next) step(ldg_stream_u4(reinterpret_cast<const uint4*>(p)), sqs[dd]);
    }
    if (!qn_visible) {  // first tile of this CTA (CTA-uniform)
      __syncthreads();
      qn_visible = true;
      const float qr = sc->qn_ref, qu = sc->qn_up;
      if (!(qu <= 0x1p100f) || (MODE == PDX_COSINE_FUSED && !(qr >= NORM_EPS))) {
        if (threadIdx.x == 0) a.ctl[1] = 1u;
        return;
      }
    }
#pragma unroll
    for (int h = 0; h < SC_VPT / 4; ++h) {
      const unsigned ih = i0 + 4 * h;
      float lo[4] = {0.0f, 0.0f, 0.0f, 0.0f}, up[4] = {0.0f, 0.0f, 0.0f, 0.0f};
      if (active) {
        const float4 s4 = *reinterpret_cast<const float4*>(a.sk.scale + ih);
        const float4 r4 = *reinterpret_cast<const float4*>(a.sk.resid + ih);
        const float4 n4 = *reinterpret_cast<const float4*>(a.norms + ih);
        const float s[4] = {s4.x, s4.y, s4.z, s4.w}, r[4] = {r4.x, r4.y, r4.z, r4.w}, nv[4] = {n4.x, n4.y, n4.z, n4.w};
        float x[4];
        unpack2(acc[2 * h], x[0], x[1]);
        unpack2(acc[2 * h + 1], x[2], x[3]);
#pragma unroll
        for (int j = 0; j < 4; ++j) screen_bounds<MODE>(x[j], s[j], r[j], nv[j], *sc, a, lo[j], up[j]);
        const float* ob = (MODE == PDX_L2) ? lo : up;
        *reinterpret_cast<float4*>(a.opt + ih) = make_float4(ob[0], ob[1], ob[2], ob[3]);
        if (a.pess) {
          const float* pb = (MODE == PDX_L2) ? up : lo;
          for (int j = 0; j < 4; ++j) a.pess[ih + j] = pb[j];
        }
      }
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const unsigned i = ih + j;
        const uint64_t key = (MODE == PDX_L2) ? make_key_asc(up[j], a.index_base + i) : make_key_desc(lo[j], a.index_base + i);
        lists[0].offer(key, active && i < a.n, thr, a.k, lane);
      }
    }
  }
  block_finish<R, 1>(lists, 1, a.k, smem_keys, a.partials, a.group_partials, a.tkeys, a.tickets);
}

// rows whose optimistic bound reaches T (a NaN bound counts as reaching it), in any order: the rescoring selects on keys
__global__ void __launch_bounds__(SCAN_THREADS) screen_compact_kernel(const float* __restrict__ opt, unsigned n, int l2,
                                                                      const uint64_t* __restrict__ tkeys, int k,
                                                                      unsigned index_base, uint32_t* __restrict__ cand,
                                                                      unsigned* ctl) {
  if (ctl[1]) return;
  const uint64_t kth = tkeys[k - 1];
  float t;
  if (kth == KEY_SENTINEL) t = l2 ? INFINITY : -INFINITY;
  else t = __uint_as_float(order_bits_to_f32_bits(l2 ? (uint32_t)(kth >> 32) : ~(uint32_t)(kth >> 32)));
  const int lane = threadIdx.x & 31;
  const unsigned stride = gridDim.x * blockDim.x, n_round = (n + 31u) / 32u * 32u;
  for (unsigned i = blockIdx.x * blockDim.x + threadIdx.x; i < n_round; i += stride) {
    bool hit = false;
    if (i < n) {
      const float b = opt[i];
      hit = l2 ? !(b > t) : !(b < t);
    }
    const unsigned m = __ballot_sync(FULL_MASK, hit);
    if (!m) continue;
    unsigned base = 0;
    if (lane == 0) base = atomicAdd(&ctl[0], (unsigned)__popc(m));
    base = __shfl_sync(FULL_MASK, base, 0);
    const unsigned pos = base + __popc(m & ((1u << lane) - 1u));
    if (hit && pos < SCREEN_CAP) cand[pos] = index_base + i;
  }
}

// One warp per candidate: the 32 lanes gather both planes of the row at once into shared memory, then one lane runs the
// reference's sequential chain (cosine divides by RN(qn * nrm) with the cached norm: the same bits as the fused scan's).
// Writes SCREEN_CAP ready-made keys (KEY_SENTINEL past the candidates); more than SCREEN_CAP candidates raise ctl[1].
template <int MODE>
__global__ void __launch_bounds__(RS_WARPS * 32) screen_rescore_kernel(const PdxView v, const float* __restrict__ query,
                                                                       const float* __restrict__ norms,
                                                                       const uint32_t* __restrict__ cand,
                                                                       unsigned* ctl, uint64_t* __restrict__ keys) {
  extern __shared__ __align__(16) unsigned char smem_raw[];
  const unsigned d = (unsigned)v.d, d_pad = (d + 3u) & ~3u;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  float* sq = reinterpret_cast<float*>(smem_raw) + (size_t)2 * d_pad * warp;  // this warp's query copy, then its row
  float* buf = sq + d_pad;
  const unsigned j = blockIdx.x * RS_WARPS + warp;
  const unsigned cnt = ctl[0], stop = ctl[1];
  if (j == 0 && lane == 0 && cnt > SCREEN_CAP) ctl[1] = 1u;
  if (stop || j >= min(cnt, (unsigned)SCREEN_CAP)) {
    if (lane == 0) keys[j] = KEY_SENTINEL;
    return;
  }
  for (unsigned dd = lane; dd < d; dd += 32) sq[dd] = query[dd];
  const unsigned gid = cand[j], i = gid - v.index_base;
  for (unsigned dd = lane; dd < d; dd += 32) buf[dd] = pdx_load1(v, (size_t)dd * v.ld + i);
  __syncwarp();
  if (lane != 0) return;
  float acc = 0.0f, qss = 0.0f;
  for (unsigned dd = 0; dd < d; ++dd) {
    const float q = sq[dd], x = buf[dd];
    accumulate<MODE == PDX_COSINE_FUSED ? PDX_DOT : MODE>(q, x, acc);
    if (MODE == PDX_COSINE_FUSED) qss = __fadd_rn(qss, __fmul_rn(q, q));
  }
  float sc = acc;
  if (MODE == PDX_COSINE_FUSED) {
    const float qn = __fsqrt_rn(qss), nrm = norms[i];
    sc = (!(qn < NORM_EPS) && nrm > NORM_EPS) ? __fdiv_rn(acc, __fmul_rn(qn, nrm)) : 0.0f;
  }
  keys[j] = MODE == PDX_L2 ? make_key_asc(sc, gid) : make_key_desc(sc, gid);
}

ScreenArgs screen_args(const PdxView& v, const float* dev_norms, const PdxSketch& sk, const float* dev_query, size_t k,
                       Workspace& ws) {
  ScreenArgs a{};
  a.sk = sk;
  a.ld = v.ld;
  a.n = (unsigned)v.n;
  a.d = (unsigned)v.d;
  a.ld16 = (unsigned)std::min<size_t>(v.ld, (v.n + 15) / 16 * 16);
  a.n_tiles = (unsigned)(((size_t)a.ld16 + SC_TILE - 1) / SC_TILE);
  a.index_base = v.index_base;
  a.k = (int)k;
  a.query = dev_query;
  a.norms = dev_norms;
  // gamma_(d+2) = (d + 2) u / (1 - (d + 2) u), u = 2^-24, rounded up to f32 (double has room to spare)
  const double du = (double)(v.d + 2) * 0x1p-24;
  a.gamma = (float)(du / (1.0 - du)) * (1.0f + 0x1p-20f);
  a.eta = (float)((double)v.d * 0x1p-148) * (1.0f + 0x1p-20f) + 0x1p-149f;
  a.nu = (float)std::sqrt((double)v.d * 0x1p-149) * (1.0f + 0x1p-20f);
  a.partials = ws.partials;
  a.group_partials = ws.group_partials;
  a.tickets = ws.tickets;
  a.tkeys = ws.sc_keys + SCREEN_CAP;
  a.opt = ws.sc_bounds;
  a.ctl = ws.sc_ctl;
  return a;
}

template <int MODE, int R>
cudaError_t launch_screen(const ScreenArgs& a, int num_sms, cudaStream_t s) {
  auto kern = pdx_screen_kernel<MODE, R>;
  const size_t smem = (size_t)2 * ((a.d + 31u) / 32u * 32u) * sizeof(float) + sizeof(ScreenQuery) +
                      (size_t)(SCAN_THREADS / 32) * a.k * sizeof(uint64_t);
  static size_t smem_set_dev[16] = {};
  size_t& smem_set = smem_set_dev[current_device_slot()];
  if (smem > 48 * 1024 && smem > smem_set) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    smem_set = smem;
  }
  int occ = 0;
  cudaError_t e = cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, SCAN_THREADS, smem);
  if (e != cudaSuccess) return e;
  if (occ < 1) return cudaErrorInvalidConfiguration;
  kern<<<balanced_grid(a.n_tiles, (unsigned)occ * (unsigned)num_sms), SCAN_THREADS, smem, s>>>(a);
  return cudaGetLastError();
}

cudaError_t launch_screen_mode(int mode, const ScreenArgs& a, int num_sms, cudaStream_t s) {
  const bool big = a.k > 32;
  switch (mode) {
    case PDX_DOT: return big ? launch_screen<PDX_DOT, 4>(a, num_sms, s) : launch_screen<PDX_DOT, 1>(a, num_sms, s);
    case PDX_COSINE_FUSED:
      return big ? launch_screen<PDX_COSINE_FUSED, 4>(a, num_sms, s) : launch_screen<PDX_COSINE_FUSED, 1>(a, num_sms, s);
    case PDX_L2: return big ? launch_screen<PDX_L2, 4>(a, num_sms, s) : launch_screen<PDX_L2, 1>(a, num_sms, s);
  }
  return cudaErrorInvalidValue;
}

}  // namespace

cudaError_t launch_pdx_knn_screened(const PdxView& v, int mode, const float* dev_norms, const PdxSketch& sk,
                                    const float* dev_query, size_t k, uint64_t* dev_keys, Workspace& ws, cudaStream_t s,
                                    LaunchCounter* launches) {
  if (!v.hi || !sk.codes || k == 0 || k > 128 || v.d == 0 || v.d > SCREEN_MAX_D || v.n < k || ws.sc_bounds_cap < v.ld)
    return cudaErrorInvalidValue;
  const ScreenArgs a = screen_args(v, dev_norms, sk, dev_query, k, ws);
  cudaError_t e = cudaMemsetAsync(ws.sc_ctl, 0, 2 * sizeof(unsigned), s);
  if (e != cudaSuccess) return e;
  if ((e = launch_screen_mode(mode, a, ws.num_sms, s)) != cudaSuccess) return e;
  screen_compact_kernel<<<(unsigned)std::min<size_t>((v.n + SCAN_THREADS - 1) / SCAN_THREADS, (size_t)ws.num_sms * 8), SCAN_THREADS, 0, s>>>(
      ws.sc_bounds, (unsigned)v.n, mode == PDX_L2, a.tkeys, (int)k, v.index_base, ws.sc_cand, ws.sc_ctl);
  const size_t rs_smem = (size_t)(2 * RS_WARPS) * ((v.d + 3) & ~(size_t)3) * sizeof(float);
#define INNR_RESCORE(MODE)                                                                                              \
  {                                                                                                                     \
    auto kern = screen_rescore_kernel<MODE>;                                                                            \
    if (rs_smem > 48 * 1024 && (e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)rs_smem)) != cudaSuccess) \
      return e;                                                                                                         \
    kern<<<(unsigned)(SCREEN_CAP / RS_WARPS), RS_WARPS * 32, rs_smem, s>>>(v, dev_query, dev_norms, ws.sc_cand, ws.sc_ctl, ws.sc_keys); \
  }
  if (mode == PDX_DOT) INNR_RESCORE(PDX_DOT)
  else if (mode == PDX_L2) INNR_RESCORE(PDX_L2)
  else INNR_RESCORE(PDX_COSINE_FUSED)
#undef INNR_RESCORE
  *launches += 3;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  if ((e = launch_topk_from_scores(ws.sc_keys, 3, SCREEN_CAP, 0, k, dev_keys, ws, s, launches)) != cudaSuccess) return e;
  // the exact full-read scan, which returns at once unless the screen handed the query over
  return launch_pdx_knn(v, mode, dev_query, 1, k, dev_keys, ws, s, launches, ws.sc_ctl + 1);
}

cudaError_t launch_pdx_screen_debug_bounds(const PdxView& v, int mode, const float* dev_norms, const PdxSketch& sk,
                                           const float* dev_query, float* host_lower, float* host_upper, Workspace& ws,
                                           cudaStream_t s, LaunchCounter* launches) {
  if (!v.hi || !sk.codes || v.n == 0 || v.d == 0 || v.d > SCREEN_MAX_D || 2 * v.ld > ws.sc_bounds_cap)
    return cudaErrorInvalidValue;
  ScreenArgs a = screen_args(v, dev_norms, sk, dev_query, 1, ws);
  a.pess = ws.sc_bounds + v.ld;
  cudaError_t e = cudaMemsetAsync(ws.sc_ctl, 0, 2 * sizeof(unsigned), s);
  if (e != cudaSuccess) return e;
  if ((e = launch_screen_mode(mode, a, ws.num_sms, s)) != cudaSuccess) return e;
  ++*launches;
  unsigned flag[2];
  if ((e = cudaMemcpyAsync(flag, ws.sc_ctl, sizeof(flag), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaStreamSynchronize(s)) != cudaSuccess) return e;
  if (flag[1]) return cudaErrorNotSupported;
  float* lower = mode == PDX_L2 ? a.opt : a.pess;
  float* upper = mode == PDX_L2 ? a.pess : a.opt;
  if ((e = cudaMemcpyAsync(host_lower, lower, v.n * sizeof(float), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  if ((e = cudaMemcpyAsync(host_upper, upper, v.n * sizeof(float), cudaMemcpyDeviceToHost, s)) != cudaSuccess) return e;
  return cudaStreamSynchronize(s);
}

}  // namespace innr
