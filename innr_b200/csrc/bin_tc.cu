// bin_tc.cu -- top-k of packed binary codes for query batches on the tensor cores (DESIGN.md section 3.11): Hamming,
// binary_dot and binary_jaccard with the keys of the CUDA-core kernels (hamming.cu), bit for bit.
//
// A code's bits, unpacked to bytes in {0, 1}, make the integer product of a code and a query the exact intersection count
// inter = sum_j a_j b_j. With the popcounts pa (row, cached per corpus) and pb (query):
//   Hamming  dist = pa + pb - 2 inter                     key make_key_u32(dist, index), ascending
//   dot      inter                                        key make_key_u32(~inter, index)
//   Jaccard  RN(inter / uni), uni = pa + pb - inter       key make_key_desc(quotient, index) (1.0 when uni == 0)
// No bound and no rescoring: the filter appends the reference's own keys. The passes follow tc_filter.cuh (prefixes of
// the corpus; the first is dense); a pass appends every pair whose KEY is <= the query's threshold key, and the k-th
// smallest stored key becomes the next threshold. Rows past a prefix have larger indices than every row in it, so a tie at
// the threshold's distance never qualifies them: only strictly better rows are appended, and a corpus of exact duplicates
// does not overflow. A query whose final list overflows is flagged on the device and answered by the exact CUDA-core
// scan (launch_binary_flagged_topk) in the same stream: nothing here waits for the host or makes it wait.
//
// Filter kernel: persistent, one CTA per SM, 448 threads: 4 epilogue warps, bulk-copy producer warp, MMA issuer warp,
// two groups of 4 unpack warps (even / odd stages). Work unit = 128 rows x up to 256 queries, query group fastest; one K
// block = one 128-bit chunk of the codes. The producer bulk-copies the chunk of the unit's 128 rows (2 KB,
// codes[c * ld + i] is contiguous along i) into the stage's staging buffer and the query group's block of the operand
// (contiguous, up to 32 KB) into its B block: two copies per K block. Each unpack thread expands one row's 128 bits into
// 8 x 16 {0,1} bytes of the stage's A block, the K-major no-swizzle layout u8_tc.cu reads straight from the u8 corpus
// (8-row x 16-byte core matrices, LBO 2 KB, SBO 128 B). 4 MMAs (M128 N<=256 K32, kind::i8) per K block, two 256-column
// s32 accumulators in TMEM. No unpacked copy of the corpus exists anywhere.
#include <climits>
#include <cstdio>

#include "common.cuh"
#include "kernels.cuh"
#include "tc_common.cuh"
#include "tc_filter.cuh"

namespace innr {

namespace {

using namespace tc;
using tcf::CAND_CAP;

constexpr int BT_THREADS = 448;
constexpr int VT = 128;   // rows per work unit (UMMA M)
constexpr int QT = 256;   // queries per work unit (UMMA N, up to)
constexpr int KC = 8;     // 16-dimension sub-chunks per K block (one 128-bit code chunk)
constexpr int STAGES = 4;
constexpr int A_CHUNK_BYTES = VT * 16;      // 2 KB: 16 unpacked dimensions of a 128-row tile
constexpr int A_BYTES = KC * A_CHUNK_BYTES;  // 16 KB
constexpr int B_BYTES = KC * QT * 16;        // 32 KB: 128 dimensions of a 256-query group
constexpr int BITS_BYTES = VT * 16;          // 2 KB: the packed chunk of the tile
constexpr int STAGE_BYTES = A_BYTES + B_BYTES + BITS_BYTES;
constexpr unsigned MAX_NQ = BIN_TC_CHUNK_QUERIES;  // queries per filter launch: their per-query values stay in shared memory
constexpr unsigned NQ_SLACK = 32;  // per-query arrays run one 32-column load past the last group

struct BtShared {
  uint64_t full[STAGES], ready[STAGES], empty[STAGES], acc_full[2], acc_empty[2];
  alignas(16) uint64_t thr[MAX_NQ + NQ_SLACK];  // threshold key of the pass
  alignas(16) int pre[MAX_NQ + NQ_SLACK];       // pre-test bound (see pre_bound)
  alignas(16) int pb[MAX_NQ + NQ_SLACK];        // query popcount
  uint32_t tmem_base;
};

struct BtArgs {
  const uint8_t* codes;  // chunk-major codes: chunk c of row i at (c * ld + i) * 16
  const uint8_t* qop;    // {0,1} query bytes, per query group g (qt_g queries) one block per K block: see qop_offset
  unsigned long long ld;
  unsigned n_rows, n_qgroups, kblocks, nq_pad, index_base;
  int dense;             // first pass: every pair kept, slot = row, no counters
  const uint32_t* popc;  // pa per row
  const int* qpopc;      // pb per (padded) query
  const uint64_t* thr;   // nq_pad threshold keys
  unsigned* cand_count;
  uint64_t* cand_key;
};

// 4 bits -> 4 bytes in {0, 1}, bit b to byte b (the four shifted copies of n do not overlap: no carries)
__device__ __forceinline__ uint32_t expand4(uint32_t n) { return (n * 0x00204081u) & 0x01010101u; }
// 16 bits -> 16 bytes, bit e to byte e
__device__ __forceinline__ uint4 expand16(uint32_t x) {
  return make_uint4(expand4(x & 0xFu), expand4((x >> 4) & 0xFu), expand4((x >> 8) & 0xFu), expand4((x >> 12) & 0xFu));
}

// 16-byte piece of the query operand: query group g (QT queries each, the last one qt_g), then K block, then 16-dimension
// sub-chunk, then query -- the B block of a (K block, group) is one contiguous run of KC * qt_g * 16 bytes
__host__ __device__ __forceinline__ size_t qop_offset(unsigned g, unsigned qt_g, unsigned kblocks, unsigned sub, unsigned qi) {
  return (size_t)g * QT * kblocks * KC + (size_t)sub * qt_g + qi;
}

template <int OP>
__device__ __forceinline__ uint64_t pair_key(unsigned inter, unsigned pa, unsigned pb, uint32_t gidx) {
  if (OP == 0) return make_key_u32(pa + pb - 2u * inter, gidx);
  if (OP == 1) return make_key_u32(~inter, gidx);
  const unsigned uni = pa + pb - inter;
  return make_key_desc(uni == 0 ? 1.0f : __fdiv_rn(__uint2float_rn(inter), __uint2float_rn(uni)), gidx);
}

// An integer / f32 test that holds for every pair whose key is <= thr (it may hold for others too):
//   Hamming  pa - 2 inter <= pre,  pre = min(thr_dist, 2^30) - pb
//   dot      -inter <= pre,        pre = -min(~thr_hi, 2^30)
//   Jaccard  inter >= RD(uni m),   m = the f32 below the threshold quotient T, pre = its bits. RN(inter / uni) >= T
//            implies inter / uni >= (m + T) / 2 > m, and RD only lowers the product (uni, inter < 2^24 are exact).
// Columns past the last query get a bound no pair meets.
template <int OP>
__device__ __forceinline__ int pre_bound(uint64_t thr, int pb, bool never) {
  const uint32_t hi = (uint32_t)(thr >> 32);
  if (OP == 0) return never ? INT_MIN : (int)min(hi, 1u << 30) - pb;
  if (OP == 1) return never ? INT_MIN : -(int)min(~hi, 1u << 30);
  if (never) return __float_as_int(INFINITY);
  if (thr == KEY_SENTINEL) return __float_as_int(-1.0f);
  const float t = __uint_as_float(order_bits_to_f32_bits(~hi));
  return __float_as_int(nextafterf(t, -INFINITY));
}
template <int OP>
__device__ __forceinline__ bool pre_test(unsigned inter, unsigned pa, int pb, int pre) {
  if (OP == 0) return (int)pa - 2 * (int)inter <= pre;
  if (OP == 1) return -(int)inter <= pre;
  return __uint2float_rn(inter) >= __fmul_rd(__uint2float_rn(pa + (unsigned)pb - inter), __int_as_float(pre));
}

template <int OP>
__global__ void __launch_bounds__(BT_THREADS, 1) bin_tc_filter_kernel(const BtArgs a) {
  extern __shared__ __align__(1024) uint8_t smem[];
  BtShared* st = reinterpret_cast<BtShared*>(smem + STAGES * STAGE_BYTES);
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
      mbar_init(&st->ready[s], 4);
      mbar_init(&st->empty[s], 1);
    }
    for (int b = 0; b < 2; ++b) {
      mbar_init(&st->acc_full[b], 1);
      mbar_init(&st->acc_empty[b], 4);
    }
    fence_barrier_init();
  }
  if (warp == 5) tmem_alloc<512>(&st->tmem_base);
  for (unsigned q = threadIdx.x; q < a.nq_pad + NQ_SLACK; q += blockDim.x) {
    const bool never = q >= a.nq_pad;
    const uint64_t t = never ? 0ull : a.thr[q];
    const int pb = never ? 0 : a.qpopc[q];
    st->thr[q] = t;
    st->pb[q] = pb;
    st->pre[q] = pre_bound<OP>(t, pb, never);
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
        const int s = it % STAGES;
        mbar_wait(&st->empty[s], ((it / STAGES) & 1) ^ 1);
        mbar_arrive_expect_tx(&st->full[s], rows * 16 + KC * qt_u * 16);
        uint8_t* sa = smem + s * STAGE_BYTES;
        uint8_t* sb = sa + A_BYTES;
        uint8_t* sbits = sb + B_BYTES;
        bulk_load(sbits, a.codes + ((unsigned long long)kb * a.ld + row0) * 16, rows * 16, &st->full[s]);
        bulk_load(sb, a.qop + qop_offset(qg, qt_u, a.kblocks, kb * KC, 0) * 16, KC * qt_u * 16, &st->full[s]);
      }
    }
  } else if (warp >= 6) {
    // =========================== unpack: one row's 128 bits per thread, two groups on alternate stages =============
    const unsigned t = (threadIdx.x - 192) % VT;
    for (unsigned it = (warp - 6) / 4; it < n_iters; it += 2) {
      const int s = it % STAGES;
      mbar_wait(&st->full[s], (it / STAGES) & 1);
      uint8_t* sa = smem + s * STAGE_BYTES;
      const uint4 w = reinterpret_cast<const uint4*>(sa + A_BYTES + B_BYTES)[t];
      const uint32_t words[4] = {w.x, w.y, w.z, w.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        *reinterpret_cast<uint4*>(sa + (2 * j) * A_CHUNK_BYTES + t * 16) = expand16(words[j] & 0xFFFFu);
        *reinterpret_cast<uint4*>(sa + (2 * j + 1) * A_CHUNK_BYTES + t * 16) = expand16(words[j] >> 16);
      }
      fence_proxy_async_smem();  // the generic-proxy stores -> visible to the MMA's operand reads
      __syncwarp();
      if (lane == 0) mbar_arrive(&st->ready[s]);
    }
  } else if (warp == 5) {
    // =========================== MMA issuer ===========================
    const uint64_t a_desc0 = make_smem_desc_kmajor_noswizzle(smem_u32(smem), A_CHUNK_BYTES, 128);
    unsigned it = 0;
    for (unsigned ul = 0; ul < n_units; ++ul) {
      const unsigned qg = (u_lo + ul) % a.n_qgroups;
      const unsigned qt_u = min((unsigned)QT, a.nq_pad - qg * QT);
      const uint32_t idesc = make_idesc_u8s8(VT, (int)qt_u);
      const uint32_t b_chunk = qt_u * 16;  // LBO of the group's B block: one 16-dimension sub-chunk of qt_u queries
      const uint64_t b_desc0 = make_smem_desc_kmajor_noswizzle(smem_u32(smem + A_BYTES), b_chunk, 128);
      const uint32_t acc = tmem + (ul & 1) * QT;
      mbar_wait(&st->acc_empty[ul & 1], ((ul >> 1) & 1) ^ 1);
      for (unsigned kb = 0; kb < a.kblocks; ++kb, ++it) {
        const int s = it % STAGES;
        mbar_wait(&st->ready[s], (it / STAGES) & 1);
        tc_fence_after_sync();
        if (elect_one_sync()) {
          const uint64_t ad = desc_advance(a_desc0, (uint32_t)s * STAGE_BYTES);
          const uint64_t bd = desc_advance(b_desc0, (uint32_t)s * STAGE_BYTES);
          if (kb == 0) umma_i8_c<false>(acc, ad, bd, idesc);
          else umma_i8_c<true>(acc, ad, bd, idesc);
#pragma unroll
          for (int ks = 1; ks < KC / 2; ++ks)  // K = 32 bytes = two sub-chunks per MMA
            umma_i8_c<true>(acc, desc_advance(ad, ks * 2 * A_CHUNK_BYTES), desc_advance(bd, ks * 2 * b_chunk), idesc);
          umma_commit(&st->empty[s]);
          if (kb == a.kblocks - 1) umma_commit(&st->acc_full[ul & 1]);
        }
        __syncwarp();
      }
    }
  } else {
    // =========================== epilogue: pre-test, exact key, append ===========================
    auto row_of = [&](unsigned ul) { return (u_lo + ul) / a.n_qgroups * VT + warp * 32 + lane; };
    unsigned pa_next = (n_units && row_of(0) < a.n_rows) ? a.popc[row_of(0)] : 0u;
    for (unsigned ul = 0; ul < n_units; ++ul) {
      const unsigned unit = u_lo + ul;
      const unsigned vt = unit / a.n_qgroups, qg = unit % a.n_qgroups;
      const unsigned qt_u = min((unsigned)QT, a.nq_pad - qg * QT);
      const int ab = ul & 1;
      const unsigned v = vt * VT + warp * 32 + lane;
      const bool vvalid = v < a.n_rows;
      const unsigned pa = pa_next;
      if (ul + 1 < n_units) pa_next = row_of(ul + 1) < a.n_rows ? a.popc[row_of(ul + 1)] : 0u;  // in flight meanwhile
      const uint32_t gidx = a.index_base + v;
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
        const unsigned qc = qg * QT + c0;
        if (a.dense) {  // every pair is kept: its key to slot v of its query, no atomics (the counters are preset)
          if (vvalid) {
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (c0 + j < qt_u)
                a.cand_key[(size_t)(qc + j) * CAND_CAP + v] = pair_key<OP>(r[j], pa, (unsigned)st->pb[qc + j], gidx);
          }
          continue;
        }
        const int4* p4 = reinterpret_cast<const int4*>(&st->pre[qc]);
        const int4* b4 = reinterpret_cast<const int4*>(&st->pb[qc]);
        unsigned pass = 0;
#pragma unroll
        for (int j4 = 0; j4 < 8; ++j4) {
          const int4 t = p4[j4];
          int4 pb = make_int4(0, 0, 0, 0);
          if (OP == 2) pb = b4[j4];
          pass |= (unsigned)pre_test<OP>(r[4 * j4 + 0], pa, pb.x, t.x) << (4 * j4 + 0);
          pass |= (unsigned)pre_test<OP>(r[4 * j4 + 1], pa, pb.y, t.y) << (4 * j4 + 1);
          pass |= (unsigned)pre_test<OP>(r[4 * j4 + 2], pa, pb.z, t.z) << (4 * j4 + 2);
          pass |= (unsigned)pre_test<OP>(r[4 * j4 + 3], pa, pb.w, t.w) << (4 * j4 + 3);
        }
        if (pass && vvalid) {  // rare outside the dense pass: the exact key of every pair that passed
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (!((pass >> j) & 1u)) continue;
            const unsigned q = qc + j;
            const uint64_t key = pair_key<OP>(r[j], pa, (unsigned)st->pb[q], gidx);
            if (key > st->thr[q]) continue;
            const unsigned pos = atomicAdd(&a.cand_count[q], 1u);
            if (pos < CAND_CAP) a.cand_key[(size_t)q * CAND_CAP + pos] = key;
          }
        }
      }
    }
  }

  tc_fence_before_sync();
  __syncthreads();
  if (warp == 5) tmem_dealloc<512>(tmem);
}

// ---- once per corpus: the popcount of every code -------------------------------------------------------------------
__global__ void bin_tc_popc_kernel(const uint4* __restrict__ codes, size_t ld, unsigned n, unsigned chunks,
                                   uint32_t* __restrict__ popc) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
    unsigned p = 0;
    for (unsigned c = 0; c < chunks; ++c) {
      const uint4 w = codes[(size_t)c * ld + i];
      p += __popc(w.x) + __popc(w.y) + __popc(w.z) + __popc(w.w);
    }
    popc[i] = p;
  }
}

// ---- per call: the {0,1} query operand, query popcounts, first-pass thresholds, counters and tickets ----------------
// one thread per 16-byte piece (query q, sub-chunk `sub` = kb * KC + j); the query words are zero padded and masked
__global__ void bin_tc_prep_kernel(const uint64_t* __restrict__ qwords, unsigned nq, unsigned nq_pad, unsigned chunks,
                                   uint8_t* __restrict__ qop, int* __restrict__ qpopc, uint64_t* __restrict__ thr,
                                   unsigned* __restrict__ cand_count, unsigned* __restrict__ tickets,
                                   unsigned first_pass_rows) {
  const size_t total = (size_t)chunks * KC * nq_pad;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const unsigned q = (unsigned)(t % nq_pad);
    const unsigned sub = (unsigned)(t / nq_pad);  // kb * KC + j: dimensions 16 sub .. 16 sub + 15
    uint32_t bits = 0;
    if (q < nq) bits = (uint32_t)(qwords[(size_t)q * 2 * chunks + sub / 4] >> (16 * (sub % 4))) & 0xFFFFu;
    const unsigned g = q / QT;
    reinterpret_cast<uint4*>(qop)[qop_offset(g, min((unsigned)QT, nq_pad - g * QT), chunks, sub, q % QT)] = expand16(bits);
    if (sub == 0) {
      unsigned p = 0;
      if (q < nq)
        for (unsigned w = 0; w < 2 * chunks; ++w) p += __popcll(qwords[(size_t)q * 2 * chunks + w]);
      qpopc[q] = (int)p;
      thr[q] = q < nq ? KEY_SENTINEL : 0ull;  // padding queries: never a candidate after the dense pass
      cand_count[q] = first_pass_rows;        // the dense first pass stores the pair (q, row v) in slot v
      tickets[q] = 0u;
    }
  }
}

// ---- after the final pass: each query's k smallest keys, or its overflow flag (count > CAND_CAP, left for the scan) --
template <int R>
__global__ void bin_tc_final_kernel(unsigned nq, unsigned k, const unsigned* __restrict__ cand_count,
                                    const uint64_t* __restrict__ cand_key, uint64_t* __restrict__ out_keys,
                                    BinTcDevStats* __restrict__ stats) {
  const unsigned q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (q >= nq) return;
  const unsigned cnt = cand_count[q];
  if (cnt > CAND_CAP) {
    if (lane == 0) atomicAdd(&stats->overflowed, 1u);
    return;
  }
  WarpList<R> list;
  list.init();
  uint64_t t = KEY_SENTINEL;
  for (unsigned c0 = 0; c0 < cnt; c0 += 32) {
    const unsigned c = c0 + lane;
    const bool valid = c < cnt;
    list.offer(valid ? cand_key[(size_t)q * CAND_CAP + c] : KEY_SENTINEL, valid, t, (int)k, lane);
  }
  list.store(out_keys + (size_t)q * k, (int)k, lane);
  if (lane == 0) atomicAdd(&stats->candidates, (unsigned long long)cnt);
}

// workspace layout ------------------------------------------------------------------------------------------------------
struct BinTcPlan {
  unsigned nq_pad, kblocks;
  size_t off_qop, off_qpopc, off_thr, off_cnt, off_tickets, off_key, off_partials, total;
};

BinTcPlan make_plan(size_t chunks, size_t nq, size_t k) {
  BinTcPlan p{};
  p.nq_pad = (unsigned)((nq + 15) / 16 * 16);
  p.kblocks = (unsigned)chunks;
  tcf::WsCursor w;
  p.off_qop = w.take((size_t)p.kblocks * KC * p.nq_pad * 16);
  p.off_qpopc = w.take((size_t)p.nq_pad * 4);
  p.off_thr = w.take((size_t)p.nq_pad * 8);
  p.off_cnt = w.take((size_t)p.nq_pad * 4);
  p.off_tickets = w.take((size_t)p.nq_pad * 4);
  p.off_key = w.take((size_t)p.nq_pad * CAND_CAP * 8);
  p.off_partials = w.take((size_t)p.nq_pad * BIN_FLAGGED_CTAS * k * 8);
  p.total = w.o;
  return p;
}

constexpr size_t FILTER_SMEM = (size_t)STAGES * STAGE_BYTES + sizeof(BtShared);
static_assert(FILTER_SMEM <= 227 * 1024, "filter shared memory");

template <int OP>
cudaError_t set_filter_smem() {
  static bool done_dev[16] = {};
  bool& done = done_dev[current_device_slot()];
  if (done) return cudaSuccess;
  cudaError_t e = cudaFuncSetAttribute(bin_tc_filter_kernel<OP>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)FILTER_SMEM);
  if (e == cudaSuccess) done = true;
  return e;
}

template <int OP>
cudaError_t launch_filter(const BtArgs& a, int num_sms, cudaStream_t s) {
  cudaError_t e = set_filter_smem<OP>();
  if (e != cudaSuccess) return e;
  const unsigned long long units = (unsigned long long)((a.n_rows + VT - 1) / VT) * a.n_qgroups;
  unsigned grid = (unsigned)num_sms;
  if (grid > units) grid = (unsigned)units;
  bin_tc_filter_kernel<OP><<<grid, BT_THREADS, FILTER_SMEM, s>>>(a);
  return cudaGetLastError();
}

// one launch sequence for up to MAX_NQ queries: prep, passes, final selection, the flagged queries on the scan
cudaError_t bin_tc_chunk(const BinView& v, int op, const uint32_t* dev_popc, const uint64_t* dev_query_words, size_t nq,
                         size_t k, uint64_t* dev_keys, void* workspace, BinTcDevStats* dev_stats, cudaEvent_t ev_begin,
                         cudaEvent_t ev_end, int num_sms, cudaStream_t s, LaunchCounter* launches, BinTcCall* call) {
  const BinTcPlan p = make_plan(v.chunks, nq, k);
  uint8_t* w = (uint8_t*)workspace;
  uint8_t* qop = w + p.off_qop;
  int* qpopc = (int*)(w + p.off_qpopc);
  uint64_t* thr = (uint64_t*)(w + p.off_thr);
  unsigned* cnt = (unsigned*)(w + p.off_cnt);
  unsigned* tickets = (unsigned*)(w + p.off_tickets);
  uint64_t* cand_key = (uint64_t*)(w + p.off_key);
  uint64_t* partials = (uint64_t*)(w + p.off_partials);
  cudaError_t e;

  // 1. operand, first-pass thresholds, counters preset for the dense pass
  const size_t first_rows = tcf::first_rows(v.n, k, 0);
  const size_t pieces = (size_t)p.kblocks * KC * p.nq_pad;
  unsigned grid = (unsigned)((pieces + 255) / 256);
  if (grid > 148 * 8) grid = 148 * 8;
  bin_tc_prep_kernel<<<grid, 256, 0, s>>>(dev_query_words, (unsigned)nq, p.nq_pad, (unsigned)v.chunks, qop, qpopc, thr, cnt,
                                          tickets, (unsigned)first_rows);
  ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;

  // 2. filter passes over growing prefixes (tc_filter.cuh)
  size_t levels[6];
  const int n_levels = tcf::levels(v.n, k, first_rows, 0, levels);
  BtArgs a{};
  a.codes = (const uint8_t*)v.data;
  a.qop = qop;
  a.ld = v.ld;
  a.n_qgroups = (p.nq_pad + QT - 1) / QT;
  a.kblocks = p.kblocks;
  a.nq_pad = p.nq_pad;
  a.index_base = v.index_base;
  a.popc = dev_popc;
  a.qpopc = qpopc;
  a.thr = thr;
  a.cand_count = cnt;
  a.cand_key = cand_key;
  for (int l = 0; l < n_levels; ++l) {
    const bool last = l == n_levels - 1;
    a.n_rows = (unsigned)levels[l];
    a.dense = l == 0;
    if (last && ev_begin) cudaEventRecord(ev_begin, s);
    e = op == 0 ? launch_filter<0>(a, num_sms, s) : op == 1 ? launch_filter<1>(a, num_sms, s) : launch_filter<2>(a, num_sms, s);
    if (e != cudaSuccess) return e;
    ++*launches;
    if (last) {
      if (ev_end) cudaEventRecord(ev_end, s);
    } else {
      tcf::launch_select_keys(nq, k, cnt, cand_key, thr, s);
      ++*launches;
      if ((e = cudaGetLastError()) != cudaSuccess) return e;
    }
  }
  // 3. the k smallest keys of every list that did not overflow
  if (k <= 32) bin_tc_final_kernel<1><<<(unsigned)((nq + 3) / 4), 128, 0, s>>>((unsigned)nq, (unsigned)k, cnt, cand_key, dev_keys, dev_stats);
  else bin_tc_final_kernel<4><<<(unsigned)((nq + 3) / 4), 128, 0, s>>>((unsigned)nq, (unsigned)k, cnt, cand_key, dev_keys, dev_stats);
  ++*launches;
  if ((e = cudaGetLastError()) != cudaSuccess) return e;
  // 4. the overflowed ones on the exact scan (a launch of fixed shape that does nothing when no list overflowed)
  if ((e = launch_binary_flagged_topk(v, op, dev_query_words, nq, k, cnt, CAND_CAP, partials, tickets, dev_keys, s,
                                      launches)) != cudaSuccess)
    return e;
  call->filter_ops += 2.0 * (double)((v.n + VT - 1) / VT * VT) * (double)(p.kblocks * KC * 16) * (double)p.nq_pad;
  call->passes = n_levels;
  return cudaSuccess;
}

}  // namespace

bool bin_tc_supported(const BinView& v, size_t nq, size_t k) {
  return nq >= 1 && k >= 1 && k <= 128 && k <= v.n && v.n < 0x7FFFFF00ull && v.words >= 1 && v.dim_bits <= BIN_TC_MAX_DIM_BITS;
}

size_t bin_tc_workspace_bytes(size_t chunks, size_t nq, size_t k) { return make_plan(chunks, nq < MAX_NQ ? nq : MAX_NQ, k).total; }

cudaError_t launch_bin_tc_popc(const BinView& v, uint32_t* dev_popc, cudaStream_t s, LaunchCounter* launches) {
  if (v.n == 0) return cudaSuccess;
  unsigned grid = (unsigned)((v.n + 255) / 256);
  if (grid > 148 * 16) grid = 148 * 16;
  bin_tc_popc_kernel<<<grid, 256, 0, s>>>(v.data, v.ld, (unsigned)v.n, (unsigned)v.chunks, dev_popc);
  ++*launches;
  return cudaGetLastError();
}

// ev: [0] call begin, [1] call end, then one (final-pass begin, end) pair per chunk of MAX_NQ queries (null: not timed)
cudaError_t launch_bin_tc(const BinView& v, int op, const uint32_t* dev_popc, const uint64_t* dev_query_words, size_t nq,
                          size_t k, uint64_t* dev_keys, void* workspace, BinTcDevStats* dev_stats, cudaEvent_t* ev, int num_sms,
                          cudaStream_t s, LaunchCounter* launches, BinTcCall* call) {
  if (!bin_tc_supported(v, nq, k) || op < 0 || op > 2) return cudaErrorInvalidValue;
  cudaError_t e;
  if (ev) cudaEventRecord(ev[0], s);
  if ((e = cudaMemsetAsync(dev_stats, 0, sizeof(BinTcDevStats), s)) != cudaSuccess) return e;
  *call = BinTcCall();
  for (size_t q0 = 0, c = 0; q0 < nq; q0 += MAX_NQ, ++c) {  // chunks of MAX_NQ queries, one after the other
    const size_t m = nq - q0 < MAX_NQ ? nq - q0 : MAX_NQ;
    if ((e = bin_tc_chunk(v, op, dev_popc, dev_query_words + q0 * 2 * v.chunks, m, k, dev_keys + q0 * k, workspace, dev_stats,
                          ev ? ev[2 + 2 * c] : nullptr, ev ? ev[3 + 2 * c] : nullptr, num_sms, s, launches, call)) != cudaSuccess)
      return e;
  }
  if (ev) cudaEventRecord(ev[1], s);
  return cudaSuccess;
}

}  // namespace innr
