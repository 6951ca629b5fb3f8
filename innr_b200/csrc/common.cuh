// common.cuh -- shared device helpers for libinnr_cuda (sm_100a).
//
//  * composite 64-bit selection keys (SURVEY.md 7/H1): (order_bits(score) << 32) | global_index, so that
//    "stable sort, truncate k" (src/batch.rs:756-758, src/scalar.rs:390-391, examples/binary_demo.rs:178)
//    becomes "k smallest distinct keys";
//  * WarpList<R>: a per-warp register-resident sorted list of 32*R keys (the fused top-k tracker that
//    replaces TopK::insert, src/topk.rs:96-121, and the full sorts);
//  * block merge + last-CTA merge so one launch yields the final top-k.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

namespace innr {

// function attributes, events and similar driver state are per device: launchers keep them in [16]-arrays indexed by
// the calling thread's current device (one host process may drive every GPU of the box)
inline int current_device_slot() {
  int d = 0;
  cudaGetDevice(&d);
  return d & 15;
}


constexpr uint64_t KEY_SENTINEL = 0xFFFFFFFFFFFFFFFFull;
constexpr unsigned FULL_MASK = 0xFFFFFFFFu;

// f32::total_cmp order -> unsigned ascending order (Rust core::f32::total_cmp transform, then sign flip)
__device__ __forceinline__ uint32_t f32_order_bits(float x) {
  uint32_t b = __float_as_uint(x);
  b ^= ((uint32_t)((int32_t)b >> 31)) >> 1;
  return b ^ 0x80000000u;
}
__host__ __device__ __forceinline__ uint32_t order_bits_to_f32_bits(uint32_t u) {
  uint32_t o = u ^ 0x80000000u;
  o ^= ((uint32_t)((int32_t)o >> 31)) >> 1;
  return o;
}
// ascending score (L2, Hamming-as-float never used): smaller score first, ties -> lower index
__device__ __forceinline__ uint64_t make_key_asc(float score, uint32_t gidx) {
  return ((uint64_t)f32_order_bits(score) << 32) | gidx;
}
// descending score (dot, cosine, u8): larger score first, ties -> lower index
__device__ __forceinline__ uint64_t make_key_desc(float score, uint32_t gidx) {
  return ((uint64_t)(~f32_order_bits(score)) << 32) | gidx;
}
__device__ __forceinline__ uint64_t make_key_u32(uint32_t dist, uint32_t gidx) {
  return ((uint64_t)dist << 32) | gidx;
}

__device__ __forceinline__ uint64_t shfl_u64(uint64_t v, int src) {
  uint32_t lo = __shfl_sync(FULL_MASK, (uint32_t)v, src);
  uint32_t hi = __shfl_sync(FULL_MASK, (uint32_t)(v >> 32), src);
  return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_xor_u64(uint64_t v, int mask) {
  uint32_t lo = __shfl_xor_sync(FULL_MASK, (uint32_t)v, mask);
  uint32_t hi = __shfl_xor_sync(FULL_MASK, (uint32_t)(v >> 32), mask);
  return ((uint64_t)hi << 32) | lo;
}
__device__ __forceinline__ uint64_t shfl_up_u64(uint64_t v, int delta) {
  uint32_t lo = __shfl_up_sync(FULL_MASK, (uint32_t)v, delta);
  uint32_t hi = __shfl_up_sync(FULL_MASK, (uint32_t)(v >> 32), delta);
  return ((uint64_t)hi << 32) | lo;
}

// streaming 128-bit global load: read-only path, do not allocate in L1 (each corpus byte is used once)
__device__ __forceinline__ float4 ldg_stream_f4(const float* p) {
  float4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.f32 {%0, %1, %2, %3}, [%4];"
               : "=f"(r.x), "=f"(r.y), "=f"(r.z), "=f"(r.w)
               : "l"(p));
  return r;
}
__device__ __forceinline__ uint4 ldg_stream_u4(const uint4* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// ---- packed f32x2 arithmetic (sm_100): two independent IEEE round-to-nearest operations per instruction. Results are
// bit-identical to the scalar __fmul_rn / __fadd_rn / __fsub_rn (no contraction can happen across an asm boundary).
__device__ __forceinline__ uint64_t pack2(float lo, float hi) {
  uint64_t r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(uint64_t v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t mul2_rn(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
// a + b as fma(a, one, b) with `one` = {1.0f, 1.0f} held in a register the compiler cannot see through (a kernel
// argument): a * 1 is exact, so this is exactly the rounded sum -- but unlike add.rn.f32x2 it cannot be contracted
// with a preceding multiply. ptxas fuses mul.rn.f32x2 + add.rn.f32x2 into ONE FFMA2 despite the explicit rounding
// modifiers (seen in the SASS, also with -fmad=false), which would break the reference's unfused mul-then-add.
__device__ __forceinline__ uint64_t add2_unfusable(uint64_t a, uint64_t b, uint64_t one2) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(one2), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t fma2_rn(uint64_t a, uint64_t b, uint64_t c) {
  uint64_t r;
  asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c));
  return r;
}
__device__ __forceinline__ uint64_t add2_rn(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}
__device__ __forceinline__ uint64_t sub2_rn(uint64_t a, uint64_t b) {
  uint64_t r;
  asm("sub.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b));
  return r;
}

// ---- stateless synthetic generators (SURVEY.md 8d); the oracle has the same functions on the CPU ----
__host__ __device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
  x += 0x9E3779B97F4A7C15ull;
  x = (x ^ (x >> 30)) * 0xBF58476D1CE4E5B9ull;
  x = (x ^ (x >> 27)) * 0x94D049BB133111EBull;
  return x ^ (x >> 31);
}
// G-hash: float(u >> 40) * 2^-23 - 1 : 24-bit integer -> exact f32, exact scale, exact subtract
__device__ __forceinline__ float ghash_value(uint64_t salt, uint64_t idx) {
  uint64_t u = splitmix64(salt + idx);
  return __fadd_rn(__fmul_rn(__uint2float_rn((unsigned)(u >> 40)), 1.0f / 8388608.0f), -1.0f);
}
// G-ref: generate_embedding (examples/batch_demo.rs:233-242), bit-identical to the Rust code
__device__ __forceinline__ float gref_value(uint64_t seed, uint64_t j) {
  uint64_t x = seed * 6364136223846793005ull + j * 1442695040888963407ull;
  float f = __uint2float_rn((unsigned)(x >> 33));  // (x >> 33) as f32
  f = __fmul_rn(f, 1.0f / 2147483648.0f);          // / (1u64 << 31) as f32  (exact)
  return __fadd_rn(__fmul_rn(f, 2.0f), -1.0f);     // * 2.0 - 1.0
}

// Sorted ascending list of 32*R keys held in registers: element p = r*32 + lane lives in v[r] of `lane`.
template <int R>
struct WarpList {
  uint64_t v[R];

  __device__ __forceinline__ void init() {
#pragma unroll
    for (int r = 0; r < R; ++r) v[r] = KEY_SENTINEL;
  }
  // element at position p (uniform), broadcast to the warp. The register is picked with uniform branches
  // (a select chain is turned into an indexed local-memory load by the compiler).
  __device__ __forceinline__ uint64_t at(int p) const {
    const int l = p & 31;
    if (R == 1) return shfl_u64(v[0], l);
    uint64_t x;
    switch (p >> 5) {
      case 0: x = shfl_u64(v[0], l); break;
      case 1: x = shfl_u64(v[R > 1 ? 1 : 0], l); break;
      case 2: x = shfl_u64(v[R > 2 ? 2 : 0], l); break;
      default: x = shfl_u64(v[R > 3 ? 3 : 0], l); break;
    }
    return x;
  }
  // insert a warp-uniform key x (distinct from all present keys); the largest element falls off
  __device__ __forceinline__ void insert(uint64_t x, int lane) {
#pragma unroll
    for (int r = R - 1; r >= 0; --r) {
      uint64_t cur = v[r];
      uint64_t up = shfl_up_u64(cur, 1);
      bool prev_lt = true;
      if (r > 0) {
        uint64_t prev_last = shfl_u64(v[r - 1], 31);
        if (lane == 0) up = prev_last;
        prev_lt = up < x;
      } else {
        prev_lt = (lane == 0) ? true : (up < x);
      }
      v[r] = (cur < x) ? cur : (prev_lt ? x : up);
    }
  }
  // bitonic clean-up of a list that holds the 32*R smallest keys as a bitonic sequence: register-level
  // compare-exchange for strides >= 32, shfl_xor for the rest
  __device__ __forceinline__ void bitonic_cleanup(int lane) {
#pragma unroll
    for (int m = R / 2; m >= 1; m >>= 1) {
#pragma unroll
      for (int r = 0; r < R; ++r)
        if ((r & m) == 0) {
          const uint64_t lo = v[r] < v[r + m] ? v[r] : v[r + m];
          const uint64_t hi = v[r] < v[r + m] ? v[r + m] : v[r];
          v[r] = lo;
          v[r + m] = hi;
        }
    }
#pragma unroll
    for (int s = 16; s >= 1; s >>= 1) {
#pragma unroll
      for (int r = 0; r < R; ++r) {
        const uint64_t o = shfl_xor_u64(v[r], s);
        const bool take_max = (lane & s) != 0;
        v[r] = ((v[r] < o) != take_max) ? v[r] : o;
      }
    }
  }
  // insert up to 32 keys at once (one per lane, KEY_SENTINEL = none): sort them across the lanes (bitonic network, 15
  // steps), fold them into the tail of the list (C[p] = min(A[p], B[N-1-p]) keeps the N smallest as a bitonic sequence)
  // and clean up. ~280 instructions whatever the count, against ~60 per key one at a time (R = 4): the early phase of a
  // scan, when most of a ballot still beats the threshold, is where a warp's selection time goes.
  __device__ __forceinline__ void insert_batch(uint64_t x, int lane) {
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        const uint64_t o = shfl_xor_u64(x, stride);
        const bool keep_min = ((lane & stride) == 0) == ((lane & size) == 0);
        x = ((x < o) == keep_min) ? x : o;
      }
    }
    const uint64_t rev = shfl_u64(x, 31 - lane);  // B[N-1-p] for the last register of the list
    v[R - 1] = rev < v[R - 1] ? rev : v[R - 1];
    bitonic_cleanup(lane);
  }
  // offer one candidate per lane; thr = current k-th key (uniform), updated in place. `cap` (uniform) is an outside
  // bound on the k-th key of the WHOLE selection (SharedThreshold below): keys at or above it cannot be in the result.
  __device__ __forceinline__ void offer(uint64_t key, bool valid, uint64_t& thr, int k, int lane, uint64_t cap = KEY_SENTINEL) {
    uint64_t lim = thr < cap ? thr : cap;
    unsigned m = __ballot_sync(FULL_MASK, valid && key < lim);
    if (__popc(m) >= (R == 1 ? 10 : 6)) {  // warp-uniform
      insert_batch((valid && key < lim) ? key : KEY_SENTINEL, lane);
      thr = at(k - 1);
      return;
    }
    while (m) {
      int src = __ffs(m) - 1;
      uint64_t x = shfl_u64(key, src);
      insert(x, lane);
      thr = at(k - 1);
      lim = thr < cap ? thr : cap;
      if (lane == src) valid = false;
      m = __ballot_sync(FULL_MASK, valid && key < lim);
    }
  }
  // Merge a sorted ascending list src[0..len) (len <= 32*R) into this list, keeping the 32*R smallest of the
  // union: C[p] = min(A[p], B[N-1-p]) is bitonic and holds them; a bitonic merge network (strides N/2 .. 1)
  // sorts it. Register-level compare-exchange for strides >= 32, shfl_xor for the rest. ~300 cycles for R=4
  // versus ~150 cycles PER KEY for one-by-one insertion.
  template <bool GLOBAL>
  __device__ __forceinline__ void merge_from(const uint64_t* src, int len, int lane) {
    constexpr int N = 32 * R;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int j = N - 1 - (r * 32 + lane);
      uint64_t b = KEY_SENTINEL;
      if (j < len) b = GLOBAL ? (uint64_t)__ldcg((const unsigned long long*)(src + j)) : src[j];
      v[r] = b < v[r] ? b : v[r];
    }
    bitonic_cleanup(lane);
  }
  // write the first k keys to dst[0..k)
  __device__ __forceinline__ void store(uint64_t* dst, int k, int lane) const {
#pragma unroll
    for (int r = 0; r < R; ++r) {
      int p = r * 32 + lane;
      if (p < k) dst[p] = v[r];
    }
  }
};

// One candidate per lane for each of QB lists at once (the same vector scored against QB queries). When at least half of
// the lists would take the batch path, ALL of them run it in lock step: the QB sorting networks are independent chains of
// shuffles in one basic block, so their latencies overlap instead of adding up (a warp of the 8-query scan spends most
// of a small shard's time here: every ballot still beats the thresholds). Otherwise each list takes its own path.
template <int R, int QB>
__device__ __forceinline__ void offer_multi(WarpList<R> (&lists)[QB], const uint64_t (&key)[QB], bool valid,
                                            uint64_t (&thr)[QB], int nq_valid, int k, int lane) {
  unsigned m[QB];
  int heavy = 0;
#pragma unroll
  for (int q = 0; q < QB; ++q) {
    m[q] = __ballot_sync(FULL_MASK, valid && q < nq_valid && key[q] < thr[q]);
    heavy += __popc(m[q]) >= (R == 1 ? 10 : 6);
  }
  if (heavy * 2 >= QB) {  // warp-uniform
    uint64_t x[QB];
#pragma unroll
    for (int q = 0; q < QB; ++q) x[q] = ((m[q] >> lane) & 1u) ? key[q] : KEY_SENTINEL;
#pragma unroll
    for (int size = 2; size <= 32; size <<= 1) {
#pragma unroll
      for (int stride = size >> 1; stride > 0; stride >>= 1) {
        const bool keep_min = ((lane & stride) == 0) == ((lane & size) == 0);
#pragma unroll
        for (int q = 0; q < QB; ++q) {
          const uint64_t o = shfl_xor_u64(x[q], stride);
          x[q] = ((x[q] < o) == keep_min) ? x[q] : o;
        }
      }
    }
#pragma unroll
    for (int q = 0; q < QB; ++q) {
      const uint64_t rev = shfl_u64(x[q], 31 - lane);
      lists[q].v[R - 1] = rev < lists[q].v[R - 1] ? rev : lists[q].v[R - 1];
    }
    if (R == 1) {  // clean-up of all lists, stage by stage
#pragma unroll
      for (int st = 16; st >= 1; st >>= 1) {
        const bool take_max = (lane & st) != 0;
#pragma unroll
        for (int q = 0; q < QB; ++q) {
          const uint64_t o = shfl_xor_u64(lists[q].v[0], st);
          lists[q].v[0] = ((lists[q].v[0] < o) != take_max) ? lists[q].v[0] : o;
        }
      }
    } else {
#pragma unroll
      for (int q = 0; q < QB; ++q) lists[q].bitonic_cleanup(lane);
    }
#pragma unroll
    for (int q = 0; q < QB; ++q) thr[q] = lists[q].at(k - 1);
    return;
  }
#pragma unroll
  for (int q = 0; q < QB; ++q)
    if (m[q]) lists[q].offer(key[q], valid && q < nq_valid, thr[q], k, lane);
}

// Merge `n_lists` sorted key lists of length k (stride `stride` u64) from `src` into `list` with bitonic merges.
// GLOBAL: src is global memory written by other CTAs of this launch -> read through L2 (ld.global.cg).
template <int R, bool GLOBAL>
__device__ __forceinline__ void warp_merge_lists(WarpList<R>& list, const uint64_t* src, int first, int step,
                                                 int n_lists, size_t stride, int k, int lane) {
  for (int g = first; g < n_lists; g += step) list.template merge_from<GLOBAL>(src + (size_t)g * stride, k, lane);
}

// Tree-merge the lists of all warps of the CTA into warp 0 (log2(warps) rounds through shared memory).
// smem must hold (warps * k) u64. All threads of the CTA must call it.
template <int R>
__device__ __forceinline__ void block_tree_merge(WarpList<R>& list, int k, uint64_t* smem_keys) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  for (int span = 1; span < n_warps; span <<= 1) {
    __syncthreads();  // smem free (previous round / previous user done)
    if ((warp & (2 * span - 1)) == span) list.store(smem_keys + (size_t)warp * k, k, lane);
    __syncthreads();
    if ((warp & (2 * span - 1)) == 0 && warp + span < n_warps)
      list.template merge_from<false>(smem_keys + (size_t)(warp + span) * k, k, lane);
  }
}

// A launch-wide bound on the k-th key, shared by every warp of every CTA of a single-query selection. A warp's own
// k-th key bounds the k-th key of the whole selection from above (the whole set contains that warp's k keys), so the
// minimum over all warps is a valid filter for everybody: a key above it cannot be in the result, and the warp that
// published the bound keeps the k keys that justify it (they only leave its list for smaller ones). Without it every
// warp fills its own list -- k (1 + ln(n_warp / k)) insertions per warp, which at k = 100 is most of a warp's
// instructions on a small shard; with it the whole launch makes about that many insertions in total.
// One 64-bit word per launch in the workspace, KEY_SENTINEL between launches (reset by block_finish's last CTA).
// Every warp of every SM polling one global word would serialise in a single L2 slice (measured: 100 M codes, one
// read per warp and tile = 3 M same-address reads, scan 1.84 -> 2.08 ms), so the traffic is two-level: warps talk to
// two words in SHARED memory (the CTA's view of the bound, the CTA's own best k-th key); one thread per CTA reconciles
// them with the global word every SHARED_THR_PERIOD tiles.
constexpr int SHARED_THR_PERIOD = 4;
struct SharedThreshold {
  unsigned long long* word;   // global, one per launch (null: disabled)
  unsigned long long* s_cap;  // shared: what this CTA last saw (min of global and its own)
  unsigned long long* s_min;  // shared: smallest k-th key any warp of this CTA has reached
  // call by all threads before the CTA's first barrier
  __device__ __forceinline__ void init(unsigned long long* w, unsigned long long* cap, unsigned long long* mn) {
    word = w;
    s_cap = cap;
    s_min = mn;
    if (threadIdx.x == 0) {
      *s_cap = KEY_SENTINEL;
      *s_min = KEY_SENTINEL;
    }
  }
  // once per tile (iteration `it` of the CTA's tile loop), before the tile's loads are consumed
  __device__ __forceinline__ uint64_t read(unsigned it) {
    if (!word) return KEY_SENTINEL;
    if (threadIdx.x == 0 && (it % SHARED_THR_PERIOD) == 0) {
      unsigned long long g;
      asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(g) : "l"(word));
      const unsigned long long mine = *reinterpret_cast<volatile unsigned long long*>(s_min);
      if (mine < g) {
        asm volatile("red.relaxed.gpu.global.min.u64 [%0], %1;" ::"l"(word), "l"(mine) : "memory");
        g = mine;
      }
      *reinterpret_cast<volatile unsigned long long*>(s_cap) = g;
    }
    // the CTA's own best k-th key is visible to its warps at once, the other CTAs' at the next refresh
    const unsigned long long c = *reinterpret_cast<volatile unsigned long long*>(s_cap);
    const unsigned long long m = *reinterpret_cast<volatile unsigned long long*>(s_min);
    return c < m ? c : m;
  }
  // after an offer: this warp's k-th key (uniform), if it undercuts what the CTA knows
  __device__ __forceinline__ void publish(uint64_t thr, uint64_t cap, int lane) {
    if (word && thr < cap && lane == 0) atomicMin(s_min, (unsigned long long)thr);
  }
};

// Ticket counters used by block_finish: tickets[0] = top level, tickets[1 + g] = group g.
constexpr int FINISH_GROUP = 32;  // CTAs per first-level merge group

// Block-level finish shared by all selection kernels (one launch -> final top-k):
//  1. tree-merge the warps' lists -> CTA top-k, written to partials[(blockIdx.x * nq + q) * k ...]
//  2. two-level ticketing: the last CTA of each group of 32 merges the group's lists into group_partials,
//     the last group to finish merges the group lists and writes out_keys[q * k ...] (sorted, sentinel padded).
// Buffers: partials (gridDim * nq * k), group_partials (n_groups * nq * k), tickets (1 + n_groups, zeroed, self-resetting).
template <int R, int QB>
__device__ __forceinline__ void block_finish(WarpList<R> (&lists)[QB], int nq_valid, int k, uint64_t* smem_keys,
                                             uint64_t* partials, uint64_t* group_partials, uint64_t* out_keys,
                                             unsigned* tickets, unsigned long long* shared_thr = nullptr) {
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, n_warps = blockDim.x >> 5;
  __shared__ unsigned s_flag;
  const unsigned n_groups = (gridDim.x + FINISH_GROUP - 1) / FINISH_GROUP;
  const unsigned group = blockIdx.x / FINISH_GROUP;
  const unsigned group_size = min((unsigned)FINISH_GROUP, gridDim.x - group * FINISH_GROUP);
  // Multi-query kernels (QB > 1, QB <= warps): ONE warp per query at every level instead of the whole CTA on one query
  // after the other -- every warp parks its QB lists in shared memory (QB * warps * k keys, sized by the launcher),
  // warp q merges the lists of query q; the group and top levels are merged the same way. A quarter of the
  // synchronisations and no serial loop over queries (what the latency of small launches such as C1 is made of).
  if (QB > 1) {
#pragma unroll
    for (int q = 0; q < QB; ++q)
      if (q < nq_valid) lists[q].store(smem_keys + ((size_t)q * n_warps + warp) * k, k, lane);
    __syncthreads();
    if (warp < nq_valid) {
      WarpList<R> acc;
      acc.init();
      warp_merge_lists<R, false>(acc, smem_keys + (size_t)warp * n_warps * k, 0, 1, n_warps, (size_t)k, k, lane);
      acc.store(partials + ((size_t)blockIdx.x * nq_valid + warp) * k, k, lane);
    }
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_flag = (atomicAdd(&tickets[1 + group], 1u) == group_size - 1) ? 1u : 0u;
    __syncthreads();
    if (!s_flag) return;
    __threadfence();
    if (warp < nq_valid) {  // last CTA of this group
      WarpList<R> acc;
      acc.init();
      warp_merge_lists<R, true>(acc, partials + ((size_t)group * FINISH_GROUP * nq_valid + warp) * k, 0, 1, (int)group_size,
                                (size_t)nq_valid * k, k, lane);
      acc.store((n_groups == 1 ? out_keys + (size_t)warp * k : group_partials + ((size_t)group * nq_valid + warp) * k), k,
                lane);
    }
    if (threadIdx.x == 0) tickets[1 + group] = 0u;  // ready for the next launch
    if (n_groups == 1) return;
    __threadfence();
    __syncthreads();
    if (threadIdx.x == 0) s_flag = (atomicAdd(&tickets[0], 1u) == n_groups - 1) ? 1u : 0u;
    __syncthreads();
    if (!s_flag) return;
    __threadfence();
    if (warp < nq_valid) {  // last group
      WarpList<R> acc;
      acc.init();
      warp_merge_lists<R, true>(acc, group_partials + (size_t)warp * k, 0, 1, (int)n_groups, (size_t)nq_valid * k, k, lane);
      acc.store(out_keys + (size_t)warp * k, k, lane);
    }
    if (threadIdx.x == 0) tickets[0] = 0u;
    return;
  }
#pragma unroll
  for (int q = 0; q < QB; ++q) {
    if (q >= nq_valid) break;
    block_tree_merge<R>(lists[q], k, smem_keys);
    if (warp == 0) lists[q].store(partials + ((size_t)blockIdx.x * nq_valid + q) * k, k, lane);
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_flag = (atomicAdd(&tickets[1 + group], 1u) == group_size - 1) ? 1u : 0u;
  __syncthreads();
  if (!s_flag) return;
  __threadfence();
  // ---- last CTA of this group: merge the group's CTA lists ----
#pragma unroll
  for (int q = 0; q < QB; ++q) {
    if (q >= nq_valid) break;
    WarpList<R> acc;
    acc.init();
    warp_merge_lists<R, true>(acc, partials + ((size_t)group * FINISH_GROUP * nq_valid + q) * k, warp, n_warps,
                              (int)group_size, (size_t)nq_valid * k, k, lane);
    block_tree_merge<R>(acc, k, smem_keys);
    if (warp == 0) acc.store((n_groups == 1 ? out_keys + (size_t)q * k
                                            : group_partials + ((size_t)group * nq_valid + q) * k), k, lane);
  }
  if (threadIdx.x == 0) tickets[1 + group] = 0u;  // ready for the next launch
  if (n_groups == 1) {
    // the last CTA of the launch (every other CTA has left its scan loop): the shared bound is KEY_SENTINEL again
    if (threadIdx.x == 0 && shared_thr) *shared_thr = KEY_SENTINEL;
    return;
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) s_flag = (atomicAdd(&tickets[0], 1u) == n_groups - 1) ? 1u : 0u;
  __syncthreads();
  if (!s_flag) return;
  __threadfence();
  if (threadIdx.x == 0 && shared_thr) *shared_thr = KEY_SENTINEL;
  // ---- last group: merge the group lists ----
#pragma unroll
  for (int q = 0; q < QB; ++q) {
    if (q >= nq_valid) break;
    WarpList<R> acc;
    acc.init();
    warp_merge_lists<R, true>(acc, group_partials + (size_t)q * k, warp, n_warps, (int)n_groups,
                              (size_t)nq_valid * k, k, lane);
    block_tree_merge<R>(acc, k, smem_keys);
    if (warp == 0) acc.store(out_keys + (size_t)q * k, k, lane);
  }
  if (threadIdx.x == 0) tickets[0] = 0u;
}

}  // namespace innr
