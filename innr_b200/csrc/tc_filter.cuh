// tc_filter.cuh -- the parts of the exact-result tensor-core filters that do not depend on the corpus encoding, shared by
// the f32 path (knn_tc.cu), the u8 path (u8_tc.cu) and the binary path (bin_tc.cu): the candidate list capacity, the
// prefix schedule of the filter passes and the selection of the next pass's threshold.
//
// A pass over rows [0, n_i) appends (row, lower bound) of every pair whose UPPER bound reaches the query's threshold; the
// k-th largest LOWER bound of the appended pairs is a valid lower bound of the reference's k-th best score and becomes the
// threshold of the next, larger pass. The first pass is dense (every pair kept, slot = row).
#pragma once
#include <algorithm>
#include <cstddef>

#include "common.cuh"

namespace innr {
namespace tcf {
namespace {  // internal linkage: each translation unit that launches the kernel owns its instantiation

constexpr unsigned CAND_CAP = 4096;  // candidate slots per query and pass
constexpr size_t ROW_TILE = 128;     // prefixes are whole 128-row tiles (the UMMA M of both filters)

// carves a call's workspace into 1 KB-aligned arrays
struct WsCursor {
  size_t o = 0;
  size_t take(size_t bytes) {
    const size_t r = o;
    o += (bytes + 1023) / 1024 * 1024;
    return r;
  }
};

// Rows of the dense first pass. For k <= 32, 1024 rows are enough: the k-th best of a 1024-row sample lets about
// rows_next / 1024 * k pairs per query through the next pass, and the selection over 1024 pairs costs a quarter of what it
// cost over 4096 (0.15 ms of the 1024-query f32 call). Larger k keep 4096. first_override > 0 replaces the rule.
inline size_t first_rows(size_t n, size_t k, int first_override) {
  return std::min<size_t>(n, first_override > 0 ? std::min<size_t>((size_t)first_override, CAND_CAP)
                                                : (k <= 32 ? (size_t)1024 : (size_t)CAND_CAP));
}

// Prefix lengths of the passes, the last one n; returns their number (<= 6).
// Prefixes between the dense pass and the whole corpus. Measured at 10M x 768, 1024 f32 queries, k = 10 (whole call, ms;
// `profiles/r02_knn_tc_schedules.log`): n/256, n/32 14.8-15.3 | n/128, n/16 (round 1) 15.6-15.9 | n/32 only 15.0-15.4 |
// n/64 only 15.5 | n/128 only 16.8. Fewer / smaller prefixes cost less themselves but leave a looser threshold: the next
// pass appends more pairs, and every append drags its whole warp through the 32-column slow path (1.7 M pairs: +2.3 ms on
// the final pass).
// sched 0 (default): n/256, n/32 for k <= 32, n/128, n/16 above | 1: n/32 | 2: n/64, n/8 | 3: n/128 | 4: n/64 | 6: n/128, n/16
inline int levels(size_t n, size_t k, size_t first, int sched, size_t out[6]) {
  int n_levels = 0;
  size_t cur = first;
  out[n_levels++] = cur;
  const bool fine = sched == 0 ? k <= 32 : false;
  const size_t mids[2] = {sched == 1 ? 0 : (sched == 2 || sched == 4 ? n / 64 : (fine ? n / 256 : n / 128)),
                          sched == 1 ? n / 32 : (sched == 2 ? n / 8 : (sched == 3 || sched == 4 ? 0 : (fine ? n / 32 : n / 16)))};
  for (size_t nx : mids)
    if (nx >= 4 * cur) {
      cur = (nx + ROW_TILE - 1) / ROW_TILE * ROW_TILE;
      out[n_levels++] = cur;
    }
  // a pass over `next` rows with the threshold of a `cur`-row sample appends about next / cur * k pairs per query:
  // keep that under half of the list (CAND_CAP) with extra prefixes where the standard ones leave a larger step
  // (small corpora, where n/256 and n/32 are below the 4 x rule)
  const size_t g_safe = std::max<size_t>(4, (size_t)(CAND_CAP / 2) / k);
  size_t extra[3];
  int n_extra = 0;
  for (size_t top = n; top / cur > g_safe && n_extra < 3;) {  // from the top down: the extra prefixes stay small
    top = ((top + g_safe - 1) / g_safe + ROW_TILE - 1) / ROW_TILE * ROW_TILE;
    if (top <= cur) break;
    extra[n_extra++] = top;
  }
  while (n_extra > 0 && n_levels < 5) {
    cur = extra[--n_extra];
    out[n_levels++] = cur;
  }
  if (n > cur) out[n_levels++] = n;
  return n_levels;
}

// ---- between passes: threshold of the next pass = k-th largest lower bound among the appended pairs ------------------
// one warp per query; also resets the counter for the next pass. Queries with qflag set keep their threshold (+inf).
template <int R>
__global__ void select_kernel(unsigned nq, unsigned k, const unsigned* __restrict__ qflag, unsigned* __restrict__ cand_count,
                              const float* __restrict__ cand_lb, float* __restrict__ thr) {
  const unsigned q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (q >= nq) return;
  if (qflag[q]) return;  // thr stays +inf
  unsigned cnt = cand_count[q];
  if (cnt > CAND_CAP) cnt = CAND_CAP;  // any k stored pairs give a valid bound
  WarpList<R> list;
  list.init();
  uint64_t t = KEY_SENTINEL;
  for (unsigned c0 = 0; c0 < cnt; c0 += 32) {
    const unsigned c = c0 + lane;
    const bool valid = c < cnt;
    const float lb = valid ? cand_lb[(size_t)q * CAND_CAP + c] : 0.0f;
    list.offer(make_key_desc(lb, c), valid, t, (int)k, lane);
  }
  const uint64_t kth = list.at((int)k - 1);
  if (lane == 0) {
    thr[q] = (kth == KEY_SENTINEL) ? -INFINITY : __uint_as_float(order_bits_to_f32_bits(~(uint32_t)(kth >> 32)));
    cand_count[q] = 0;
  }
}

inline void launch_select(size_t nq, size_t k, const unsigned* qflag, unsigned* cnt, const float* cand_lb, float* thr,
                          cudaStream_t s) {
  if (k <= 32) select_kernel<1><<<(unsigned)((nq + 3) / 4), 128, 0, s>>>((unsigned)nq, (unsigned)k, qflag, cnt, cand_lb, thr);
  else select_kernel<4><<<(unsigned)((nq + 3) / 4), 128, 0, s>>>((unsigned)nq, (unsigned)k, qflag, cnt, cand_lb, thr);
}

// ---- the same step for filters that append exact keys (bin_tc.cu): the next threshold is the k-th smallest stored KEY ---
// An overflowed list still gives a valid threshold: any k stored keys belong to real rows. KEY_SENTINEL when fewer than k
// keys are stored (the next pass then keeps every pair).
template <int R>
__global__ void select_keys_kernel(unsigned nq, unsigned k, unsigned* __restrict__ cand_count,
                                   const uint64_t* __restrict__ cand_key, uint64_t* __restrict__ thr_key) {
  const unsigned q = blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (q >= nq) return;
  unsigned cnt = cand_count[q];
  if (cnt > CAND_CAP) cnt = CAND_CAP;
  WarpList<R> list;
  list.init();
  uint64_t t = KEY_SENTINEL;
  for (unsigned c0 = 0; c0 < cnt; c0 += 32) {
    const unsigned c = c0 + lane;
    const bool valid = c < cnt;
    list.offer(valid ? cand_key[(size_t)q * CAND_CAP + c] : KEY_SENTINEL, valid, t, (int)k, lane);
  }
  const uint64_t kth = list.at((int)k - 1);
  if (lane == 0) {
    thr_key[q] = kth;
    cand_count[q] = 0;
  }
}

inline void launch_select_keys(size_t nq, size_t k, unsigned* cnt, const uint64_t* cand_key, uint64_t* thr_key,
                               cudaStream_t s) {
  if (k <= 32) select_keys_kernel<1><<<(unsigned)((nq + 3) / 4), 128, 0, s>>>((unsigned)nq, (unsigned)k, cnt, cand_key, thr_key);
  else select_keys_kernel<4><<<(unsigned)((nq + 3) / 4), 128, 0, s>>>((unsigned)nq, (unsigned)k, cnt, cand_key, thr_key);
}

}  // namespace
}  // namespace tcf
}  // namespace innr
