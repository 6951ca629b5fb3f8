// api.cu -- the C-ABI of libinnr_cuda.so (include/innr_cuda.h): handles, per-device stream + workspace,
// host<->device staging, argument checks that mirror the reference's panics. No torch, no CPU fallback.
#include "../../include/innr_cuda.h"

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <string>
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <functional>
#include <map>
#include <memory>
#include <thread>
#include <vector>

#include "common.cuh"
#include "kernels.cuh"

using namespace innr;

struct innr_cuda_corpus {
  int kind = 0;  // 0 f32 pdx, 1 binary, 2 u8, 3 tokens, 4 ternary
  int device = 0;
  bool owns = true;
  void* dev = nullptr;
  size_t bytes = 0;
  size_t n = 0, d = 0, ld = 0;
  uint64_t index_base = 0;
  // binary
  size_t words = 0, chunks = 0, dim_bits = 0;
  // u8
  float alpha = 1.0f, offset = 0.0f;
  // tokens
  uint64_t* dev_offsets = nullptr;
  size_t total_tokens = 0, uniform_tokens = 0;
  CUtensorMap tmap;
  bool tmap_valid = false;
  // f32 PDX, split layout (pdx.cuh): the low-half plane (the high halves start at `dev`); null for plain corpora
  uint16_t* lo_plane = nullptr;
  // f32 PDX, split corpora: the screened kNN's sidecar (built with the corpus): dev_norms (the reference's norm bits) and
  // the 8-bit sketch (PdxSketch: d * ld code bytes, then ld scales and ld residual bounds; sketch_of); `screen` = norms,
  // scales and bounds finite for every row
  uint8_t* dev_sketch = nullptr;
  bool screen = false;
  // f32 PDX: lazily built operands of the tensor-core filter path (knn_tc.cu): exact norms, f16 unit vectors + TMA map;
  // u8: the row radii of its filter path (u8_tc.cu, dev_radius); binary: the row popcounts of its filter path (bin_tc.cu,
  // dev_popc)
  int tc_state = 0;  // 0 not built, 1 ready, -1 unusable (non-finite norms / no memory): exact scan only
  float* dev_radius = nullptr;
  uint32_t* dev_popc = nullptr;
  float* dev_norms = nullptr;
  void* dev_xh = nullptr;
  CUtensorMap tm_xh;
  // f32 PDX: per-dimension variances and the order batch_knn_reordered walks the rows in, computed on first use (the
  // corpus is immutable, so recomputing them per call as the reference does would give the same values)
  bool var_ready = false;
  std::vector<float> variances;
  uint32_t* dev_order = nullptr;
};

constexpr int MAX_SHARD_DEVICES = 16;
// One asynchronous host-buffer call in flight (innr_cuda_*_async -> innr_cuda_ticket_wait). A device owns two of
// these, one per workspace lane: stream, event and staging buffers live as long as the device context.
struct innr_cuda_ticket {
  int device = -1;
  bool in_flight = false;
  int kind = 0;            // corpus kind of the call: 0 f32, 1 binary, 2 u8
  int metric = 0;
  size_t nq = 0, k = 0, kk = 0;
  cudaStream_t stream = nullptr;
  cudaEvent_t done = nullptr;
  void *d_query = nullptr, *d_keys = nullptr, *h_in = nullptr, *h_out = nullptr;  // h_*: pinned
  size_t d_query_cap = 0, d_keys_cap = 0, h_in_cap = 0, h_out_cap = 0;
  // MaxSim top-k: the slot's own score vectors (a chunk of queries x n_docs), so two calls in flight never share them
  void* d_scores = nullptr;
  size_t d_scores_cap = 0;
  // a sharded call (innr_cuda_*_sharded_async): this is the root's ticket, `siblings` are the other devices' (released
  // with it), the merged keys come out of the exchange launch into d_merged, rows are k wide, and the exchange's status
  // word travels behind the keys
  bool sharded = false;
  size_t krow = 0;
  void* d_merged = nullptr;
  size_t d_merged_cap = 0;
  innr_cuda_ticket* siblings[MAX_SHARD_DEVICES] = {};
  int n_siblings = 0;
  std::atomic<int>* group_busy = nullptr;  // the group's in-flight counter (decremented at the wait)
};

// One rank's end of the peer-mapped key exchange (exchange.cu).
struct innr_cuda_exchange {
  int device = 0, n_ranks = 1, rank = 0;
  size_t slot_keys = 0;
  void* mailbox = nullptr;                 // cudaMalloc'd on `device`
  std::vector<void*> peers;                // every rank's mailbox as mapped here (peers[rank] == mailbox)
  std::vector<char> ipc_opened;            // peers[i] came from cudaIpcOpenMemHandle
  void** dev_peer_table = nullptr;
  unsigned* dev_status = nullptr;
  uint64_t calls = 0;                      // number of the last call made on this rank
  uint64_t timeout_ns = 10ull * 1000 * 1000 * 1000;
  bool connected = false;
};

namespace {

constexpr int MAX_DEVICES = 16;
constexpr size_t MAX_FUSED_K = 128;

struct Buf {  // growable device or pinned-host scratch
  void* p = nullptr;
  size_t cap = 0;
  bool pinned = false;
  cudaError_t reserve(size_t bytes) {
    if (bytes <= cap) return cudaSuccess;
    if (p) {
      if (pinned) cudaFreeHost(p); else cudaFree(p);
      p = nullptr;
      cap = 0;
    }
    size_t want = bytes < 4096 ? 4096 : bytes + bytes / 4;
    cudaError_t e = pinned ? cudaMallocHost(&p, want) : cudaMalloc(&p, want);
    if (e == cudaSuccess) cap = want;
    return e;
  }
  void release() {
    if (p) {
      if (pinned) cudaFreeHost(p); else cudaFree(p);
    }
    p = nullptr;
    cap = 0;
  }
};

struct DeviceCtx {
  bool ready = false;
  int device = -1;
  cudaStream_t stream = nullptr;
  cudaEvent_t ev0 = nullptr, ev1 = nullptr;
  // The workspaces and the scratch buffers below are shared by everything that runs on this device. Host-facing entries
  // run on `stream` and synchronise before they return; `_dev` entries enqueue on the CALLER's stream and return at
  // once, so they leave an event behind (ws_event[lane] on ws_stream[lane]) that the next user of that lane on any
  // other stream waits for. Lane 0 = `ws` + every scratch buffer (all entries may use it); lane 1 = `ws_alt`, used only
  // by the fused k <= 128 scans of `_dev` entries, which need nothing but a Workspace: two independent scans on two
  // caller streams then overlap (the ramp at the end of one launch is filled by the head of the next -- what makes a
  // 1/8-corpus shard scan as fast per byte as a whole-corpus one, DESIGN.md section 6).
  cudaEvent_t ws_event[2] = {nullptr, nullptr};
  cudaStream_t ws_stream[2] = {nullptr, nullptr};
  bool ws_pending[2] = {false, false};
  uint64_t ws_seq[2] = {0, 0};
  uint64_t seq = 0;
  Workspace ws, ws_alt;
  Workspace& lane_ws(int lane) { return lane ? ws_alt : ws; }
  innr_cuda_ticket async_slot[2];  // asynchronous host-buffer calls in flight (at most one per lane)
  unsigned async_next = 0;
  Buf d_query, d_keys, d_scores, d_aux, d_tcws, h_pin, h_counts;
  float last_ms = 0.0f;
  // the binary filter's statistics stay on the device until innr_cuda_bin_tc_last_stats asks (bin_tc.cu: launch_bin_tc)
  BinTcDevStats* bt_stats = nullptr;
  std::vector<cudaEvent_t> bt_ev;
};

struct Options {
  bool knn_tc = true;
  size_t knn_tc_min_n = 100000;
  size_t knn_tc_min_queries = 2;  // measured at 10M x 768: filter call 2.6 ms for 2..64 queries, 8-query scan pass 6.3 ms
  size_t f32_split_min_rows = 1000000;  // owned f32 corpora from this many rows are stored split (DESIGN.md section 2)
  bool maxsim_tc = true;
  bool u8_tc = true;
  // measured at C5 (50M x 384, DESIGN.md section 3.10): k = 10, 8 queries 7.8 ms against 18.8 ms on the pair kernel, 2 queries
  // 7.8 against 4.8. Above k = 32 the candidate lists overflow for most queries (k = 100, 1024 queries: 978 re-run on the
  // scan, slower than the pair kernel), so larger k stay on the scan.
  size_t u8_tc_min_n = 100000;
  size_t u8_tc_min_queries = 8;
  size_t u8_tc_max_k = 32;
  bool bin_tc = true;
  // measured at C4 (100M x 1024 bit, DESIGN.md section 3.11): a filter call costs ~15 ms up to 64 queries; the CUDA-core
  // route takes 12.6 ms for 16 queries and 25.2 ms for 32 at k = 10 (k = 100: 10.4 ms for 8, 20.8 ms for 16), so batches
  // start at 32 queries. Every k <= 128 measured faster from 32 queries on.
  size_t bin_tc_min_n = 100000;
  size_t bin_tc_min_queries = 32;
  size_t bin_tc_max_k = 128;
  bool kernel_timing = false;
} g_opt;

// One mutex per device: calls on different GPUs run concurrently from different host threads (one stream + one
// workspace per device are what a call owns); g_mu guards the process-wide options and statistics only.
std::mutex g_mu;
std::mutex g_dev_mu[MAX_DEVICES];
DeviceCtx g_ctx[MAX_DEVICES];
LaunchCounter g_launches{0};
KnnTcStats g_tc_stats;
KnnTcStats g_u8tc_stats;  // the last u8 filter call (kept apart: knn_tc_last_stats reports f32 calls only)
// the last binary filter call: its device, what the host knew at launch and how many query chunks it had (the rest of its
// statistics is read from the device's bt_stats / bt_ev when asked)
int g_bintc_device = -1;
BinTcCall g_bintc_call;
size_t g_bintc_chunks = 0;
thread_local int t_device = -1;
thread_local std::string t_err;
std::mutex& dev_mu(int d) { return g_dev_mu[(d >= 0 && d < MAX_DEVICES) ? d : 0]; }
// Device of entries that take no corpus: the one this thread bound with innr_cuda_init, else the thread's current CUDA
// device (a host runtime such as torch has usually set it), else 0.
int cur_dev() {
  if (t_device >= 0) return t_device;
  int d = 0;
  if (cudaGetDevice(&d) != cudaSuccess) {
    cudaGetLastError();
    d = 0;
  }
  return (d >= 0 && d < MAX_DEVICES) ? d : 0;
}
// Every entry holds the device's mutex for its duration and leaves the calling thread's current CUDA device as it found
// it (the library switches devices internally; a host runtime's own notion of the current device must not change).
struct EntryGuard {
  std::lock_guard<std::mutex> lk;
  int prev = -1;
  explicit EntryGuard(int device) : lk(dev_mu(device)) {
    if (cudaGetDevice(&prev) != cudaSuccess) {
      cudaGetLastError();
      prev = -1;
    }
  }
  ~EntryGuard() {
    if (prev >= 0) cudaSetDevice(prev);
  }
};

void shard_groups_shutdown();  // defined with the in-process sharding state below

int fail(int code, const std::string& msg) {
  t_err = msg;
  return code;
}
int cuda_fail(cudaError_t e, const char* what) {
  cudaGetLastError();  // clear sticky-less error state
  return fail(e == cudaErrorMemoryAllocation ? INNR_ENOMEM : INNR_ECUDA,
              std::string(what) + ": " + cudaGetErrorString(e));
}
#define CU(call)                                   \
  do {                                             \
    cudaError_t e__ = (call);                      \
    if (e__ != cudaSuccess) return cuda_fail(e__, #call); \
  } while (0)

// per-CTA partial lists: up to 8 CTAs/SM x 8 queries x 32 keys, or 1 query x 128 keys
// (the same buffers hold several query groups of one launch when the grid is small: scan_f32.cu, grid.y)
int alloc_workspace(Workspace& w, int num_sms) {
  w.num_sms = num_sms;
  w.partials_cap = (size_t)num_sms * 8 * 8 * 32 * 4;
  CU(cudaMalloc(&w.partials, w.partials_cap * sizeof(uint64_t)));
  w.group_cap = (size_t)(num_sms * 8 / 32 + 2) * 8 * 128 * 4;
  CU(cudaMalloc(&w.group_partials, w.group_cap * sizeof(uint64_t)));
  w.tickets_cap = 16384;
  CU(cudaMalloc(&w.tickets, w.tickets_cap * sizeof(unsigned)));
  CU(cudaMemset(w.tickets, 0, w.tickets_cap * sizeof(unsigned)));
  CU(cudaMalloc(&w.shared_thr, 64 * sizeof(unsigned long long)));
  CU(cudaMemset(w.shared_thr, 0xFF, 64 * sizeof(unsigned long long)));
  return INNR_OK;
}
void free_workspace(Workspace& w) {
  cudaFree(w.sc_bounds);
  cudaFree(w.sc_cand);
  cudaFree(w.sc_keys);
  cudaFree(w.sc_ctl);
  cudaFree(w.partials);
  cudaFree(w.group_partials);
  cudaFree(w.tickets);
  cudaFree(w.shared_thr);
}

// How an entry uses the device's shared state: WS_HOST = host-facing (lane 0, runs on the context's stream and
// synchronises), WS_DEV = `_dev` entry that may touch the scratch buffers (lane 0, caller's stream), WS_DEV_SCAN = `_dev`
// entry that needs a Workspace and nothing else (either lane), WS_NONE = neither.
enum WsUse { WS_HOST, WS_DEV, WS_DEV_SCAN, WS_NONE };

int ensure_ctx(int device, DeviceCtx** out, WsUse use = WS_HOST, cudaStream_t user = nullptr, int* lane_out = nullptr) {
  if (device < 0 || device >= MAX_DEVICES) return fail(INNR_EINVAL, "device index out of range");
  DeviceCtx& c = g_ctx[device];
  if (!c.ready) {
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0) {
      cudaGetLastError();
      return fail(INNR_ECUDA, "no CUDA device available (libinnr_cuda has no CPU fallback)");
    }
    if (device >= count) return fail(INNR_EINVAL, "device index >= device count");
    CU(cudaSetDevice(device));
    cudaDeviceProp prop;
    CU(cudaGetDeviceProperties(&prop, device));
    c.device = device;
    CU(cudaStreamCreateWithFlags(&c.stream, cudaStreamNonBlocking));
    CU(cudaEventCreate(&c.ev0));
    CU(cudaEventCreate(&c.ev1));
    for (int l = 0; l < 2; ++l) CU(cudaEventCreateWithFlags(&c.ws_event[l], cudaEventDisableTiming));
    int rc = alloc_workspace(c.ws, prop.multiProcessorCount);
    if (rc == INNR_OK) rc = alloc_workspace(c.ws_alt, prop.multiProcessorCount);
    if (rc) return rc;
    c.h_pin.pinned = true;
    c.h_counts.pinned = true;
    c.ready = true;
  } else {
    CU(cudaSetDevice(device));
  }
  // order this call after the last `_dev` call that is still using the same lane on another stream
  int lane = 0;
  if (use == WS_DEV_SCAN) {
    for (int l = 0; l < 2; ++l)
      if (c.ws_pending[l] && cudaEventQuery(c.ws_event[l]) == cudaSuccess) c.ws_pending[l] = false;
    cudaGetLastError();  // cudaErrorNotReady from the queries above is not an error
    if (c.ws_pending[0] && c.ws_stream[0] == user) lane = 0;        // stream order already covers it
    else if (c.ws_pending[1] && c.ws_stream[1] == user) lane = 1;
    else if (!c.ws_pending[0]) lane = 0;
    else if (!c.ws_pending[1]) lane = 1;
    else lane = c.ws_seq[0] <= c.ws_seq[1] ? 0 : 1;                // both busy elsewhere: queue behind the older one
  }
  if (use == WS_HOST) {
    if (c.ws_pending[0]) {
      CU(cudaStreamWaitEvent(c.stream, c.ws_event[0], 0));
      c.ws_pending[0] = false;  // host-facing entries synchronise c.stream before they return
    }
  } else if (use != WS_NONE) {
    if (c.ws_pending[lane] && c.ws_stream[lane] != user) CU(cudaStreamWaitEvent(user, c.ws_event[lane], 0));
  }
  if (lane_out) *lane_out = lane;
  *out = &c;
  return INNR_OK;
}

// `_dev` entries: the work stays in flight on the caller's stream when the entry returns
struct DevRelease {
  DeviceCtx& c;
  cudaStream_t s;
  int lane;
  DevRelease(DeviceCtx& ctx, cudaStream_t stream, int lane_ = 0) : c(ctx), s(stream), lane(lane_) {}
  ~DevRelease() {
    if (cudaEventRecord(c.ws_event[lane], s) == cudaSuccess) {
      c.ws_pending[lane] = true;
      c.ws_stream[lane] = s;
      c.ws_seq[lane] = ++c.seq;
    } else {
      cudaGetLastError();
    }
  }
};

int current_ctx(DeviceCtx** out) { return ensure_ctx(cur_dev(), out); }

int ctx_for(const innr_cuda_corpus* c, DeviceCtx** out) { return ensure_ctx(c->device, out); }
int ctx_for_dev(const innr_cuda_corpus* c, DeviceCtx** out, cudaStream_t user, bool scan_only = false, int* lane = nullptr) {
  return ensure_ctx(c->device, out, scan_only ? WS_DEV_SCAN : WS_DEV, user, lane);
}

size_t round_up(size_t x, size_t m) { return (x + m - 1) / m * m; }

int check_index_range(size_t n, uint64_t index_base) {
  if (index_base + n >= 0xFFFFFFFFull) return fail(INNR_EUNSUPPORTED, "global indices must be < 2^32 - 1");
  return INNR_OK;
}

struct Timed {  // records the device time of the kernels launched in its scope
  DeviceCtx& c;
  // off unless innr_cuda_set_option("kernel_timing", 1): the two timed event records cost a 70 us call 15 us
  bool on;
  explicit Timed(DeviceCtx& ctx) : c(ctx), on(g_opt.kernel_timing) { if (on) cudaEventRecord(c.ev0, c.stream); }
  void stop() { if (on) cudaEventRecord(c.ev1, c.stream); }
  void finish() { if (on) cudaEventElapsedTime(&c.last_ms, c.ev0, c.ev1); }
};

// decode sorted composite keys on the host
void decode_keys_f32(const uint64_t* keys, size_t count, bool descending, uint64_t* out_idx, float* out_score) {
  for (size_t j = 0; j < count; ++j) {
    uint32_t hi = (uint32_t)(keys[j] >> 32);
    if (descending) hi = ~hi;
    uint32_t bits = order_bits_to_f32_bits(hi);
    float f;
    std::memcpy(&f, &bits, 4);
    out_idx[j] = keys[j] & 0xFFFFFFFFull;
    out_score[j] = f;
  }
}

// frees everything a corpus handle owns (the device's mutex is held by the caller)
void destroy_corpus(innr_cuda_corpus* c) {
  if (!c) return;
  cudaSetDevice(c->device);
  if (c->owns && c->dev) cudaFree(c->dev);
  if (c->dev_offsets) cudaFree(c->dev_offsets);
  if (c->dev_norms) cudaFree(c->dev_norms);
  if (c->dev_sketch) cudaFree(c->dev_sketch);
  if (c->dev_xh) cudaFree(c->dev_xh);
  if (c->dev_radius) cudaFree(c->dev_radius);
  if (c->dev_popc) cudaFree(c->dev_popc);
  if (c->dev_order) cudaFree(c->dev_order);
  delete c;
}
// Upload / generate entries: a failure after the handle exists frees it again and hands back NULL (a mid-upload error
// must not strand a multi-GB allocation behind a pointer the caller will never wrap).
struct CorpusGuard {
  innr_cuda_corpus** out;
  bool ok = false;
  explicit CorpusGuard(innr_cuda_corpus** o) : out(o) {}
  ~CorpusGuard() {
    if (!ok && out && *out) {
      destroy_corpus(*out);
      *out = nullptr;
    }
  }
};

int new_corpus(int kind, int device, innr_cuda_corpus** out) {
  *out = new (std::nothrow) innr_cuda_corpus();
  if (!*out) return fail(INNR_ENOMEM, "host allocation failed");
  (*out)->kind = kind;
  (*out)->device = device;
  return INNR_OK;
}

PdxView pdx_view(const innr_cuda_corpus* c) {
  if (c->lo_plane) return PdxView{nullptr, c->n, c->d, c->ld, (uint32_t)c->index_base, (const uint16_t*)c->dev, c->lo_plane};
  return PdxView{(const float*)c->dev, c->n, c->d, c->ld, (uint32_t)c->index_base};
}
PdxDst pdx_dst(innr_cuda_corpus* c) {
  if (c->lo_plane) return PdxDst{nullptr, (uint16_t*)c->dev, c->lo_plane, c->ld};
  return PdxDst{(float*)c->dev, nullptr, nullptr, c->ld};
}
BinView bin_view(const innr_cuda_corpus* c) {
  return BinView{(const uint4*)c->dev, c->n, c->ld, c->words, c->chunks, c->dim_bits, (uint32_t)c->index_base};
}
U8View u8_view(const innr_cuda_corpus* c) {
  return U8View{(const uint4*)c->dev, c->n, c->d, c->ld, c->chunks, c->alpha, c->offset, (uint32_t)c->index_base};
}
TokView tok_view(const innr_cuda_corpus* c) {
  return TokView{(const float*)c->dev, c->dev_offsets, c->n, c->d, c->total_tokens, c->uniform_tokens, c->tmap,
                 c->tmap_valid, c->dev_norms};
}

// Shared tail of every host-facing top-k call: keys device -> pinned -> decode.
template <class Decode>
int fetch_keys(DeviceCtx& ctx, size_t nq, size_t kk, Timed& tm, Decode decode, bool already_on_host = false) {
  CU(ctx.h_pin.reserve(nq * kk * sizeof(uint64_t)));
  if (!already_on_host)
    CU(cudaMemcpyAsync(ctx.h_pin.p, ctx.d_keys.p, nq * kk * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx.stream));
  CU(cudaStreamSynchronize(ctx.stream));
  tm.finish();
  decode((const uint64_t*)ctx.h_pin.p);
  return INNR_OK;
}

}  // namespace

extern "C" {

int innr_cuda_device_count(int* out_count) {
  if (!out_count) return fail(INNR_EINVAL, "null out_count");
  int count = 0;
  cudaError_t e = cudaGetDeviceCount(&count);
  if (e != cudaSuccess) {
    cudaGetLastError();
    count = 0;
  }
  *out_count = count;
  return INNR_OK;
}

int innr_cuda_init(int device) {
  EntryGuard lk(device);
  DeviceCtx* c;
  int rc = ensure_ctx(device, &c);
  if (rc == INNR_OK) t_device = device;
  return rc;
}

int innr_cuda_shutdown(void) {
  shard_groups_shutdown();  // worker threads, mailboxes and staging of the in-process sharded entries
  for (int i = 0; i < MAX_DEVICES; ++i) {
    std::lock_guard<std::mutex> lk(g_dev_mu[i]);
    DeviceCtx& c = g_ctx[i];
    if (!c.ready) continue;
    cudaSetDevice(i);
    cudaStreamSynchronize(c.stream);
    c.d_query.release(); c.d_keys.release(); c.d_scores.release(); c.d_aux.release(); c.d_tcws.release(); c.h_pin.release(); c.h_counts.release();
    free_workspace(c.ws);
    free_workspace(c.ws_alt);
    cudaEventDestroy(c.ev0);
    cudaEventDestroy(c.ev1);
    for (int l = 0; l < 2; ++l) cudaEventDestroy(c.ws_event[l]);
    for (cudaEvent_t e : c.bt_ev) cudaEventDestroy(e);
    if (c.bt_stats) cudaFree(c.bt_stats);
    for (innr_cuda_ticket& t : c.async_slot) {
      if (t.stream) cudaStreamSynchronize(t.stream);
      if (t.d_query) cudaFree(t.d_query);
      if (t.d_keys) cudaFree(t.d_keys);
      if (t.h_in) cudaFreeHost(t.h_in);
      if (t.h_out) cudaFreeHost(t.h_out);
      if (t.d_merged) cudaFree(t.d_merged);
      if (t.d_scores) cudaFree(t.d_scores);
      if (t.done) cudaEventDestroy(t.done);
      if (t.stream) cudaStreamDestroy(t.stream);
    }
    cudaStreamDestroy(c.stream);
    c = DeviceCtx();
  }
  return INNR_OK;
}

const char* innr_cuda_last_error(void) { return t_err.c_str(); }
const char* innr_cuda_backend_name(void) { return "cuda"; }
int innr_cuda_dense_backend(size_t len, int* out_is_cuda) {
  (void)len;
  if (!out_is_cuda) return fail(INNR_EINVAL, "null out");
  *out_is_cuda = 1;
  return INNR_OK;
}
int innr_cuda_set_option(const char* name, double value) {
  if (!name) return fail(INNR_EINVAL, "null option name");
  std::lock_guard<std::mutex> lk(g_mu);
  const std::string n(name);
  if (n == "knn_tc") g_opt.knn_tc = value != 0;
  else if (n == "knn_tc_min_n") g_opt.knn_tc_min_n = (size_t)value;
  else if (n == "knn_tc_min_queries") g_opt.knn_tc_min_queries = (size_t)value;
  else if (n == "f32_split_min_rows") g_opt.f32_split_min_rows = (size_t)value;
  else if (n == "maxsim_tc") g_opt.maxsim_tc = value != 0;
  else if (n == "u8_tc") g_opt.u8_tc = value != 0;
  else if (n == "u8_tc_min_n") g_opt.u8_tc_min_n = (size_t)value;
  else if (n == "u8_tc_min_queries") g_opt.u8_tc_min_queries = (size_t)value;
  else if (n == "u8_tc_max_k") g_opt.u8_tc_max_k = (size_t)value;
  else if (n == "bin_tc") g_opt.bin_tc = value != 0;
  else if (n == "bin_tc_min_n") g_opt.bin_tc_min_n = (size_t)value;
  else if (n == "bin_tc_min_queries") g_opt.bin_tc_min_queries = (size_t)value;
  else if (n == "bin_tc_max_k") g_opt.bin_tc_max_k = (size_t)value;
  else if (n == "kernel_timing") g_opt.kernel_timing = value != 0;
  else if (n == "u8_scaled_chains") u8_set_scaled_chains(value != 0);
  else return fail(INNR_EINVAL, "unknown option: " + n);
  return INNR_OK;
}
int innr_cuda_knn_tc_last_stats(float* out_filter_ms, float* out_total_ms, double* out_filter_flops,
                                uint64_t* out_candidates, uint32_t* out_exact_scan_queries, int* out_passes) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (out_filter_ms) *out_filter_ms = g_tc_stats.filter_ms;
  if (out_total_ms) *out_total_ms = g_tc_stats.total_ms;
  if (out_filter_flops) *out_filter_flops = g_tc_stats.filter_flops;
  if (out_candidates) *out_candidates = g_tc_stats.candidates;
  if (out_exact_scan_queries) *out_exact_scan_queries = g_tc_stats.overflowed;
  if (out_passes) *out_passes = g_tc_stats.passes;
  return INNR_OK;
}
int innr_cuda_u8_tc_last_stats(float* out_filter_ms, float* out_total_ms, double* out_filter_ops,
                               uint64_t* out_candidates, uint32_t* out_exact_scan_queries, int* out_passes) {
  std::lock_guard<std::mutex> lk(g_mu);
  if (out_filter_ms) *out_filter_ms = g_u8tc_stats.filter_ms;
  if (out_total_ms) *out_total_ms = g_u8tc_stats.total_ms;
  if (out_filter_ops) *out_filter_ops = g_u8tc_stats.filter_flops;
  if (out_candidates) *out_candidates = g_u8tc_stats.candidates;
  if (out_exact_scan_queries) *out_exact_scan_queries = g_u8tc_stats.overflowed;
  if (out_passes) *out_passes = g_u8tc_stats.passes;
  return INNR_OK;
}
int innr_cuda_bin_tc_last_stats(float* out_filter_ms, float* out_total_ms, double* out_filter_ops,
                                uint64_t* out_candidates, uint32_t* out_exact_scan_queries, int* out_passes) {
  int device;
  BinTcCall call;
  size_t chunks;
  {
    std::lock_guard<std::mutex> lk(g_mu);
    device = g_bintc_device;
    call = g_bintc_call;
    chunks = g_bintc_chunks;
  }
  float filter_ms = 0.0f, total_ms = 0.0f;
  BinTcDevStats ds{};
  if (device >= 0) {  // waits for that call (and only for it) to finish on the device
    EntryGuard lk(device);
    DeviceCtx& c = g_ctx[device];
    CU(cudaSetDevice(device));
    CU(cudaEventSynchronize(c.bt_ev[1]));
    CU(cudaEventElapsedTime(&total_ms, c.bt_ev[0], c.bt_ev[1]));
    for (size_t i = 0; i < chunks; ++i) {
      float ms = 0.0f;
      CU(cudaEventElapsedTime(&ms, c.bt_ev[2 + 2 * i], c.bt_ev[3 + 2 * i]));
      filter_ms += ms;
    }
    CU(cudaMemcpy(&ds, c.bt_stats, sizeof(ds), cudaMemcpyDeviceToHost));
  }
  if (out_filter_ms) *out_filter_ms = filter_ms;
  if (out_total_ms) *out_total_ms = total_ms;
  if (out_filter_ops) *out_filter_ops = call.filter_ops;
  if (out_candidates) *out_candidates = ds.candidates;
  if (out_exact_scan_queries) *out_exact_scan_queries = ds.overflowed;
  if (out_passes) *out_passes = call.passes;
  return INNR_OK;
}
int innr_cuda_launch_count(uint64_t* out_count) {
  if (!out_count) return fail(INNR_EINVAL, "null out");
  *out_count = g_launches;
  return INNR_OK;
}
int innr_cuda_last_kernel_ms(float* out_ms) {
  if (!out_ms) return fail(INNR_EINVAL, "null out");
  DeviceCtx* c;
  int rc = current_ctx(&c);
  if (rc) return rc;
  *out_ms = c->last_ms;
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ f32 PDX corpus
static int alloc_pdx(DeviceCtx& ctx, size_t n, size_t d, uint64_t index_base, innr_cuda_corpus** out) {
  int rc = check_index_range(n, index_base);
  if (rc) return rc;
  rc = new_corpus(0, ctx.device, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  c->n = n;
  c->d = d;
  c->ld = round_up(n, 64);
  c->index_base = index_base;
  c->bytes = c->ld * d * sizeof(float);
  if (c->bytes) {
    cudaError_t e = cudaMalloc(&c->dev, c->bytes);
    if (e != cudaSuccess) {
      delete c;
      *out = nullptr;
      return cuda_fail(e, "cudaMalloc(corpus)");
    }
    if (n >= g_opt.f32_split_min_rows) c->lo_plane = (uint16_t*)c->dev + c->ld * d;
  }
  guard.ok = true;
  return INNR_OK;
}

static PdxSketch sketch_of(const innr_cuda_corpus* c) {
  float* rows = (float*)(c->dev_sketch + c->d * c->ld);  // d * ld is a multiple of 64: 16 B aligned
  return PdxSketch{c->dev_sketch, rows, rows + c->ld};
}

// After a split corpus is written: its sidecar. The norms pass writes whole float4 groups (up to ld entries), the
// screen reads whole groups of 16: the per-row arrays have ld (+ the tensor-core path's 16 B of scratch) entries.
static int build_sidecar(innr_cuda_corpus* c, DeviceCtx* ctx) {
  if (!c->lo_plane) return INNR_OK;
  CU(cudaMalloc((void**)&c->dev_norms, c->ld * sizeof(float) + 16));
  CU(cudaMalloc((void**)&c->dev_sketch, c->d * c->ld + 2 * c->ld * sizeof(float)));
  const PdxView v = pdx_view(c);
  CU(launch_pdx_scores(v, PDX_NORMS, nullptr, nullptr, c->dev_norms, ctx->ws, ctx->stream, &g_launches));
  CU(ctx->h_counts.reserve(64));
  unsigned* flag = (unsigned*)(c->dev_norms + c->ld);
  CU(launch_pdx_sketch(v, c->dev_norms, sketch_of(c), flag, ctx->stream, &g_launches));
  CU(cudaMemcpyAsync(ctx->h_counts.p, flag, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  c->screen = *(unsigned*)ctx->h_counts.p == 0;
  return INNR_OK;
}

int innr_cuda_upload_f32_pdx(const float* host_pdx, size_t n, size_t d, uint64_t index_base,
                             innr_cuda_corpus** out) {
  if (!out || (!host_pdx && n * d)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_pdx(*ctx, n, d, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes && !c->lo_plane) {
    CU(cudaMemsetAsync(c->dev, 0, c->bytes, ctx->stream));
    CU(cudaMemcpy2DAsync(c->dev, c->ld * sizeof(float), host_pdx, n * sizeof(float), n * sizeof(float), d,
                         cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  } else if (c->bytes) {
    // split: dimension rows in chunks through one 256 MB staging buffer, split into the two planes on the device
    size_t chunk = (size_t)(256u << 20) / (n * sizeof(float));
    if (chunk < 1) chunk = 1;
    if (chunk > d) chunk = d;
    void* stage = nullptr;
    cudaError_t e = cudaMalloc(&stage, chunk * n * sizeof(float));
    for (size_t d0 = 0; d0 < d && e == cudaSuccess; d0 += chunk) {
      const size_t rows = d - d0 < chunk ? d - d0 : chunk;
      e = cudaMemcpyAsync(stage, host_pdx + d0 * n, rows * n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
      if (e == cudaSuccess) e = launch_pdx_rows_to_dst((const float*)stage, rows, n, pdx_dst(c).at_column(d0 * c->ld), ctx->stream, &g_launches);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (stage) cudaFree(stage);
    if (e != cudaSuccess) return cuda_fail(e, "upload_f32_pdx");
  }
  rc = build_sidecar(c, ctx);
  if (rc) return rc;
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_upload_f32_rows(const float* host_rows, size_t n, size_t d, uint64_t index_base,
                              innr_cuda_corpus** out) {
  if (!out || (!host_rows && n * d)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_pdx(*ctx, n, d, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    // ingest in chunks of rows through one 256 MB device staging buffer (stream order keeps copy and transpose of
    // consecutive chunks apart): the device never holds a second copy of the corpus
    size_t chunk = (size_t)(256u << 20) / (d * sizeof(float));
    chunk = chunk / 32 * 32;
    if (chunk < 32) chunk = 32;
    if (chunk > n) chunk = n;
    void* stage = nullptr;
    cudaError_t e = cudaMalloc(&stage, chunk * d * sizeof(float));
    for (size_t i0 = 0; i0 < n && e == cudaSuccess; i0 += chunk) {
      const size_t rows = n - i0 < chunk ? n - i0 : chunk;
      const bool last = i0 + rows == n;
      e = cudaMemcpyAsync(stage, host_rows + i0 * d, rows * d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream);
      if (e == cudaSuccess)
        e = launch_transpose_rows_to_pdx((const float*)stage, rows, d, pdx_dst(c).at_column(i0),
                                         last ? c->ld - i0 : rows, ctx->stream, &g_launches);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    if (stage) cudaFree(stage);
    if (e != cudaSuccess) return cuda_fail(e, "upload_f32_rows");
  }
  rc = build_sidecar(c, ctx);
  if (rc) return rc;
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_wrap_f32_pdx_dev(const float* dev_pdx, size_t n, size_t d, size_t ld, uint64_t index_base,
                               innr_cuda_corpus** out) {
  if (!out) return fail(INNR_EINVAL, "null out");
  if (ld < n || (ld % 4) != 0 || ((uintptr_t)dev_pdx % 16) != 0)
    return fail(INNR_EINVAL, "wrap_f32_pdx_dev: need ld >= n, ld % 4 == 0, 16-byte aligned base");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = check_index_range(n, index_base);
  if (rc) return rc;
  rc = new_corpus(0, ctx->device, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  c->owns = false;
  c->dev = (void*)dev_pdx;
  c->n = n;
  c->d = d;
  c->ld = ld;
  c->index_base = index_base;
  c->bytes = ld * d * sizeof(float);
  guard.ok = true;
  return INNR_OK;
}

// Matryoshka prefix (src/dense.rs:436-462 are the pairwise functions): in the PDX layout the first `prefix_dim`
// dimensions of every vector ARE the first prefix_dim rows, so a truncated corpus is a zero-copy view. Every f32 entry
// works on the view and equals the reference's batch function on VerticalBatch::from_rows of the truncated vectors.
// The view does not own the memory: free it before its parent.
int innr_cuda_prefix_view(const innr_cuda_corpus* c, size_t prefix_dim, innr_cuda_corpus** out) {
  if (!out || !c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  const size_t d = prefix_dim < c->d ? prefix_dim : c->d;  // prefix_len.min(a.len())
  EntryGuard lk(c->device);
  int rc = new_corpus(0, c->device, out);
  if (rc) return rc;
  innr_cuda_corpus* v = *out;
  v->owns = false;
  v->dev = c->dev;
  v->lo_plane = c->lo_plane;  // the parent's planes; its sidecar is for the full d, so the view has none
  v->n = c->n;
  v->d = d;
  v->ld = c->ld;
  v->index_base = c->index_base;
  v->bytes = c->ld * d * sizeof(float);
  return INNR_OK;
}

int innr_cuda_generate_f32_pdx(int generator, uint64_t salt, uint64_t first_row, size_t n, size_t d,
                               uint64_t index_base, innr_cuda_corpus** out) {
  if (!out || (generator != 0 && generator != 1)) return fail(INNR_EINVAL, "bad argument");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_pdx(*ctx, n, d, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    CU(launch_generate_f32_pdx(generator, salt, first_row, n, d, pdx_dst(c), ctx->stream, &g_launches));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  rc = build_sidecar(c, ctx);
  if (rc) return rc;
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_free(innr_cuda_corpus* c) {
  if (!c) return INNR_OK;
  EntryGuard lk(c->device);
  destroy_corpus(c);
  return INNR_OK;
}

int innr_cuda_corpus_info(const innr_cuda_corpus* c, int* kind, size_t* n, size_t* d, size_t* ld,
                          uint64_t* index_base, size_t* device_bytes) {
  if (!c) return fail(INNR_EINVAL, "null corpus");
  if (kind) *kind = c->kind;
  if (n) *n = c->n;
  if (d) *d = c->kind == 1 ? c->dim_bits : c->d;
  if (ld) *ld = c->ld;
  if (index_base) *index_base = c->index_base;
  if (device_bytes) *device_bytes = c->bytes;
  return INNR_OK;
}

int innr_cuda_extract_vector(const innr_cuda_corpus* c, size_t i, float* out_host) {
  if (!c || c->kind != 0 || !out_host) return fail(INNR_EINVAL, "extract_vector: need an f32 corpus");
  if (i >= c->n) return fail(INNR_EINVAL, "extract_vector: index out of bounds");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  if (c->d == 0) return INNR_OK;
  if (c->lo_plane) {  // the two halves of every element, joined here
    std::vector<uint16_t> h(c->d), l(c->d);
    CU(cudaMemcpy2DAsync(h.data(), sizeof(uint16_t), (const uint16_t*)c->dev + i, c->ld * sizeof(uint16_t), sizeof(uint16_t),
                         c->d, cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaMemcpy2DAsync(l.data(), sizeof(uint16_t), c->lo_plane + i, c->ld * sizeof(uint16_t), sizeof(uint16_t), c->d,
                         cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    for (size_t dd = 0; dd < c->d; ++dd) {
      const uint32_t b = ((uint32_t)h[dd] << 16) | l[dd];
      std::memcpy(out_host + dd, &b, sizeof(b));
    }
    return INNR_OK;
  }
  CU(cudaMemcpy2DAsync(out_host, sizeof(float), (const float*)c->dev + i, c->ld * sizeof(float), sizeof(float),
                       c->d, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ full score vectors
static int pdx_scores(const innr_cuda_corpus* c, int mode, const float* query, size_t query_len,
                      const float* norms, size_t norms_len, float* out_host) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  if (mode == PDX_COSINE_NORMS && norms_len != c->n)
    return fail(INNR_EINVAL, "batch_cosine: norms.len() != batch.num_vectors");     // src/batch.rs:711
  if (mode != PDX_NORMS && query_len != c->d)
    return fail(INNR_EINVAL, "query.len() != batch.dimension");                       // src/batch.rs:251,285
  if (c->n == 0) return INNR_OK;
  if (!out_host || (mode != PDX_NORMS && !query && c->d)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(ctx->d_scores.reserve(c->ld * sizeof(float)));
  if (mode != PDX_NORMS && c->d)
    CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if (mode == PDX_COSINE_NORMS) {
    CU(ctx->d_aux.reserve(c->n * sizeof(float)));
    CU(cudaMemcpyAsync(ctx->d_aux.p, norms, c->n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  }
  Timed tm(*ctx);
  CU(launch_pdx_scores(pdx_view(c), mode, (const float*)ctx->d_query.p, (const float*)ctx->d_aux.p,
                       (float*)ctx->d_scores.p, ctx->ws, ctx->stream, &g_launches));
  tm.stop();
  CU(cudaMemcpyAsync(out_host, ctx->d_scores.p, c->n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  tm.finish();
  return INNR_OK;
}

int innr_cuda_batch_dot(const innr_cuda_corpus* c, const float* query, size_t query_len, float* out_host) {
  return pdx_scores(c, PDX_DOT, query, query_len, nullptr, 0, out_host);
}
int innr_cuda_batch_l2_squared(const innr_cuda_corpus* c, const float* query, size_t query_len, float* out_host) {
  return pdx_scores(c, PDX_L2, query, query_len, nullptr, 0, out_host);
}
int innr_cuda_batch_norms(const innr_cuda_corpus* c, float* out_host) {
  return pdx_scores(c, PDX_NORMS, nullptr, 0, nullptr, 0, out_host);
}
int innr_cuda_batch_cosine(const innr_cuda_corpus* c, const float* query, size_t query_len, const float* norms,
                           size_t norms_len, float* out_host) {
  return pdx_scores(c, PDX_COSINE_NORMS, query, query_len, norms, norms_len, out_host);
}

// ------------------------------------------------------------------------------------------ kNN
// Queries on the device -> keys on the device. Large batches of dot / cosine queries go through the tensor-core
// filter (knn_tc.cu: exact results, see there); everything else through the bit-exact scan with fused top-k.
// innr_cuda_set_option("knn_tc", 0) disables the tensor-core path.
// Builds the per-corpus operands of the filter path on first use; on any failure the corpus stays on the exact scan.
static int knn_tc_prepare(innr_cuda_corpus* c, DeviceCtx* ctx, const PdxView& v, cudaStream_t s) {
  if (c->tc_state != 0) return INNR_OK;
  c->tc_state = -1;
  const size_t xh_bytes = c->n * knn_tc_dpad(c->d) * 2;
  const bool have_norms = c->dev_norms != nullptr;  // a split corpus' sidecar: the same bits
  if ((!have_norms && cudaMalloc(&c->dev_norms, c->n * sizeof(float) + 16) != cudaSuccess) ||
      cudaMalloc(&c->dev_xh, xh_bytes) != cudaSuccess) {
    cudaGetLastError();  // out of memory is not an error of the call: exact scan
    if (!have_norms && c->dev_norms) cudaFree(c->dev_norms);
    if (!have_norms) c->dev_norms = nullptr;
    c->dev_xh = nullptr;
    return INNR_OK;
  }
  if (!have_norms) {
    CU(ctx->d_scores.reserve(c->ld * sizeof(float)));
    CU(launch_pdx_scores(v, PDX_NORMS, nullptr, nullptr, (float*)ctx->d_scores.p, ctx->ws, s, &g_launches));
    CU(cudaMemcpyAsync(c->dev_norms, ctx->d_scores.p, c->n * sizeof(float), cudaMemcpyDeviceToDevice, s));
  }
  CU(ctx->h_counts.reserve(64));
  unsigned* nonfinite = (unsigned*)ctx->h_counts.p;
  CU(launch_knn_tc_build(v, c->dev_norms, c->dev_xh, (unsigned*)(c->dev_norms + c->n), &c->tm_xh, nonfinite, s, &g_launches));
  if (*nonfinite == 0) {
    c->tc_state = 1;
  } else {
    cudaFree(c->dev_xh);
    c->dev_xh = nullptr;
  }
  return INNR_OK;
}

// k > 128: one scores pass per query, then rounds of the generic selection over the score vector (scan_f32.cu:
// launch_topk_from_scores). Exact for any k <= N; the corpus is read once per query, the 4 B/vector score array
// once per 128 results.
static int big_k_from_scores(DeviceCtx* ctx, const void* dev_scores, int kind, size_t n, uint64_t index_base, size_t k,
                             uint64_t* dev_keys, cudaStream_t s) {
  CU(launch_topk_from_scores(dev_scores, kind, n, (uint32_t)index_base, k, dev_keys, ctx->ws, s, &g_launches));
  return INNR_OK;
}

// Writes min(k, n) keys per query at row stride `k` (k <= 128: the fused lists are sentinel-initialised, so the rows come
// out sentinel-padded to k by themselves; k > 128: the caller pre-fills dev_keys with sentinels when k > n).
static bool knn_takes_tc_filter(const innr_cuda_corpus* c, const PdxView& v, int mode, size_t nq, size_t k) {
  return g_opt.knn_tc && c->n >= g_opt.knn_tc_min_n && nq >= g_opt.knn_tc_min_queries && knn_tc_supported(v, mode, nq, k);
}
// single queries on a split corpus with a finite sidecar take the screened kNN (scan_f32.cu)
static bool knn_takes_screen(const innr_cuda_corpus* c, size_t nq, size_t k) {
  return nq == 1 && c->screen && k <= MAX_FUSED_K && k <= c->n && c->d <= SCREEN_MAX_D;
}
// its scratch lives in the lane's Workspace (both lanes may run one), sized for `rows` rows (2 x rows for the test hook)
static int ensure_screen_scratch(Workspace& w, size_t rows) {
  if (!w.sc_cand) {
    CU(cudaMalloc((void**)&w.sc_cand, SCREEN_CAP * sizeof(uint32_t)));
    CU(cudaMalloc((void**)&w.sc_keys, (SCREEN_CAP + MAX_FUSED_K) * sizeof(uint64_t)));
    CU(cudaMalloc((void**)&w.sc_ctl, 2 * sizeof(unsigned)));
  }
  if (w.sc_bounds_cap < rows) {
    if (w.sc_bounds) cudaFree(w.sc_bounds);  // waits for the device: a launch in flight may still read it
    w.sc_bounds = nullptr;
    w.sc_bounds_cap = 0;
    CU(cudaMalloc((void**)&w.sc_bounds, rows * sizeof(float)));
    w.sc_bounds_cap = rows;
  }
  return INNR_OK;
}
static int knn_screened(innr_cuda_corpus* c, Workspace& w, int mode, const float* dev_query, size_t k, uint64_t* dev_keys,
                        cudaStream_t s) {
  int rc = ensure_screen_scratch(w, c->ld);
  if (rc) return rc;
  CU(launch_pdx_knn_screened(pdx_view(c), mode, c->dev_norms, sketch_of(c), dev_query, k, dev_keys, w, s, &g_launches));
  return INNR_OK;
}
// the plain fused scan (k <= 128, no tensor-core filter) needs a Workspace and nothing else: either lane will do
// (so does the screened kNN)
static bool knn_is_scan_only(const innr_cuda_corpus* c, int mode, size_t nq, size_t k) {
  return k <= MAX_FUSED_K && !knn_takes_tc_filter(c, pdx_view(c), mode, nq, k);
}
static int knn_keys_dev(innr_cuda_corpus* c, DeviceCtx* ctx, int mode, const float* dev_queries, size_t nq, size_t k,
                        uint64_t* dev_keys, cudaStream_t s, int lane = 0) {
  PdxView v = pdx_view(c);
  if (k > MAX_FUSED_K) {
    const size_t kk = k < c->n ? k : c->n;
    if (kk < k) CU(cudaMemsetAsync(dev_keys, 0xFF, nq * k * sizeof(uint64_t), s));
    CU(ctx->d_scores.reserve(c->ld * sizeof(float)));
    for (size_t q = 0; q < nq; ++q) {
      CU(launch_pdx_scores(v, mode, dev_queries + q * c->d, nullptr, (float*)ctx->d_scores.p, ctx->ws, s, &g_launches));
      int rc = big_k_from_scores(ctx, ctx->d_scores.p, mode == PDX_L2 ? 0 : 1, c->n, c->index_base, kk, dev_keys + q * k, s);
      if (rc) return rc;
    }
    return INNR_OK;
  }
  const bool tc = knn_takes_tc_filter(c, v, mode, nq, k);
  if (tc) {
    int rc = knn_tc_prepare(c, ctx, v, s);
    if (rc) return rc;
  }
  if (tc && c->tc_state == 1) {
    CU(ctx->d_tcws.reserve(knn_tc_workspace_bytes(c->n, c->d, nq, k)));
    CU(ctx->h_counts.reserve(nq * sizeof(unsigned)));
    std::vector<unsigned> overflow;
    KnnTcStats st;
    CU(launch_pdx_knn_tc(v, c->tm_xh, c->dev_norms, mode, dev_queries, nq, k, dev_keys, ctx->d_tcws.p,
                         (unsigned*)ctx->h_counts.p, ctx->ws, s, &g_launches, &overflow, &st));
    {
      std::lock_guard<std::mutex> lg(g_mu);
      g_tc_stats = st;
    }
    for (unsigned q : overflow) {
      if (knn_takes_screen(c, 1, k)) {
        int rc = knn_screened(c, ctx->ws, mode, dev_queries + (size_t)q * c->d, k, dev_keys + (size_t)q * k, s);
        if (rc) return rc;
      } else {
        CU(launch_pdx_knn(v, mode, dev_queries + (size_t)q * c->d, 1, k, dev_keys + (size_t)q * k, ctx->ws, s, &g_launches));
      }
    }
    return INNR_OK;
  }
  if (!tc && knn_takes_screen(c, nq, k)) return knn_screened(c, ctx->lane_ws(lane), mode, dev_queries, k, dev_keys, s);
  CU(launch_pdx_knn(v, mode, dev_queries, nq, k, dev_keys, ctx->lane_ws(tc ? 0 : lane), s, &g_launches));
  return INNR_OK;
}

static int metric_to_mode(int metric, int* mode);

// Test hook for the tensor-core filter's error bound (tests/test_gpu_parity.py::test_knn_tc_bound_*): the lower bounds of
// the dense first pass for rows < min(n, 4096), row-major n_queries x *out_rows, plus eps and the per-query flag
// (1 = the filter does not answer this query: zero / non-finite norm). The corpus needs >= 4096 rows; returns
// INNR_EUNSUPPORTED when the corpus cannot take the filter path (non-finite norms, no memory).
extern "C" int innr_cuda_knn_tc_debug_bounds(const innr_cuda_corpus* c, int metric, const float* queries, size_t n_queries,
                                             size_t query_len, float* out_lower, size_t* out_rows, float* out_eps,
                                             uint32_t* out_qflags) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");
  if (!queries || !out_lower || !out_rows || !out_eps || !out_qflags || n_queries == 0) return fail(INNR_EINVAL, "null argument");
  PdxView v = pdx_view(c);
  if (!knn_tc_supported(v, mode, n_queries, 10)) return fail(INNR_EUNSUPPORTED, "corpus too small for the filter path");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  rc = ctx_for(c, &ctx);
  if (rc) return rc;
  rc = knn_tc_prepare(const_cast<innr_cuda_corpus*>(c), ctx, v, ctx->stream);
  if (rc) return rc;
  if (c->tc_state != 1) return fail(INNR_EUNSUPPORTED, "corpus cannot take the filter path (non-finite norms or no memory)");
  CU(ctx->d_query.reserve((n_queries * c->d + 4) * sizeof(float)));
  CU(ctx->d_tcws.reserve(knn_tc_workspace_bytes(c->n, c->d, n_queries, 10)));
  CU(cudaMemcpyAsync(ctx->d_query.p, queries, n_queries * c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(launch_knn_tc_debug_bounds(v, c->tm_xh, c->dev_norms, mode, (const float*)ctx->d_query.p, n_queries, ctx->d_tcws.p, out_lower,
                                out_rows, out_eps, out_qflags, ctx->ws.num_sms, ctx->stream, &g_launches));
  return INNR_OK;
}

extern "C" int innr_cuda_knn_screen_debug_bounds(const innr_cuda_corpus* c, int metric, const float* query,
                                                 size_t query_len, float* out_lower, float* out_upper) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");
  if (!query || !out_lower || !out_upper) return fail(INNR_EINVAL, "null argument");
  if (!c->screen || c->d > SCREEN_MAX_D || c->n == 0) return fail(INNR_EUNSUPPORTED, "corpus cannot take the screened kNN");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  rc = ctx_for(c, &ctx);
  if (rc) return rc;
  rc = ensure_screen_scratch(ctx->ws, 2 * c->ld);
  if (rc) return rc;
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  cudaError_t e = launch_pdx_screen_debug_bounds(pdx_view(c), mode, c->dev_norms, sketch_of(c), (const float*)ctx->d_query.p,
                                                 out_lower, out_upper, ctx->ws, ctx->stream, &g_launches);
  if (e == cudaErrorNotSupported) return fail(INNR_EUNSUPPORTED, "the query cannot be screened");
  CU(e);
  return INNR_OK;
}

static int metric_to_mode(int metric, int* mode) {
  switch (metric) {
    case INNR_METRIC_DOT: *mode = PDX_DOT; return INNR_OK;
    case INNR_METRIC_COSINE: *mode = PDX_COSINE_FUSED; return INNR_OK;
    case INNR_METRIC_L2: *mode = PDX_L2; return INNR_OK;
  }
  return fail(INNR_EINVAL, "unknown metric");
}

int innr_cuda_batch_knn(const innr_cuda_corpus* c, int metric, const float* queries, size_t n_queries,
                        size_t query_len, size_t k, uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");  // src/batch.rs:386,743,778
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0 || n_queries == 0) return INNR_OK;                           // src/batch.rs:388-393
  if (!out_idx || !out_score || (!queries && c->d)) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < c->n ? k : c->n;                                               // k.min(num_vectors)
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  rc = ctx_for(c, &ctx);
  if (rc) return rc;
  CU(ctx->d_query.reserve((n_queries * c->d + 4) * sizeof(float)));
  CU(ctx->d_keys.reserve(n_queries * kk * sizeof(uint64_t)));
  if (c->d)
    CU(cudaMemcpyAsync(ctx->d_query.p, queries, n_queries * c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  // small results: the finishing CTA stores the keys straight into pinned host memory (mapped under UVA), which saves
  // the device-to-host copy's own launch
  const bool mapped = n_queries * kk * sizeof(uint64_t) <= (64u << 10) && knn_is_scan_only(c, mode, n_queries, kk);
  if (mapped) CU(ctx->h_pin.reserve(n_queries * kk * sizeof(uint64_t)));
  Timed tm(*ctx);
  rc = knn_keys_dev(const_cast<innr_cuda_corpus*>(c), ctx, mode, (const float*)ctx->d_query.p, n_queries, kk,
                    (uint64_t*)(mapped ? ctx->h_pin.p : ctx->d_keys.p), ctx->stream);
  if (rc) return rc;
  tm.stop();
  rc = fetch_keys(*ctx, n_queries, kk, tm, [&](const uint64_t* keys) {
    for (size_t q = 0; q < n_queries; ++q)
      decode_keys_f32(keys + q * kk, kk, metric != INNR_METRIC_L2, out_idx + q * k, out_score + q * k);
  }, mapped);
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// batch_dimension_variance + variance_order (src/batch.rs:572-603) of a resident corpus, cached in the handle.
static int ensure_variance_order(innr_cuda_corpus* c, DeviceCtx* ctx) {
  if (c->var_ready) return INNR_OK;
  std::vector<float> var(c->d, 0.0f);
  if (c->d) {
    CU(ctx->d_aux.reserve(c->d * sizeof(float)));
    CU(launch_dimension_variance(pdx_view(c), (float*)ctx->d_aux.p, ctx->stream, &g_launches));
    CU(cudaMemcpyAsync(var.data(), ctx->d_aux.p, c->d * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
    // order.sort_by(|&a, &b| variances[b].total_cmp(&variances[a])): stable, decreasing under f32::total_cmp
    auto ordered = [](float f) {
      uint32_t b;
      std::memcpy(&b, &f, 4);
      return (int32_t)(b ^ ((uint32_t)((int32_t)b >> 31) >> 1));
    };
    std::vector<uint32_t> order(c->d);
    for (size_t i = 0; i < c->d; ++i) order[i] = (uint32_t)i;
    std::stable_sort(order.begin(), order.end(), [&](uint32_t a, uint32_t b) { return ordered(var[b]) < ordered(var[a]); });
    if (!c->dev_order) CU(cudaMalloc((void**)&c->dev_order, c->d * sizeof(uint32_t)));
    CU(cudaMemcpyAsync(c->dev_order, order.data(), c->d * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  c->variances.swap(var);
  c->var_ready = true;
  return INNR_OK;
}

int innr_cuda_batch_dimension_variance(const innr_cuda_corpus* c, float* out, size_t out_len) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  if (out_len != c->d) return fail(INNR_EINVAL, "out_len != batch.dimension");
  if (c->d == 0) return INNR_OK;
  if (!out) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  rc = ensure_variance_order(const_cast<innr_cuda_corpus*>(c), ctx);
  if (rc) return rc;
  std::memcpy(out, c->variances.data(), c->d * sizeof(float));
  return INNR_OK;
}

int innr_cuda_batch_knn_reordered(const innr_cuda_corpus* c, const float* query, size_t query_len, size_t k,
                                  uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");  // src/batch.rs:622
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0) return INNR_OK;                                             // src/batch.rs:624-629
  if (!out_idx || !out_score || (!query && c->d)) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < c->n ? k : c->n;
  if (c->d == 0) {  // no row is ever added: every distance is 0.0 and the stable sort keeps index order
    for (size_t j = 0; j < kk; ++j) { out_idx[j] = c->index_base + j; out_score[j] = 0.0f; }
    if (out_count) *out_count = kk;
    return INNR_OK;
  }
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  rc = ensure_variance_order(const_cast<innr_cuda_corpus*>(c), ctx);
  if (rc) return rc;
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(ctx->d_keys.reserve(kk * sizeof(uint64_t)));
  CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  const PdxView v = pdx_view(c);
  if (kk <= MAX_FUSED_K) {
    CU(launch_pdx_knn_reordered(v, (const float*)ctx->d_query.p, c->dev_order, kk, (uint64_t*)ctx->d_keys.p, ctx->ws,
                                ctx->stream, &g_launches));
  } else {
    CU(ctx->d_scores.reserve(c->ld * sizeof(float)));
    CU(launch_pdx_scores(v, PDX_L2_PERM, (const float*)ctx->d_query.p, nullptr, (float*)ctx->d_scores.p, ctx->ws, ctx->stream,
                         &g_launches, 0.0f, c->dev_order));
    rc = big_k_from_scores(ctx, ctx->d_scores.p, 0, c->n, c->index_base, kk, (uint64_t*)ctx->d_keys.p, ctx->stream);
    if (rc) return rc;
  }
  tm.stop();
  rc = fetch_keys(*ctx, 1, kk, tm, [&](const uint64_t* keys) { decode_keys_f32(keys, kk, false, out_idx, out_score); });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// batch_knn_adaptive (src/batch.rs:441-564): the reference's approximate early-termination kNN, reproduced exactly --
// same candidate set, same distances (the sequential sum over all dimensions), same order. One pass per threshold
// epoch (scan_f32.cu); the host only reads one counter per epoch to apply the reference's `alive_count > k` guard.
int innr_cuda_batch_knn_adaptive(const innr_cuda_corpus* c, const float* query, size_t query_len, size_t k,
                                 size_t warmup_dims, uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");  // src/batch.rs:447
  if (warmup_dims == 0) return fail(INNR_EINVAL, "warmup_dims must be > 0");           // :448
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0) return INNR_OK;                                             // :450-455
  if (!out_idx || !out_score || (!query && c->d)) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < c->n ? k : c->n;
  if (c->d == 0) {                                                                      // :458-463
    for (size_t j = 0; j < kk; ++j) { out_idx[j] = c->index_base + j; out_score[j] = 0.0f; }
    if (out_count) *out_count = kk;
    return INNR_OK;
  }
  const size_t w = warmup_dims < c->d ? warmup_dims : c->d;
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  cudaStream_t s = ctx->stream;
  const size_t words = c->ld / 32 + 2;
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(ctx->d_scores.reserve(c->ld * sizeof(float)));
  CU(ctx->d_keys.reserve(2 * kk * sizeof(uint64_t)));
  CU(ctx->d_aux.reserve((2 * words + 8 + c->ld) * sizeof(uint32_t)));
  CU(ctx->h_counts.reserve(64));
  uint32_t* mask_a = (uint32_t*)ctx->d_aux.p;
  uint32_t* mask_b = mask_a + words;
  float* thr = (float*)(mask_b + words);
  unsigned* pruned = (unsigned*)(thr + 4);
  uint32_t* ev = (uint32_t*)(thr + 8);
  float* dist = (float*)ctx->d_scores.p;
  uint64_t* keys = (uint64_t*)ctx->d_keys.p;
  const float* dq = (const float*)ctx->d_query.p;
  unsigned* h_pruned = (unsigned*)ctx->h_counts.p;
  CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, s));
  Timed tm(*ctx);
  const PdxView v = pdx_view(c);
  auto read_pruned = [&](size_t* out) -> int {
    CU(cudaMemcpyAsync(h_pruned, pruned, sizeof(unsigned), cudaMemcpyDeviceToHost, s));
    CU(cudaStreamSynchronize(s));
    *out = *h_pruned;
    return INNR_OK;
  };
  // warm-up: the first w dimensions of every vector (a prefix of the same sequential sum)
  PdxView vw = v;
  vw.d = w;
  CU(launch_pdx_scores(vw, PDX_L2, dq, nullptr, dist, ctx->ws, s, &g_launches));
  CU(launch_topk_from_scores(dist, 0, c->n, 0, kk, keys, ctx->ws, s, &g_launches));
  const float ratio = (float)c->d / (float)w;                                           // :486
  CU(launch_adaptive_threshold(keys + kk - 1, ratio, thr, s, &g_launches));
  CU(cudaMemsetAsync(pruned, 0, sizeof(unsigned), s));
  CU(launch_adaptive_mark(v, dist, ratio, thr, mask_a, pruned, s, &g_launches));
  size_t alive = c->n, p = 0;
  rc = read_pruned(&p);
  if (rc) return rc;
  alive -= p;  // the k smallest estimates never exceed 1.5 x the k-th: at least k candidates stay
  for (size_t d0 = w; d0 < c->d;) {
    size_t last = (d0 + 31) / 32 * 32;  // the next dimension after which the reference refreshes the threshold
    if (last >= c->d) last = c->d - 1;
    const size_t d1 = last + 1;
    const int no_prune = alive <= kk;
    CU(cudaMemsetAsync(pruned, 0, sizeof(unsigned), s));
    CU(launch_adaptive_epoch(v, dq, d0, d1, dist, mask_a, mask_b, thr, ev, pruned, no_prune, s, &g_launches));
    if (!no_prune) {
      rc = read_pruned(&p);
      if (rc) return rc;
      if (alive - p < kk) {
        // The reference stops pruning when k candidates are left, and it meets the candidates in (dimension, index)
        // order: of the p that exceeded the threshold in this epoch only the first alive - k die; the last
        // k - (alive - p) of them in that order stay for good.
        const size_t m = kk - (alive - p);
        CU(ctx->d_tcws.reserve(c->n * sizeof(uint64_t)));
        CU(launch_adaptive_event_keys(mask_a, mask_b, ev, c->n, (uint64_t*)ctx->d_tcws.p, s, &g_launches));
        CU(launch_topk_from_scores(ctx->d_tcws.p, 3, c->n, 0, m, keys + kk, ctx->ws, s, &g_launches, nullptr, nullptr,
                                   (unsigned)c->n, (unsigned)c->n));
        CU(launch_adaptive_revive(keys + kk, m, mask_b, s, &g_launches));
        alive = kk;
      } else {
        alive -= p;
      }
    }
    if (last % 32 == 0 && alive > kk) {                                                  // :528-543
      CU(launch_topk_from_scores(dist, 0, c->n, 0, kk, keys, ctx->ws, s, &g_launches, nullptr, mask_b));
      CU(launch_adaptive_threshold(keys + kk - 1, 1.0f, thr, s, &g_launches));
    }
    std::swap(mask_a, mask_b);
    d0 = d1;
  }
  CU(launch_topk_from_scores(dist, 0, c->n, (uint32_t)c->index_base, kk, keys, ctx->ws, s, &g_launches, nullptr, mask_a));
  tm.stop();
  rc = fetch_keys(*ctx, 1, kk, tm, [&](const uint64_t* hk) { decode_keys_f32(hk, kk, false, out_idx, out_score); });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// Re-rank stage of the reference's two-stage pipeline (src/scalar.rs:366-368, examples/binary_demo.rs:235-237): exact
// batch_knn / batch_knn_dot / batch_knn_cosine restricted to `candidates` (global indices, distinct), i.e. the result of
// the reference function on the sub-batch of those vectors with their original indices reported; ties -> lower index.
int innr_cuda_batch_knn_subset(const innr_cuda_corpus* c, int metric, const float* query, size_t query_len,
                               const uint64_t* candidates, size_t n_candidates, size_t k, uint64_t* out_idx,
                               float* out_score, size_t* out_count) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0 || n_candidates == 0) return INNR_OK;
  if (!out_idx || !out_score || !candidates || (!query && c->d)) return fail(INNR_EINVAL, "null argument");
  for (size_t j = 0; j < n_candidates; ++j)
    if (candidates[j] < c->index_base || candidates[j] - c->index_base >= c->n)
      return fail(INNR_EINVAL, "batch_knn_subset: candidate index out of bounds");
  const size_t kk = k < n_candidates ? k : n_candidates;
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  rc = ctx_for(c, &ctx);
  if (rc) return rc;
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(ctx->d_keys.reserve(kk * sizeof(uint64_t)));
  CU(ctx->d_aux.reserve(n_candidates * sizeof(uint32_t)));
  CU(ctx->d_scores.reserve(n_candidates * sizeof(float)));
  CU(ctx->h_pin.reserve(n_candidates * sizeof(uint32_t)));
  uint32_t* h = (uint32_t*)ctx->h_pin.p;
  for (size_t j = 0; j < n_candidates; ++j) h[j] = (uint32_t)candidates[j];
  CU(cudaMemcpyAsync(ctx->d_aux.p, h, n_candidates * sizeof(uint32_t), cudaMemcpyHostToDevice, ctx->stream));
  if (c->d) CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  CU(launch_subset_scores(pdx_view(c), mode, (const float*)ctx->d_query.p, (const uint32_t*)ctx->d_aux.p, n_candidates,
                          (float*)ctx->d_scores.p, ctx->stream, &g_launches));
  CU(launch_topk_from_scores(ctx->d_scores.p, mode == PDX_L2 ? 0 : 1, n_candidates, 0, kk, (uint64_t*)ctx->d_keys.p,
                             ctx->ws, ctx->stream, &g_launches, (const uint32_t*)ctx->d_aux.p));
  tm.stop();
  rc = fetch_keys(*ctx, 1, kk, tm, [&](const uint64_t* keys) {
    decode_keys_f32(keys, kk, metric != INNR_METRIC_L2, out_idx, out_score);
  });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// batch_knn_filtered (src/batch.rs:820-882): the closure predicate crosses the ABI as a bitmask (bit i of word i/64,
// LSB first, like PackedBinary). L2, stable ascending sort of the passing vectors, k clamped to their number.
int innr_cuda_batch_knn_filtered(const innr_cuda_corpus* c, const float* query, size_t query_len, size_t k,
                                 const uint64_t* mask_words, size_t mask_len_words, uint64_t* out_idx,
                                 float* out_score, size_t* out_count) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");  // src/batch.rs:829
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0) return INNR_OK;                                              // :831-836
  if (!mask_words || mask_len_words < (c->n + 63) / 64) return fail(INNR_EINVAL, "mask shorter than the batch");
  if (!out_idx || !out_score || (!query && c->d)) return fail(INNR_EINVAL, "null argument");
  const size_t words = (c->n + 63) / 64;
  size_t passing = 0;
  for (size_t w = 0; w < words; ++w) {
    uint64_t m = mask_words[w];
    if (w == words - 1 && (c->n & 63)) m &= (~0ull) >> (64 - (c->n & 63));  // bits past num_vectors are not vectors
    passing += (size_t)__builtin_popcountll(m);
  }
  if (passing == 0) return INNR_OK;                                                     // :842-847
  const size_t kk = k < passing ? k : passing;                                          // k.min(num_passing)
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  const size_t dev_words64 = c->ld / 64 + 2;  // the kernel reads whole u32 words up to the row pitch
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(ctx->d_keys.reserve(kk * sizeof(uint64_t)));
  CU(ctx->d_aux.reserve(dev_words64 * sizeof(uint64_t)));
  CU(cudaMemsetAsync(ctx->d_aux.p, 0, dev_words64 * sizeof(uint64_t), ctx->stream));
  CU(cudaMemcpyAsync(ctx->d_aux.p, mask_words, words * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  if (c->d) CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  if (kk <= MAX_FUSED_K) {
    CU(launch_pdx_knn_filtered(pdx_view(c), (const float*)ctx->d_query.p, (const uint32_t*)ctx->d_aux.p, kk,
                               (uint64_t*)ctx->d_keys.p, ctx->ws, ctx->stream, &g_launches));
  } else {  // any k: all distances (the passing vectors' are the same sums), then rounds of <= 128 over the passing ones
    CU(ctx->d_scores.reserve(c->ld * sizeof(float)));
    CU(launch_pdx_scores(pdx_view(c), PDX_L2, (const float*)ctx->d_query.p, nullptr, (float*)ctx->d_scores.p, ctx->ws,
                         ctx->stream, &g_launches));
    CU(launch_topk_from_scores(ctx->d_scores.p, 0, c->n, (uint32_t)c->index_base, kk, (uint64_t*)ctx->d_keys.p, ctx->ws,
                               ctx->stream, &g_launches, nullptr, (const uint32_t*)ctx->d_aux.p));
  }
  tm.stop();
  rc = fetch_keys(*ctx, 1, kk, tm, [&](const uint64_t* keys) { decode_keys_f32(keys, kk, false, out_idx, out_score); });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// batch_l2_squared_pruning (src/batch.rs:320-365): (index, squared distance) of every vector none of whose partial
// distances exceeded `threshold`, ascending index. Writes min(count, capacity) pairs; *out_count = count.
int innr_cuda_batch_l2_squared_pruning(const innr_cuda_corpus* c, const float* query, size_t query_len, float threshold,
                                       uint64_t* out_idx, float* out_dist, size_t capacity, size_t* out_count) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");  // src/batch.rs:325
  if (!out_count) return fail(INNR_EINVAL, "null out_count");
  *out_count = 0;
  if (c->n == 0) return INNR_OK;
  if (capacity && (!out_idx || !out_dist)) return fail(INNR_EINVAL, "null argument");
  if (c->d == 0) {  // no dimension is ever processed: every vector survives with distance 0.0
    for (size_t i = 0; i < c->n && i < capacity; ++i) { out_idx[i] = c->index_base + i; out_dist[i] = 0.0f; }
    *out_count = c->n;
    return INNR_OK;
  }
  if (!query) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  const size_t nb = compact_blocks(c->n);
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(ctx->d_scores.reserve(c->ld * sizeof(float)));
  CU(ctx->d_aux.reserve((nb + 1) * sizeof(unsigned)));
  CU(ctx->h_counts.reserve(64));
  CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  CU(launch_pdx_scores(pdx_view(c), PDX_L2_PRUNE, (const float*)ctx->d_query.p, nullptr, (float*)ctx->d_scores.p,
                       ctx->ws, ctx->stream, &g_launches, threshold));
  CU(launch_compact_count((const float*)ctx->d_scores.p, c->n, (unsigned*)ctx->d_aux.p, ctx->stream, &g_launches));
  CU(cudaMemcpyAsync(ctx->h_counts.p, (unsigned*)ctx->d_aux.p + nb, sizeof(unsigned), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  const size_t count = *(unsigned*)ctx->h_counts.p;
  *out_count = count;
  const size_t take = count < capacity ? count : capacity;
  if (count) {
    CU(ctx->d_keys.reserve(count * (sizeof(uint64_t) + sizeof(float))));
    uint64_t* d_idx = (uint64_t*)ctx->d_keys.p;
    float* d_dist = (float*)(d_idx + count);
    CU(launch_compact_scatter((const float*)ctx->d_scores.p, c->n, c->index_base, (const unsigned*)ctx->d_aux.p, d_idx,
                              d_dist, ctx->stream, &g_launches));
    tm.stop();
    if (take) {
      CU(cudaMemcpyAsync(out_idx, d_idx, take * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
      CU(cudaMemcpyAsync(out_dist, d_dist, take * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
    }
    CU(cudaStreamSynchronize(ctx->stream));
  } else {
    tm.stop();
    CU(cudaStreamSynchronize(ctx->stream));
  }
  tm.finish();
  return INNR_OK;
}

int innr_cuda_batch_knn_keys_dev(const innr_cuda_corpus* c, int metric, const float* dev_queries,
                                 size_t n_queries, size_t k, uint64_t* dev_keys, void* stream) {
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  if (k == 0 || n_queries == 0) return INNR_OK;
  EntryGuard lk(c->device);
  cudaStream_t s = (cudaStream_t)stream;
  DeviceCtx* ctx;
  int lane = 0;
  rc = ctx_for_dev(c, &ctx, s, knn_is_scan_only(c, mode, n_queries, k), &lane);
  if (rc) return rc;
  DevRelease rel(*ctx, s, lane);
  if (c->n == 0) {  // rows are n_queries x k, sentinel-padded (header contract)
    CU(cudaMemsetAsync(dev_keys, 0xFF, n_queries * k * sizeof(uint64_t), s));
    return INNR_OK;
  }
  return knn_keys_dev(const_cast<innr_cuda_corpus*>(c), ctx, mode, dev_queries, n_queries, k, dev_keys, s, lane);
}

int innr_cuda_merge_keys_dev(const uint64_t* dev_keys_in, size_t n_lists, size_t n_queries, size_t k, int metric,
                             uint64_t* dev_keys_out, uint64_t* dev_idx, float* dev_score, void* stream) {
  if (k == 0 || n_queries == 0 || n_lists == 0) return INNR_OK;
  // the device is the one the key lists live on (the calling thread need not have bound it with innr_cuda_init)
  int device = cur_dev();
  cudaPointerAttributes attr;
  if (cudaPointerGetAttributes(&attr, dev_keys_in) == cudaSuccess && attr.type == cudaMemoryTypeDevice) device = attr.device;
  else cudaGetLastError();
  EntryGuard lk(device);
  cudaStream_t us = (cudaStream_t)stream;
  DeviceCtx* ctx;
  if (k <= MAX_FUSED_K) {  // one launch, no workspace and no scratch: nothing to order against
    int rc = ensure_ctx(device, &ctx, WS_NONE, us);
    if (rc) return rc;
    CU(launch_merge_keys(dev_keys_in, n_lists, n_queries, k, metric != INNR_METRIC_L2, dev_keys_out, dev_idx, dev_score,
                         us, &g_launches));
    return INNR_OK;
  }
  int rc = ensure_ctx(device, &ctx, WS_DEV, us);
  if (rc) return rc;
  DevRelease rel(*ctx, us);
  {
    uint64_t* keys_out = dev_keys_out;
    if (!keys_out) {
      CU(ctx->d_tcws.reserve(n_queries * k * sizeof(uint64_t)));
      keys_out = (uint64_t*)ctx->d_tcws.p;
    }
    CU(launch_merge_keys_big(dev_keys_in, n_lists, n_queries, k, metric != INNR_METRIC_L2, keys_out, dev_idx, dev_score,
                             ctx->ws, (cudaStream_t)stream, &g_launches));
    return INNR_OK;
  }
}

int innr_cuda_topk_from_distances(const float* distances, size_t n, size_t k, uint32_t* out_id, float* out_distance,
                                  size_t* out_count) {
  if (out_count) *out_count = 0;
  if (n == 0 || k == 0) return INNR_OK;
  if (!distances || !out_id || !out_distance) return fail(INNR_EINVAL, "null argument");
  int rc = check_index_range(n, 0);
  if (rc) return rc;
  const size_t kk = k < n ? k : n;
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  rc = current_ctx(&ctx);
  if (rc) return rc;
  CU(ctx->d_scores.reserve(n * sizeof(float)));
  CU(ctx->d_keys.reserve(kk * sizeof(uint64_t)));
  CU(cudaMemcpyAsync(ctx->d_scores.p, distances, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  CU(launch_topk_from_distances((const float*)ctx->d_scores.p, n, kk, (uint64_t*)ctx->d_keys.p, ctx->ws,
                                ctx->stream, &g_launches));
  tm.stop();
  rc = fetch_keys(*ctx, 1, kk, tm, [&](const uint64_t* keys) {
    std::vector<uint64_t> idx(kk);
    decode_keys_f32(keys, kk, false, idx.data(), out_distance);
    for (size_t j = 0; j < kk; ++j) out_id[j] = (uint32_t)idx[j];
  });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ binary codes
static int alloc_binary(DeviceCtx& ctx, size_t n, size_t dim_bits, uint64_t index_base, innr_cuda_corpus** out) {
  int rc = check_index_range(n, index_base);
  if (rc) return rc;
  rc = new_corpus(1, ctx.device, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  c->n = n;
  c->dim_bits = dim_bits;
  c->words = (dim_bits + 63) / 64;
  c->chunks = (c->words + 1) / 2;
  c->d = dim_bits;
  c->ld = round_up(n, 16);
  c->index_base = index_base;
  c->bytes = c->chunks * c->ld * sizeof(uint4);
  if (c->bytes) {
    cudaError_t e = cudaMalloc(&c->dev, c->bytes);
    if (e != cudaSuccess) {
      delete c;
      *out = nullptr;
      return cuda_fail(e, "cudaMalloc(binary corpus)");
    }
  }
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_upload_binary(const uint64_t* words, size_t n, size_t dim_bits, uint64_t index_base,
                            innr_cuda_corpus** out) {
  if (!out) return fail(INNR_EINVAL, "null out");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_binary(*ctx, n, dim_bits, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    if (!words) return fail(INNR_EINVAL, "null words");
    void* stage = nullptr;
    CU(cudaMalloc(&stage, n * c->words * sizeof(uint64_t)));
    cudaError_t e = cudaMemcpyAsync(stage, words, n * c->words * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
      e = launch_binary_pack((const uint64_t*)stage, n, c->words, dim_bits, (uint4*)c->dev, c->ld, ctx->stream, &g_launches);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(stage);
    if (e != cudaSuccess) return cuda_fail(e, "upload_binary");
  }
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_generate_binary(uint64_t salt, uint64_t first_row, size_t n, size_t dim_bits, uint64_t index_base,
                              innr_cuda_corpus** out) {
  if (!out) return fail(INNR_EINVAL, "null out");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_binary(*ctx, n, dim_bits, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    CU(launch_generate_binary(salt, first_row, n, c->words, dim_bits, (uint4*)c->dev, c->ld, ctx->stream, &g_launches));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  guard.ok = true;
  return INNR_OK;
}

// copies nq query codes (row-major words) to the device, padded to 2*chunks words each and masked
static int stage_binary_queries(DeviceCtx& ctx, const innr_cuda_corpus* c, const uint64_t* query_words, size_t nq) {
  const size_t qw = 2 * c->chunks;
  CU(ctx.h_pin.reserve(nq * qw * sizeof(uint64_t)));
  uint64_t* h = (uint64_t*)ctx.h_pin.p;
  const size_t rem = c->dim_bits % 64;
  for (size_t q = 0; q < nq; ++q)
    for (size_t w = 0; w < qw; ++w) {
      uint64_t x = w < c->words ? query_words[q * c->words + w] : 0;
      if (w + 1 == c->words && rem) x &= (1ull << rem) - 1;  // PackedBinary::new masks padding
      h[q * qw + w] = x;
    }
  CU(ctx.d_query.reserve(nq * qw * sizeof(uint64_t) + 16));
  CU(cudaMemcpyAsync(ctx.d_query.p, h, nq * qw * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx.stream));
  return INNR_OK;
}

int innr_cuda_hamming_all(const innr_cuda_corpus* c, const uint64_t* query_words, size_t query_dim_bits,
                          uint32_t* out_host) {
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (query_dim_bits != c->dim_bits)
    return fail(INNR_EINVAL, "innr::binary_hamming: dimension mismatch");             // src/binary.rs:155-159
  if (c->n == 0) return INNR_OK;
  if (!out_host || (!query_words && c->words)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  if (c->words == 0) {
    std::memset(out_host, 0, c->n * sizeof(uint32_t));
    return INNR_OK;
  }
  rc = stage_binary_queries(*ctx, c, query_words, 1);
  if (rc) return rc;
  CU(ctx->d_scores.reserve(c->n * sizeof(uint32_t)));
  Timed tm(*ctx);
  CU(launch_hamming_all(bin_view(c), (const uint64_t*)ctx->d_query.p, (uint32_t*)ctx->d_scores.p, ctx->stream,
                        &g_launches));
  tm.stop();
  CU(cudaMemcpyAsync(out_host, ctx->d_scores.p, c->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  tm.finish();
  return INNR_OK;
}

// encode_binary (src/binary.rs:133-141) of every vector of a device-resident f32 corpus, on the device: the derived
// code set shares the f32 corpus' index_base, so first-pass indices feed innr_cuda_batch_knn_subset directly.
int innr_cuda_binary_from_f32(const innr_cuda_corpus* f32_corpus, float threshold, innr_cuda_corpus** out) {
  if (!out || !f32_corpus || f32_corpus->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  EntryGuard lk(f32_corpus->device);
  DeviceCtx* ctx;
  int rc = ctx_for(f32_corpus, &ctx);
  if (rc) return rc;
  rc = alloc_binary(*ctx, f32_corpus->n, f32_corpus->d, f32_corpus->index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    CU(launch_binary_from_pdx(pdx_view(f32_corpus), threshold,
                              (uint4*)c->dev, c->ld, ctx->stream, &g_launches));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  guard.ok = true;
  return INNR_OK;
}

// binary_dot / binary_jaccard of one query against every code (src/binary.rs:178-213)
static int binary_setop_all(const innr_cuda_corpus* c, const uint64_t* query_words, size_t query_dim_bits, bool jaccard,
                            void* out_host) {
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (query_dim_bits != c->dim_bits) return fail(INNR_EINVAL, "dimension mismatch");  // assert_eq!(a.dimension, b.dimension)
  if (c->n == 0) return INNR_OK;
  if (!out_host || (!query_words && c->words)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  if (c->words == 0) {  // no words: intersection 0, union 0 -> dot 0, jaccard 1.0
    for (size_t i = 0; i < c->n; ++i) {
      if (jaccard) ((float*)out_host)[i] = 1.0f; else ((uint32_t*)out_host)[i] = 0u;
    }
    return INNR_OK;
  }
  rc = stage_binary_queries(*ctx, c, query_words, 1);
  if (rc) return rc;
  CU(ctx->d_scores.reserve(c->n * sizeof(uint32_t)));
  Timed tm(*ctx);
  if (jaccard)
    CU(launch_binary_jaccard_all(bin_view(c), (const uint64_t*)ctx->d_query.p, (float*)ctx->d_scores.p, ctx->stream, &g_launches));
  else
    CU(launch_binary_dot_all(bin_view(c), (const uint64_t*)ctx->d_query.p, (uint32_t*)ctx->d_scores.p, ctx->stream, &g_launches));
  tm.stop();
  CU(cudaMemcpyAsync(out_host, ctx->d_scores.p, c->n * sizeof(uint32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  tm.finish();
  return INNR_OK;
}
int innr_cuda_binary_dot_all(const innr_cuda_corpus* c, const uint64_t* query_words, size_t query_dim_bits,
                             uint32_t* out_host) {
  return binary_setop_all(c, query_words, query_dim_bits, false, out_host);
}
int innr_cuda_binary_jaccard_all(const innr_cuda_corpus* c, const uint64_t* query_words, size_t query_dim_bits,
                                 float* out_host) {
  return binary_setop_all(c, query_words, query_dim_bits, true, out_host);
}

// Query batches go through the tensor-core filter (bin_tc.cu: the exact keys, see there) when the corpus qualifies;
// innr_cuda_set_option("bin_tc", 0) disables it. Single queries always take the scan.
static bool bin_takes_tc_filter(const innr_cuda_corpus* c, size_t nq, size_t k) {
  return g_opt.bin_tc && c->n >= g_opt.bin_tc_min_n && nq >= g_opt.bin_tc_min_queries && nq >= 2 && k <= g_opt.bin_tc_max_k &&
         bin_tc_supported(bin_view(c), nq, k);
}
// the Hamming scans need a Workspace and nothing else: either lane will do
static bool hamming_is_scan_only(const innr_cuda_corpus* c, size_t nq, size_t k) {
  return k <= MAX_FUSED_K && !bin_takes_tc_filter(c, nq, k);
}
static bool setops_fused(const innr_cuda_corpus* c, size_t k) {
  return k <= MAX_FUSED_K && c->chunks * sizeof(uint4) + 8 * k * sizeof(uint64_t) <= 48 * 1024;
}
static bool setops_is_scan_only(const innr_cuda_corpus* c, size_t nq, size_t k) {
  return setops_fused(c, k) && !bin_takes_tc_filter(c, nq, k);
}
// The row popcounts of the filter path, built on first use (the handle stays immutable: a cache of the same data). On
// failure (no memory) the corpus stays on the CUDA-core scans.
static int bin_tc_prepare(innr_cuda_corpus* c, cudaStream_t s) {
  if (c->tc_state != 0) return INNR_OK;
  c->tc_state = -1;
  if (cudaMalloc(&c->dev_popc, c->n * sizeof(uint32_t)) != cudaSuccess) {
    cudaGetLastError();  // out of memory is not an error of the call: the scans answer
    c->dev_popc = nullptr;
    return INNR_OK;
  }
  CU(launch_bin_tc_popc(bin_view(c), c->dev_popc, s, &g_launches));
  c->tc_state = 1;
  return INNR_OK;
}
// op 0 Hamming, 1 binary_dot, 2 binary_jaccard; *taken = false when the corpus cannot take the filter (no memory). Lane 0:
// the filter's scratch. Enqueues only: the statistics stay on the device.
static int bin_tc_keys(const innr_cuda_corpus* c, DeviceCtx* ctx, int op, const uint64_t* dev_query_words, size_t nq, size_t k,
                       uint64_t* dev_keys, cudaStream_t s, bool* taken) {
  *taken = false;
  int rc = bin_tc_prepare(const_cast<innr_cuda_corpus*>(c), s);
  if (rc) return rc;
  if (c->tc_state != 1) return INNR_OK;
  CU(ctx->d_tcws.reserve(bin_tc_workspace_bytes(c->chunks, nq, k)));
  if (!ctx->bt_stats) CU(cudaMalloc((void**)&ctx->bt_stats, sizeof(BinTcDevStats)));
  const size_t chunks = (nq + BIN_TC_CHUNK_QUERIES - 1) / BIN_TC_CHUNK_QUERIES;
  while (ctx->bt_ev.size() < 2 + 2 * chunks) {
    cudaEvent_t e;
    CU(cudaEventCreate(&e));
    ctx->bt_ev.push_back(e);
  }
  BinTcCall call;
  CU(launch_bin_tc(bin_view(c), op, c->dev_popc, dev_query_words, nq, k, dev_keys, ctx->d_tcws.p, ctx->bt_stats,
                   ctx->bt_ev.data(), ctx->ws.num_sms, s, &g_launches, &call));
  {
    std::lock_guard<std::mutex> lg(g_mu);
    g_bintc_device = ctx->device;
    g_bintc_call = call;
    g_bintc_chunks = chunks;
  }
  *taken = true;
  return INNR_OK;
}
// binary_dot (op 0) / binary_jaccard (op 1) keys of nq queries, rows of k keys (sentinel padded past n): the filter for
// batches that qualify, else the single-query route once per query
static int setop_keys(const innr_cuda_corpus* c, DeviceCtx* ctx, int op, const uint64_t* dev_query_words, size_t nq, size_t k,
                      uint64_t* dev_keys, cudaStream_t s, int lane = 0) {
  if (bin_takes_tc_filter(c, nq, k)) {
    bool taken;
    int rc = bin_tc_keys(c, ctx, 1 + op, dev_query_words, nq, k, dev_keys, s, &taken);
    if (rc || taken) return rc;
  }
  const size_t qw = 2 * c->chunks;
  if (setops_fused(c, k)) {
    for (size_t q = 0; q < nq; ++q)
      CU(launch_binary_setops_topk(bin_view(c), op, dev_query_words + q * qw, k, dev_keys + q * k, ctx->lane_ws(lane), s,
                                   &g_launches));
    return INNR_OK;
  }
  const size_t kk = k < c->n ? k : c->n;
  if (kk < k) CU(cudaMemsetAsync(dev_keys, 0xFF, nq * k * sizeof(uint64_t), s));
  CU(ctx->d_scores.reserve(c->n * sizeof(uint32_t)));
  for (size_t q = 0; q < nq; ++q) {
    if (op)
      CU(launch_binary_jaccard_all(bin_view(c), dev_query_words + q * qw, (float*)ctx->d_scores.p, s, &g_launches));
    else
      CU(launch_binary_dot_all(bin_view(c), dev_query_words + q * qw, (uint32_t*)ctx->d_scores.p, s, &g_launches));
    CU(launch_topk_from_scores(ctx->d_scores.p, op ? 1 : 4, c->n, (uint32_t)c->index_base, kk, dev_keys + q * k, ctx->ws, s,
                               &g_launches));
  }
  return INNR_OK;
}

// Top-k by binary_dot (op 0) or binary_jaccard (op 1) over a code set: the caller composition the reference shows for
// Hamming (examples/binary_demo.rs:174-180) with the similarity ranked descending, ties -> lower index. Scores as f32
// (dot counts are exact: dimension < 2^24).
int innr_cuda_binary_topk(const innr_cuda_corpus* c, int op, const uint64_t* query_words, size_t query_dim_bits, size_t k,
                          uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (op != 0 && op != 1) return fail(INNR_EINVAL, "binary_topk: op must be 0 (dot) or 1 (jaccard)");
  if (query_dim_bits != c->dim_bits) return fail(INNR_EINVAL, "dimension mismatch");  // assert_eq!(a.dimension, b.dimension)
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0) return INNR_OK;
  if (!out_idx || !out_score || (!query_words && c->words)) return fail(INNR_EINVAL, "null argument");
  if (c->dim_bits >= (1u << 24)) return fail(INNR_EUNSUPPORTED, "binary_topk: dimension >= 2^24");
  const size_t kk = k < c->n ? k : c->n;
  if (c->words == 0) {  // no words: dot 0 / jaccard 1.0 for every code, index order
    for (size_t j = 0; j < kk; ++j) { out_idx[j] = c->index_base + j; out_score[j] = op ? 1.0f : 0.0f; }
    if (out_count) *out_count = kk;
    return INNR_OK;
  }
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  rc = stage_binary_queries(*ctx, c, query_words, 1);
  if (rc) return rc;
  CU(ctx->d_scores.reserve(c->n * sizeof(uint32_t)));
  CU(ctx->d_keys.reserve(kk * sizeof(uint64_t)));
  Timed tm(*ctx);
  const size_t fused_smem = c->chunks * sizeof(uint4) + 8 * kk * sizeof(uint64_t);
  if (kk <= MAX_FUSED_K && fused_smem <= 48 * 1024) {
    // one pass: the selection rides on the scan (same keys as the two-step route below), nothing of size n is written
    CU(launch_binary_setops_topk(bin_view(c), op, (const uint64_t*)ctx->d_query.p, kk, (uint64_t*)ctx->d_keys.p, ctx->ws,
                                 ctx->stream, &g_launches));
  } else {
    if (op)
      CU(launch_binary_jaccard_all(bin_view(c), (const uint64_t*)ctx->d_query.p, (float*)ctx->d_scores.p, ctx->stream, &g_launches));
    else
      CU(launch_binary_dot_all(bin_view(c), (const uint64_t*)ctx->d_query.p, (uint32_t*)ctx->d_scores.p, ctx->stream, &g_launches));
    CU(launch_topk_from_scores(ctx->d_scores.p, op ? 1 : 4, c->n, (uint32_t)c->index_base, kk, (uint64_t*)ctx->d_keys.p, ctx->ws,
                               ctx->stream, &g_launches));
  }
  tm.stop();
  rc = fetch_keys(*ctx, 1, kk, tm, [&](const uint64_t* keys) {
    if (op) {
      decode_keys_f32(keys, kk, true, out_idx, out_score);
    } else {
      for (size_t j = 0; j < kk; ++j) {
        out_idx[j] = keys[j] & 0xFFFFFFFFull;
        out_score[j] = (float)(~(uint32_t)(keys[j] >> 32));
      }
    }
  });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

static int hamming_keys(const innr_cuda_corpus* c, DeviceCtx* ctx, const uint64_t* dev_query_words, size_t nq, size_t k,
                        uint64_t* dev_keys, cudaStream_t s, int lane = 0) {
  if (bin_takes_tc_filter(c, nq, k)) {
    bool taken;
    int rc = bin_tc_keys(c, ctx, 0, dev_query_words, nq, k, dev_keys, s, &taken);
    if (rc || taken) return rc;
  }
  if (k <= MAX_FUSED_K) {
    CU(launch_hamming_topk(bin_view(c), dev_query_words, nq, k, dev_keys, ctx->lane_ws(lane), s, &g_launches));
    return INNR_OK;
  }
  const size_t kk = k < c->n ? k : c->n;  // rows stay k wide, sentinel-padded
  if (kk < k) CU(cudaMemsetAsync(dev_keys, 0xFF, nq * k * sizeof(uint64_t), s));
  CU(ctx->d_scores.reserve(c->n * sizeof(uint32_t)));
  for (size_t q = 0; q < nq; ++q) {
    CU(launch_hamming_all(bin_view(c), dev_query_words + q * 2 * c->chunks, (uint32_t*)ctx->d_scores.p, s, &g_launches));
    int rc = big_k_from_scores(ctx, ctx->d_scores.p, 2, c->n, c->index_base, kk, dev_keys + q * k, s);
    if (rc) return rc;
  }
  return INNR_OK;
}

int innr_cuda_hamming_topk(const innr_cuda_corpus* c, const uint64_t* query_words, size_t n_queries,
                           size_t query_dim_bits, size_t k, uint64_t* out_idx, uint32_t* out_dist,
                           size_t* out_count) {
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (query_dim_bits != c->dim_bits) return fail(INNR_EINVAL, "innr::binary_hamming: dimension mismatch");
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0 || n_queries == 0) return INNR_OK;
  if (!out_idx || !out_dist || (!query_words && c->words)) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < c->n ? k : c->n;
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  if (c->words == 0) {  // zero-dimensional codes: every distance is 0 -> first kk indices
    for (size_t q = 0; q < n_queries; ++q)
      for (size_t j = 0; j < kk; ++j) {
        out_idx[q * k + j] = c->index_base + j;
        out_dist[q * k + j] = 0;
      }
    if (out_count) *out_count = kk;
    return INNR_OK;
  }
  rc = stage_binary_queries(*ctx, c, query_words, n_queries);
  if (rc) return rc;
  CU(ctx->d_keys.reserve(n_queries * kk * sizeof(uint64_t)));
  Timed tm(*ctx);
  rc = hamming_keys(c, ctx, (const uint64_t*)ctx->d_query.p, n_queries, kk, (uint64_t*)ctx->d_keys.p, ctx->stream);
  if (rc) return rc;
  tm.stop();
  rc = fetch_keys(*ctx, n_queries, kk, tm, [&](const uint64_t* keys) {
    for (size_t q = 0; q < n_queries; ++q)
      for (size_t j = 0; j < kk; ++j) {
        out_idx[q * k + j] = keys[q * kk + j] & 0xFFFFFFFFull;
        out_dist[q * k + j] = (uint32_t)(keys[q * kk + j] >> 32);
      }
  });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

int innr_cuda_hamming_topk_keys_dev(const innr_cuda_corpus* c, const uint64_t* dev_query_words, size_t n_queries,
                                    size_t k, uint64_t* dev_keys, void* stream) {
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (k == 0 || n_queries == 0) return INNR_OK;
  EntryGuard lk(c->device);
  cudaStream_t s = (cudaStream_t)stream;
  DeviceCtx* ctx;
  int lane = 0;
  int rc = ctx_for_dev(c, &ctx, s, hamming_is_scan_only(c, n_queries, k), &lane);
  if (rc) return rc;
  DevRelease rel(*ctx, s, lane);
  if (c->n == 0 || c->words == 0) {
    CU(cudaMemsetAsync(dev_keys, 0xFF, n_queries * k * sizeof(uint64_t), s));
    return INNR_OK;
  }
  return hamming_keys(c, ctx, dev_query_words, n_queries, k, dev_keys, s, lane);
}

// n_queries calls of innr_cuda_binary_topk in one: query batches take the tensor-core filter (bin_tc.cu) when they qualify
int innr_cuda_binary_topk_batch(const innr_cuda_corpus* c, int op, const uint64_t* query_words, size_t n_queries,
                                size_t query_dim_bits, size_t k, uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (op != 0 && op != 1) return fail(INNR_EINVAL, "binary_topk: op must be 0 (dot) or 1 (jaccard)");
  if (query_dim_bits != c->dim_bits) return fail(INNR_EINVAL, "dimension mismatch");  // assert_eq!(a.dimension, b.dimension)
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0 || n_queries == 0) return INNR_OK;
  if (!out_idx || !out_score || (!query_words && c->words)) return fail(INNR_EINVAL, "null argument");
  if (c->dim_bits >= (1u << 24)) return fail(INNR_EUNSUPPORTED, "binary_topk: dimension >= 2^24");
  const size_t kk = k < c->n ? k : c->n;
  if (c->words == 0) {  // no words: dot 0 / jaccard 1.0 for every code, index order
    for (size_t q = 0; q < n_queries; ++q)
      for (size_t j = 0; j < kk; ++j) {
        out_idx[q * k + j] = c->index_base + j;
        out_score[q * k + j] = op ? 1.0f : 0.0f;
      }
    if (out_count) *out_count = kk;
    return INNR_OK;
  }
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  rc = stage_binary_queries(*ctx, c, query_words, n_queries);
  if (rc) return rc;
  CU(ctx->d_keys.reserve(n_queries * kk * sizeof(uint64_t)));
  Timed tm(*ctx);
  rc = setop_keys(c, ctx, op, (const uint64_t*)ctx->d_query.p, n_queries, kk, (uint64_t*)ctx->d_keys.p, ctx->stream);
  if (rc) return rc;
  tm.stop();
  rc = fetch_keys(*ctx, n_queries, kk, tm, [&](const uint64_t* keys) {
    for (size_t q = 0; q < n_queries; ++q) {
      const uint64_t* kq = keys + q * kk;
      if (op) {
        decode_keys_f32(kq, kk, true, out_idx + q * k, out_score + q * k);
      } else {
        for (size_t j = 0; j < kk; ++j) {
          out_idx[q * k + j] = kq[j] & 0xFFFFFFFFull;
          out_score[q * k + j] = (float)(~(uint32_t)(kq[j] >> 32));
        }
      }
    }
  });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

int innr_cuda_binary_topk_keys_dev(const innr_cuda_corpus* c, int op, const uint64_t* dev_query_words, size_t n_queries,
                                   size_t k, uint64_t* dev_keys, void* stream) {
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (op != 0 && op != 1) return fail(INNR_EINVAL, "binary_topk: op must be 0 (dot) or 1 (jaccard)");
  if (k == 0 || n_queries == 0) return INNR_OK;
  if (c->n > 0 && c->words == 0) return fail(INNR_EUNSUPPORTED, "zero-dimensional codes: use innr_cuda_binary_topk_batch");
  if (c->dim_bits >= (1u << 24)) return fail(INNR_EUNSUPPORTED, "binary_topk: dimension >= 2^24");
  EntryGuard lk(c->device);
  cudaStream_t s = (cudaStream_t)stream;
  DeviceCtx* ctx;
  int lane = 0;
  int rc = ctx_for_dev(c, &ctx, s, setops_is_scan_only(c, n_queries, k), &lane);
  if (rc) return rc;
  DevRelease rel(*ctx, s, lane);
  if (c->n == 0) {
    CU(cudaMemsetAsync(dev_keys, 0xFF, n_queries * k * sizeof(uint64_t), s));
    return INNR_OK;
  }
  return setop_keys(c, ctx, op, dev_query_words, n_queries, k, dev_keys, s, lane);
}

int innr_cuda_encode_binary(const float* values, size_t n, float threshold, uint64_t* out_words) {
  if (n == 0) return INNR_OK;
  if (!values || !out_words) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  const size_t nw = (n + 63) / 64;
  CU(ctx->d_scores.reserve(n * sizeof(float)));
  CU(ctx->d_aux.reserve(nw * sizeof(uint64_t)));
  CU(cudaMemcpyAsync(ctx->d_scores.p, values, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(launch_encode_binary((const float*)ctx->d_scores.p, n, threshold, (uint64_t*)ctx->d_aux.p, ctx->stream, &g_launches));
  CU(cudaMemcpyAsync(out_words, ctx->d_aux.p, nw * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ u8 codes
static int alloc_u8(DeviceCtx& ctx, size_t n, size_t d, float alpha, float offset, uint64_t index_base,
                    innr_cuda_corpus** out) {
  int rc = check_index_range(n, index_base);
  if (rc) return rc;
  rc = new_corpus(2, ctx.device, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  c->n = n;
  c->d = d;
  c->chunks = (d + 15) / 16;
  c->ld = round_up(n, 16);
  c->alpha = alpha;
  c->offset = offset;
  c->index_base = index_base;
  c->bytes = c->chunks * c->ld * sizeof(uint4);
  if (c->bytes) {
    cudaError_t e = cudaMalloc(&c->dev, c->bytes);
    if (e != cudaSuccess) {
      delete c;
      *out = nullptr;
      return cuda_fail(e, "cudaMalloc(u8 corpus)");
    }
  }
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_upload_u8(const uint8_t* rows, size_t n, size_t d, float alpha, float offset, uint64_t index_base,
                        innr_cuda_corpus** out) {
  if (!out) return fail(INNR_EINVAL, "null out");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_u8(*ctx, n, d, alpha, offset, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    if (!rows) return fail(INNR_EINVAL, "null rows");
    void* stage = nullptr;
    CU(cudaMalloc(&stage, n * d));
    cudaError_t e = cudaMemcpyAsync(stage, rows, n * d, cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess) e = launch_u8_pack((const uint8_t*)stage, n, d, (uint4*)c->dev, c->ld, ctx->stream, &g_launches);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(stage);
    if (e != cudaSuccess) return cuda_fail(e, "upload_u8");
  }
  guard.ok = true;
  return INNR_OK;
}

// quantize_u8 (src/scalar.rs:212-225) of every vector of a device-resident f32 corpus, on the device
int innr_cuda_u8_from_f32(const innr_cuda_corpus* f32_corpus, float alpha, float offset, innr_cuda_corpus** out) {
  if (!out || !f32_corpus || f32_corpus->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  EntryGuard lk(f32_corpus->device);
  DeviceCtx* ctx;
  int rc = ctx_for(f32_corpus, &ctx);
  if (rc) return rc;
  rc = alloc_u8(*ctx, f32_corpus->n, f32_corpus->d, alpha, offset, f32_corpus->index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    CU(launch_u8_from_pdx(pdx_view(f32_corpus), alpha, offset,
                          (uint4*)c->dev, c->ld, ctx->stream, &g_launches));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_generate_u8(uint64_t salt, uint64_t first_row, size_t n, size_t d, float alpha, float offset,
                          uint64_t index_base, innr_cuda_corpus** out) {
  if (!out) return fail(INNR_EINVAL, "null out");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_u8(*ctx, n, d, alpha, offset, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    CU(launch_generate_u8(salt, first_row, n, d, alpha, offset, (uint4*)c->dev, c->ld, ctx->stream, &g_launches));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_quantize_u8(const float* values, size_t n, float alpha, float offset, uint8_t* out_codes) {
  if (n == 0) return INNR_OK;
  if (!values || !out_codes) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  CU(ctx->d_scores.reserve(n * sizeof(float)));
  CU(ctx->d_aux.reserve(n));
  CU(cudaMemcpyAsync(ctx->d_scores.p, values, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(launch_quantize_u8((const float*)ctx->d_scores.p, n, alpha, offset, (uint8_t*)ctx->d_aux.p, ctx->stream, &g_launches));
  CU(cudaMemcpyAsync(out_codes, ctx->d_aux.p, n, cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return INNR_OK;
}

static int u8_scores(const innr_cuda_corpus* c, int mode, const float* query, size_t query_len, float* out_host,
                     const char* mismatch_msg) {
  if (!c || c->kind != 2) return fail(INNR_EINVAL, "need a u8 corpus");
  if (query_len != c->d) return fail(INNR_EINVAL, mismatch_msg);
  if (c->n == 0) return INNR_OK;
  if (!out_host || (!query && c->d)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
  CU(ctx->d_scores.reserve(c->n * sizeof(float)));
  if (c->d) CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  if (c->d == 0) {
    // mixed dot of empty vectors is 0.0; asymmetric adds offset * 0.0
    for (size_t i = 0; i < c->n; ++i) out_host[i] = 0.0f;
    return INNR_OK;
  }
  Timed tm(*ctx);
  CU(launch_u8_scores(u8_view(c), mode, (const float*)ctx->d_query.p, (float*)ctx->d_scores.p, ctx->stream, &g_launches));
  tm.stop();
  CU(cudaMemcpyAsync(out_host, ctx->d_scores.p, c->n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  tm.finish();
  return INNR_OK;
}

int innr_cuda_mixed_dot_u8_all(const innr_cuda_corpus* c, const float* query, size_t query_len, float* out_host) {
  return u8_scores(c, 0, query, query_len, out_host, "mixed_dot_u8_f32: slice length mismatch");
}
int innr_cuda_asymmetric_dot_u8_all(const innr_cuda_corpus* c, const float* query, size_t query_len, float* out_host) {
  return u8_scores(c, 1, query, query_len, out_host, "asymmetric_dot_u8: dimension mismatch");
}

// Large batches go through the tensor-core filter (u8_tc.cu: exact results, see there) when the corpus qualifies;
// innr_cuda_set_option("u8_tc", 0) disables it. Single queries always take the scan.
static bool u8_takes_tc_filter(const innr_cuda_corpus* c, size_t nq, size_t k) {
  return g_opt.u8_tc && c->n >= g_opt.u8_tc_min_n && nq >= g_opt.u8_tc_min_queries && nq >= 2 && k <= g_opt.u8_tc_max_k &&
         u8_tc_supported(u8_view(c), nq, k);
}
// the pair / single-query scans need a Workspace and nothing else: either lane will do
static bool u8_is_scan_only(const innr_cuda_corpus* c, size_t nq, size_t k) {
  return k <= MAX_FUSED_K && !u8_takes_tc_filter(c, nq, k);
}
// The row radii of the filter path, built on first use (the handle stays immutable: a cache of the same data). On failure
// (no memory) the corpus stays on the exact scan.
static int u8_tc_prepare(innr_cuda_corpus* c, cudaStream_t s) {
  if (c->tc_state != 0) return INNR_OK;
  c->tc_state = -1;
  if (cudaMalloc(&c->dev_radius, c->n * sizeof(float)) != cudaSuccess) {
    cudaGetLastError();  // out of memory is not an error of the call: exact scan
    c->dev_radius = nullptr;
    return INNR_OK;
  }
  CU(launch_u8_tc_radius(u8_view(c), c->dev_radius, s, &g_launches));
  c->tc_state = 1;
  return INNR_OK;
}
static int u8_keys(const innr_cuda_corpus* c, DeviceCtx* ctx, const float* dev_queries, size_t nq, size_t k,
                   uint64_t* dev_keys, cudaStream_t s, int lane = 0) {
  if (u8_takes_tc_filter(c, nq, k)) {  // lane 0: the filter's scratch
    innr_cuda_corpus* cm = const_cast<innr_cuda_corpus*>(c);
    int rc = u8_tc_prepare(cm, s);
    if (rc) return rc;
    if (c->tc_state == 1) {
      CU(ctx->d_tcws.reserve(u8_tc_workspace_bytes(c->d, nq, false)));
      CU(ctx->h_counts.reserve((nq < 1024 ? nq : 1024) * sizeof(unsigned)));
      std::vector<unsigned> overflow;
      KnnTcStats st;
      CU(launch_u8_knn_tc(u8_view(c), c->dev_radius, dev_queries, nq, k, dev_keys, ctx->d_tcws.p, (unsigned*)ctx->h_counts.p,
                          ctx->ws, s, &g_launches, &overflow, &st));
      {
        std::lock_guard<std::mutex> lg(g_mu);
        g_u8tc_stats = st;
      }
      for (unsigned q : overflow)
        CU(launch_u8_knn(u8_view(c), dev_queries + (size_t)q * c->d, 1, k, dev_keys + (size_t)q * k, ctx->ws, s, &g_launches));
      return INNR_OK;
    }
  }
  if (k <= MAX_FUSED_K) {
    CU(launch_u8_knn(u8_view(c), dev_queries, nq, k, dev_keys, ctx->lane_ws(lane), s, &g_launches));
    return INNR_OK;
  }
  const size_t kk = k < c->n ? k : c->n;  // rows stay k wide, sentinel-padded
  if (kk < k) CU(cudaMemsetAsync(dev_keys, 0xFF, nq * k * sizeof(uint64_t), s));
  CU(ctx->d_scores.reserve(c->n * sizeof(float)));
  for (size_t q = 0; q < nq; ++q) {
    CU(launch_u8_scores(u8_view(c), 1, dev_queries + q * c->d, (float*)ctx->d_scores.p, s, &g_launches));
    int rc = big_k_from_scores(ctx, ctx->d_scores.p, 1, c->n, c->index_base, kk, dev_keys + q * k, s);
    if (rc) return rc;
  }
  return INNR_OK;
}

int innr_cuda_batch_knn_u8(const innr_cuda_corpus* c, const float* queries, size_t n_queries, size_t query_len,
                           size_t k, uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 2) return fail(INNR_EINVAL, "need a u8 corpus");
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0 || n_queries == 0) return INNR_OK;  // src/scalar.rs:376-378 (before any length check)
  if (query_len != c->d) return fail(INNR_EINVAL, "asymmetric_dot_u8_precomputed: dimension mismatch");
  if (!out_idx || !out_score || (!queries && c->d)) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < c->n ? k : c->n;
  if (c->d == 0) return fail(INNR_EUNSUPPORTED, "zero-dimensional u8 corpus");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  CU(ctx->d_query.reserve((n_queries * c->d + 4) * sizeof(float)));
  CU(ctx->d_keys.reserve(n_queries * kk * sizeof(uint64_t)));
  CU(cudaMemcpyAsync(ctx->d_query.p, queries, n_queries * c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  rc = u8_keys(c, ctx, (const float*)ctx->d_query.p, n_queries, kk, (uint64_t*)ctx->d_keys.p, ctx->stream);
  if (rc) return rc;
  tm.stop();
  rc = fetch_keys(*ctx, n_queries, kk, tm, [&](const uint64_t* keys) {
    for (size_t q = 0; q < n_queries; ++q) decode_keys_f32(keys + q * kk, kk, true, out_idx + q * k, out_score + q * k);
  });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

int innr_cuda_batch_knn_u8_keys_dev(const innr_cuda_corpus* c, const float* dev_queries, size_t n_queries, size_t k,
                                    uint64_t* dev_keys, void* stream) {
  if (!c || c->kind != 2) return fail(INNR_EINVAL, "need a u8 corpus");
  if (k == 0 || n_queries == 0) return INNR_OK;
  EntryGuard lk(c->device);
  cudaStream_t s = (cudaStream_t)stream;
  DeviceCtx* ctx;
  int lane = 0;
  int rc = ctx_for_dev(c, &ctx, s, u8_is_scan_only(c, n_queries, k), &lane);
  if (rc) return rc;
  DevRelease rel(*ctx, s, lane);
  if (c->n == 0 || c->d == 0) {
    CU(cudaMemsetAsync(dev_keys, 0xFF, n_queries * k * sizeof(uint64_t), s));
    return INNR_OK;
  }
  return u8_keys(c, ctx, dev_queries, n_queries, k, dev_keys, s, lane);
}

// Test hook for the u8 filter's bound (tests/test_gpu_u8_tc.py): the score interval [lower, upper] of the dense first
// pass for rows < min(n, 4096), row-major n_queries x *out_rows, exactly as the filter computes it, plus the per-query flag
// (1 = the filter does not answer this query: it goes to the exact scan). INNR_EUNSUPPORTED when the corpus cannot take
// the filter path (alpha / 255 not finite and positive, d > 8192, no memory).
extern "C" int innr_cuda_u8_tc_debug_bounds(const innr_cuda_corpus* c, const float* queries, size_t n_queries, size_t query_len,
                                            float* out_lower, float* out_upper, size_t* out_rows, uint32_t* out_qflags) {
  if (!c || c->kind != 2) return fail(INNR_EINVAL, "need a u8 corpus");
  if (query_len != c->d) return fail(INNR_EINVAL, "asymmetric_dot_u8_precomputed: dimension mismatch");
  if (!queries || !out_lower || !out_upper || !out_rows || !out_qflags || n_queries == 0) return fail(INNR_EINVAL, "null argument");
  if (n_queries > 1024) return fail(INNR_EINVAL, "at most 1024 queries per call");
  if (!u8_tc_supported(u8_view(c), n_queries, 1)) return fail(INNR_EUNSUPPORTED, "corpus cannot take the u8 filter path");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  rc = u8_tc_prepare(const_cast<innr_cuda_corpus*>(c), ctx->stream);
  if (rc) return rc;
  if (c->tc_state != 1) return fail(INNR_EUNSUPPORTED, "corpus cannot take the u8 filter path (no memory)");
  CU(ctx->d_query.reserve((n_queries * c->d + 4) * sizeof(float)));
  CU(ctx->d_tcws.reserve(u8_tc_workspace_bytes(c->d, n_queries, true)));
  CU(cudaMemcpyAsync(ctx->d_query.p, queries, n_queries * c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(launch_u8_tc_debug_bounds(u8_view(c), c->dev_radius, (const float*)ctx->d_query.p, n_queries, ctx->d_tcws.p, out_lower,
                               out_upper, out_rows, out_qflags, ctx->ws.num_sms, ctx->stream, &g_launches));
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ ternary codes
static int alloc_ternary(DeviceCtx& ctx, size_t n, size_t dim, uint64_t index_base, innr_cuda_corpus** out) {
  int rc = check_index_range(n, index_base);
  if (rc) return rc;
  rc = new_corpus(4, ctx.device, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  c->n = n;
  c->dim_bits = dim;  // dimension (values)
  c->d = dim;
  c->words = (dim + 31) / 32;
  c->chunks = (c->words + 1) / 2;
  c->ld = round_up(n, 16);
  c->index_base = index_base;
  c->bytes = c->chunks * c->ld * sizeof(uint4);
  if (c->bytes) {
    cudaError_t e = cudaMalloc(&c->dev, c->bytes);
    if (e != cudaSuccess) {
      delete c;
      *out = nullptr;
      return cuda_fail(e, "cudaMalloc(ternary corpus)");
    }
  }
  guard.ok = true;
  return INNR_OK;
}
static TerView ter_view(const innr_cuda_corpus* c) {
  return TerView{(const uint4*)c->dev, c->n, c->ld, c->words, c->chunks, c->d, (uint32_t)c->index_base};
}

int innr_cuda_upload_ternary(const uint64_t* words, size_t n, size_t dimension, uint64_t index_base,
                             innr_cuda_corpus** out) {
  if (!out) return fail(INNR_EINVAL, "null out");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = alloc_ternary(*ctx, n, dimension, index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    if (!words) return fail(INNR_EINVAL, "null words");
    void* stage = nullptr;
    CU(cudaMalloc(&stage, n * c->words * sizeof(uint64_t)));
    cudaError_t e = cudaMemcpyAsync(stage, words, n * c->words * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream);
    if (e == cudaSuccess)
      e = launch_ternary_pack((const uint64_t*)stage, n, c->words, dimension, (uint4*)c->dev, c->ld, ctx->stream, &g_launches);
    if (e == cudaSuccess) e = cudaStreamSynchronize(ctx->stream);
    cudaFree(stage);
    if (e != cudaSuccess) return cuda_fail(e, "upload_ternary");
  }
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_ternary_from_f32(const innr_cuda_corpus* f32_corpus, float threshold, innr_cuda_corpus** out) {
  if (!out || !f32_corpus || f32_corpus->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  EntryGuard lk(f32_corpus->device);
  DeviceCtx* ctx;
  int rc = ctx_for(f32_corpus, &ctx);
  if (rc) return rc;
  rc = alloc_ternary(*ctx, f32_corpus->n, f32_corpus->d, f32_corpus->index_base, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  if (c->bytes) {
    CU(launch_ternary_from_pdx(pdx_view(f32_corpus), threshold,
                               (uint4*)c->dev, c->ld, ctx->stream, &g_launches));
    CU(cudaStreamSynchronize(ctx->stream));
  }
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_encode_ternary(const float* values, size_t n, float threshold, uint64_t* out_words) {
  if (n == 0) return INNR_OK;
  if (!values || !out_words) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  const size_t n_words = (n + 31) / 32;
  CU(ctx->d_scores.reserve(n * sizeof(float)));
  CU(ctx->d_aux.reserve(n_words * sizeof(uint64_t)));
  CU(cudaMemcpyAsync(ctx->d_scores.p, values, n * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  CU(launch_encode_ternary((const float*)ctx->d_scores.p, n, threshold, (uint64_t*)ctx->d_aux.p, ctx->stream, &g_launches));
  CU(cudaMemcpyAsync(out_words, ctx->d_aux.p, n_words * sizeof(uint64_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  return INNR_OK;
}

// op 0: ternary_dot (query = packed words), 1: ternary_hamming (packed words), 2: ternary::asymmetric_dot (f32 query).
// Stages the query, runs the scan into d_scores (f32) and optionally d_aux (i32).
static int ternary_scores_dev(const innr_cuda_corpus* c, DeviceCtx* ctx, int op, const void* query, size_t query_dim,
                              bool want_i32, bool stage_only = false) {
  if (op < 0 || op > 2) return fail(INNR_EINVAL, "unknown ternary op");
  if (query_dim != c->d)  // src/ternary.rs:192-196 / :287 assert_eq!
    return fail(INNR_EINVAL, op == 0 ? "innr::ternary_dot: dimension mismatch" : "dimension mismatch");
  CU(ctx->d_scores.reserve(c->n * sizeof(float)));
  if (want_i32) CU(ctx->d_aux.reserve(c->n * sizeof(int32_t)));
  if (op == 2) {
    CU(ctx->d_query.reserve((c->d + 4) * sizeof(float)));
    CU(cudaMemcpyAsync(ctx->d_query.p, query, c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  } else {
    const size_t padded = 2 * c->chunks;  // words, zero padded to whole chunks
    CU(ctx->d_query.reserve(padded * sizeof(uint64_t)));
    CU(cudaMemsetAsync(ctx->d_query.p, 0, padded * sizeof(uint64_t), ctx->stream));
    std::vector<uint64_t> w((const uint64_t*)query, (const uint64_t*)query + c->words);
    const size_t rem = c->d % 32;
    if (rem && !w.empty()) w.back() &= (1ull << (rem * 2)) - 1;  // PackedTernary::new masks the query's padding too
    CU(cudaMemcpyAsync(ctx->d_query.p, w.data(), c->words * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
    CU(cudaStreamSynchronize(ctx->stream));  // w is a stack-owned staging copy
  }
  if (stage_only) return INNR_OK;
  CU(launch_ternary_scores(ter_view(c), op, (const uint64_t*)ctx->d_query.p, (const float*)ctx->d_query.p,
                           (float*)ctx->d_scores.p, want_i32 ? (int32_t*)ctx->d_aux.p : nullptr, ctx->stream, &g_launches));
  return INNR_OK;
}

int innr_cuda_ternary_scores_all(const innr_cuda_corpus* c, int op, const void* query, size_t query_dim,
                                 float* out_f32_host, int32_t* out_i32_host) {
  if (!c || c->kind != 4) return fail(INNR_EINVAL, "need a ternary corpus");
  if (c->n == 0) return INNR_OK;
  if ((!out_f32_host && !out_i32_host) || (!query && c->d)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  if (c->d == 0) {  // no dimensions: every score is 0
    if (query_dim != 0) return fail(INNR_EINVAL, "dimension mismatch");
    for (size_t i = 0; i < c->n; ++i) {
      if (out_f32_host) out_f32_host[i] = 0.0f;
      if (out_i32_host) out_i32_host[i] = 0;
    }
    return INNR_OK;
  }
  Timed tm(*ctx);
  rc = ternary_scores_dev(c, ctx, op, query, query_dim, out_i32_host != nullptr && op != 2);
  if (rc) return rc;
  tm.stop();
  if (out_f32_host) CU(cudaMemcpyAsync(out_f32_host, ctx->d_scores.p, c->n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  if (out_i32_host && op != 2)
    CU(cudaMemcpyAsync(out_i32_host, ctx->d_aux.p, c->n * sizeof(int32_t), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  tm.finish();
  return INNR_OK;
}

// top-k over the ternary scores: dot / asymmetric dot descending, Hamming ascending; ties -> lower index (stable sort)
int innr_cuda_ternary_topk(const innr_cuda_corpus* c, int op, const void* query, size_t query_dim, size_t k,
                           uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 4) return fail(INNR_EINVAL, "need a ternary corpus");
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0) return INNR_OK;
  if (!out_idx || !out_score || (!query && c->d)) return fail(INNR_EINVAL, "null argument");
  if (c->d == 0) return fail(INNR_EUNSUPPORTED, "zero-dimensional ternary corpus");
  const size_t kk = k < c->n ? k : c->n;
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  CU(ctx->d_keys.reserve(kk * sizeof(uint64_t)));
  Timed tm(*ctx);
  const size_t q_bytes = op == 2 ? c->chunks * 64 * sizeof(float) : c->chunks * sizeof(uint4);
  if (kk <= MAX_FUSED_K && q_bytes + 8 * kk * sizeof(uint64_t) <= 200 * 1024) {
    // one pass: query staged, scan with the selection fused in (same keys as the two-step route below)
    rc = ternary_scores_dev(c, ctx, op, query, query_dim, false, true);
    if (rc) return rc;
    CU(launch_ternary_topk(ter_view(c), op, (const uint64_t*)ctx->d_query.p, (const float*)ctx->d_query.p, kk,
                           (uint64_t*)ctx->d_keys.p, ctx->ws, ctx->stream, &g_launches));
  } else {
    rc = ternary_scores_dev(c, ctx, op, query, query_dim, false);
    if (rc) return rc;
    CU(launch_topk_from_scores(ctx->d_scores.p, op == 1 ? 0 : 1, c->n, (uint32_t)c->index_base, kk, (uint64_t*)ctx->d_keys.p,
                               ctx->ws, ctx->stream, &g_launches));
  }
  tm.stop();
  rc = fetch_keys(*ctx, 1, kk, tm, [&](const uint64_t* keys) { decode_keys_f32(keys, kk, op != 1, out_idx, out_score); });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ MaxSim
int innr_cuda_upload_tokens(const float* tokens, const uint64_t* doc_offsets, size_t n_docs, size_t dim,
                            uint64_t index_base, innr_cuda_corpus** out) {
  if (!out || (n_docs && !doc_offsets)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  size_t total = n_docs ? (size_t)doc_offsets[n_docs] : 0;
  if (n_docs && doc_offsets[0] != 0) return fail(INNR_EINVAL, "doc_offsets[0] must be 0");
  for (size_t j = 0; j < n_docs; ++j)
    if (doc_offsets[j + 1] < doc_offsets[j]) return fail(INNR_EINVAL, "doc_offsets must be non-decreasing");
  if (total * dim && !tokens) return fail(INNR_EINVAL, "null tokens");
  rc = new_corpus(3, ctx->device, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  c->n = n_docs;
  c->d = dim;
  c->index_base = index_base;
  c->total_tokens = total;
  c->bytes = total * dim * sizeof(float);
  if (c->bytes) {
    CU(cudaMalloc(&c->dev, c->bytes));
    CU(cudaMemcpyAsync(c->dev, tokens, c->bytes, cudaMemcpyHostToDevice, ctx->stream));
    c->tmap_valid = make_token_tmap(&c->tmap, (const float*)c->dev, total, dim);
    if (c->tmap_valid) {  // token-norm cache of the tcgen05 path (SURVEY 8e: lives with its shard)
      CU(cudaMalloc((void**)&c->dev_norms, total * sizeof(float)));
      CU(launch_token_inv_norms((const float*)c->dev, total, dim, c->dev_norms, ctx->stream, &g_launches));
    }
  }
  if (n_docs) {
    CU(cudaMalloc(&c->dev_offsets, (n_docs + 1) * sizeof(uint64_t)));
    CU(cudaMemcpyAsync(c->dev_offsets, doc_offsets, (n_docs + 1) * sizeof(uint64_t), cudaMemcpyHostToDevice, ctx->stream));
  }
  CU(cudaStreamSynchronize(ctx->stream));
  guard.ok = true;
  return INNR_OK;
}

int innr_cuda_generate_tokens(uint64_t salt, uint64_t first_doc, size_t n_docs, size_t tokens_per_doc, size_t dim,
                              uint64_t index_base, innr_cuda_corpus** out) {
  if (!out) return fail(INNR_EINVAL, "null out");
  EntryGuard lk(cur_dev());
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  rc = new_corpus(3, ctx->device, out);
  if (rc) return rc;
  innr_cuda_corpus* c = *out;
  CorpusGuard guard(out);
  c->n = n_docs;
  c->d = dim;
  c->index_base = index_base;
  c->total_tokens = n_docs * tokens_per_doc;
  c->uniform_tokens = tokens_per_doc;
  c->bytes = c->total_tokens * dim * sizeof(float);
  if (c->bytes) {
    CU(cudaMalloc(&c->dev, c->bytes));
    CU(launch_generate_tokens(salt, first_doc * tokens_per_doc, c->total_tokens, dim, (float*)c->dev, ctx->stream, &g_launches));
    c->tmap_valid = make_token_tmap(&c->tmap, (const float*)c->dev, c->total_tokens, dim);
    if (c->tmap_valid) {
      CU(cudaMalloc((void**)&c->dev_norms, c->total_tokens * sizeof(float)));
      CU(launch_token_inv_norms((const float*)c->dev, c->total_tokens, dim, c->dev_norms, ctx->stream, &g_launches));
    }
    CU(cudaStreamSynchronize(ctx->stream));
  }
  guard.ok = true;
  return INNR_OK;
}

static int maxsim_common(const innr_cuda_corpus* c, DeviceCtx* ctx, const float* dev_q, size_t n_q, int cosine,
                         float* dev_scores, cudaStream_t s) {
  if (n_q == 0 || c->total_tokens == 0 || c->d == 0) {
    // empty query or all-empty docs -> 0.0 (src/maxsim.rs:97-99); zero-dim tokens dot to 0.0 as well
    if (c->n) CU(cudaMemsetAsync(dev_scores, 0, c->n * sizeof(float), s));
    return INNR_OK;
  }
  // tcgen05/TMEM path when the shape fits (dim <= 128, a multiple of 4; query tokens in groups of 32); option "maxsim_tc" = 0 forces the CUDA-core kernel
  TokView tv = tok_view(c);
  cudaError_t e = (g_opt.maxsim_tc && maxsim_tc_supported(tv, n_q))
                      ? launch_maxsim_tc(tv, dev_q, n_q, cosine, dev_scores, ctx->ws.num_sms, s, &g_launches)
                      : launch_maxsim(tv, dev_q, n_q, cosine, dev_scores, s, &g_launches);
  if (e == cudaErrorInvalidValue) return fail(INNR_EUNSUPPORTED, "maxsim: dim / n_q exceed the shared-memory tile");
  if (e != cudaSuccess) return cuda_fail(e, "launch_maxsim");
  (void)ctx;
  return INNR_OK;
}

int innr_cuda_maxsim(const innr_cuda_corpus* c, const float* q_tokens, size_t n_q, size_t q_dim, int cosine_flag,
                     float* out_scores_host) {
  if (!c || c->kind != 3) return fail(INNR_EINVAL, "need a token corpus");
  if (n_q && c->total_tokens && q_dim != c->d) return fail(INNR_EINVAL, "dimension mismatch (doc)");  // src/maxsim.rs:107-110
  if (c->n == 0) return INNR_OK;
  if (!out_scores_host || (n_q * q_dim && !q_tokens)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  CU(ctx->d_query.reserve((n_q * c->d + 4) * sizeof(float)));
  CU(ctx->d_scores.reserve(c->n * sizeof(float)));
  if (n_q * c->d && c->total_tokens)
    CU(cudaMemcpyAsync(ctx->d_query.p, q_tokens, n_q * c->d * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  rc = maxsim_common(c, ctx, (const float*)ctx->d_query.p, n_q, cosine_flag, (float*)ctx->d_scores.p, ctx->stream);
  if (rc) return rc;
  tm.stop();
  CU(cudaMemcpyAsync(out_scores_host, ctx->d_scores.p, c->n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  tm.finish();
  return INNR_OK;
}

// A batch of queries against the document set (the caller loop of examples/maxsim_colbert.rs:171-174 over several
// queries): q_tokens is n_queries x n_q x dim, scores n_queries x n_docs. On the tcgen05 path two queries of <= 32 tokens
// share every corpus pass; other shapes run query by query.
static int maxsim_batch_common(const innr_cuda_corpus* c, DeviceCtx* ctx, const float* dev_q, size_t n_queries, size_t n_q,
                               int cosine, float* dev_scores, cudaStream_t s) {
  TokView tv = tok_view(c);
  if (n_q >= 1 && n_q <= 32 && c->total_tokens && c->d && g_opt.maxsim_tc && maxsim_tc_supported(tv, n_q)) {
    cudaError_t e = launch_maxsim_tc_batch(tv, dev_q, n_queries, n_q, cosine, dev_scores, ctx->ws.num_sms, s, &g_launches);
    if (e != cudaSuccess) return cuda_fail(e, "launch_maxsim_tc_batch");
    return INNR_OK;
  }
  for (size_t i = 0; i < n_queries; ++i) {
    int rc = maxsim_common(c, ctx, dev_q + i * n_q * c->d, n_q, cosine, dev_scores + i * c->n, s);
    if (rc) return rc;
  }
  return INNR_OK;
}

int innr_cuda_maxsim_batch(const innr_cuda_corpus* c, const float* q_tokens, size_t n_queries, size_t n_q, size_t q_dim,
                           int cosine_flag, float* out_scores_host) {
  if (!c || c->kind != 3) return fail(INNR_EINVAL, "need a token corpus");
  if (n_q && c->total_tokens && q_dim != c->d) return fail(INNR_EINVAL, "dimension mismatch (doc)");  // src/maxsim.rs:107-110
  if (c->n == 0 || n_queries == 0) return INNR_OK;
  if (!out_scores_host || (n_q * q_dim && !q_tokens)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  const size_t qfloats = n_queries * n_q * c->d;
  CU(ctx->d_query.reserve((qfloats + 4) * sizeof(float)));
  CU(ctx->d_scores.reserve(n_queries * c->n * sizeof(float)));
  if (qfloats && c->total_tokens)
    CU(cudaMemcpyAsync(ctx->d_query.p, q_tokens, qfloats * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  rc = maxsim_batch_common(c, ctx, (const float*)ctx->d_query.p, n_queries, n_q, cosine_flag, (float*)ctx->d_scores.p,
                           ctx->stream);
  if (rc) return rc;
  tm.stop();
  CU(cudaMemcpyAsync(out_scores_host, ctx->d_scores.p, n_queries * c->n * sizeof(float), cudaMemcpyDeviceToHost, ctx->stream));
  CU(cudaStreamSynchronize(ctx->stream));
  tm.finish();
  return INNR_OK;
}

int innr_cuda_maxsim_batch_dev(const innr_cuda_corpus* c, const float* dev_q_tokens, size_t n_queries, size_t n_q,
                               int cosine_flag, float* dev_scores, void* stream) {
  if (!c || c->kind != 3) return fail(INNR_EINVAL, "need a token corpus");
  if (c->n == 0 || n_queries == 0) return INNR_OK;
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for_dev(c, &ctx, (cudaStream_t)stream);
  if (rc) return rc;
  DevRelease rel(*ctx, (cudaStream_t)stream);
  return maxsim_batch_common(c, ctx, dev_q_tokens, n_queries, n_q, cosine_flag, dev_scores, (cudaStream_t)stream);
}

int innr_cuda_maxsim_dev(const innr_cuda_corpus* c, const float* dev_q_tokens, size_t n_q, int cosine_flag,
                         float* dev_scores, void* stream) {
  if (!c || c->kind != 3) return fail(INNR_EINVAL, "need a token corpus");
  if (c->n == 0) return INNR_OK;
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for_dev(c, &ctx, (cudaStream_t)stream);
  if (rc) return rc;
  DevRelease rel(*ctx, (cudaStream_t)stream);
  return maxsim_common(c, ctx, dev_q_tokens, n_q, cosine_flag, dev_scores, (cudaStream_t)stream);
}

// MaxSim top-k: the score vectors of a chunk of queries (maxsim_batch_common: pairs of <= 32-token queries still share
// a corpus pass), then one selection per query over its vector (launch_topk_from_scores kind 1: descending under
// total_cmp, ties -> lower index, rounds of 128 for any k). The keys are those of a stable descending sort of
// innr_cuda_maxsim's output. The scratch holds one chunk, so it is bounded by MAXSIM_TOPK_SCRATCH (or two score vectors)
// whatever the batch size.
constexpr size_t MAXSIM_TOPK_SCRATCH = 64ull << 20;
static size_t maxsim_topk_chunk(const innr_cuda_corpus* c, size_t nq) {
  size_t rows = MAXSIM_TOPK_SCRATCH / (c->n * sizeof(float));
  rows = rows < 2 ? 2 : rows & ~(size_t)1;  // even: a chunk boundary never splits a pair
  return rows < nq ? rows : nq;
}
// Writes min(k, n) keys per query at row stride k, the rest of each row sentinel-padded; dev_scores holds
// maxsim_topk_chunk(c, nq) * n floats. Needs c->n > 0 and lane 0 of ctx (launch_topk_from_scores uses ctx->ws).
static int maxsim_topk_keys(const innr_cuda_corpus* c, DeviceCtx* ctx, const float* dev_q, size_t nq, size_t n_q, int cosine,
                            size_t k, uint64_t* dev_keys, float* dev_scores, cudaStream_t s) {
  const size_t kk = k < c->n ? k : c->n;
  if (kk < k) CU(cudaMemsetAsync(dev_keys, 0xFF, nq * k * sizeof(uint64_t), s));
  const size_t chunk = maxsim_topk_chunk(c, nq);
  for (size_t q0 = 0; q0 < nq; q0 += chunk) {
    const size_t m = nq - q0 < chunk ? nq - q0 : chunk;
    int rc = maxsim_batch_common(c, ctx, dev_q + q0 * n_q * c->d, m, n_q, cosine, dev_scores, s);
    if (rc) return rc;
    for (size_t j = 0; j < m; ++j) {
      rc = big_k_from_scores(ctx, dev_scores + j * c->n, 1, c->n, c->index_base, kk, dev_keys + (q0 + j) * k, s);
      if (rc) return rc;
    }
  }
  return INNR_OK;
}

int innr_cuda_maxsim_topk(const innr_cuda_corpus* c, const float* q_tokens, size_t n_queries, size_t n_q, size_t q_dim,
                          int cosine_flag, size_t k, uint64_t* out_idx, float* out_score, size_t* out_count) {
  if (!c || c->kind != 3) return fail(INNR_EINVAL, "need a token corpus");
  if (n_q && c->total_tokens && q_dim != c->d) return fail(INNR_EINVAL, "dimension mismatch (doc)");  // src/maxsim.rs:107-110
  if (out_count) *out_count = 0;
  if (c->n == 0 || k == 0 || n_queries == 0) return INNR_OK;
  if (!out_idx || !out_score || (n_q * q_dim && !q_tokens)) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < c->n ? k : c->n;
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  int rc = ctx_for(c, &ctx);
  if (rc) return rc;
  const size_t qfloats = n_queries * n_q * c->d;
  CU(ctx->d_query.reserve((qfloats + 4) * sizeof(float)));
  CU(ctx->d_keys.reserve(n_queries * kk * sizeof(uint64_t)));
  CU(ctx->d_scores.reserve(maxsim_topk_chunk(c, n_queries) * c->n * sizeof(float)));
  if (qfloats && c->total_tokens)
    CU(cudaMemcpyAsync(ctx->d_query.p, q_tokens, qfloats * sizeof(float), cudaMemcpyHostToDevice, ctx->stream));
  Timed tm(*ctx);
  rc = maxsim_topk_keys(c, ctx, (const float*)ctx->d_query.p, n_queries, n_q, cosine_flag, kk, (uint64_t*)ctx->d_keys.p,
                        (float*)ctx->d_scores.p, ctx->stream);
  if (rc) return rc;
  tm.stop();
  rc = fetch_keys(*ctx, n_queries, kk, tm, [&](const uint64_t* keys) {
    for (size_t q = 0; q < n_queries; ++q) decode_keys_f32(keys + q * kk, kk, true, out_idx + q * k, out_score + q * k);
  });
  if (rc) return rc;
  if (out_count) *out_count = kk;
  return INNR_OK;
}

int innr_cuda_maxsim_topk_keys_dev(const innr_cuda_corpus* c, const float* dev_q_tokens, size_t n_queries, size_t n_q,
                                   int cosine_flag, size_t k, uint64_t* dev_keys, void* stream) {
  if (!c || c->kind != 3) return fail(INNR_EINVAL, "need a token corpus");
  if (k == 0 || n_queries == 0) return INNR_OK;
  if (!dev_keys || (n_q * c->d && c->total_tokens && !dev_q_tokens)) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(c->device);
  cudaStream_t s = (cudaStream_t)stream;
  DeviceCtx* ctx;
  int rc = ctx_for_dev(c, &ctx, s);  // lane 0: the score vectors live in the device's scratch
  if (rc) return rc;
  DevRelease rel(*ctx, s);
  if (c->n == 0) {
    CU(cudaMemsetAsync(dev_keys, 0xFF, n_queries * k * sizeof(uint64_t), s));
    return INNR_OK;
  }
  CU(ctx->d_scores.reserve(maxsim_topk_chunk(c, n_queries) * c->n * sizeof(float)));
  return maxsim_topk_keys(c, ctx, dev_q_tokens, n_queries, n_q, cosine_flag, k, dev_keys, (float*)ctx->d_scores.p, s);
}

// ------------------------------------------------------------------------------------------ asynchronous host-buffer calls
// The host-facing top-k entries synchronise before they return, so a caller with one query per call pays the ramp at
// both ends of every launch and leaves the GPU idle while it decodes. The _async forms queue the same work (query
// staged through pinned memory, shard scan on one of the device's two lanes, keys back into pinned memory) on a stream
// of their own and return a ticket; innr_cuda_ticket_wait blocks on that call only. Two tickets per device can be in
// flight: submit(i + 1) before wait(i) keeps two scans overlapping on the device (DESIGN.md section 6).
static int grow(void** p, size_t* cap, size_t bytes, bool pinned) {
  if (bytes <= *cap) return INNR_OK;
  if (*p) {
    if (pinned) cudaFreeHost(*p); else cudaFree(*p);
    *p = nullptr;
    *cap = 0;
  }
  const size_t want = bytes < 4096 ? 4096 : bytes + bytes / 4;
  CU(pinned ? cudaMallocHost(p, want) : cudaMalloc(p, want));
  *cap = want;
  return INNR_OK;
}
// picks a free ticket of the corpus' device (the caller holds the device mutex) and sizes its buffers
static int async_begin(const innr_cuda_corpus* c, DeviceCtx** ctx_out, innr_cuda_ticket** out, size_t query_bytes,
                       size_t nq, size_t k, size_t kk) {
  DeviceCtx* ctx;
  int rc = ensure_ctx(c->device, &ctx, WS_NONE);
  if (rc) return rc;
  innr_cuda_ticket* t = nullptr;
  for (unsigned j = 0; j < 2 && !t; ++j) {
    innr_cuda_ticket& cand = ctx->async_slot[(ctx->async_next + j) & 1];
    if (!cand.in_flight) t = &cand;
  }
  if (!t) return fail(INNR_EBUSY, "two asynchronous calls are already in flight on this device: wait for a ticket first");
  ctx->async_next = (unsigned)((t - ctx->async_slot) + 1) & 1;
  if (!t->stream) {
    CU(cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking));
    // spin-wait unless asked otherwise: a blocking wait puts the host thread to sleep and adds its wake-up latency
    // (tens of microseconds) to every short call
    static const bool blocking = getenv("INNR_ASYNC_BLOCKING_WAIT") != nullptr;
    CU(cudaEventCreateWithFlags(&t->done, cudaEventDisableTiming | (blocking ? cudaEventBlockingSync : 0)));
  }
  t->device = c->device;
  t->kind = c->kind;
  t->nq = nq;
  t->k = k;
  t->kk = kk;
  t->sharded = false;  // the slot may have served a sharded call before
  t->n_siblings = 0;
  t->group_busy = nullptr;
  if ((rc = grow(&t->h_in, &t->h_in_cap, query_bytes, true))) return rc;
  if ((rc = grow(&t->d_query, &t->d_query_cap, query_bytes + 16, false))) return rc;
  if ((rc = grow(&t->d_keys, &t->d_keys_cap, nq * kk * sizeof(uint64_t), false))) return rc;
  if ((rc = grow(&t->h_out, &t->h_out_cap, nq * kk * sizeof(uint64_t), true))) return rc;
  *ctx_out = ctx;
  *out = t;
  return INNR_OK;
}
// keys -> pinned memory, completion event; the ticket is in flight from here on
static int async_finish(innr_cuda_ticket* t) {
  if (t->nq * t->kk)
    CU(cudaMemcpyAsync(t->h_out, t->d_keys, t->nq * t->kk * sizeof(uint64_t), cudaMemcpyDeviceToHost, t->stream));
  CU(cudaEventRecord(t->done, t->stream));
  t->in_flight = true;
  return INNR_OK;
}

int innr_cuda_batch_knn_async(const innr_cuda_corpus* c, int metric, const float* queries, size_t n_queries,
                              size_t query_len, size_t k, innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  if (!c || c->kind != 0) return fail(INNR_EINVAL, "need an f32 PDX corpus");
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  if (query_len != c->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");  // src/batch.rs:386,743,778
  const bool empty = c->n == 0 || k == 0 || n_queries == 0;                            // src/batch.rs:388-393
  if (!empty && !queries && c->d) return fail(INNR_EINVAL, "null argument");
  const size_t kk = empty ? 0 : (k < c->n ? k : c->n);
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  innr_cuda_ticket* t;
  const size_t qbytes = empty ? 0 : n_queries * c->d * sizeof(float);
  rc = async_begin(c, &ctx, &t, qbytes, n_queries, k, kk);
  if (rc) return rc;
  t->metric = metric;
  if (!empty) {
    if (qbytes) {
      std::memcpy(t->h_in, queries, qbytes);
      CU(cudaMemcpyAsync(t->d_query, t->h_in, qbytes, cudaMemcpyHostToDevice, t->stream));
    }
    int lane = 0;
    rc = ensure_ctx(c->device, &ctx, knn_is_scan_only(c, mode, n_queries, kk) ? WS_DEV_SCAN : WS_DEV, t->stream, &lane);
    if (rc) return rc;
    DevRelease rel(*ctx, t->stream, lane);
    rc = knn_keys_dev(const_cast<innr_cuda_corpus*>(c), ctx, mode, (const float*)t->d_query, n_queries, kk,
                      (uint64_t*)t->d_keys, t->stream, lane);
    if (rc) return rc;
  }
  rc = async_finish(t);
  if (rc) return rc;
  *out_ticket = t;
  return INNR_OK;
}

int innr_cuda_hamming_topk_async(const innr_cuda_corpus* c, const uint64_t* query_words, size_t n_queries,
                                 size_t query_dim_bits, size_t k, innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  if (!c || c->kind != 1) return fail(INNR_EINVAL, "need a binary corpus");
  if (query_dim_bits != c->dim_bits) return fail(INNR_EINVAL, "innr::binary_hamming: dimension mismatch");
  const bool empty = c->n == 0 || k == 0 || n_queries == 0;
  if (!empty && c->words == 0) return fail(INNR_EUNSUPPORTED, "zero-dimensional codes: use innr_cuda_hamming_topk");
  if (!empty && !query_words) return fail(INNR_EINVAL, "null argument");
  const size_t kk = empty ? 0 : (k < c->n ? k : c->n);
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  innr_cuda_ticket* t;
  const size_t qw = 2 * c->chunks;
  const size_t qbytes = empty ? 0 : n_queries * qw * sizeof(uint64_t);
  int rc = async_begin(c, &ctx, &t, qbytes, n_queries, k, kk);
  if (rc) return rc;
  if (!empty) {
    uint64_t* h = (uint64_t*)t->h_in;
    const size_t rem = c->dim_bits % 64;
    for (size_t q = 0; q < n_queries; ++q)
      for (size_t w = 0; w < qw; ++w) {
        uint64_t x = w < c->words ? query_words[q * c->words + w] : 0;
        if (w + 1 == c->words && rem) x &= (1ull << rem) - 1;  // PackedBinary::new masks padding
        h[q * qw + w] = x;
      }
    CU(cudaMemcpyAsync(t->d_query, t->h_in, qbytes, cudaMemcpyHostToDevice, t->stream));
    int lane = 0;
    rc = ensure_ctx(c->device, &ctx, hamming_is_scan_only(c, n_queries, kk) ? WS_DEV_SCAN : WS_DEV, t->stream, &lane);
    if (rc) return rc;
    DevRelease rel(*ctx, t->stream, lane);
    rc = hamming_keys(c, ctx, (const uint64_t*)t->d_query, n_queries, kk, (uint64_t*)t->d_keys, t->stream, lane);
    if (rc) return rc;
  }
  rc = async_finish(t);
  if (rc) return rc;
  *out_ticket = t;
  return INNR_OK;
}

int innr_cuda_batch_knn_u8_async(const innr_cuda_corpus* c, const float* queries, size_t n_queries, size_t query_len,
                                 size_t k, innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  if (!c || c->kind != 2) return fail(INNR_EINVAL, "need a u8 corpus");
  const bool empty = c->n == 0 || k == 0 || n_queries == 0;  // src/scalar.rs:376-378 (before any length check)
  if (!empty && query_len != c->d) return fail(INNR_EINVAL, "asymmetric_dot_u8_precomputed: dimension mismatch");
  if (!empty && c->d == 0) return fail(INNR_EUNSUPPORTED, "zero-dimensional u8 corpus");
  if (!empty && !queries) return fail(INNR_EINVAL, "null argument");
  const size_t kk = empty ? 0 : (k < c->n ? k : c->n);
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  innr_cuda_ticket* t;
  const size_t qbytes = empty ? 0 : n_queries * c->d * sizeof(float);
  int rc = async_begin(c, &ctx, &t, qbytes, n_queries, k, kk);
  if (rc) return rc;
  if (!empty) {
    std::memcpy(t->h_in, queries, qbytes);
    CU(cudaMemcpyAsync(t->d_query, t->h_in, qbytes, cudaMemcpyHostToDevice, t->stream));
    int lane = 0;
    rc = ensure_ctx(c->device, &ctx, u8_is_scan_only(c, n_queries, kk) ? WS_DEV_SCAN : WS_DEV, t->stream, &lane);
    if (rc) return rc;
    DevRelease rel(*ctx, t->stream, lane);
    rc = u8_keys(c, ctx, (const float*)t->d_query, n_queries, kk, (uint64_t*)t->d_keys, t->stream, lane);
    if (rc) return rc;
  }
  rc = async_finish(t);
  if (rc) return rc;
  *out_ticket = t;
  return INNR_OK;
}

int innr_cuda_maxsim_topk_async(const innr_cuda_corpus* c, const float* q_tokens, size_t n_queries, size_t n_q,
                                size_t q_dim, int cosine_flag, size_t k, innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  if (!c || c->kind != 3) return fail(INNR_EINVAL, "need a token corpus");
  if (n_q && c->total_tokens && q_dim != c->d) return fail(INNR_EINVAL, "dimension mismatch (doc)");  // src/maxsim.rs:107-110
  const bool empty = c->n == 0 || k == 0 || n_queries == 0;
  if (!empty && n_q * q_dim && !q_tokens) return fail(INNR_EINVAL, "null argument");
  const size_t kk = empty ? 0 : (k < c->n ? k : c->n);
  EntryGuard lk(c->device);
  DeviceCtx* ctx;
  innr_cuda_ticket* t;
  const size_t qbytes = (empty || !c->total_tokens) ? 0 : n_queries * n_q * c->d * sizeof(float);
  int rc = async_begin(c, &ctx, &t, qbytes, n_queries, k, kk);
  if (rc) return rc;
  t->metric = INNR_METRIC_DOT;  // descending keys
  if (!empty) {
    if (qbytes) {
      std::memcpy(t->h_in, q_tokens, qbytes);
      CU(cudaMemcpyAsync(t->d_query, t->h_in, qbytes, cudaMemcpyHostToDevice, t->stream));
    }
    if ((rc = grow(&t->d_scores, &t->d_scores_cap, maxsim_topk_chunk(c, n_queries) * c->n * sizeof(float), false))) return rc;
    rc = ensure_ctx(c->device, &ctx, WS_DEV, t->stream);  // lane 0: the selection uses ctx->ws
    if (rc) return rc;
    DevRelease rel(*ctx, t->stream);
    rc = maxsim_topk_keys(c, ctx, (const float*)t->d_query, n_queries, n_q, cosine_flag, kk, (uint64_t*)t->d_keys,
                          (float*)t->d_scores, t->stream);
    if (rc) return rc;
  }
  rc = async_finish(t);
  if (rc) return rc;
  *out_ticket = t;
  return INNR_OK;
}

int innr_cuda_ticket_wait(innr_cuda_ticket* t, uint64_t* out_idx, float* out_score, uint32_t* out_dist,
                          size_t* out_count) {
  if (out_count) *out_count = 0;
  if (!t || !t->in_flight) return fail(INNR_EINVAL, "ticket is not in flight");
  if (t->kk && (!out_idx || (t->kind == 1 ? !out_dist : !out_score))) return fail(INNR_EINVAL, "null argument");
  // block on this call only, outside the device mutex: other threads keep submitting meanwhile
  cudaError_t e = cudaEventSynchronize(t->done);
  for (int j = 0; j < t->n_siblings; ++j) {  // the other devices' parts of a sharded call: long finished, release them
    innr_cuda_ticket* sib = t->siblings[j];
    cudaError_t es = cudaEventSynchronize(sib->done);
    if (e == cudaSuccess) e = es;
    EntryGuard slk(sib->device);
    sib->in_flight = false;
  }
  EntryGuard lk(t->device);
  t->in_flight = false;
  t->n_siblings = 0;
  if (t->sharded && t->group_busy) t->group_busy->fetch_sub(1);
  if (e != cudaSuccess) return cuda_fail(e, "cudaEventSynchronize(ticket)");
  const uint64_t* keys = (const uint64_t*)t->h_out;
  const size_t row = t->sharded ? t->krow : t->kk;
  if (t->sharded && t->kk && *(const unsigned*)(keys + t->nq * t->krow) != 0)
    return fail(INNR_ECUDA, "sharded call: a shard did not publish its keys within the exchange timeout");
  for (size_t q = 0; q < t->nq && t->kk; ++q) {
    if (t->kind == 1) {
      for (size_t j = 0; j < t->kk; ++j) {
        out_idx[q * t->k + j] = keys[q * row + j] & 0xFFFFFFFFull;
        out_dist[q * t->k + j] = (uint32_t)(keys[q * row + j] >> 32);
      }
    } else {
      decode_keys_f32(keys + q * row, t->kk, t->kind == 2 || t->metric != INNR_METRIC_L2, out_idx + q * t->k,
                      out_score + q * t->k);
    }
  }
  if (out_count) *out_count = t->kk;
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ peer-mapped exchange
static ExchangeView ex_view(const innr_cuda_exchange* x) {
  return ExchangeView{(uint64_t*)x->mailbox, (uint64_t* const*)x->dev_peer_table, x->n_ranks, x->rank, x->slot_keys,
                      x->dev_status, x->timeout_ns};
}

int innr_cuda_exchange_create(int n_ranks, int rank, size_t slot_keys, innr_cuda_exchange** out) {
  if (!out || n_ranks < 1 || n_ranks > 64 || rank < 0 || rank >= n_ranks) return fail(INNR_EINVAL, "exchange_create: bad rank / n_ranks");
  if (slot_keys == 0) slot_keys = 16384;
  const int device = cur_dev();
  EntryGuard lk(device);
  DeviceCtx* ctx;
  int rc = current_ctx(&ctx);
  if (rc) return rc;
  innr_cuda_exchange* x = new (std::nothrow) innr_cuda_exchange();
  if (!x) return fail(INNR_ENOMEM, "host allocation failed");
  x->device = device;
  x->n_ranks = n_ranks;
  x->rank = rank;
  x->slot_keys = slot_keys;
  x->peers.assign(n_ranks, nullptr);
  x->ipc_opened.assign(n_ranks, 0);
  const size_t bytes = exchange_mailbox_bytes(n_ranks, slot_keys);
  cudaError_t e = cudaMalloc(&x->mailbox, bytes);
  if (e == cudaSuccess) e = cudaMemset(x->mailbox, 0, bytes);
  if (e == cudaSuccess) e = cudaMalloc((void**)&x->dev_peer_table, n_ranks * sizeof(void*));
  if (e == cudaSuccess) e = cudaMalloc((void**)&x->dev_status, sizeof(unsigned));
  if (e == cudaSuccess) e = cudaMemset(x->dev_status, 0, sizeof(unsigned));
  if (e != cudaSuccess) {
    if (x->mailbox) cudaFree(x->mailbox);
    if (x->dev_peer_table) cudaFree(x->dev_peer_table);
    if (x->dev_status) cudaFree(x->dev_status);
    delete x;
    return cuda_fail(e, "exchange_create");
  }
  x->peers[rank] = x->mailbox;
  if (n_ranks == 1) {
    e = cudaMemcpy(x->dev_peer_table, x->peers.data(), sizeof(void*), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return cuda_fail(e, "exchange_create");
    x->connected = true;
  }
  *out = x;
  return INNR_OK;
}

int innr_cuda_exchange_ipc_handle(const innr_cuda_exchange* x, void* out_handle64) {
  if (!x || !out_handle64) return fail(INNR_EINVAL, "null argument");
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "cudaIpcMemHandle_t is 64 bytes");
  EntryGuard lk(x->device);
  CU(cudaSetDevice(x->device));
  cudaIpcMemHandle_t h;
  CU(cudaIpcGetMemHandle(&h, x->mailbox));
  std::memcpy(out_handle64, &h, 64);
  return INNR_OK;
}

static int exchange_finish_connect(innr_cuda_exchange* x) {
  CU(cudaSetDevice(x->device));
  CU(cudaMemcpy(x->dev_peer_table, x->peers.data(), x->n_ranks * sizeof(void*), cudaMemcpyHostToDevice));
  x->connected = true;
  return INNR_OK;
}

int innr_cuda_exchange_connect_ipc(innr_cuda_exchange* x, const void* handles) {
  if (!x || !handles) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(x->device);
  CU(cudaSetDevice(x->device));
  for (int r = 0; r < x->n_ranks; ++r) {
    if (r == x->rank || x->peers[r]) continue;
    cudaIpcMemHandle_t h;
    std::memcpy(&h, (const char*)handles + (size_t)r * 64, 64);
    void* p = nullptr;
    CU(cudaIpcOpenMemHandle(&p, h, cudaIpcMemLazyEnablePeerAccess));
    x->peers[r] = p;
    x->ipc_opened[r] = 1;
  }
  return exchange_finish_connect(x);
}

int innr_cuda_exchange_connect_local(innr_cuda_exchange* const* all, int n_ranks) {
  if (!all || n_ranks < 1) return fail(INNR_EINVAL, "null argument");
  for (int r = 0; r < n_ranks; ++r)
    if (!all[r] || all[r]->n_ranks != n_ranks || all[r]->rank != r || all[r]->slot_keys != all[0]->slot_keys)
      return fail(INNR_EINVAL, "exchange_connect_local: objects must be ranks 0..n-1 of one exchange");
  int prev = -1;
  cudaGetDevice(&prev);
  for (int r = 0; r < n_ranks; ++r) {
    innr_cuda_exchange* x = all[r];
    std::lock_guard<std::mutex> lk(dev_mu(x->device));
    cudaSetDevice(x->device);
    for (int p = 0; p < n_ranks; ++p) {
      if (all[p]->device != x->device) {
        int can = 0;
        cudaDeviceCanAccessPeer(&can, x->device, all[p]->device);
        if (!can) {
          if (prev >= 0) cudaSetDevice(prev);
          return fail(INNR_EUNSUPPORTED, "exchange_connect_local: no peer access between the devices");
        }
        cudaError_t e = cudaDeviceEnablePeerAccess(all[p]->device, 0);
        if (e != cudaSuccess && e != cudaErrorPeerAccessAlreadyEnabled) {
          if (prev >= 0) cudaSetDevice(prev);
          return cuda_fail(e, "cudaDeviceEnablePeerAccess");
        }
        cudaGetLastError();
      }
      x->peers[p] = all[p]->mailbox;
    }
    int rc = exchange_finish_connect(x);
    if (rc) {
      if (prev >= 0) cudaSetDevice(prev);
      return rc;
    }
  }
  if (prev >= 0) cudaSetDevice(prev);
  return INNR_OK;
}

int innr_cuda_exchange_free(innr_cuda_exchange* x) {
  if (!x) return INNR_OK;
  EntryGuard lk(x->device);
  cudaSetDevice(x->device);
  cudaDeviceSynchronize();
  for (int r = 0; r < x->n_ranks; ++r)
    if (x->ipc_opened[r] && x->peers[r]) cudaIpcCloseMemHandle(x->peers[r]);
  cudaFree(x->mailbox);
  cudaFree(x->dev_peer_table);
  cudaFree(x->dev_status);
  cudaGetLastError();
  delete x;
  return INNR_OK;
}

int innr_cuda_exchange_set_timeout_ms(innr_cuda_exchange* x, double ms) {
  if (!x || !(ms > 0)) return fail(INNR_EINVAL, "bad argument");
  x->timeout_ns = (uint64_t)(ms * 1e6);
  return INNR_OK;
}

int innr_cuda_exchange_status(innr_cuda_exchange* x, int* out_status) {
  if (!x || !out_status) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(x->device);
  CU(cudaSetDevice(x->device));
  unsigned v = 0;
  CU(cudaMemcpy(&v, x->dev_status, sizeof(unsigned), cudaMemcpyDeviceToHost));
  *out_status = (int)v;
  return INNR_OK;
}

int innr_cuda_exchange_merge_dev(innr_cuda_exchange* x, const uint64_t* dev_local_keys, size_t n_queries, size_t k,
                                 int metric, int publish_only, uint64_t* dev_keys_out, uint64_t* dev_idx,
                                 float* dev_score, uint32_t* dev_dist, void* stream) {
  if (!x || !x->connected) return fail(INNR_EINVAL, "exchange is not connected");
  if (k == 0 || n_queries == 0) return INNR_OK;
  if (k > MAX_FUSED_K) return fail(INNR_EUNSUPPORTED, "exchange_merge_dev: k > 128 (gather the lists and use innr_cuda_merge_keys_dev)");
  if (n_queries * k > x->slot_keys) return fail(INNR_EUNSUPPORTED, "exchange_merge_dev: n_queries * k exceeds the mailbox slot");
  if (!dev_local_keys) return fail(INNR_EINVAL, "null argument");
  EntryGuard lk(x->device);
  DeviceCtx* ctx;
  int rc = ensure_ctx(x->device, &ctx, WS_NONE, (cudaStream_t)stream);  // mailboxes only: no workspace, no scratch
  if (rc) return rc;
  ++x->calls;
  CU(launch_exchange_merge(ex_view(x), dev_local_keys, n_queries, k, x->calls, publish_only, metric != INNR_METRIC_L2,
                           dev_keys_out, dev_idx, dev_score, dev_dist, (cudaStream_t)stream, &g_launches));
  return INNR_OK;
}

// ------------------------------------------------------------------------------------------ one process, several GPUs
// Row shards on different devices, one host thread per shard (the per-device mutexes let them run concurrently), each
// computing its local top-k through the single-device entry; the k x n_shards (key, index) pairs are merged on the
// host in key order -- the same composite keys as on the device, so "lower global index wins" holds across shards.
// This is the single-process counterpart of the torch.distributed / NCCL harness (SURVEY 8e): a Rust host that owns all
// GPUs of a box needs no collective library for an exchange of k keys per device.
}  // extern "C"
namespace {
uint32_t host_order_bits(float x) {
  uint32_t b;
  std::memcpy(&b, &x, 4);
  b ^= ((uint32_t)((int32_t)b >> 31)) >> 1;
  return b ^ 0x80000000u;
}
struct ShardOut {
  std::vector<uint64_t> idx;
  std::vector<float> score;
  std::vector<uint32_t> dist;
  size_t count = 0;
  int rc = INNR_OK;
  std::string err;
};
// ---- in-process sharding over distinct devices: persistent worker threads + the peer-mapped exchange -------------
// One worker per shard stays alive between calls (thread creation costs more than an eighth-of-a-corpus scan); a call
// hands every worker one closure and waits for all of them. Workers spin briefly after a job before they block, so
// back-to-back calls find them hot.
class ShardPool {
 public:
  explicit ShardPool(size_t n) : n_(n) {
    for (size_t i = 0; i < n; ++i) th_.emplace_back([this, i] { loop(i); });
  }
  ~ShardPool() {
    {
      std::lock_guard<std::mutex> lk(m_);
      stop_ = true;
      ++gen_;
    }
    cv_.notify_all();
    for (auto& t : th_) t.join();
  }
  void run(const std::function<void(size_t)>& job) {
    job_ = &job;
    done_.store(0, std::memory_order_relaxed);
    {
      std::lock_guard<std::mutex> lk(m_);
      gen_.fetch_add(1, std::memory_order_release);
    }
    cv_.notify_all();
    while (done_.load(std::memory_order_acquire) != n_) std::this_thread::yield();
  }

 private:
  void loop(size_t i) {
    uint64_t seen = 0;
    for (;;) {
      // hot phase: poll the generation counter for a while, then block
      bool got = false;
      for (int spin = 0; spin < 20000 && !got; ++spin) got = gen_.load(std::memory_order_acquire) != seen;
      if (!got) {
        std::unique_lock<std::mutex> lk(m_);
        cv_.wait(lk, [&] { return gen_.load(std::memory_order_acquire) != seen; });
      }
      seen = gen_.load(std::memory_order_acquire);
      if (stop_) return;
      (*job_)(i);
      done_.fetch_add(1, std::memory_order_release);
    }
  }
  size_t n_;
  std::vector<std::thread> th_;
  std::mutex m_;
  std::condition_variable cv_;
  std::atomic<uint64_t> gen_{0};
  std::atomic<size_t> done_{0};
  const std::function<void(size_t)>* job_ = nullptr;
  bool stop_ = false;
};

struct ShardGroup {  // one per distinct ordered device list
  std::vector<innr_cuda_exchange*> ex;
  std::unique_ptr<ShardPool> pool;
  std::vector<Buf> pin_q, pin_out;  // per shard pinned staging (queries in, root results out)
  std::vector<Buf> d_idx, d_score;  // root outputs
  std::mutex mu;                    // one sharded call at a time per group (the exchange numbers its calls)
  // asynchronous calls: at most two in flight (one per mailbox parity); `consumed[p]` is recorded on the root's stream
  // behind its merge of the call with parity p -- the other devices wait for it before they publish into that parity again
  std::atomic<int> async_in_flight{0};
  cudaEvent_t consumed[2] = {nullptr, nullptr};
};
std::mutex g_groups_mu;
std::map<std::vector<int>, std::unique_ptr<ShardGroup>> g_groups;

void shard_groups_shutdown() {
  std::lock_guard<std::mutex> lk(g_groups_mu);
  for (auto& kv : g_groups) {
    ShardGroup* g = kv.second.get();
    if (!g) continue;
    g->pool.reset();  // joins the workers
    for (int p = 0; p < 2; ++p)
      if (g->consumed[p]) cudaEventDestroy(g->consumed[p]);
    for (size_t i = 0; i < g->ex.size(); ++i) {
      cudaSetDevice(g->ex[i]->device);
      g->pin_q[i].release();
      g->pin_out[i].release();
      g->d_idx[i].release();
      g->d_score[i].release();
      innr_cuda_exchange_free(g->ex[i]);
    }
  }
  g_groups.clear();
}

// Devices of the shards if they are pairwise distinct and a group can be (or was) set up, else nullptr (the caller
// then takes the thread-per-shard + host-merge route, which also serves several shards on one device).
ShardGroup* shard_group_for(const innr_cuda_corpus* const* shards, size_t n_shards) {
  if (n_shards < 2) return nullptr;
  std::vector<int> devs(n_shards);
  for (size_t i = 0; i < n_shards; ++i) devs[i] = shards[i]->device;
  std::vector<int> sorted_devs = devs;
  std::sort(sorted_devs.begin(), sorted_devs.end());
  if (std::adjacent_find(sorted_devs.begin(), sorted_devs.end()) != sorted_devs.end()) return nullptr;
  std::lock_guard<std::mutex> lk(g_groups_mu);
  auto it = g_groups.find(devs);
  if (it != g_groups.end()) return it->second.get();  // may hold nullptr: set-up failed once, do not retry per call
  std::unique_ptr<ShardGroup> g(new ShardGroup());
  bool ok = true;
  const int saved = t_device;
  for (size_t i = 0; i < n_shards && ok; ++i) {
    t_device = devs[i];
    innr_cuda_exchange* x = nullptr;
    ok = innr_cuda_exchange_create((int)n_shards, (int)i, 0, &x) == INNR_OK;
    if (ok) g->ex.push_back(x);
  }
  t_device = saved;
  if (ok) ok = innr_cuda_exchange_connect_local(g->ex.data(), (int)n_shards) == INNR_OK;
  if (!ok) {
    for (auto* x : g->ex) innr_cuda_exchange_free(x);
    g_groups[devs] = nullptr;
    return nullptr;
  }
  g->pool.reset(new ShardPool(n_shards));
  g->pin_q.resize(n_shards);
  g->pin_out.resize(n_shards);
  g->d_idx.resize(n_shards);
  g->d_score.resize(n_shards);
  for (size_t i = 0; i < n_shards; ++i) g->pin_q[i].pinned = g->pin_out[i].pinned = true;
  ShardGroup* raw = g.get();
  g_groups[devs] = std::move(g);
  return raw;
}

// The exchange route of the three sharded entries. `enqueue_keys(i, ctx, dev_query, dev_keys)` queues shard i's local
// top-k on ctx->stream. Shard 0's device is the root: it merges and its result travels back; the others only publish.
// Returns INNR_EUNSUPPORTED when the request does not fit the mailboxes (caller falls back).
template <class EnqueueKeys>
int sharded_via_exchange(ShardGroup* g, const innr_cuda_corpus* const* shards, size_t n_shards, const void* queries,
                         size_t query_bytes, size_t nq, size_t k, int metric, bool want_dist, EnqueueKeys enqueue_keys,
                         uint64_t* out_idx, float* out_score, uint32_t* out_dist) {
  if (k > MAX_FUSED_K || nq * k > g->ex[0]->slot_keys) return INNR_EUNSUPPORTED;
  std::lock_guard<std::mutex> call_lk(g->mu);
  if (g->async_in_flight.load()) return fail(INNR_EBUSY, "asynchronous sharded calls are in flight on these devices: wait for their tickets first");
  std::vector<int> rcs(n_shards, INNR_OK);
  std::vector<std::string> errs(n_shards);
  const size_t out_bytes = nq * k * (sizeof(uint64_t) + sizeof(uint32_t));
  std::function<void(size_t)> job = [&](size_t i) {
    auto body = [&]() -> int {
      const innr_cuda_corpus* c = shards[i];
      innr_cuda_exchange* x = g->ex[i];
      ++x->calls;  // first thing: a shard that fails below must not leave the ranks' call numbers out of step
      EntryGuard lk(c->device);
      DeviceCtx* ctx;
      int rc = ctx_for(c, &ctx);
      if (rc) return rc;
      cudaStream_t s = ctx->stream;
      // the non-root shards leave their work in flight on the device's stream: later host-facing calls are ordered behind
      // it by that stream, `_dev` calls on caller streams by the lane-0 event this records
      DevRelease rel(*ctx, s, 0);
      CU(g->pin_q[i].reserve(query_bytes));
      std::memcpy(g->pin_q[i].p, queries, query_bytes);
      CU(ctx->d_query.reserve(query_bytes + 16));
      CU(ctx->d_keys.reserve(nq * k * sizeof(uint64_t)));
      CU(cudaMemcpyAsync(ctx->d_query.p, g->pin_q[i].p, query_bytes, cudaMemcpyHostToDevice, s));
      rc = enqueue_keys(i, ctx, ctx->d_query.p, (uint64_t*)ctx->d_keys.p);
      if (rc) return rc;
      if (i != 0) {
        CU(launch_exchange_merge(ex_view(x), (const uint64_t*)ctx->d_keys.p, nq, k, x->calls, 1, 0, nullptr, nullptr, nullptr,
                                 nullptr, s, &g_launches));
        return INNR_OK;  // stays in flight on this device's stream; the root's merge is what waits for it
      }
      CU(g->d_idx[0].reserve(nq * k * sizeof(uint64_t)));
      CU(g->d_score[0].reserve(nq * k * sizeof(uint32_t)));
      CU(g->pin_out[0].reserve(out_bytes));
      CU(launch_exchange_merge(ex_view(x), (const uint64_t*)ctx->d_keys.p, nq, k, x->calls, 0, metric != INNR_METRIC_L2, nullptr,
                               (uint64_t*)g->d_idx[0].p, want_dist ? nullptr : (float*)g->d_score[0].p,
                               want_dist ? (uint32_t*)g->d_score[0].p : nullptr, s, &g_launches));
      char* h = (char*)g->pin_out[0].p;
      CU(cudaMemcpyAsync(h, g->d_idx[0].p, nq * k * sizeof(uint64_t), cudaMemcpyDeviceToHost, s));
      CU(cudaMemcpyAsync(h + nq * k * sizeof(uint64_t), g->d_score[0].p, nq * k * sizeof(uint32_t), cudaMemcpyDeviceToHost, s));
      CU(cudaStreamSynchronize(s));
      unsigned st = 0;
      CU(cudaMemcpy(&st, x->dev_status, sizeof(unsigned), cudaMemcpyDeviceToHost));
      if (st) return fail(INNR_ECUDA, "sharded call: a shard did not publish its keys within the exchange timeout");
      return INNR_OK;
    };
    rcs[i] = body();
    if (rcs[i]) errs[i] = t_err;
  };
  g->pool->run(job);
  for (size_t i = 0; i < n_shards; ++i)
    if (rcs[i]) return fail(rcs[i], "shard " + std::to_string(i) + ": " + errs[i]);
  const char* h = (const char*)g->pin_out[0].p;
  std::memcpy(out_idx, h, nq * k * sizeof(uint64_t));
  if (want_dist) std::memcpy(out_dist, h + nq * k * sizeof(uint64_t), nq * k * sizeof(uint32_t));
  else std::memcpy(out_score, h + nq * k * sizeof(uint64_t), nq * k * sizeof(float));
  return INNR_OK;
}

// Asynchronous form of the exchange route: every device queues its part on the stream of one of its two asynchronous
// slots (the slot = the mailbox parity of this call, so consecutive calls alternate and two can be in flight), the root
// keeps the merged KEYS in device memory and copies them to pinned memory behind the merge; nothing synchronises. The
// returned ticket is the root's; innr_cuda_ticket_wait releases the other devices' slots with it. `enqueue_keys(i, ctx,
// dev_query, dev_keys, stream, lane)` queues shard i's local top-k.
template <class ScanOnly, class EnqueueKeys>
int sharded_async_via_exchange(ShardGroup* g, const innr_cuda_corpus* const* shards, size_t n_shards, const void* queries,
                               size_t query_bytes, size_t nq, size_t k, size_t kk, int metric, ScanOnly scan_only,
                               EnqueueKeys enqueue_keys, innr_cuda_ticket** out_ticket) {
  if (k > MAX_FUSED_K || nq * k > g->ex[0]->slot_keys || n_shards > (size_t)MAX_SHARD_DEVICES)
    return fail(INNR_EUNSUPPORTED, "asynchronous sharded call: k > 128 or the batch does not fit the mailboxes (use the synchronous entry)");
  std::lock_guard<std::mutex> call_lk(g->mu);
  if (g->async_in_flight.load() >= 2) return fail(INNR_EBUSY, "two asynchronous sharded calls are already in flight: wait for a ticket first");
  const int p = (int)((g->ex[0]->calls + 1) & 1);  // slot = mailbox parity of this call
  // reserve slot p on every device and make its stream wait until the root has consumed the previous call of this parity
  std::vector<innr_cuda_ticket*> tk(n_shards, nullptr);
  int rc = INNR_OK;
  for (size_t i = 0; i < n_shards && rc == INNR_OK; ++i) {
    EntryGuard lk(shards[i]->device);
    DeviceCtx* ctx;
    rc = ensure_ctx(shards[i]->device, &ctx, WS_NONE);
    if (rc) break;
    innr_cuda_ticket* t = &ctx->async_slot[p];
    if (t->in_flight) {
      rc = fail(INNR_EBUSY, "an asynchronous call is in flight in the slot this sharded call needs: wait for its ticket first");
      break;
    }
    auto prepare = [&]() -> int {
      if (!t->stream) {
        static const bool blocking = getenv("INNR_ASYNC_BLOCKING_WAIT") != nullptr;
        CU(cudaStreamCreateWithFlags(&t->stream, cudaStreamNonBlocking));
        CU(cudaEventCreateWithFlags(&t->done, cudaEventDisableTiming | (blocking ? cudaEventBlockingSync : 0)));
      }
      if (i == 0 && !g->consumed[p]) CU(cudaEventCreateWithFlags(&g->consumed[p], cudaEventDisableTiming));
      return INNR_OK;
    };
    rc = prepare();
    if (rc) break;
    t->in_flight = true;  // reserved
    tk[i] = t;
  }
  if (rc == INNR_OK)
    for (size_t i = 1; i < n_shards && rc == INNR_OK; ++i) {
      cudaError_t e = cudaStreamWaitEvent(tk[i]->stream, g->consumed[p], 0);  // a never-recorded event counts as complete
      if (e != cudaSuccess) rc = cuda_fail(e, "cudaStreamWaitEvent(consumed)");
    }
  if (rc) {
    for (size_t i = 0; i < n_shards; ++i)
      if (tk[i]) {
        EntryGuard lk(shards[i]->device);
        tk[i]->in_flight = false;
      }
    return rc;
  }
  std::vector<int> rcs(n_shards, INNR_OK);
  std::vector<std::string> errs(n_shards);
  std::function<void(size_t)> job = [&](size_t i) {
    auto body = [&]() -> int {
      const innr_cuda_corpus* c = shards[i];
      innr_cuda_exchange* x = g->ex[i];
      innr_cuda_ticket* t = tk[i];
      ++x->calls;  // first thing: a shard that fails below must not leave the ranks' call numbers out of step
      EntryGuard lk(c->device);
      DeviceCtx* ctx;
      int r = ensure_ctx(c->device, &ctx, WS_NONE);
      if (r) return r;
      t->device = c->device;
      t->kind = c->kind;
      t->metric = metric;
      t->nq = nq;
      t->k = k;
      t->kk = kk;
      t->krow = k;
      t->sharded = i == 0;
      t->n_siblings = 0;
      if ((r = grow(&t->h_in, &t->h_in_cap, query_bytes, true))) return r;
      if ((r = grow(&t->d_query, &t->d_query_cap, query_bytes + 16, false))) return r;
      if ((r = grow(&t->d_keys, &t->d_keys_cap, nq * k * sizeof(uint64_t), false))) return r;
      std::memcpy(t->h_in, queries, query_bytes);
      CU(cudaMemcpyAsync(t->d_query, t->h_in, query_bytes, cudaMemcpyHostToDevice, t->stream));
      int lane = 0;
      r = ensure_ctx(c->device, &ctx, scan_only(i) ? WS_DEV_SCAN : WS_DEV, t->stream, &lane);
      if (r) return r;
      {
        DevRelease rel(*ctx, t->stream, lane);
        r = enqueue_keys(i, ctx, t->d_query, (uint64_t*)t->d_keys, t->stream, lane);
        if (r) return r;
      }
      if (i != 0) {
        CU(launch_exchange_merge(ex_view(x), (const uint64_t*)t->d_keys, nq, k, x->calls, 1, 0, nullptr, nullptr, nullptr,
                                 nullptr, t->stream, &g_launches));
        CU(cudaEventRecord(t->done, t->stream));
        return INNR_OK;
      }
      if ((r = grow(&t->d_merged, &t->d_merged_cap, nq * k * sizeof(uint64_t), false))) return r;
      if ((r = grow(&t->h_out, &t->h_out_cap, nq * k * sizeof(uint64_t) + 16, true))) return r;
      CU(launch_exchange_merge(ex_view(x), (const uint64_t*)t->d_keys, nq, k, x->calls, 0, metric != INNR_METRIC_L2,
                               (uint64_t*)t->d_merged, nullptr, nullptr, nullptr, t->stream, &g_launches));
      CU(cudaEventRecord(g->consumed[p], t->stream));
      CU(cudaMemcpyAsync(t->h_out, t->d_merged, nq * k * sizeof(uint64_t), cudaMemcpyDeviceToHost, t->stream));
      CU(cudaMemcpyAsync((char*)t->h_out + nq * k * sizeof(uint64_t), x->dev_status, sizeof(unsigned), cudaMemcpyDeviceToHost,
                         t->stream));
      CU(cudaEventRecord(t->done, t->stream));
      return INNR_OK;
    };
    rcs[i] = body();
    if (rcs[i]) errs[i] = t_err;
  };
  g->pool->run(job);
  for (size_t i = 0; i < n_shards; ++i)
    if (rcs[i]) {
      // what was queued stays queued; give the slots back once their streams have drained
      for (size_t j = 0; j < n_shards; ++j) {
        cudaStreamSynchronize(tk[j]->stream);
        EntryGuard lk(shards[j]->device);
        tk[j]->in_flight = false;
      }
      return fail(rcs[i], "shard " + std::to_string(i) + ": " + errs[i]);
    }
  innr_cuda_ticket* root = tk[0];
  for (size_t i = 1; i < n_shards; ++i) root->siblings[root->n_siblings++] = tk[i];
  root->group_busy = &g->async_in_flight;
  g->async_in_flight.fetch_add(1);
  *out_ticket = root;
  return INNR_OK;
}

template <class Call>
int run_shards(size_t n_shards, Call call, std::vector<ShardOut>& outs) {
  std::vector<std::thread> th;
  th.reserve(n_shards);
  for (size_t i = 0; i < n_shards; ++i)
    th.emplace_back([&, i] {
      outs[i].rc = call(i, outs[i]);
      if (outs[i].rc) outs[i].err = t_err;  // the message is thread-local
    });
  for (auto& t : th) t.join();
  for (size_t i = 0; i < n_shards; ++i)
    if (outs[i].rc) return fail(outs[i].rc, "shard " + std::to_string(i) + ": " + outs[i].err);
  return INNR_OK;
}
}  // namespace
extern "C" {

int innr_cuda_batch_knn_sharded(const innr_cuda_corpus* const* shards, size_t n_shards, int metric, const float* queries,
                                size_t n_queries, size_t query_len, size_t k, uint64_t* out_idx, float* out_score,
                                size_t* out_count) {
  if (out_count) *out_count = 0;
  if (!shards || n_shards == 0) return fail(INNR_EINVAL, "no shards");
  size_t n_total = 0;
  for (size_t i = 0; i < n_shards; ++i) {
    if (!shards[i] || shards[i]->kind != 0) return fail(INNR_EINVAL, "need f32 PDX shards");
    if (shards[i]->d != shards[0]->d) return fail(INNR_EINVAL, "shards differ in dimension");
    n_total += shards[i]->n;
  }
  if (query_len != shards[0]->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;
  if (!out_idx || !out_score) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < n_total ? k : n_total;
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  // distinct devices: every shard scans on its own stream, the lists meet in the root's mailbox over NVLink and are
  // merged there in the same launch (csrc/exchange.cu); one D2H of k results, no host merge
  if (ShardGroup* g = shard_group_for(shards, n_shards)) {
    rc = sharded_via_exchange(g, shards, n_shards, queries, n_queries * query_len * sizeof(float), n_queries, k, metric, false,
                              [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk) -> int {
                                innr_cuda_corpus* c = const_cast<innr_cuda_corpus*>(shards[i]);
                                if (c->n == 0) {
                                  CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), ctx->stream));
                                  return INNR_OK;
                                }
                                return knn_keys_dev(c, ctx, mode, (const float*)dq, n_queries, k, dk, ctx->stream);
                              },
                              out_idx, out_score, nullptr);
    if (rc == INNR_OK) {
      if (out_count) *out_count = kk;
      return INNR_OK;
    }
    if (rc != INNR_EUNSUPPORTED) return rc;
  }
  std::vector<ShardOut> outs(n_shards);
  rc = run_shards(n_shards, [&](size_t i, ShardOut& o) {
    o.idx.assign(n_queries * k, 0);
    o.score.assign(n_queries * k, 0.0f);
    return innr_cuda_batch_knn(shards[i], metric, queries, n_queries, query_len, k, o.idx.data(), o.score.data(), &o.count);
  }, outs);
  if (rc) return rc;
  const bool desc = metric != INNR_METRIC_L2;
  std::vector<std::pair<uint64_t, float>> all;
  for (size_t q = 0; q < n_queries; ++q) {
    all.clear();
    for (size_t i = 0; i < n_shards; ++i)
      for (size_t j = 0; j < outs[i].count; ++j) {
        const float sc = outs[i].score[q * k + j];
        const uint32_t ob = desc ? ~host_order_bits(sc) : host_order_bits(sc);
        all.emplace_back(((uint64_t)ob << 32) | outs[i].idx[q * k + j], sc);
      }
    std::sort(all.begin(), all.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
    for (size_t j = 0; j < kk; ++j) {
      out_idx[q * k + j] = all[j].first & 0xFFFFFFFFull;
      out_score[q * k + j] = all[j].second;
    }
  }
  if (out_count) *out_count = kk;
  return INNR_OK;
}

int innr_cuda_hamming_topk_sharded(const innr_cuda_corpus* const* shards, size_t n_shards, const uint64_t* query_words,
                                   size_t n_queries, size_t query_dim_bits, size_t k, uint64_t* out_idx,
                                   uint32_t* out_dist, size_t* out_count) {
  if (out_count) *out_count = 0;
  if (!shards || n_shards == 0) return fail(INNR_EINVAL, "no shards");
  size_t n_total = 0;
  for (size_t i = 0; i < n_shards; ++i) {
    if (!shards[i] || shards[i]->kind != 1) return fail(INNR_EINVAL, "need binary shards");
    n_total += shards[i]->n;
  }
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;
  if (!out_idx || !out_dist) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < n_total ? k : n_total;
  int rc = INNR_OK;
  bool same_dim = true;
  for (size_t i = 0; i < n_shards; ++i) same_dim = same_dim && shards[i]->dim_bits == query_dim_bits;
  if (ShardGroup* g = (same_dim && shards[0]->words) ? shard_group_for(shards, n_shards) : nullptr) {
    // the query codes in the form the scan reads them: padded to whole 128-bit chunks, padding bits masked
    const innr_cuda_corpus* c0 = shards[0];
    const size_t qw = 2 * c0->chunks, rem = c0->dim_bits % 64;
    std::vector<uint64_t> padded(n_queries * qw, 0);
    for (size_t q = 0; q < n_queries; ++q)
      for (size_t w = 0; w < c0->words; ++w) {
        uint64_t x = query_words[q * c0->words + w];
        if (w + 1 == c0->words && rem) x &= (1ull << rem) - 1;
        padded[q * qw + w] = x;
      }
    rc = sharded_via_exchange(g, shards, n_shards, padded.data(), padded.size() * sizeof(uint64_t), n_queries, k, INNR_METRIC_L2, true,
                              [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk) -> int {
                                const innr_cuda_corpus* c = shards[i];
                                if (c->n == 0) {
                                  CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), ctx->stream));
                                  return INNR_OK;
                                }
                                return hamming_keys(c, ctx, (const uint64_t*)dq, n_queries, k, dk, ctx->stream);
                              },
                              out_idx, nullptr, out_dist);
    if (rc == INNR_OK) {
      if (out_count) *out_count = kk;
      return INNR_OK;
    }
    if (rc != INNR_EUNSUPPORTED) return rc;
  }
  std::vector<ShardOut> outs(n_shards);
  rc = run_shards(n_shards, [&](size_t i, ShardOut& o) {
    o.idx.assign(n_queries * k, 0);
    o.dist.assign(n_queries * k, 0);
    return innr_cuda_hamming_topk(shards[i], query_words, n_queries, query_dim_bits, k, o.idx.data(), o.dist.data(), &o.count);
  }, outs);
  if (rc) return rc;
  std::vector<uint64_t> all;
  for (size_t q = 0; q < n_queries; ++q) {
    all.clear();
    for (size_t i = 0; i < n_shards; ++i)
      for (size_t j = 0; j < outs[i].count; ++j)
        all.push_back(((uint64_t)outs[i].dist[q * k + j] << 32) | outs[i].idx[q * k + j]);
    std::sort(all.begin(), all.end());
    for (size_t j = 0; j < kk; ++j) {
      out_idx[q * k + j] = all[j] & 0xFFFFFFFFull;
      out_dist[q * k + j] = (uint32_t)(all[j] >> 32);
    }
  }
  if (out_count) *out_count = kk;
  return INNR_OK;
}

int innr_cuda_batch_knn_u8_sharded(const innr_cuda_corpus* const* shards, size_t n_shards, const float* queries,
                                   size_t n_queries, size_t query_len, size_t k, uint64_t* out_idx, float* out_score,
                                   size_t* out_count) {
  if (out_count) *out_count = 0;
  if (!shards || n_shards == 0) return fail(INNR_EINVAL, "no shards");
  size_t n_total = 0;
  for (size_t i = 0; i < n_shards; ++i) {
    if (!shards[i] || shards[i]->kind != 2) return fail(INNR_EINVAL, "need u8 shards");
    n_total += shards[i]->n;
  }
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;
  if (!out_idx || !out_score) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < n_total ? k : n_total;
  int rc = INNR_OK;
  bool same_dim = true;
  for (size_t i = 0; i < n_shards; ++i) same_dim = same_dim && shards[i]->d == query_len && shards[i]->d > 0;
  if (ShardGroup* g = same_dim ? shard_group_for(shards, n_shards) : nullptr) {
    rc = sharded_via_exchange(g, shards, n_shards, queries, n_queries * query_len * sizeof(float), n_queries, k, INNR_METRIC_DOT, false,
                              [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk) -> int {
                                const innr_cuda_corpus* c = shards[i];
                                if (c->n == 0) {
                                  CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), ctx->stream));
                                  return INNR_OK;
                                }
                                return u8_keys(c, ctx, (const float*)dq, n_queries, k, dk, ctx->stream);
                              },
                              out_idx, out_score, nullptr);
    if (rc == INNR_OK) {
      if (out_count) *out_count = kk;
      return INNR_OK;
    }
    if (rc != INNR_EUNSUPPORTED) return rc;
  }
  std::vector<ShardOut> outs(n_shards);
  rc = run_shards(n_shards, [&](size_t i, ShardOut& o) {
    o.idx.assign(n_queries * k, 0);
    o.score.assign(n_queries * k, 0.0f);
    return innr_cuda_batch_knn_u8(shards[i], queries, n_queries, query_len, k, o.idx.data(), o.score.data(), &o.count);
  }, outs);
  if (rc) return rc;
  std::vector<std::pair<uint64_t, float>> all;
  for (size_t q = 0; q < n_queries; ++q) {
    all.clear();
    for (size_t i = 0; i < n_shards; ++i)
      for (size_t j = 0; j < outs[i].count; ++j) {
        const float sc = outs[i].score[q * k + j];
        all.emplace_back(((uint64_t)(~host_order_bits(sc)) << 32) | outs[i].idx[q * k + j], sc);
      }
    std::sort(all.begin(), all.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
    for (size_t j = 0; j < kk; ++j) {
      out_idx[q * k + j] = all[j].first & 0xFFFFFFFFull;
      out_score[q * k + j] = all[j].second;
    }
  }
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// Token shards (one document range each): the argument checks of innr_cuda_maxsim_topk over the union of the shards.
static int check_token_shards(const innr_cuda_corpus* const* shards, size_t n_shards, size_t n_q, size_t q_dim,
                              size_t* n_total) {
  if (!shards || n_shards == 0) return fail(INNR_EINVAL, "no shards");
  size_t tokens = 0;
  *n_total = 0;
  for (size_t i = 0; i < n_shards; ++i) {
    if (!shards[i] || shards[i]->kind != 3) return fail(INNR_EINVAL, "need token shards");
    if (shards[i]->d != shards[0]->d) return fail(INNR_EINVAL, "shards differ in dimension");
    *n_total += shards[i]->n;
    tokens += shards[i]->total_tokens;
  }
  if (n_q && tokens && q_dim != shards[0]->d) return fail(INNR_EINVAL, "dimension mismatch (doc)");  // src/maxsim.rs:107-110
  return INNR_OK;
}

int innr_cuda_maxsim_topk_sharded(const innr_cuda_corpus* const* shards, size_t n_shards, const float* q_tokens,
                                  size_t n_queries, size_t n_q, size_t q_dim, int cosine_flag, size_t k, uint64_t* out_idx,
                                  float* out_score, size_t* out_count) {
  if (out_count) *out_count = 0;
  size_t n_total = 0;
  int rc = check_token_shards(shards, n_shards, n_q, q_dim, &n_total);
  if (rc) return rc;
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;
  if (!out_idx || !out_score || (n_q * q_dim && !q_tokens)) return fail(INNR_EINVAL, "null argument");
  const size_t kk = k < n_total ? k : n_total;
  // distinct devices: every shard scores and selects on its own stream, the lists meet in the root's mailbox
  if (ShardGroup* g = shard_group_for(shards, n_shards)) {
    const float none = 0.0f;
    const size_t qbytes = n_queries * n_q * shards[0]->d * sizeof(float);
    rc = sharded_via_exchange(g, shards, n_shards, qbytes ? (const void*)q_tokens : (const void*)&none, qbytes, n_queries, k,
                              INNR_METRIC_DOT, false,
                              [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk) -> int {
                                const innr_cuda_corpus* c = shards[i];
                                if (c->n == 0) {
                                  CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), ctx->stream));
                                  return INNR_OK;
                                }
                                CU(ctx->d_scores.reserve(maxsim_topk_chunk(c, n_queries) * c->n * sizeof(float)));
                                return maxsim_topk_keys(c, ctx, (const float*)dq, n_queries, n_q, cosine_flag, k, dk,
                                                        (float*)ctx->d_scores.p, ctx->stream);
                              },
                              out_idx, out_score, nullptr);
    if (rc == INNR_OK) {
      if (out_count) *out_count = kk;
      return INNR_OK;
    }
    if (rc != INNR_EUNSUPPORTED) return rc;
  }
  std::vector<ShardOut> outs(n_shards);
  rc = run_shards(n_shards, [&](size_t i, ShardOut& o) {
    o.idx.assign(n_queries * k, 0);
    o.score.assign(n_queries * k, 0.0f);
    return innr_cuda_maxsim_topk(shards[i], q_tokens, n_queries, n_q, q_dim, cosine_flag, k, o.idx.data(), o.score.data(),
                                 &o.count);
  }, outs);
  if (rc) return rc;
  std::vector<std::pair<uint64_t, float>> all;
  for (size_t q = 0; q < n_queries; ++q) {
    all.clear();
    for (size_t i = 0; i < n_shards; ++i)
      for (size_t j = 0; j < outs[i].count; ++j) {
        const float sc = outs[i].score[q * k + j];
        all.emplace_back(((uint64_t)(~host_order_bits(sc)) << 32) | outs[i].idx[q * k + j], sc);
      }
    std::sort(all.begin(), all.end(), [](const auto& a, const auto& b) { return a.first < b.first; });
    for (size_t j = 0; j < kk; ++j) {
      out_idx[q * k + j] = all[j].first & 0xFFFFFFFFull;
      out_score[q * k + j] = all[j].second;
    }
  }
  if (out_count) *out_count = kk;
  return INNR_OK;
}

// ---- asynchronous forms of the sharded entries (exchange route only: shards on pairwise distinct devices) ------------
int innr_cuda_batch_knn_sharded_async(const innr_cuda_corpus* const* shards, size_t n_shards, int metric,
                                      const float* queries, size_t n_queries, size_t query_len, size_t k,
                                      innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  if (!shards || n_shards == 0) return fail(INNR_EINVAL, "no shards");
  size_t n_total = 0;
  for (size_t i = 0; i < n_shards; ++i) {
    if (!shards[i] || shards[i]->kind != 0) return fail(INNR_EINVAL, "need f32 PDX shards");
    if (shards[i]->d != shards[0]->d) return fail(INNR_EINVAL, "shards differ in dimension");
    n_total += shards[i]->n;
  }
  if (query_len != shards[0]->d) return fail(INNR_EINVAL, "query.len() != batch.dimension");
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;  // empty result: no ticket
  if (!queries) return fail(INNR_EINVAL, "null argument");
  int mode;
  int rc = metric_to_mode(metric, &mode);
  if (rc) return rc;
  ShardGroup* g = shard_group_for(shards, n_shards);
  if (!g) return fail(INNR_EUNSUPPORTED, "asynchronous sharded calls need two or more shards on pairwise distinct devices with peer access");
  return sharded_async_via_exchange(
      g, shards, n_shards, queries, n_queries * query_len * sizeof(float), n_queries, k, k < n_total ? k : n_total, metric,
      [&](size_t i) { return shards[i]->n == 0 || knn_is_scan_only(shards[i], mode, n_queries, k); },
      [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk, cudaStream_t s, int lane) -> int {
        innr_cuda_corpus* c = const_cast<innr_cuda_corpus*>(shards[i]);
        if (c->n == 0) {
          CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), s));
          return INNR_OK;
        }
        return knn_keys_dev(c, ctx, mode, (const float*)dq, n_queries, k, dk, s, lane);
      },
      out_ticket);
}

int innr_cuda_hamming_topk_sharded_async(const innr_cuda_corpus* const* shards, size_t n_shards, const uint64_t* query_words,
                                         size_t n_queries, size_t query_dim_bits, size_t k, innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  if (!shards || n_shards == 0) return fail(INNR_EINVAL, "no shards");
  size_t n_total = 0;
  for (size_t i = 0; i < n_shards; ++i) {
    if (!shards[i] || shards[i]->kind != 1) return fail(INNR_EINVAL, "need binary shards");
    if (shards[i]->dim_bits != query_dim_bits) return fail(INNR_EINVAL, "innr::binary_hamming: dimension mismatch");
    n_total += shards[i]->n;
  }
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;  // empty result: no ticket
  if (!query_words) return fail(INNR_EINVAL, "null argument");
  if (shards[0]->words == 0) return fail(INNR_EUNSUPPORTED, "zero-dimensional codes: use innr_cuda_hamming_topk_sharded");
  ShardGroup* g = shard_group_for(shards, n_shards);
  if (!g) return fail(INNR_EUNSUPPORTED, "asynchronous sharded calls need two or more shards on pairwise distinct devices with peer access");
  const innr_cuda_corpus* c0 = shards[0];
  const size_t qw = 2 * c0->chunks, rem = c0->dim_bits % 64;
  std::vector<uint64_t> padded(n_queries * qw, 0);  // padded to whole 128-bit chunks, padding bits masked
  for (size_t q = 0; q < n_queries; ++q)
    for (size_t w = 0; w < c0->words; ++w) {
      uint64_t x = query_words[q * c0->words + w];
      if (w + 1 == c0->words && rem) x &= (1ull << rem) - 1;
      padded[q * qw + w] = x;
    }
  return sharded_async_via_exchange(
      g, shards, n_shards, padded.data(), padded.size() * sizeof(uint64_t), n_queries, k, k < n_total ? k : n_total,
      INNR_METRIC_L2, [&](size_t i) { return shards[i]->n == 0 || hamming_is_scan_only(shards[i], n_queries, k); },
      [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk, cudaStream_t s, int lane) -> int {
        const innr_cuda_corpus* c = shards[i];
        if (c->n == 0) {
          CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), s));
          return INNR_OK;
        }
        return hamming_keys(c, ctx, (const uint64_t*)dq, n_queries, k, dk, s, lane);
      },
      out_ticket);
}

int innr_cuda_batch_knn_u8_sharded_async(const innr_cuda_corpus* const* shards, size_t n_shards, const float* queries,
                                         size_t n_queries, size_t query_len, size_t k, innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  if (!shards || n_shards == 0) return fail(INNR_EINVAL, "no shards");
  size_t n_total = 0;
  for (size_t i = 0; i < n_shards; ++i) {
    if (!shards[i] || shards[i]->kind != 2) return fail(INNR_EINVAL, "need u8 shards");
    if (shards[i]->d != shards[0]->d) return fail(INNR_EINVAL, "shards differ in dimension");
    n_total += shards[i]->n;
  }
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;  // src/scalar.rs:376-378 (before any length check): no ticket
  if (query_len != shards[0]->d) return fail(INNR_EINVAL, "asymmetric_dot_u8_precomputed: dimension mismatch");
  if (!queries) return fail(INNR_EINVAL, "null argument");
  if (shards[0]->d == 0) return fail(INNR_EUNSUPPORTED, "zero-dimensional u8 corpus");
  ShardGroup* g = shard_group_for(shards, n_shards);
  if (!g) return fail(INNR_EUNSUPPORTED, "asynchronous sharded calls need two or more shards on pairwise distinct devices with peer access");
  return sharded_async_via_exchange(
      g, shards, n_shards, queries, n_queries * query_len * sizeof(float), n_queries, k, k < n_total ? k : n_total,
      INNR_METRIC_DOT, [&](size_t i) { return shards[i]->n == 0 || u8_is_scan_only(shards[i], n_queries, k); },
      [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk, cudaStream_t s, int lane) -> int {
        const innr_cuda_corpus* c = shards[i];
        if (c->n == 0) {
          CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), s));
          return INNR_OK;
        }
        return u8_keys(c, ctx, (const float*)dq, n_queries, k, dk, s, lane);
      },
      out_ticket);
}

int innr_cuda_maxsim_topk_sharded_async(const innr_cuda_corpus* const* shards, size_t n_shards, const float* q_tokens,
                                        size_t n_queries, size_t n_q, size_t q_dim, int cosine_flag, size_t k,
                                        innr_cuda_ticket** out_ticket) {
  if (!out_ticket) return fail(INNR_EINVAL, "null out_ticket");
  *out_ticket = nullptr;
  size_t n_total = 0;
  int rc = check_token_shards(shards, n_shards, n_q, q_dim, &n_total);
  if (rc) return rc;
  if (n_total == 0 || k == 0 || n_queries == 0) return INNR_OK;  // empty result: no ticket
  if (n_q * q_dim && !q_tokens) return fail(INNR_EINVAL, "null argument");
  ShardGroup* g = shard_group_for(shards, n_shards);
  if (!g) return fail(INNR_EUNSUPPORTED, "asynchronous sharded calls need two or more shards on pairwise distinct devices with peer access");
  const float none = 0.0f;
  const size_t qbytes = n_queries * n_q * shards[0]->d * sizeof(float);
  return sharded_async_via_exchange(
      g, shards, n_shards, qbytes ? (const void*)q_tokens : (const void*)&none, qbytes, n_queries, k,
      k < n_total ? k : n_total, INNR_METRIC_DOT, [&](size_t) { return false; },  // lane 0: scratch score vectors
      [&](size_t i, DeviceCtx* ctx, void* dq, uint64_t* dk, cudaStream_t s, int) -> int {
        const innr_cuda_corpus* c = shards[i];
        if (c->n == 0) {
          CU(cudaMemsetAsync(dk, 0xFF, n_queries * k * sizeof(uint64_t), s));
          return INNR_OK;
        }
        // the score vectors belong to the asynchronous slot this call runs in (the one whose stream is `s`)
        innr_cuda_ticket* t = ctx->async_slot[0].stream == s ? &ctx->async_slot[0] : &ctx->async_slot[1];
        int r = grow(&t->d_scores, &t->d_scores_cap, maxsim_topk_chunk(c, n_queries) * c->n * sizeof(float), false);
        if (r) return r;
        return maxsim_topk_keys(c, ctx, (const float*)dq, n_queries, n_q, cosine_flag, k, dk, (float*)t->d_scores, s);
      },
      out_ticket);
}

}  // extern "C"
