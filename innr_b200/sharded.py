"""Row-sharded corpora across the GPUs of one box: one process per GPU, `torch.distributed` for the plumbing.

SURVEY.md 8e: vectors are independent and top-k selection is a monoid, so each rank scans a contiguous row range
(global index = shard base + local; contiguous ranges keep "lower global index wins" consistent across shards),
emits its local top-k as sorted 64-bit composite keys, and ONE allgather of k keys per rank per query exchanges
them; every rank then runs the same n_ranks*k -> k merge. No other collective is on the data path.

torch is used for device buffers, streams and the allgather only; the scan and the merge are libinnr_cuda kernels
launched on torch's current stream through the `_dev` entry points of the C-ABI.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


def shard_range(n: int, rank: int, world: int):
    """Contiguous row range [lo, hi) of shard `rank` (SURVEY.md 8d: shard s owns rows [s*N/G, (s+1)*N/G))."""
    return (n * rank) // world, (n * (rank + 1)) // world


# ---- host-side key codec (same bit layout as csrc/common.cuh; used by the CPU/gloo tests and for decoding) ----
def order_bits(scores: np.ndarray) -> np.ndarray:
    b = np.ascontiguousarray(scores, dtype=np.float32).view(np.uint32).astype(np.uint32)
    mask = ((b.view(np.int32) >> 31).view(np.uint32)) >> np.uint32(1)
    return (b ^ mask) ^ np.uint32(0x80000000)


def encode_keys(scores: np.ndarray, indices: np.ndarray, descending: bool) -> np.ndarray:
    o = order_bits(scores)
    if descending:
        o = ~o
    return (o.astype(np.uint64) << np.uint64(32)) | np.asarray(indices, dtype=np.uint64)


def decode_keys(keys: np.ndarray, descending: bool):
    keys = np.asarray(keys, dtype=np.uint64)
    hi = (keys >> np.uint64(32)).astype(np.uint32)
    if descending:
        hi = ~hi
    o = hi ^ np.uint32(0x80000000)
    mask = ((o.view(np.int32) >> 31).view(np.uint32)) >> np.uint32(1)
    return (keys & np.uint64(0xFFFFFFFF)), (o ^ mask).view(np.float32)


def merge_keys_host(key_lists: np.ndarray, k: int) -> np.ndarray:
    """Reference semantics of the merge (K10): the k smallest keys of the union. key_lists: (n_lists, k)."""
    flat = np.asarray(key_lists, dtype=np.uint64).reshape(-1)
    flat = flat[flat != np.uint64(0xFFFFFFFFFFFFFFFF)]
    return np.sort(flat)[:k]


class PeerExchange:
    """One rank's end of the peer-mapped key exchange (csrc/exchange.cu, include/innr_cuda.h): a mailbox in this rank's
    device memory that every peer writes into over NVLink, and ONE kernel per call that publishes, waits and merges --
    the replacement of `all_gather_into_tensor` + merge launch on the sharded top-k path. Built on the calling thread's
    device (innr_b200.init)."""

    def __init__(self, n_ranks: int, rank: int, slot_keys: int = 0):
        self.n_ranks, self.rank = int(n_ranks), int(rank)
        h = C.c_void_p()
        L.call("innr_cuda_exchange_create", self.n_ranks, self.rank, slot_keys, C.byref(h))
        self.h = h
        self.slot_keys = slot_keys or 16384

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h:
            try:
                L.lib().innr_cuda_exchange_free(h)
            except Exception:
                pass

    def ipc_handle(self) -> bytes:
        buf = C.create_string_buffer(64)
        L.call("innr_cuda_exchange_ipc_handle", self.h, buf)
        return buf.raw

    def connect_ipc(self, handles) -> None:
        """handles: the 64-byte handles of all ranks, in rank order (each rank's own entry is ignored)."""
        blob = b"".join(handles)
        assert len(blob) == 64 * self.n_ranks
        L.call("innr_cuda_exchange_connect_ipc", self.h, C.create_string_buffer(blob, len(blob)))

    @staticmethod
    def connect_local(exchanges) -> None:
        """All ranks of one exchange living in THIS process (possibly on different devices)."""
        arr = (C.c_void_p * len(exchanges))(*[x.h for x in exchanges])
        L.call("innr_cuda_exchange_connect_local", arr, len(exchanges))

    @classmethod
    def for_process_group(cls, dist, group=None, slot_keys: int = 0) -> "PeerExchange":
        """One process per GPU (torch.distributed): every rank creates its mailbox, the IPC handles travel through the
        process group once, every rank maps all peers."""
        world, rank = dist.get_world_size(group), dist.get_rank(group)
        ex = cls(world, rank, slot_keys)
        if world > 1:
            handles = [None] * world
            dist.all_gather_object(handles, ex.ipc_handle(), group=group)
            ex.connect_ipc(handles)
        return ex

    def set_timeout_ms(self, ms: float) -> None:
        L.call("innr_cuda_exchange_set_timeout_ms", self.h, C.c_double(ms))

    def status(self) -> int:
        v = C.c_int(0)
        L.call("innr_cuda_exchange_status", self.h, C.byref(v))
        return int(v.value)

    def fits(self, nq: int, k: int) -> bool:
        return 0 < k <= 128 and nq * k <= self.slot_keys

    def merge_dev(self, local_keys_ptr: int, nq: int, k: int, metric_id: int, stream, keys_out=None, idx=None,
                  score=None, dist_out=None, publish_only: bool = False) -> None:
        vp = lambda t: None if t is None else C.c_void_p(t.data_ptr())  # noqa: E731
        L.call("innr_cuda_exchange_merge_dev", self.h, C.c_void_p(local_keys_ptr), nq, k, metric_id, int(publish_only),
               vp(keys_out), vp(idx), vp(score), vp(dist_out), stream)


class ShardedKnn:
    """One rank's view of a row-sharded corpus. kind: 'f32' (DeviceBatch), 'u8' (U8Corpus), 'binary' (BinaryCorpus),
    'maxsim' (TokenCorpus, a document range; metric 'dot' or 'cosine'; queries of `query_tokens` tokens each, passed as
    nq x query_tokens x dim floats). `exchange`: a connected PeerExchange (keys travel through peer-mapped mailboxes, one
    launch) or None (one NCCL `all_gather_into_tensor` of k keys per rank + the merge launch)."""

    def __init__(self, shard, kind: str = "f32", metric: str = "cosine", group=None, exchange=None, query_tokens: int = 0):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.shard, self.kind, self.metric, self.group = shard, kind, metric, group
        self.world = dist.get_world_size(group) if dist.is_initialized() else 1
        self.exchange = exchange
        self._metric_id = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
        assert kind != "maxsim" or metric in ("dot", "cosine"), "MaxSim ranks by dot or cosine"
        self.query_tokens = int(query_tokens)
        self._bufs = {}

    def _buffers(self, nq: int, k: int, device):
        key = (nq, k)
        if key not in self._bufs:
            t = self.torch
            b = dict(
                local=t.empty(nq * k, dtype=t.int64, device=device),
                gathered=t.empty(self.world * nq * k, dtype=t.int64, device=device),
                idx=t.empty(nq * k, dtype=t.int64, device=device),
                score=t.empty(nq * k, dtype=t.float32 if self.kind != "binary" else t.int32, device=device),
                keys=t.empty(nq * k, dtype=t.int64, device=device))
            # the pointers never change: build the ctypes objects once (a step of a small corpus is host-bound)
            b["p"] = {name: C.c_void_p(b[name].data_ptr()) for name in ("local", "gathered", "idx", "score", "keys")}
            b["views"] = (b["idx"].view(nq, k), b["score"].view(nq, k))
            self._bufs[key] = b
        return self._bufs[key]

    def knn_dev(self, dev_queries, nq: int, k: int):
        """dev_queries: torch tensor on this rank's GPU (f32 nq x d, or int64 words for 'binary'). Returns
        (idx int64[nq,k], score[nq,k]) tensors on the device, identical on every rank. All work is queued on
        torch's current stream."""
        t = self.torch
        stream = C.c_void_p(t.cuda.current_stream().cuda_stream)
        b = self._buffers(nq, k, dev_queries.device)
        self._keys(dev_queries, nq, k, b["local"], stream)
        if self.exchange is not None and self.exchange.fits(nq, k):
            # publish / wait / merge / decode in ONE launch, no collective call
            if self.kind == "binary":
                self.exchange.merge_dev(b["local"].data_ptr(), nq, k, L.METRIC_L2, stream, idx=b["idx"], dist_out=b["score"])
            else:
                m = L.METRIC_L2 if (self.kind == "f32" and self.metric == "l2") else L.METRIC_DOT
                self.exchange.merge_dev(b["local"].data_ptr(), nq, k, m, stream, idx=b["idx"], score=b["score"])
            return b["idx"].view(nq, k), b["score"].view(nq, k)
        if self.world > 1:
            self.dist.all_gather_into_tensor(b["gathered"], b["local"], group=self.group)
            src, n_lists = b["gathered"], self.world
        else:
            src, n_lists = b["local"], 1
        if self.kind == "binary":
            # distance is the high half of the key itself
            L.call("innr_cuda_merge_keys_dev", C.c_void_p(src.data_ptr()), n_lists, nq, k, L.METRIC_L2,
                   C.c_void_p(b["keys"].data_ptr()), C.c_void_p(b["idx"].data_ptr()), None, stream)
            return b["idx"].view(nq, k), (b["keys"] >> 32).view(nq, k)
        m = L.METRIC_L2 if (self.kind == "f32" and self.metric == "l2") else L.METRIC_DOT
        L.call("innr_cuda_merge_keys_dev", b["p"]["gathered" if self.world > 1 else "local"], n_lists, nq, k, m,
               None, b["p"]["idx"], b["p"]["score"], stream)
        return b["views"]

    # ---- pipelined form: consecutive scans overlap, the exchange of query i runs under the scan of query i + 1 ---------
    def _keys(self, dev_queries, nq, k, local, stream):
        qp, lp = C.c_void_p(dev_queries.data_ptr()), C.c_void_p(local.data_ptr())
        if self.kind == "f32":
            L.call("innr_cuda_batch_knn_keys_dev", self.shard.h, self._metric_id, qp, nq, k, lp, stream)
        elif self.kind == "u8":
            L.call("innr_cuda_batch_knn_u8_keys_dev", self.shard.h, qp, nq, k, lp, stream)
        elif self.kind == "maxsim":
            L.call("innr_cuda_maxsim_topk_keys_dev", self.shard.h, qp, nq, self.query_tokens, int(self.metric == "cosine"), k,
                   lp, stream)
        else:
            L.call("innr_cuda_hamming_topk_keys_dev", self.shard.h, qp, nq, k, lp, stream)

    def knn_dev_pipelined(self, dev_queries, nq: int, k: int, overlap_scans: bool = True, host_queries=None,
                          host_out: bool = False):
        """Throughput form of knn_dev for a stream of independent queries. Two things overlap here that knn_dev serialises
        (kind 'maxsim': only the second -- its tcgen05 kernel fills every SM and its score vectors live in the library's
        one scratch lane, so two MaxSim scans cannot overlap; overlap_scans is ignored and the scans stay on torch's
        current stream, while the exchange still runs on the side stream):

        * consecutive shard scans. They alternate between two scan streams (the library keeps two workspaces per device
          for exactly this, api.cu `lane`), so the CTAs of scan i + 1 fill the SMs as the last CTAs of scan i retire and
          while its merge runs: the ramp at both ends of a launch -- 4 % (f32) to 10 % (Hamming) of a 1/8-corpus shard
          scan -- disappears;
        * scan and exchange. The exchange is a barrier between the ranks: on the scan's stream it adds its latency AND
          the ranks' per-step skew to every step. Here it is queued on a high-priority side stream (one CTA; it finds a
          slot next to the next scan's CTAs), so a rank only ever waits for data that is two calls old.

        The scan streams first wait for everything queued so far on torch's current stream (the queries may have been
        produced there). Returns (idx, score, event): the tensors are valid once `event` has completed
        (`torch.cuda.current_stream().wait_event(event)` or `drain()`); they are reused by the call after next.
        Without a peer exchange at world > 1 (NCCL route), or for requests that do not fit the mailboxes, falls back to
        knn_dev (event None). `overlap_scans=False` keeps the scans on torch's current stream (only the exchange moves
        to the side stream): fewer host calls per step, the better choice when a scan is so short that the step is bound
        by the host's launch rate (BASELINE C1: a 5 MB corpus).

        Host-buffer streaming: `host_queries` (a PINNED torch tensor; dev_queries is then ignored) is copied to the
        device on torch's current stream in front of the scan, and with `host_out=True` the results are copied into
        pinned host tensors behind the merge, on its stream -- the returned (idx, score) are then those HOST tensors,
        complete when `event` is. One host synchronisation per batch of calls instead of one per call."""
        t = self.torch
        if self.kind == "maxsim":
            overlap_scans = False
        if host_queries is not None and ((self.exchange is None and self.world > 1) or k > 128
                                         or (self.exchange is not None and not self.exchange.fits(nq, k))):
            dev_queries = host_queries.to(f"cuda:{t.cuda.current_device()}", non_blocking=True)
            host_queries = None
        if (self.exchange is None and (self.world > 1 or not overlap_scans)) \
                or (self.exchange is not None and not self.exchange.fits(nq, k)) or k > 128:
            idx, sc = self.knn_dev(dev_queries, nq, k)
            if host_out:
                idx, sc = idx.cpu(), sc.cpu()
            return idx, sc, None
        key = ("pipe", nq, k)
        if key not in self._bufs:
            dev = dev_queries.device if host_queries is None else t.device("cuda", t.cuda.current_device())
            mk = lambda dt: t.empty(nq * k, dtype=dt, device=dev)  # noqa: E731
            self._bufs[key] = {"slots": [dict(local=mk(t.int64), idx=mk(t.int64), keys=mk(t.int64),
                                              score=mk(t.float32 if self.kind != "binary" else t.int32),
                                              scan_done=t.cuda.Event(), ex_done=t.cuda.Event(), ready=t.cuda.Event(),
                                              used=False) for _ in range(2)],
                               "calls": 0}
            if getattr(self, "_ex_stream", None) is None:
                self._ex_stream = t.cuda.Stream(device=dev, priority=-1)
                self._scan_streams = [t.cuda.Stream(device=dev), t.cuda.Stream(device=dev)]
        st = self._bufs[key]
        parity = st["calls"] & 1
        slot = st["slots"][parity]
        st["calls"] += 1
        main = t.cuda.current_stream()
        if host_queries is not None:
            if "dq" not in slot:
                slot["dq"] = t.empty(host_queries.shape, dtype=host_queries.dtype, device=slot["local"].device)
            if slot["used"]:
                main.wait_event(slot["scan_done"])   # the scan of two calls ago has read this slot's query copy
            slot["dq"].copy_(host_queries, non_blocking=True)
            dev_queries = slot["dq"]
        if host_out and "h_idx" not in slot:
            slot["h_idx"] = t.empty(nq * k, dtype=t.int64).pin_memory()
            slot["h_score"] = t.empty(nq * k, dtype=slot["score"].dtype).pin_memory()
        if overlap_scans:
            scan = self._scan_streams[parity]
            slot["ready"].record(main)
            scan.wait_event(slot["ready"])
        else:
            scan = main
        if slot["used"]:
            scan.wait_event(slot["ex_done"])   # the exchange of two calls ago has read `local` (long done)
        self._keys(dev_queries, nq, k, slot["local"], C.c_void_p(scan.cuda_stream))
        m = L.METRIC_L2 if (self.kind == "binary" or (self.kind == "f32" and self.metric == "l2")) else L.METRIC_DOT
        if self.exchange is None:  # one rank: decode the list behind the scan, on the scan's stream
            L.call("innr_cuda_merge_keys_dev", C.c_void_p(slot["local"].data_ptr()), 1, nq, k, m,
                   C.c_void_p(slot["keys"].data_ptr()), C.c_void_p(slot["idx"].data_ptr()),
                   None if self.kind == "binary" else C.c_void_p(slot["score"].data_ptr()), C.c_void_p(scan.cuda_stream))
            slot["scan_done"].record(scan)
            if self.kind == "binary" or host_out:
                with t.cuda.stream(scan):
                    if self.kind == "binary":  # the distance is the high half of the key itself
                        slot["score"].copy_(slot["keys"] >> 32)
                    if host_out:
                        slot["h_idx"].copy_(slot["idx"], non_blocking=True)
                        slot["h_score"].copy_(slot["score"], non_blocking=True)
            slot["ex_done"].record(scan)
            slot["used"] = True
            if host_out:
                return slot["h_idx"].view(nq, k), slot["h_score"].view(nq, k), slot["ex_done"]
            return slot["idx"].view(nq, k), slot["score"].view(nq, k), slot["ex_done"]
        slot["scan_done"].record(scan)
        ex = self._ex_stream
        ex.wait_event(slot["scan_done"])
        exs = C.c_void_p(ex.cuda_stream)
        if self.kind == "binary":
            self.exchange.merge_dev(slot["local"].data_ptr(), nq, k, m, exs, idx=slot["idx"], dist_out=slot["score"])
        else:
            self.exchange.merge_dev(slot["local"].data_ptr(), nq, k, m, exs, idx=slot["idx"], score=slot["score"])
        if host_out:
            with t.cuda.stream(ex):
                slot["h_idx"].copy_(slot["idx"], non_blocking=True)
                slot["h_score"].copy_(slot["score"], non_blocking=True)
        slot["ex_done"].record(ex)
        slot["used"] = True
        if host_out:
            return slot["h_idx"].view(nq, k), slot["h_score"].view(nq, k), slot["ex_done"]
        return slot["idx"].view(nq, k), slot["score"].view(nq, k), slot["ex_done"]

    def drain(self):
        """Makes torch's current stream wait for every exchange queued by knn_dev_pipelined."""
        main = self.torch.cuda.current_stream()
        for key, st in self._bufs.items():
            if isinstance(key, tuple) and key and key[0] == "pipe":
                for slot in st["slots"]:
                    if slot["used"]:
                        main.wait_event(slot["ex_done"])

    def knn(self, queries_host: np.ndarray, k: int, pinned_stage=None):
        """End-to-end call with HOST buffers: H2D of the queries, shard scan, allgather, merge, D2H of the result."""
        t = self.torch
        q = np.ascontiguousarray(queries_host)
        if q.ndim == 1 or (self.kind == "maxsim" and q.ndim == 2):
            q = q.reshape((1,) + q.shape)
        nq = q.shape[0]
        src = t.from_numpy(q.view(np.int64) if self.kind == "binary" else q)
        dq = src.to(f"cuda:{t.cuda.current_device()}", non_blocking=True)
        idx, score = self.knn_dev(dq, nq, k)
        return idx.cpu().numpy().astype(np.uint64), score.cpu().numpy()


# ---- one process, several GPUs: the C-ABI's own sharded entries (no torch.distributed, no NCCL) -------------------------
def _handle_array(shards):
    arr = (C.c_void_p * len(shards))(*[sh.h for sh in shards])
    return arr


def batch_knn_sharded(metric: str, queries, shards, k: int):
    """`shards`: DeviceBatch row shards (possibly on different devices, each with its index_base). One host thread per
    shard inside the library; the k keys per shard are merged on the host. Returns (idx, scores) of shape (nq, <=k)."""
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    sc = np.zeros((nq, kk), np.float32)
    cnt = C.c_size_t(0)
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    L.call("innr_cuda_batch_knn_sharded", _handle_array(shards), len(shards), m, qs.ctypes.data_as(L.f32p), nq, qlen, k,
           idx.ctypes.data_as(L.u64p), sc.ctypes.data_as(L.f32p), C.byref(cnt))
    return idx[:, :cnt.value], sc[:, :cnt.value]


def hamming_topk_sharded(query_words, shards, k: int):
    qs = np.ascontiguousarray(query_words, dtype=np.uint64)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq = qs.shape[0]
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    ds = np.zeros((nq, kk), np.uint32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_hamming_topk_sharded", _handle_array(shards), len(shards), qs.ctypes.data_as(L.u64p), nq,
           shards[0].dimension, k, idx.ctypes.data_as(L.u64p), ds.ctypes.data_as(L.u32p), C.byref(cnt))
    return idx[:, :cnt.value], ds[:, :cnt.value]


def batch_knn_u8_sharded(queries, shards, k: int):
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    sc = np.zeros((nq, kk), np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_batch_knn_u8_sharded", _handle_array(shards), len(shards), qs.ctypes.data_as(L.f32p), nq, qlen, k,
           idx.ctypes.data_as(L.u64p), sc.ctypes.data_as(L.f32p), C.byref(cnt))
    return idx[:, :cnt.value], sc[:, :cnt.value]


def maxsim_topk_sharded(queries, shards, k: int, cosine: bool = False):
    """maxsim_topk_batch over TokenCorpus shards (document ranges, each with its index_base; on distinct devices the
    lists meet in the peer-mapped exchange, otherwise one host thread per shard and a host merge). `queries`:
    (n_queries, n_q, dim). Equals the unsharded call over the whole document set."""
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    assert qs.ndim == 3, "queries must be (n_queries, n_q, dim)"
    nq = qs.shape[0]
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    sc = np.zeros((nq, kk), np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_maxsim_topk_sharded", _handle_array(shards), len(shards), qs.ctypes.data_as(L.f32p), nq, qs.shape[1],
           qs.shape[2], 1 if cosine else 0, k, idx.ctypes.data_as(L.u64p), sc.ctypes.data_as(L.f32p), C.byref(cnt))
    return idx[:, :cnt.value], sc[:, :cnt.value]
