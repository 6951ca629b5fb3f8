"""Asynchronous host-buffer top-k (include/innr_cuda.h: innr_cuda_*_async / innr_cuda_ticket_wait).

`submit_*` queues a call and returns a Ticket at once; `Ticket.wait()` blocks on that call only and returns what the
synchronous function returns (same arrays, same bits). Two tickets per device may be in flight: submitting call i + 1
before waiting for call i keeps two shard scans overlapping on the device.

    pending = None
    for q in queries:
        t = stream.submit_knn("cosine", q, corpus, 10)
        if pending is not None:
            use(pending.wait())
        pending = t
    use(pending.wait())
"""
import ctypes as C

import numpy as np

from . import _lib as L


class Ticket:
    def __init__(self, handle, kind: str, nq: int, k: int):
        self._h, self.kind, self.nq, self.k = handle, kind, nq, k

    def __del__(self):
        # a ticket dropped without a wait still occupies one of the device's two slots: collect it
        try:
            if getattr(self, "_h", None) is not None:
                self.wait()
        except Exception:
            pass

    def wait(self):
        """(idx[nq, min(k, N)], scores-or-distances[nq, min(k, N)]); a ticket can be waited for once."""
        if self._h is None:
            raise L.InnrCudaError("ticket was already waited for")
        if not self._h:  # the library hands out no ticket for an empty result (sharded forms)
            self._h = None
            return (np.zeros((self.nq, 0), np.uint64),
                    np.zeros((self.nq, 0), np.uint32 if self.kind == "binary" else np.float32))
        kk = max(self.k, 1)
        idx = np.zeros((self.nq, kk), np.uint64)
        cnt = C.c_size_t(0)
        h, self._h = self._h, None
        if self.kind == "binary":
            ds = np.zeros((self.nq, kk), np.uint32)
            L.call("innr_cuda_ticket_wait", h, idx.ctypes.data_as(L.u64p), None, ds.ctypes.data_as(L.u32p), C.byref(cnt))
            return idx[:, :cnt.value], ds[:, :cnt.value]
        sc = np.zeros((self.nq, kk), np.float32)
        L.call("innr_cuda_ticket_wait", h, idx.ctypes.data_as(L.u64p), sc.ctypes.data_as(L.f32p), None, C.byref(cnt))
        return idx[:, :cnt.value], sc[:, :cnt.value]


def submit_knn(metric: str, queries, batch, k: int) -> Ticket:
    """batch_knn / batch_knn_dot / batch_knn_cosine (src/batch.rs:385,742,777) over a DeviceBatch, queued."""
    from .batch import _dev, _f32
    dev = _dev(batch)
    qs = _f32(queries)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    h = C.c_void_p()
    L.call("innr_cuda_batch_knn_async", dev.h, m, qs.ctypes.data_as(L.f32p), nq, qlen, k, C.byref(h))
    return Ticket(h, "f32", nq, k)


def submit_hamming_topk(query_words, corpus, k: int) -> Ticket:
    """Hamming top-k over a BinaryCorpus (examples/binary_demo.rs:174-180), queued."""
    qs = np.ascontiguousarray(query_words, dtype=np.uint64)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    h = C.c_void_p()
    L.call("innr_cuda_hamming_topk_async", corpus.h, qs.ctypes.data_as(L.u64p), qs.shape[0], corpus.dimension, k, C.byref(h))
    return Ticket(h, "binary", qs.shape[0], k)


def submit_knn_u8(queries, corpus, k: int) -> Ticket:
    """batch_knn_u8 (src/scalar.rs:370-393) over a U8Corpus, queued."""
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    h = C.c_void_p()
    L.call("innr_cuda_batch_knn_u8_async", corpus.h, qs.ctypes.data_as(L.f32p), nq, qlen, k, C.byref(h))
    return Ticket(h, "u8", nq, k)


def submit_maxsim_topk(queries, corpus, k: int, cosine: bool = False) -> Ticket:
    """maxsim_topk_batch over a TokenCorpus (`queries`: (n_queries, n_q, dim)), queued. Each of the device's two slots
    owns its score vectors, so two calls in flight never share scratch."""
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    assert qs.ndim == 3, "queries must be (n_queries, n_q, dim)"
    h = C.c_void_p()
    L.call("innr_cuda_maxsim_topk_async", corpus.h, qs.ctypes.data_as(L.f32p), qs.shape[0], qs.shape[1], qs.shape[2],
           1 if cosine else 0, k, C.byref(h))
    return Ticket(h, "maxsim", qs.shape[0], k)


# ---- row shards on different devices of this process (innr_cuda_*_sharded_async): one ticket per call ------------------
def _shard_handles(shards):
    return (C.c_void_p * len(shards))(*[sh.h for sh in shards])


def submit_knn_sharded(metric: str, queries, shards, k: int) -> Ticket:
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    h = C.c_void_p()
    L.call("innr_cuda_batch_knn_sharded_async", _shard_handles(shards), len(shards), m, qs.ctypes.data_as(L.f32p), nq, qlen, k,
           C.byref(h))
    return Ticket(h, "f32", nq, k)


def submit_hamming_topk_sharded(query_words, shards, k: int) -> Ticket:
    qs = np.ascontiguousarray(query_words, dtype=np.uint64)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    h = C.c_void_p()
    L.call("innr_cuda_hamming_topk_sharded_async", _shard_handles(shards), len(shards), qs.ctypes.data_as(L.u64p), qs.shape[0],
           shards[0].dimension, k, C.byref(h))
    return Ticket(h, "binary", qs.shape[0], k)


def submit_knn_u8_sharded(queries, shards, k: int) -> Ticket:
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    h = C.c_void_p()
    L.call("innr_cuda_batch_knn_u8_sharded_async", _shard_handles(shards), len(shards), qs.ctypes.data_as(L.f32p), nq, qlen, k,
           C.byref(h))
    return Ticket(h, "u8", nq, k)


def submit_maxsim_topk_sharded(queries, shards, k: int, cosine: bool = False) -> Ticket:
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    assert qs.ndim == 3, "queries must be (n_queries, n_q, dim)"
    h = C.c_void_p()
    L.call("innr_cuda_maxsim_topk_sharded_async", _shard_handles(shards), len(shards), qs.ctypes.data_as(L.f32p), qs.shape[0],
           qs.shape[1], qs.shape[2], 1 if cosine else 0, k, C.byref(h))
    return Ticket(h, "maxsim", qs.shape[0], k)
