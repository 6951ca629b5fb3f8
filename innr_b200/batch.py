"""Host-side mirror of innr::batch (src/batch.rs) over the CUDA C-ABI.

Same names, argument meaning and error behaviour as the reference: `VerticalBatch`, `batch_dot`,
`batch_l2_squared`, `batch_norms`, `batch_cosine`, `batch_knn`, `batch_knn_dot`, `batch_knn_cosine`,
`BatchKnnResult`. A `VerticalBatch` keeps the reference's host-visible dimension-major buffer
(`data[d*N + i]`, src/batch.rs:69) for the accessors and owns a device-resident copy (uploaded once, lazily)
that every batch_* call scans. `DeviceBatch` is the same thing without a host copy (corpora generated on
the device or too large for host RAM).
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L


def _f32(a) -> np.ndarray:
    return np.ascontiguousarray(a, dtype=np.float32)


def _ptr(a: np.ndarray, ty):
    return a.ctypes.data_as(ty)


class _Handle:
    """Owns an innr_cuda_corpus*."""

    def __init__(self, h: C.c_void_p):
        self.h = h

    def __del__(self):
        h, self.h = getattr(self, "h", None), None
        if h:
            try:
                L.lib().innr_cuda_free(h)
            except Exception:
                pass


class DeviceBatch:
    """A device-resident PDX shard (no host copy). `index_base` makes reported indices global."""

    def __init__(self, handle: _Handle, num_vectors: int, dimension: int, index_base: int = 0):
        self._handle = handle
        self.num_vectors = int(num_vectors)
        self.dimension = int(dimension)
        self.index_base = int(index_base)

    @property
    def h(self):
        return self._handle.h

    @classmethod
    def generate(cls, generator: str, salt: int, first_row: int, n: int, d: int, index_base: int = 0):
        """generator: 'ghash' (SURVEY.md 8d) or 'gref' (examples/batch_demo.rs:233-242, seed = salt + row)."""
        h = C.c_void_p()
        L.call("innr_cuda_generate_f32_pdx", {"ghash": 0, "gref": 1}[generator], salt, first_row, n, d, index_base,
               C.byref(h))
        return cls(_Handle(h), n, d, index_base)

    @classmethod
    def from_pdx(cls, pdx, n: int, d: int, index_base: int = 0):
        pdx = _f32(pdx).reshape(-1)
        assert pdx.size == n * d
        h = C.c_void_p()
        L.call("innr_cuda_upload_f32_pdx", _ptr(pdx, L.f32p), n, d, index_base, C.byref(h))
        return cls(_Handle(h), n, d, index_base)

    @classmethod
    def from_rows_flat(cls, rows, n: int, d: int, index_base: int = 0):
        rows = _f32(rows).reshape(-1)
        assert rows.size == n * d
        h = C.c_void_p()
        L.call("innr_cuda_upload_f32_rows", _ptr(rows, L.f32p), n, d, index_base, C.byref(h))
        return cls(_Handle(h), n, d, index_base)

    @classmethod
    def wrap_device(cls, dev_ptr: int, n: int, d: int, ld: int, index_base: int = 0, keepalive=None):
        h = C.c_void_p()
        L.call("innr_cuda_wrap_f32_pdx_dev", C.c_void_p(dev_ptr), n, d, ld, index_base, C.byref(h))
        b = cls(_Handle(h), n, d, index_base)
        b._keepalive = keepalive
        return b

    def prefix(self, prefix_dim: int) -> "DeviceBatch":
        """Zero-copy view of the first `prefix_dim` dimensions (Matryoshka prefix, src/dense.rs:436-462)."""
        h = C.c_void_p()
        L.call("innr_cuda_prefix_view", self.h, prefix_dim, C.byref(h))
        v = DeviceBatch(_Handle(h), self.num_vectors, min(prefix_dim, self.dimension), self.index_base)
        v._keepalive = self  # the view does not own the device memory
        return v

    def extract_vector(self, i: int) -> np.ndarray:
        out = np.zeros(self.dimension, np.float32)
        L.call("innr_cuda_extract_vector", self.h, i, _ptr(out, L.f32p))
        return out

    def device_bytes(self) -> int:
        v = C.c_size_t(0)
        L.call("innr_cuda_corpus_info", self.h, None, None, None, None, None, C.byref(v))
        return int(v.value)


class VerticalBatch:
    """src/batch.rs:88-220. Host accessors read the dimension-major buffer; scans run on the device copy."""

    def __init__(self, data: np.ndarray, num_vectors: int, dimension: int):
        self.data = _f32(data).reshape(-1)
        self.num_vectors = int(num_vectors)
        self.dimension = int(dimension)
        assert self.data.size == self.num_vectors * self.dimension
        self._dev = None

    # --- constructors -------------------------------------------------------------------------------
    @classmethod
    def from_rows(cls, rows) -> "VerticalBatch":  # src/batch.rs:103
        if len(rows) == 0:
            return cls(np.zeros(0, np.float32), 0, 0)
        d = len(rows[0])
        for r in rows:
            assert len(r) == d, "Inconsistent vector dimension"  # src/batch.rs:120
        flat = _f32(np.array(rows, dtype=np.float32).reshape(len(rows), d))
        return cls.from_flat(flat.reshape(-1), len(rows), d)

    from_slices = from_rows  # src/batch.rs:138

    @classmethod
    def from_flat(cls, data, num_vectors: int, dimension: int) -> "VerticalBatch":  # src/batch.rs:167
        data = _f32(data).reshape(-1)
        assert data.size == num_vectors * dimension
        # The host-visible dimension-major buffer (what VerticalBatch::data() exposes, src/batch.rs:212) is a
        # plain re-striding of the caller's rows; the device copy is uploaded from it on first use.
        # (DeviceBatch.from_rows_flat does the same transpose on the device for corpora that never need
        # host accessors.)
        pdx = np.ascontiguousarray(data.reshape(num_vectors, dimension).T).reshape(-1)
        return cls(pdx, num_vectors, dimension)

    # --- accessors (src/batch.rs:187-220) -----------------------------------------------------------------
    def get(self, dim: int, vec_idx: int) -> float:
        return float(self.data[dim * self.num_vectors + vec_idx])

    def dimension_slice(self, dim: int) -> np.ndarray:
        return self.data[dim * self.num_vectors:(dim + 1) * self.num_vectors]

    def extract_vector(self, vec_idx: int) -> np.ndarray:
        if self.dimension == 0:
            return np.zeros(0, np.float32)
        return self.device().extract_vector(vec_idx)

    def device(self) -> DeviceBatch:
        if self._dev is None:
            self._dev = DeviceBatch.from_pdx(self.data, self.num_vectors, self.dimension)
        return self._dev


def _dev(batch) -> DeviceBatch:
    return batch.device() if isinstance(batch, VerticalBatch) else batch


class BatchKnnResult:  # src/batch.rs:368-377
    def __init__(self, indices, scores):
        self.indices = [int(i) for i in indices]
        self.scores = np.asarray(scores, dtype=np.float32)

    def __eq__(self, other):
        return self.indices == other.indices and self.scores.tobytes() == other.scores.tobytes()

    def __repr__(self):
        return f"BatchKnnResult(indices={self.indices}, scores={self.scores.tolist()})"


def _scores(fn: str, query, batch) -> np.ndarray:
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    out = np.zeros(dev.num_vectors, np.float32)
    L.call(fn, dev.h, _ptr(q, L.f32p), q.size, _ptr(out, L.f32p))
    return out


def batch_l2_squared(query, batch) -> np.ndarray:  # src/batch.rs:236
    return _scores("innr_cuda_batch_l2_squared", query, batch)


def batch_dot(query, batch) -> np.ndarray:  # src/batch.rs:270
    return _scores("innr_cuda_batch_dot", query, batch)


def batch_norms(batch) -> np.ndarray:  # src/batch.rs:663
    dev = _dev(batch)
    out = np.zeros(dev.num_vectors, np.float32)
    L.call("innr_cuda_batch_norms", dev.h, _ptr(out, L.f32p))
    return out


def batch_cosine(query, batch, norms) -> np.ndarray:  # src/batch.rs:690
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    nr = _f32(norms).reshape(-1)
    out = np.zeros(dev.num_vectors, np.float32)
    L.call("innr_cuda_batch_cosine", dev.h, _ptr(q, L.f32p), q.size, _ptr(nr, L.f32p), nr.size, _ptr(out, L.f32p))
    return out


def _into(out: list, values) -> None:
    """The reference's `_into` contract: the caller's buffer is cleared, then filled (resized to N)."""
    out.clear()
    out.extend(float(x) for x in values)


def batch_l2_squared_into(query, batch, out: list) -> None:  # src/batch.rs:250
    _into(out, batch_l2_squared(query, batch))


def batch_dot_into(query, batch, out: list) -> None:  # src/batch.rs:284
    _into(out, batch_dot(query, batch))


def batch_norms_into(batch, out: list) -> None:  # src/batch.rs:672
    _into(out, batch_norms(batch))


def batch_cosine_into(query, batch, norms, out: list) -> None:  # src/batch.rs:705
    _into(out, batch_cosine(query, batch, norms))


def batch_dimension_variance(batch) -> np.ndarray:  # src/batch.rs:572
    """Variance of every dimension row (the reference's sequential sums, bit for bit); zeros for <= 1 vector."""
    dev = _dev(batch)
    out = np.zeros(dev.dimension, np.float32)
    L.call("innr_cuda_batch_dimension_variance", dev.h, _ptr(out, L.f32p), out.size)
    return out


def batch_knn_reordered(query, batch, k: int) -> BatchKnnResult:  # src/batch.rs:621
    """Exact L2 kNN with the dimensions accumulated in decreasing-variance order; ties -> lower index."""
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    assert q.size == dev.dimension, "query.len() != batch.dimension"
    kk = max(min(k, dev.num_vectors), 1)
    idx = np.zeros(kk, np.uint64)
    sc = np.zeros(kk, np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_batch_knn_reordered", dev.h, _ptr(q, L.f32p), q.size, k, _ptr(idx, L.u64p), _ptr(sc, L.f32p),
           C.byref(cnt))
    return BatchKnnResult(idx[:cnt.value], sc[:cnt.value])


def batch_knn_adaptive(query, batch, k: int, warmup_dims: int) -> BatchKnnResult:  # src/batch.rs:441
    """The reference's approximate early-termination kNN, reproduced exactly (same survivors, distances and order)."""
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    assert q.size == dev.dimension, "query.len() != batch.dimension"
    assert warmup_dims > 0, "warmup_dims must be > 0"
    kk = max(min(k, dev.num_vectors), 1)
    idx = np.zeros(kk, np.uint64)
    sc = np.zeros(kk, np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_batch_knn_adaptive", dev.h, _ptr(q, L.f32p), q.size, k, warmup_dims, _ptr(idx, L.u64p),
           _ptr(sc, L.f32p), C.byref(cnt))
    return BatchKnnResult(idx[:cnt.value], sc[:cnt.value])


def batch_knn_many(metric: str, queries, batch, k: int):
    """n_queries x d queries in one call (shares corpus passes between queries). Returns (idx, scores) arrays
    of shape (n_queries, min(k, N))."""
    dev = _dev(batch)
    qs = _f32(queries)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    sc = np.zeros((nq, kk), np.float32)
    cnt = C.c_size_t(0)
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    L.call("innr_cuda_batch_knn", dev.h, m, _ptr(qs, L.f32p), nq, qlen, k, _ptr(idx, L.u64p), _ptr(sc, L.f32p),
           C.byref(cnt))
    return idx[:, :cnt.value], sc[:, :cnt.value]


def knn_tc_debug_bounds(metric: str, queries, batch):
    """Test hook (include/innr_cuda.h: innr_cuda_knn_tc_debug_bounds): the tensor-core filter's LOWER bound for every
    (query, row < min(N, 4096)) pair exactly as production computes it. Returns (lower[nq, rows], eps, qflags[nq])."""
    dev = _dev(batch)
    qs = _f32(queries)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    lower = np.zeros((nq, 4096), np.float32)
    rows, eps = C.c_size_t(0), C.c_float(0)
    flags = np.zeros(nq, np.uint32)
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    L.call("innr_cuda_knn_tc_debug_bounds", dev.h, m, _ptr(qs, L.f32p), nq, qlen, _ptr(lower, L.f32p), C.byref(rows),
           C.byref(eps), _ptr(flags, L.u32p))
    return lower.reshape(-1)[:nq * rows.value].reshape(nq, rows.value), float(eps.value), flags


def knn_screen_debug_bounds(metric: str, query, batch):
    """Test hook (include/innr_cuda.h: innr_cuda_knn_screen_debug_bounds): the screened kNN's interval for every row of a
    split corpus. Returns (lower[n], upper[n])."""
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    lower = np.zeros(dev.num_vectors, np.float32)
    upper = np.zeros(dev.num_vectors, np.float32)
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    L.call("innr_cuda_knn_screen_debug_bounds", dev.h, m, _ptr(q, L.f32p), q.size, _ptr(lower, L.f32p), _ptr(upper, L.f32p))
    return lower, upper


def _knn(metric: str, query, batch, k: int) -> BatchKnnResult:
    q = _f32(query).reshape(1, -1)
    idx, sc = batch_knn_many(metric, q, batch, k)
    return BatchKnnResult(idx[0], sc[0])


def batch_knn(query, batch, k: int) -> BatchKnnResult:  # src/batch.rs:385 (squared L2, ascending)
    return _knn("l2", query, batch, k)


def batch_knn_dot(query, batch, k: int) -> BatchKnnResult:  # src/batch.rs:742 (descending)
    return _knn("dot", query, batch, k)


def batch_knn_cosine(query, batch, k: int) -> BatchKnnResult:  # src/batch.rs:777 (descending)
    return _knn("cosine", query, batch, k)


def batch_knn_filtered(query, batch, k: int, predicate) -> BatchKnnResult:  # src/batch.rs:820-882
    """`predicate(index) -> bool` is evaluated on the host into a bitmask (the reference builds `mask: Vec<bool>` the
    same way, :839); a numpy bool array of length N is accepted directly. Squared L2 of the passing vectors only."""
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    assert q.size == dev.dimension, "query.len() != batch.dimension"
    n = dev.num_vectors
    if isinstance(predicate, np.ndarray):
        bits = predicate.astype(bool).reshape(-1)
        assert bits.size == n
    else:
        bits = np.fromiter((bool(predicate(i)) for i in range(n)), dtype=bool, count=n)
    words = np.zeros((n + 63) // 64 + 1, np.uint64)
    packed = np.packbits(bits, bitorder="little")
    words.view(np.uint8)[:packed.size] = packed
    kk = max(k, 1)
    idx = np.zeros(kk, np.uint64)
    sc = np.zeros(kk, np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_batch_knn_filtered", dev.h, _ptr(q, L.f32p), q.size, k, _ptr(words, L.u64p), words.size,
           _ptr(idx, L.u64p), _ptr(sc, L.f32p), C.byref(cnt))
    return BatchKnnResult(idx[:cnt.value], sc[:cnt.value])


def batch_l2_squared_pruning(query, batch, threshold: float):  # src/batch.rs:320-365
    """[(index, squared distance)] of the vectors none of whose partial distances exceeded `threshold`."""
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    assert q.size == dev.dimension, "query.len() != batch.dimension"
    n = dev.num_vectors
    idx = np.zeros(max(n, 1), np.uint64)
    ds = np.zeros(max(n, 1), np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_batch_l2_squared_pruning", dev.h, _ptr(q, L.f32p), q.size, float(threshold), _ptr(idx, L.u64p),
           _ptr(ds, L.f32p), n, C.byref(cnt))
    m = cnt.value
    return [(int(idx[j]), float(ds[j])) for j in range(m)]


def batch_knn_subset(metric: str, query, batch, candidates, k: int) -> BatchKnnResult:
    """Exact re-rank of `candidates` (distinct global indices): the reference's batch_knn / batch_knn_dot /
    batch_knn_cosine over the sub-batch of those vectors, original indices reported (second stage of the two-stage
    retrieval the reference documents, src/scalar.rs:366-368, examples/binary_demo.rs:235-237)."""
    dev = _dev(batch)
    q = _f32(query).reshape(-1)
    assert q.size == dev.dimension, "query.len() != batch.dimension"
    cand = np.ascontiguousarray(candidates, dtype=np.uint64).reshape(-1)
    kk = max(min(k, cand.size), 1)
    idx = np.zeros(kk, np.uint64)
    sc = np.zeros(kk, np.float32)
    cnt = C.c_size_t(0)
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    L.call("innr_cuda_batch_knn_subset", dev.h, m, _ptr(q, L.f32p), q.size, _ptr(cand, L.u64p), cand.size, k,
           _ptr(idx, L.u64p), _ptr(sc, L.f32p), C.byref(cnt))
    return BatchKnnResult(idx[:cnt.value], sc[:cnt.value])
