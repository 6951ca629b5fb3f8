"""Host-side mirror of innr::scalar (src/scalar.rs) over the CUDA C-ABI: `QuantizationParams`, `QuantizedU8`,
`quantize_u8`, `mixed_dot_u8_f32`, `asymmetric_dot_u8`, `batch_knn_u8`, plus the device-resident `U8Corpus`."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from .batch import _Handle


class QuantizationParams:  # src/scalar.rs:44-163
    def __init__(self, alpha: float, offset: float):
        self.alpha = float(np.float32(alpha))
        self.offset = float(np.float32(offset))

    @classmethod
    def from_range(cls, mn: float, mx: float):  # :54-60
        a = np.float32(mx) - np.float32(mn)
        return cls(a if a > 0.0 else 1.0, mn)

    @staticmethod
    def _range(v):
        """min / max as the reference's scan finds them (:76-84): start at f32::MAX / f32::MIN, replace on strict
        `<` / `>` only -- NaN never wins, the first of several equal extremes (e.g. +0.0 before -0.0) is kept."""
        f32max = np.float32(np.finfo(np.float32).max)
        mn, mx = f32max, -f32max
        fin = v[~np.isnan(v)]
        if fin.size:
            lo, hi = fin[np.argmin(fin)], fin[np.argmax(fin)]
            if lo < mn:
                mn = lo
            if hi > mx:
                mx = hi
        return mn, mx

    @classmethod
    def fit(cls, values):  # :68-88 (parameter fitting is a host-side scan in the reference and here)
        v = np.asarray(values, dtype=np.float32).reshape(-1)
        if v.size == 0:
            return cls(1.0, 0.0)
        mn, mx = cls._range(v)
        return cls.from_range(float(mn), float(mx))

    @classmethod
    def fit_quantile(cls, values, quantile: float):  # :104-137 (parameter fitting: a host-side sort, like the reference)
        quantile = np.float32(quantile)
        assert 0.0 < quantile <= 1.0, "quantile must be in (0.0, 1.0]"
        v = np.asarray(values, dtype=np.float32).reshape(-1)
        if v.size == 0:
            return cls(1.0, 0.0)
        if quantile >= 1.0:
            return cls.fit(v)
        v = v[np.isfinite(v)]
        if v.size == 0:
            return cls(1.0, 0.0)
        bits = v.view(np.int32)
        v = v[np.argsort(bits ^ ((bits >> 31) & 0x7FFFFFFF), kind="stable")]  # f32::total_cmp order (-0.0 < +0.0)
        one, two, n = np.float32(1.0), np.float32(2.0), np.float32(v.size)
        tail = (one - quantile) / two
        lo = int(np.floor(tail * n))
        hi = min(int(np.ceil((one - tail) * n)), v.size - 1)
        return cls.from_range(float(v[lo]), float(v[hi]))

    @classmethod
    def fit_vectors(cls, vectors):  # :143-163
        vs = [np.asarray(v, dtype=np.float32).reshape(-1) for v in vectors]
        v = np.concatenate(vs) if vs else np.zeros(0, np.float32)
        mn, mx = cls._range(v)
        if mn > mx:
            return cls(1.0, 0.0)
        return cls.from_range(float(mn), float(mx))


class QuantizedU8:  # src/scalar.rs:171-208
    def __init__(self, data, dimension: int):
        data = np.ascontiguousarray(data, dtype=np.uint8).reshape(-1)
        assert data.size == dimension, f"QuantizedU8: data length {data.size} doesn't match dimension {dimension}"
        self.data = data
        self.dimension = int(dimension)

    def memory_bytes(self) -> int:
        return self.data.size


def quantize_u8(values, params: QuantizationParams) -> QuantizedU8:  # src/scalar.rs:212-225, on the device
    v = np.ascontiguousarray(values, dtype=np.float32).reshape(-1)
    out = np.zeros(v.size, np.uint8)
    L.call("innr_cuda_quantize_u8", v.ctypes.data_as(L.f32p), v.size, C.c_float(params.alpha),
           C.c_float(params.offset), out.ctypes.data_as(L.u8p))
    return QuantizedU8(out, v.size)


class U8Corpus:
    """Device-resident scalar-quantised corpus (16-dimension chunks, chunk-major, u8.cu)."""

    def __init__(self, handle: _Handle, n: int, d: int, params: QuantizationParams, index_base: int = 0):
        self._handle = handle
        self.num_vectors, self.dimension, self.params, self.index_base = int(n), int(d), params, int(index_base)

    @property
    def h(self):
        return self._handle.h

    @classmethod
    def from_f32(cls, batch, params: QuantizationParams):
        """quantize_u8 (src/scalar.rs:212-225) of every vector of a device-resident f32 corpus, on the device."""
        from .batch import _dev
        dev = _dev(batch)
        h = C.c_void_p()
        L.call("innr_cuda_u8_from_f32", dev.h, C.c_float(params.alpha), C.c_float(params.offset), C.byref(h))
        return cls(_Handle(h), dev.num_vectors, dev.dimension, params, dev.index_base)

    @classmethod
    def from_rows(cls, rows, params: QuantizationParams, index_base: int = 0, dimension=None):
        if isinstance(rows, np.ndarray):
            mat = np.ascontiguousarray(rows, dtype=np.uint8)
            if mat.ndim == 1:
                mat = mat.reshape(1, -1)
        else:
            rows = list(rows)
            if rows:
                d0 = rows[0].dimension
                for r in rows:
                    assert r.dimension == d0, "asymmetric_dot_u8_precomputed: dimension mismatch"
                mat = np.stack([r.data for r in rows])
            else:
                mat = np.zeros((0, dimension or 0), np.uint8)
        n, d = mat.shape
        h = C.c_void_p()
        L.call("innr_cuda_upload_u8", mat.ctypes.data_as(L.u8p), n, d, C.c_float(params.alpha),
               C.c_float(params.offset), index_base, C.byref(h))
        return cls(_Handle(h), n, d, params, index_base)

    @classmethod
    def generate(cls, salt: int, first_row: int, n: int, d: int, params: QuantizationParams, index_base: int = 0):
        h = C.c_void_p()
        L.call("innr_cuda_generate_u8", salt, first_row, n, d, C.c_float(params.alpha), C.c_float(params.offset),
               index_base, C.byref(h))
        return cls(_Handle(h), n, d, params, index_base)


def _scores(fn: str, query, corpus: U8Corpus) -> np.ndarray:
    q = np.ascontiguousarray(query, dtype=np.float32).reshape(-1)
    out = np.zeros(corpus.num_vectors, np.float32)
    L.call(fn, corpus.h, q.ctypes.data_as(L.f32p), q.size, out.ctypes.data_as(L.f32p))
    return out


def mixed_dot_u8_all(query, corpus: U8Corpus) -> np.ndarray:
    return _scores("innr_cuda_mixed_dot_u8_all", query, corpus)


def asymmetric_dot_u8_all(query, corpus: U8Corpus) -> np.ndarray:
    return _scores("innr_cuda_asymmetric_dot_u8_all", query, corpus)


def mixed_dot_u8_f32(a, b) -> float:  # src/scalar.rs:314 (pairwise; 1-row corpus)
    a = np.ascontiguousarray(a, dtype=np.float32).reshape(-1)
    b = np.ascontiguousarray(b, dtype=np.uint8).reshape(-1)
    assert a.size == b.size, f"mixed_dot_u8_f32: slice length mismatch ({a.size} vs {b.size})"
    if a.size == 0:
        return 0.0
    return float(mixed_dot_u8_all(a, U8Corpus.from_rows(b.reshape(1, -1), QuantizationParams(1.0, 0.0)))[0])


def asymmetric_dot_u8(query, quantized: QuantizedU8, params: QuantizationParams) -> float:  # src/scalar.rs:261
    q = np.ascontiguousarray(query, dtype=np.float32).reshape(-1)
    assert q.size == quantized.dimension, (
        f"asymmetric_dot_u8: dimension mismatch ({q.size} vs {quantized.dimension})")
    if q.size == 0:
        return 0.0
    return float(asymmetric_dot_u8_all(q, U8Corpus.from_rows(quantized.data.reshape(1, -1), params))[0])


class QueryContext:  # src/scalar.rs:228-232
    def __init__(self, query_sum: float):
        self.query_sum = float(np.float32(query_sum))


def query_context(query) -> QueryContext:  # src/scalar.rs:236-240: sequential f32 sum
    s = np.float32(0.0)
    for x in np.ascontiguousarray(query, dtype=np.float32).reshape(-1):
        s = np.float32(s + x)
    return QueryContext(float(s))


def asymmetric_dot_u8_precomputed(query, quantized: QuantizedU8, params: QuantizationParams, ctx: QueryContext) -> float:
    """src/scalar.rs:286-300: `(alpha / 255) * mixed + offset * ctx.query_sum` with the mixed dot from the device."""
    q = np.ascontiguousarray(query, dtype=np.float32).reshape(-1)
    assert q.size == quantized.dimension, (
        f"asymmetric_dot_u8_precomputed: dimension mismatch ({q.size} vs {quantized.dimension})")
    mixed = np.float32(mixed_dot_u8_f32(q, quantized.data)) if q.size else np.float32(0.0)
    a, o = np.float32(params.alpha), np.float32(params.offset)
    return float(np.float32(np.float32(a / np.float32(255.0)) * mixed) + np.float32(o * np.float32(ctx.query_sum)))


def batch_knn_u8_many(queries, corpus: U8Corpus, k: int):
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    sc = np.zeros((nq, kk), np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_batch_knn_u8", corpus.h, qs.ctypes.data_as(L.f32p), nq, qlen, k, idx.ctypes.data_as(L.u64p),
           sc.ctypes.data_as(L.f32p), C.byref(cnt))
    return idx[:, :cnt.value], sc[:, :cnt.value]


def u8_tc_debug_bounds(queries, corpus: U8Corpus):
    """Test hook (include/innr_cuda.h: innr_cuda_u8_tc_debug_bounds): the u8 tensor-core filter's score interval for
    every (query, row < min(N, 4096)) pair exactly as production computes it. Returns (lower[nq, rows], upper[nq, rows],
    qflags[nq])."""
    qs = np.ascontiguousarray(queries, dtype=np.float32)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq, qlen = qs.shape
    lower = np.zeros((nq, 4096), np.float32)
    upper = np.zeros((nq, 4096), np.float32)
    rows = C.c_size_t(0)
    flags = np.zeros(nq, np.uint32)
    L.call("innr_cuda_u8_tc_debug_bounds", corpus.h, qs.ctypes.data_as(L.f32p), nq, qlen, lower.ctypes.data_as(L.f32p),
           upper.ctypes.data_as(L.f32p), C.byref(rows), flags.ctypes.data_as(L.u32p))
    r = rows.value
    return lower.reshape(-1)[:nq * r].reshape(nq, r), upper.reshape(-1)[:nq * r].reshape(nq, r), flags


def batch_knn_u8(query, corpus, params: QuantizationParams, k: int):  # src/scalar.rs:370-393 -> Vec<(usize, f32)>
    if not isinstance(corpus, U8Corpus):
        if len(corpus) == 0 or k == 0:
            return []
        corpus = U8Corpus.from_rows(corpus, params)
    if corpus.num_vectors == 0 or k == 0:
        return []
    idx, sc = batch_knn_u8_many(np.ascontiguousarray(query, dtype=np.float32).reshape(1, -1), corpus, k)
    return [(int(i), float(s)) for i, s in zip(idx[0], sc[0])]
