"""Host-side mirror of innr::binary (src/binary.rs) over the CUDA C-ABI: `PackedBinary`, `encode_binary`,
`binary_hamming`, `binary_dot`, `binary_jaccard`, plus the corpus-level entries the device path adds (`BinaryCorpus`, `hamming_topk`) for the
caller composition in examples/binary_demo.rs:174-180."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from .batch import _Handle


class PackedBinary:  # src/binary.rs:37-117
    def __init__(self, data, dimension: int):
        data = np.array(data, dtype=np.uint64).reshape(-1)
        expect = (dimension + 63) // 64
        assert data.size == expect, (
            f"PackedBinary: data length {data.size} doesn't match dimension {dimension} (expected {expect} words)")
        rem = dimension % 64
        if rem and data.size:  # mask padding past `dimension` (src/binary.rs:59-66)
            data[-1] &= np.uint64((1 << rem) - 1)
        self.data = data
        self.dimension = int(dimension)

    @classmethod
    def zeros(cls, dimension: int):
        return cls(np.zeros((dimension + 63) // 64, np.uint64), dimension)

    def set(self, idx: int, val: bool):
        if idx >= self.dimension:
            return
        w, b = idx // 64, idx % 64
        if val:
            self.data[w] |= np.uint64(1 << b)
        else:
            self.data[w] &= np.uint64(~(1 << b) & 0xFFFFFFFFFFFFFFFF)

    def get(self, idx: int) -> bool:
        if idx >= self.dimension:
            return False
        return bool((int(self.data[idx // 64]) >> (idx % 64)) & 1)

    def memory_bytes(self) -> int:
        return self.data.size * 8


def encode_binary(values, threshold: float) -> PackedBinary:  # src/binary.rs:133-141, on the device
    v = np.ascontiguousarray(values, dtype=np.float32).reshape(-1)
    out = np.zeros((v.size + 63) // 64, np.uint64)
    L.call("innr_cuda_encode_binary", v.ctypes.data_as(L.f32p), v.size, C.c_float(threshold),
           out.ctypes.data_as(L.u64p))
    return PackedBinary(out, v.size)


class BinaryCorpus:
    """Device-resident set of packed codes (chunk-major layout, hamming.cu)."""

    def __init__(self, handle: _Handle, n: int, dimension: int, index_base: int = 0):
        self._handle = handle
        self.num_codes = int(n)
        self.dimension = int(dimension)
        self.index_base = int(index_base)

    @property
    def h(self):
        return self._handle.h

    @classmethod
    def from_words(cls, words, n: int, dimension: int, index_base: int = 0):
        w = np.ascontiguousarray(words, dtype=np.uint64).reshape(-1)
        assert w.size == n * ((dimension + 63) // 64)
        h = C.c_void_p()
        L.call("innr_cuda_upload_binary", w.ctypes.data_as(L.u64p), n, dimension, index_base, C.byref(h))
        return cls(_Handle(h), n, dimension, index_base)

    @classmethod
    def from_codes(cls, codes, index_base: int = 0):
        codes = list(codes)
        if not codes:
            return cls.from_words(np.zeros(0, np.uint64), 0, 0, index_base)
        dim = codes[0].dimension
        for c in codes:
            assert c.dimension == dim, "innr::binary_hamming: dimension mismatch"
        return cls.from_words(np.stack([c.data for c in codes]) if dim else np.zeros(0, np.uint64), len(codes), dim,
                              index_base)

    @classmethod
    def from_f32(cls, batch, threshold: float = 0.0):
        """encode_binary (src/binary.rs:133-141) of every vector of a device-resident f32 corpus, on the device."""
        from .batch import _dev
        dev = _dev(batch)
        h = C.c_void_p()
        L.call("innr_cuda_binary_from_f32", dev.h, C.c_float(threshold), C.byref(h))
        return cls(_Handle(h), dev.num_vectors, dev.dimension, dev.index_base)

    @classmethod
    def generate(cls, salt: int, first_row: int, n: int, dimension: int, index_base: int = 0):
        h = C.c_void_p()
        L.call("innr_cuda_generate_binary", salt, first_row, n, dimension, index_base, C.byref(h))
        return cls(_Handle(h), n, dimension, index_base)


def hamming_all(query: PackedBinary, corpus: BinaryCorpus) -> np.ndarray:
    out = np.zeros(corpus.num_codes, np.uint32)
    q = np.ascontiguousarray(query.data, dtype=np.uint64)
    L.call("innr_cuda_hamming_all", corpus.h, q.ctypes.data_as(L.u64p), query.dimension, out.ctypes.data_as(L.u32p))
    return out


def binary_dot_all(query: PackedBinary, corpus: BinaryCorpus) -> np.ndarray:
    out = np.zeros(corpus.num_codes, np.uint32)
    q = np.ascontiguousarray(query.data, dtype=np.uint64)
    L.call("innr_cuda_binary_dot_all", corpus.h, q.ctypes.data_as(L.u64p), query.dimension, out.ctypes.data_as(L.u32p))
    return out


def binary_jaccard_all(query: PackedBinary, corpus: BinaryCorpus) -> np.ndarray:
    out = np.zeros(corpus.num_codes, np.float32)
    q = np.ascontiguousarray(query.data, dtype=np.uint64)
    L.call("innr_cuda_binary_jaccard_all", corpus.h, q.ctypes.data_as(L.u64p), query.dimension,
           out.ctypes.data_as(L.f32p))
    return out


def binary_topk(op: str, query: PackedBinary, corpus: BinaryCorpus, k: int):
    """Top-k codes by `binary_dot` ("dot") or `binary_jaccard` ("jaccard"), descending, ties -> lower index.
    Returns (indices uint64[m], scores float32[m])."""
    kk = max(min(k, corpus.num_codes), 1)
    idx = np.zeros(kk, np.uint64)
    sc = np.zeros(kk, np.float32)
    cnt = C.c_size_t(0)
    q = np.ascontiguousarray(query.data, dtype=np.uint64)
    L.call("innr_cuda_binary_topk", corpus.h, {"dot": 0, "jaccard": 1}[op], q.ctypes.data_as(L.u64p), query.dimension, k,
           idx.ctypes.data_as(L.u64p), sc.ctypes.data_as(L.f32p), C.byref(cnt))
    return idx[:cnt.value], sc[:cnt.value]


def binary_topk_many(op: str, queries, corpus: BinaryCorpus, k: int):
    """`binary_topk` for a batch of query codes in one call ((nq, words) uint64, or PackedBinary codes): the same
    results as one `binary_topk` per query. Returns (indices uint64[nq, m], scores float32[nq, m]), m = min(k, n)."""
    if len(queries) and isinstance(queries[0], PackedBinary):
        queries = np.stack([np.asarray(q.data, dtype=np.uint64) for q in queries])
    qs = np.ascontiguousarray(queries, dtype=np.uint64)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq = qs.shape[0]
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    sc = np.zeros((nq, kk), np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_binary_topk_batch", corpus.h, {"dot": 0, "jaccard": 1}[op], qs.ctypes.data_as(L.u64p), nq,
           corpus.dimension, k, idx.ctypes.data_as(L.u64p), sc.ctypes.data_as(L.f32p), C.byref(cnt))
    return idx[:, :cnt.value], sc[:, :cnt.value]


def binary_topk_keys_dev(op: str, dev_query_words, corpus: BinaryCorpus, k: int, dev_keys, stream=None):
    """Device-resident batch: dev_query_words a CUDA uint64 tensor (nq, 2 * ceil(dim / 128)), zero padded; dev_keys a
    CUDA int64 tensor (nq, k) receiving the keys (include/innr_cuda.h). Enqueued on `stream` (torch stream or None for
    the current one); returns at once."""
    import torch
    s = stream if stream is not None else torch.cuda.current_stream(dev_query_words.device)
    L.call("innr_cuda_binary_topk_keys_dev", corpus.h, {"dot": 0, "jaccard": 1}[op], C.c_void_p(dev_query_words.data_ptr()),
           dev_query_words.shape[0], k, C.c_void_p(dev_keys.data_ptr()), C.c_void_p(s.cuda_stream))


def binary_dot(a: PackedBinary, b: PackedBinary) -> int:  # src/binary.rs:178 (pairwise; 1-code corpus)
    assert a.dimension == b.dimension
    if a.dimension == 0:
        return 0
    return int(binary_dot_all(a, BinaryCorpus.from_codes([b]))[0])


def binary_jaccard(a: PackedBinary, b: PackedBinary) -> float:  # src/binary.rs:198
    assert a.dimension == b.dimension
    if a.dimension == 0:
        return 1.0
    return float(binary_jaccard_all(a, BinaryCorpus.from_codes([b]))[0])


def binary_hamming(a: PackedBinary, b: PackedBinary) -> int:  # src/binary.rs:154 (pairwise; 1-code corpus)
    assert a.dimension == b.dimension, (
        f"innr::binary_hamming: dimension mismatch ({a.dimension} vs {b.dimension})")
    if a.dimension == 0:
        return 0
    return int(hamming_all(a, BinaryCorpus.from_codes([b]))[0])


def hamming_topk_many(query_words, corpus: BinaryCorpus, k: int):
    qs = np.ascontiguousarray(query_words, dtype=np.uint64)
    if qs.ndim == 1:
        qs = qs.reshape(1, -1)
    nq = qs.shape[0]
    kk = max(k, 1)
    idx = np.zeros((nq, kk), np.uint64)
    ds = np.zeros((nq, kk), np.uint32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_hamming_topk", corpus.h, qs.ctypes.data_as(L.u64p), nq, corpus.dimension, k,
           idx.ctypes.data_as(L.u64p), ds.ctypes.data_as(L.u32p), C.byref(cnt))
    return idx[:, :cnt.value], ds[:, :cnt.value]


def hamming_topk(query_words, codes, k: int):
    """examples/binary_demo.rs:174-180 as one call. `codes`: BinaryCorpus, or an (n, words) uint64 array."""
    q = np.ascontiguousarray(query_words, dtype=np.uint64).reshape(-1)
    if not isinstance(codes, BinaryCorpus):
        c = np.ascontiguousarray(codes, dtype=np.uint64).reshape(-1, max(q.size, 1))
        codes = BinaryCorpus.from_words(c, c.shape[0], q.size * 64)
    idx, ds = hamming_topk_many(q.reshape(1, -1), codes, k)
    return idx[0], ds[0]
