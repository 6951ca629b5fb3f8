"""Host-side mirror of innr::maxsim (src/maxsim.rs) over the CUDA C-ABI: pairwise `maxsim` / `maxsim_cosine`
(same signatures as the reference) and the corpus-level `TokenCorpus` + `maxsim_corpus` the device path adds for
the caller loop in examples/maxsim_colbert.rs:171-174."""
from __future__ import annotations

import ctypes as C

import numpy as np

from . import _lib as L
from .batch import _Handle


def _tokens(t, what: str) -> np.ndarray:
    if isinstance(t, np.ndarray) and t.ndim == 2:
        return np.ascontiguousarray(t, dtype=np.float32)
    t = list(t)
    if len(t) == 0:
        return np.zeros((0, 0), np.float32)
    dim = len(t[0])
    assert all(len(x) == dim for x in t), f"dimension mismatch ({what})"  # src/maxsim.rs:103-110
    return np.ascontiguousarray(np.array(t, dtype=np.float32).reshape(len(t), dim))


class TokenCorpus:
    """Device-resident document set: total_tokens x dim token matrix + per-document offsets."""

    def __init__(self, handle: _Handle, n_docs: int, dim: int, index_base: int = 0):
        self._handle = handle
        self.num_docs, self.dimension, self.index_base = int(n_docs), int(dim), int(index_base)

    @property
    def h(self):
        return self._handle.h

    @classmethod
    def from_tokens(cls, tokens, doc_offsets, dim: int, index_base: int = 0):
        t = np.ascontiguousarray(tokens, dtype=np.float32).reshape(-1)
        off = np.ascontiguousarray(doc_offsets, dtype=np.uint64).reshape(-1)
        n_docs = max(off.size - 1, 0)
        h = C.c_void_p()
        L.call("innr_cuda_upload_tokens", t.ctypes.data_as(L.f32p), off.ctypes.data_as(L.u64p), n_docs, dim,
               index_base, C.byref(h))
        return cls(_Handle(h), n_docs, dim, index_base)

    @classmethod
    def generate(cls, salt: int, first_doc: int, n_docs: int, tokens_per_doc: int, dim: int, index_base: int = 0):
        h = C.c_void_p()
        L.call("innr_cuda_generate_tokens", salt, first_doc, n_docs, tokens_per_doc, dim, index_base, C.byref(h))
        return cls(_Handle(h), n_docs, dim, index_base)


def maxsim_corpus(query_tokens, corpus: TokenCorpus, cosine: bool = False, out: np.ndarray | None = None) -> np.ndarray:
    """Scores of every document. `out` (float32, num_docs, C-contiguous) lets the caller own the result buffer, as the
    C-ABI does -- a page-locked one receives the device->host copy at full PCIe speed."""
    q = _tokens(query_tokens, "query")
    if out is None:
        out = np.zeros(corpus.num_docs, np.float32)
    assert out.dtype == np.float32 and out.size == corpus.num_docs and out.flags.c_contiguous, "out: float32[num_docs]"
    L.call("innr_cuda_maxsim", corpus.h, q.ctypes.data_as(L.f32p), q.shape[0], q.shape[1] if q.shape[0] else 0,
           1 if cosine else 0, out.ctypes.data_as(L.f32p))
    return out


def maxsim_corpus_batch(queries, corpus: TokenCorpus, cosine: bool = False) -> np.ndarray:
    """`queries`: (n_queries, n_q, dim). Returns (n_queries, n_docs); row i equals maxsim_corpus(queries[i], ...)."""
    q = np.ascontiguousarray(queries, dtype=np.float32)
    assert q.ndim == 3, "queries must be (n_queries, n_q, dim)"
    out = np.zeros((q.shape[0], corpus.num_docs), np.float32)
    L.call("innr_cuda_maxsim_batch", corpus.h, q.ctypes.data_as(L.f32p), q.shape[0], q.shape[1], q.shape[2],
           1 if cosine else 0, out.ctypes.data_as(L.f32p))
    return out


def maxsim_topk(query_tokens, corpus: TokenCorpus, k: int, cosine: bool = False):
    """The k best documents for one query token set: (indices uint64[min(k, num_docs)], scores float32[...]), scores
    descending under f32::total_cmp, exact ties -> lower index (index_base + doc). The scores are maxsim_corpus's bit
    for bit: the result is a stable descending total_cmp sort of its output, truncated to k, computed on the device."""
    q = _tokens(query_tokens, "query")
    idx, sc = maxsim_topk_batch(q.reshape(1, q.shape[0], q.shape[1]), corpus, k, cosine)
    return idx[0], sc[0]


def maxsim_topk_batch(queries, corpus: TokenCorpus, k: int, cosine: bool = False):
    """`queries`: (n_queries, n_q, dim). Returns (indices uint64[n_queries, min(k, num_docs)], scores float32[...]);
    row i equals maxsim_topk(queries[i], ...)."""
    q = np.ascontiguousarray(queries, dtype=np.float32)
    assert q.ndim == 3, "queries must be (n_queries, n_q, dim)"
    nq, kk = q.shape[0], max(int(k), 1)
    idx = np.zeros((nq, kk), np.uint64)
    sc = np.zeros((nq, kk), np.float32)
    cnt = C.c_size_t(0)
    L.call("innr_cuda_maxsim_topk", corpus.h, q.ctypes.data_as(L.f32p), nq, q.shape[1], q.shape[2] if q.shape[1] else 0,
           1 if cosine else 0, k, idx.ctypes.data_as(L.u64p), sc.ctypes.data_as(L.f32p), C.byref(cnt))
    return idx[:, :cnt.value], sc[:, :cnt.value]


def _pair(query_tokens, doc_tokens, cosine: bool) -> float:
    q, d = _tokens(query_tokens, "query"), _tokens(doc_tokens, "doc")
    if q.shape[0] == 0 or d.shape[0] == 0:
        return 0.0  # src/maxsim.rs:97-99
    assert q.shape[1] == d.shape[1], "dimension mismatch (doc)"
    if q.shape[1] == 0:
        return 0.0
    corpus = TokenCorpus.from_tokens(d, [0, d.shape[0]], d.shape[1])
    return float(maxsim_corpus(q, corpus, cosine)[0])


def maxsim(query_tokens, doc_tokens) -> float:  # src/maxsim.rs:96
    return _pair(query_tokens, doc_tokens, False)


def maxsim_cosine(query_tokens, doc_tokens) -> float:  # src/maxsim.rs:168
    return _pair(query_tokens, doc_tokens, True)
