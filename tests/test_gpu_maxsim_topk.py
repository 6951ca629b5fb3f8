"""MaxSim top-k (innr_cuda_maxsim_topk and its _keys_dev, _async, _sharded and _sharded_async forms).

The contract (DESIGN section 3.4): the scores are innr_cuda_maxsim's bit for bit, so for the same corpus, query, metric and
kernel path the result equals a stable descending f32::total_cmp sort of maxsim_corpus's output, truncated to k -- in
indices (index_base + doc) and in score bits. Here that is checked on both kernel paths (tcgen05 at dim 128, the
CUDA-core kernel at dim 130), for every query-token regime (1, 32: one pass; 33, 64: two column groups; 65: two
passes), over k below, at and above one selection round (128) and above n_docs; against the oracle within the DESIGN
section 4 tolerance; with planted exact ties, NaN and -inf totals, zero-norm tokens and an empty query; and for every
other form against the host entry. Tests that need two GPUs skip on a one-GPU box, like test_gpu_multi.py."""
import ctypes as C
import os
import subprocess
import sys
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
NT = max(1, min(os.cpu_count() or 1, 16))   # oracle threads


def _n_gpus():
    import torch
    return torch.cuda.device_count()


needs2 = pytest.mark.skipif("_n_gpus() < 2", reason="needs >= 2 GPUs in one box")


@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    return innr_b200


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def want_topk(scores, k, index_base=0):
    """Stable descending total_cmp sort of a score vector, truncated to k."""
    from innr_b200 import sharded
    order = np.argsort(~sharded.order_bits(scores), kind="stable")[:k]
    return order.astype(np.uint64) + np.uint64(index_base), scores[order]


def assert_same(got, want, what=""):
    (gi, gs), (wi, ws) = got, want
    assert np.array_equal(gi, wi), (what, gi[:8], wi[:8])
    assert np.array_equal(bits(gs), bits(ws)), what


def mixed_corpus(n_docs, dim, seed, max_len=40):
    """Documents of 0..max_len tokens (about one in eight empty)."""
    rng = np.random.default_rng(seed)
    lens = rng.integers(1, max_len + 1, size=n_docs)
    lens[rng.random(n_docs) < 0.125] = 0
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    toks = rng.standard_normal((int(off[-1]), dim)).astype(np.float32)
    return toks, off


KS = (1, 10, 128, 129, 300)


# ------------------------------------------------------------------------------------------------ ranking exactness
@pytest.mark.parametrize("dim", [128, 130])
@pytest.mark.parametrize("n_q", [1, 32, 33, 64, 65])
@pytest.mark.parametrize("cosine", [False, True], ids=["dot", "cosine"])
@pytest.mark.parametrize("source", ["uploaded", "generated"])
def test_topk_is_stable_sort_of_maxsim(ib, source, cosine, n_q, dim):
    n_docs = 700
    if source == "uploaded":
        toks, off = mixed_corpus(n_docs, dim, seed=n_q * 7 + dim)
        corpus = ib.TokenCorpus.from_tokens(toks, off, dim, index_base=1000)
    else:
        corpus = ib.TokenCorpus.generate(0x7A11_0001, 5, n_docs, 24, dim, index_base=1000)
    q = np.random.default_rng(n_q + dim).standard_normal((n_q, dim)).astype(np.float32)
    scores = ib.maxsim_corpus(q, corpus, cosine=cosine)
    for k in KS + (n_docs, n_docs + 5):
        got = ib.maxsim_topk(q, corpus, k, cosine=cosine)
        assert got[0].shape == (min(k, n_docs),)
        assert_same(got, want_topk(scores, k, 1000), (source, cosine, n_q, dim, k))


def test_empty_results_and_argument_checks(ib):
    toks, off = mixed_corpus(50, 16, seed=3)
    corpus = ib.TokenCorpus.from_tokens(toks, off, 16)
    q = np.ones((4, 16), np.float32)
    assert ib.maxsim_topk(q, corpus, 0)[0].size == 0
    empty = ib.TokenCorpus.from_tokens(np.zeros((0, 16), np.float32), [0], 16)
    assert ib.maxsim_topk(q, empty, 10)[0].size == 0
    assert ib.maxsim_topk_batch(np.zeros((0, 4, 16), np.float32), corpus, 10)[0].shape == (0, 0)
    with pytest.raises(AssertionError, match="dimension mismatch"):
        ib.maxsim_topk(np.ones((4, 15), np.float32), corpus, 10)


# ------------------------------------------------------------------------------------------------ against the oracle
@pytest.mark.parametrize("cosine", [False, True], ids=["dot", "cosine"])
def test_topk_against_oracle(ib, oracle, cosine):
    n_docs, dim, k = 20_000, 128, 100
    toks, off = mixed_corpus(n_docs, dim, seed=11, max_len=60)
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    rng = np.random.default_rng(12)
    for n_q in (32, 65):
        q = rng.standard_normal((n_q, dim)).astype(np.float32)
        gi, gs = ib.maxsim_topk(q, corpus, k, cosine=cosine)
        ref = oracle.maxsim_corpus(q, toks, off, cosine_flag=cosine, n_threads=NT).astype(np.float64)
        # DESIGN section 4: |got - ref| <= 1e-5 sum_i max_j sum_k |q_ik d_jk| + 1e-6 (cosine: at most 1e-5 n_q + 1e-6)
        cond = (np.full(n_docs, float(n_q)) if cosine
                else oracle.maxsim_corpus(np.abs(q), np.abs(toks), off, n_threads=NT).astype(np.float64))
        tol = 1e-5 * cond + 1e-6
        gi = gi.astype(np.int64)
        assert np.all(np.abs(gs.astype(np.float64) - ref[gi]) <= tol[gi]), (cosine, n_q)
        wi = np.argsort(-ref, kind="stable")[:k]
        kth = ref[wi[-1]]
        for doc in set(gi.tolist()) ^ set(wi.tolist()):   # disagreement only among near-ties of the k-th score
            assert abs(ref[doc] - kth) <= tol[doc] + tol[wi[-1]], (cosine, n_q, doc)


# ------------------------------------------------------------------------------------------------ planted edges
@pytest.mark.parametrize("dim", [128, 130])
@pytest.mark.parametrize("cosine", [False, True], ids=["dot", "cosine"])
def test_planted_ties_and_special_totals(ib, cosine, dim):
    """Identical documents at the first doc, in the middle, at the last doc and on both sides of a shard boundary come
    back in index order; all-NaN documents (-inf under dot), zero-norm documents and NaN totals (dot products that
    overflow to +inf for some query tokens and to -inf for others) keep the order total_cmp gives them; an empty query ranks by index."""
    from innr_b200 import sharded
    n_docs, nt = 1001, 8
    rng = np.random.default_rng(21 + dim)
    q = rng.standard_normal((32, dim)).astype(np.float32)
    docs = rng.standard_normal((n_docs, nt, dim)).astype(np.float32) * 0.1
    best = q[:nt].copy()                              # (cosine) scores above every random document
    boundary = 600
    planted = [0, 500, boundary - 1, boundary, n_docs - 1]
    for j in planted:
        docs[j] = best
    docs[100] = np.nan                                # all-NaN documents
    docs[700] = np.nan
    docs[200] = 0.0                                   # zero-norm tokens
    docs[300] = 0.0
    if not cosine:
        # query tokens +-(e_0 + e_1) against a token (3e38, 3e38, 0, ...): the dot products overflow to +inf and -inf,
        # the maxima are +inf and -inf and their sum is NaN
        q[:] = 0.0
        q[:, :2] = np.where(np.arange(32) % 2 == 0, 1.0, -1.0)[:, None]
        docs[400] = 0.0
        docs[400, :, :2] = 3e38
        docs[800] = docs[400]
    off = np.arange(0, (n_docs + 1) * nt, nt, dtype=np.uint64)
    toks = docs.reshape(-1, dim)
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    scores = ib.maxsim_corpus(q, corpus, cosine=cosine)
    for k in (1, 5, 10, 128, 129, n_docs, n_docs + 5):
        assert_same(ib.maxsim_topk(q, corpus, k, cosine=cosine), want_topk(scores, k), (cosine, dim, k))
    gi, gs = ib.maxsim_topk(q, corpus, n_docs, cosine=cosine)
    assert len(set(bits(scores[planted]).tolist())) == 1, "identical documents score identically"
    pos = [int(np.flatnonzero(gi == j)[0]) for j in planted]
    assert pos == sorted(pos) and pos[-1] - pos[0] == len(planted) - 1, pos   # adjacent, in index order
    if cosine:
        assert gi[:len(planted)].tolist() == planted
    else:
        # the NaN totals: the positive NaN of the device, first, in index order
        assert np.isnan(scores[400]) and np.isnan(scores[800]) and not np.signbit(scores[[400, 800]]).any()
        assert gi[:2].tolist() == [400, 800] and np.all(np.isnan(gs[:2]))
        assert np.all(scores[[100, 700]] == -np.inf) and gi[-2:].tolist() == [100, 700]
    # the same ties across a shard boundary (one device: the host-merge route), with index_base
    shards = [ib.TokenCorpus.from_tokens(toks[:boundary * nt], off[:boundary + 1], dim),
              ib.TokenCorpus.from_tokens(toks[boundary * nt:], off[boundary:] - off[boundary], dim, index_base=boundary)]
    for k in (5, 10, 200, n_docs + 5):
        si, ss = sharded.maxsim_topk_sharded(q[None], shards, k, cosine=cosine)
        assert_same((si[0], ss[0]), want_topk(scores, k), ("sharded", cosine, dim, k))
    # an empty query: every score is 0.0, the ranking is by index
    ei, es = ib.maxsim_topk(np.zeros((0, dim), np.float32), corpus, 10, cosine=cosine)
    assert ei.tolist() == list(range(10)) and np.all(bits(es) == 0)


# ------------------------------------------------------------------------------------------------ other forms
@pytest.mark.parametrize("n_q", [32, 65])
def test_batch_equals_single_queries(ib, n_q):
    toks, off = mixed_corpus(3000, 128, seed=31)
    corpus = ib.TokenCorpus.from_tokens(toks, off, 128, index_base=7)
    qs = np.random.default_rng(32).standard_normal((5, n_q, 128)).astype(np.float32)
    for cosine in (False, True):
        for k in (10, 300):
            bi, bs = ib.maxsim_topk_batch(qs, corpus, k, cosine=cosine)
            for j in range(5):
                assert_same((bi[j], bs[j]), ib.maxsim_topk(qs[j], corpus, k, cosine=cosine), (n_q, cosine, k, j))


def test_batch_in_chunks(ib):
    """1,000,000 documents: the score scratch holds 16 queries (64 MB), so a batch of 37 runs as 16 + 16 + 5; every row
    equals the stable sort of the batch score entry."""
    n_docs, dim = 1_000_000, 32
    corpus = ib.TokenCorpus.generate(0x7A11_0002, 0, n_docs, 2, dim, index_base=3)
    qs = np.random.default_rng(33).standard_normal((37, 8, dim)).astype(np.float32)
    scores = ib.maxsim_corpus_batch(qs, corpus, cosine=True)
    for k in (10, 129):
        gi, gs = ib.maxsim_topk_batch(qs, corpus, k, cosine=True)
        for j in range(37):
            assert_same((gi[j], gs[j]), want_topk(scores[j], k, 3), (k, j))


def test_keys_dev_on_a_caller_stream(ib):
    import torch
    from innr_b200 import _lib as L, sharded
    n_docs = 2000
    toks, off = mixed_corpus(n_docs, 128, seed=41)
    corpus = ib.TokenCorpus.from_tokens(toks, off, 128, index_base=50)
    qs = np.random.default_rng(42).standard_normal((3, 32, 128)).astype(np.float32)
    st = torch.cuda.Stream()
    with torch.cuda.stream(st):
        dq = torch.from_numpy(qs).cuda()
        for k in (10, 129, n_docs + 5):
            keys = torch.empty(3 * k, dtype=torch.int64, device="cuda")
            L.call("innr_cuda_maxsim_topk_keys_dev", corpus.h, C.c_void_p(dq.data_ptr()), 3, 32, 1, k,
                   C.c_void_p(keys.data_ptr()), C.c_void_p(st.cuda_stream))
            st.synchronize()
            kv = keys.cpu().numpy().view(np.uint64).reshape(3, k)
            kk = min(k, n_docs)
            assert np.all(kv[:, kk:] == np.uint64(0xFFFFFFFFFFFFFFFF))     # sentinel padding past n_docs
            for j in range(3):
                idx, sc = sharded.decode_keys(kv[j, :kk], descending=True)
                assert_same((idx, sc), ib.maxsim_topk(qs[j], corpus, k, cosine=True), k)


def test_async_tickets(ib):
    from innr_b200 import _lib as L, stream
    toks, off = mixed_corpus(4000, 128, seed=51)
    corpus = ib.TokenCorpus.from_tokens(toks, off, 128)
    rng = np.random.default_rng(52)
    qa = rng.standard_normal((2, 32, 128)).astype(np.float32)
    qb = rng.standard_normal((3, 33, 128)).astype(np.float32)
    ta = stream.submit_maxsim_topk(qa, corpus, 10, cosine=True)
    tb = stream.submit_maxsim_topk(qb, corpus, 300)
    with pytest.raises(L.InnrCudaError, match="in flight"):
        stream.submit_maxsim_topk(qa, corpus, 10)
    gb, ga = tb.wait(), ta.wait()
    assert_same(ga, ib.maxsim_topk_batch(qa, corpus, 10, cosine=True), "a")
    assert_same(gb, ib.maxsim_topk_batch(qb, corpus, 300), "b")
    for rep in range(3):  # slots are reused
        t = stream.submit_maxsim_topk(qa, corpus, 129, cosine=True)
        assert_same(t.wait(), ib.maxsim_topk_batch(qa, corpus, 129, cosine=True), rep)


# ------------------------------------------------------------------------------------------------ shards
def test_shards_sharing_a_device(ib):
    """Four shards on one device (one of them empty) take the thread-per-shard + host-merge route; the async sharded
    form refuses them (the exchange route needs distinct devices)."""
    from innr_b200 import sharded, stream
    n_docs, dim = 5000, 128
    toks, off = mixed_corpus(n_docs, dim, seed=61)
    whole = ib.TokenCorpus.from_tokens(toks, off, dim)
    cuts = [0, 1200, 1200, 3100, n_docs]
    shards = [ib.TokenCorpus.from_tokens(toks[int(off[a]):int(off[b])], off[a:b + 1] - off[a], dim, index_base=a)
              for a, b in zip(cuts, cuts[1:])]
    qs = np.random.default_rng(62).standard_normal((3, 32, dim)).astype(np.float32)
    for cosine in (False, True):
        for k in (1, 10, 100, 200, n_docs + 5):
            assert_same(sharded.maxsim_topk_sharded(qs, shards, k, cosine=cosine),
                        ib.maxsim_topk_batch(qs, whole, k, cosine=cosine), (cosine, k))
    with pytest.raises(NotImplementedError):
        stream.submit_maxsim_topk_sharded(qs, shards, 10)


@needs2
def test_shards_over_devices(ib):
    """One shard per device: the exchange route (k = 10, 100), synchronous and asynchronous, and the host-merge
    fallback (k = 200) all equal the unsharded call."""
    import torch
    from innr_b200 import sharded, stream
    n_dev = min(torch.cuda.device_count(), 4)
    n_docs, dim = 30_001, 128
    toks, off = mixed_corpus(n_docs, dim, seed=71)
    whole = ib.TokenCorpus.from_tokens(toks, off, dim)
    cuts = [n_docs * r // n_dev for r in range(n_dev + 1)]
    shards = []
    for dev, (a, b) in enumerate(zip(cuts, cuts[1:])):
        ib.init(dev)
        shards.append(ib.TokenCorpus.from_tokens(toks[int(off[a]):int(off[b])], off[a:b + 1] - off[a], dim, index_base=a))
    ib.init(0)
    rng = np.random.default_rng(72)
    for rep in range(2):
        qs = rng.standard_normal((3, 32, dim)).astype(np.float32)
        for cosine in (False, True):
            for k in (10, 100, 200):
                want = ib.maxsim_topk_batch(qs, whole, k, cosine=cosine)
                assert_same(sharded.maxsim_topk_sharded(qs, shards, k, cosine=cosine), want, (rep, cosine, k))
                if k <= 128:
                    t1 = stream.submit_maxsim_topk_sharded(qs, shards, k, cosine=cosine)
                    t2 = stream.submit_maxsim_topk_sharded(qs[::-1], shards, k, cosine=cosine)
                    assert_same(t1.wait(), want, ("async", rep, cosine, k))
                    w2 = ib.maxsim_topk_batch(qs[::-1], whole, k, cosine=cosine)
                    assert_same(t2.wait(), w2, ("async2", rep, cosine, k))


@needs2
def test_sharded_knn_maxsim_under_torchrun():
    n = min(_n_gpus(), 4)
    r = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}",
                        "--master-addr", "127.0.0.1", "--master-port", "29541",
                        os.path.join(ROOT, "tests", "mp_maxsim_check.py")],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "mp_maxsim_check ok" in r.stdout, (r.stdout[-3000:], r.stderr[-3000:])


# ------------------------------------------------------------------------------------------------ scale
def test_c3_document_shape(ib):
    """125,000 generated documents of 180 tokens x 128 (11.5 GB, a 1/8 shard of C3): the top-10 of a cosine query of 32
    tokens equals the stable sort of innr_cuda_maxsim_dev's output."""
    import torch
    from innr_b200 import _lib as L, synth
    t0 = time.time()
    free0, total = torch.cuda.mem_get_info()
    n_docs, nt, dim = 125_000, 180, 128
    corpus = ib.TokenCorpus.generate(synth.SALT_CORPUS, 0, n_docs, nt, dim)
    q = synth.ghash_f32(synth.SALT_QUERY, 0, 32 * dim).reshape(32, dim)
    dq = torch.from_numpy(q).cuda()
    out = torch.empty(n_docs, dtype=torch.float32, device="cuda")
    L.call("innr_cuda_maxsim_dev", corpus.h, C.c_void_p(dq.data_ptr()), 32, 1, C.c_void_p(out.data_ptr()),
           C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    peak = total - torch.cuda.mem_get_info()[0]
    assert_same(ib.maxsim_topk(q, corpus, 10, cosine=True), want_topk(out.cpu().numpy(), 10))
    peak = max(peak, total - torch.cuda.mem_get_info()[0])
    print(f"[maxsim-topk] C3 document shape: wall {time.time() - t0:.3f} s, peak device memory in use {peak / 1e9:.1f} GB "
          f"(free at start {free0 / 1e9:.1f} GB)")
