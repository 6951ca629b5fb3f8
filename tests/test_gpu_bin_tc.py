"""The tensor-core filter for binary query batches (csrc/bin_tc.cu, DESIGN.md section 3.11) against the CUDA-core
scans and the oracle.

* Whole lists: Hamming indices and distances equal the CUDA-core route's (option bin_tc = 0) and the oracle's over the
  batch sizes, k and code widths the path serves; binary_dot / binary_jaccard lists of binary_topk_many equal one
  binary_topk call per query and the oracle, score bits included. Which path ran is asserted through bin_tc_last_stats.
* The prefix schedule, exact-duplicate tie groups larger than the candidate list, final and intermediate overflows.
* The device, asynchronous and sharded entries, and a _keys_dev call that returns while its stream is still busy.
Multi-GPU cases skip on a machine with one GPU."""
import ctypes as C
import os
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NT = max(1, min(os.cpu_count() or 1, 16))
CAND_CAP = 4096
DEFAULT_MIN_N, DEFAULT_MIN_Q, DEFAULT_MAX_K = 100_000, 32, 128


@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    innr_b200.set_option("bin_tc", 1)
    innr_b200.set_option("bin_tc_min_n", 0)
    innr_b200.set_option("bin_tc_min_queries", 2)
    innr_b200.set_option("bin_tc_max_k", 128)
    yield innr_b200
    innr_b200.set_option("bin_tc", 1)
    innr_b200.set_option("bin_tc_min_n", DEFAULT_MIN_N)
    innr_b200.set_option("bin_tc_min_queries", DEFAULT_MIN_Q)
    innr_b200.set_option("bin_tc_max_k", DEFAULT_MAX_K)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def levels(n, k, with_extra=False):
    """tc_filter.cuh: levels(n, k, first_rows(n, k, 0), 0) -- the prefixes of the filter passes (and how many of them
    are extra prefixes)."""
    cur = min(n, 1024 if k <= 32 else CAND_CAP)
    out = [cur]
    for nx in ((n // 256, n // 32) if k <= 32 else (n // 128, n // 16)):
        if nx >= 4 * cur:
            cur = (nx + 127) // 128 * 128
            out.append(cur)
    g_safe = max(4, (CAND_CAP // 2) // k)
    extra, top = [], n
    while top // cur > g_safe and len(extra) < 3:
        top = ((top + g_safe - 1) // g_safe + 127) // 128 * 128
        if top <= cur:
            break
        extra.append(top)
    n_extra = 0
    while extra and len(out) < 5:
        cur = extra.pop()
        out.append(cur)
        n_extra += 1
    if n > cur:
        out.append(n)
    return (out, n_extra) if with_extra else out


def stats():
    from innr_b200 import _lib as L
    return L.bin_tc_last_stats()


def words_of(dim):
    return (dim + 63) // 64


def masked(w, dim):
    """PackedBinary::new: padding bits of the last word cleared."""
    w = np.array(w, dtype=np.uint64, copy=True)
    if dim % 64:
        w[..., -1] &= np.uint64((1 << (dim % 64)) - 1)
    return w


def random_codes(rng, n, dim, density=0.5):
    b = rng.random((n, words_of(dim) * 64)) < density
    w = np.zeros((n, words_of(dim)), np.uint64)
    for j in range(64):
        w |= b[:, j::64].astype(np.uint64) << np.uint64(j)
    return masked(w, dim)


def near(rng, rows, dim, flips):
    """rows with `flips` random bits flipped each (inside the dimension)."""
    out = rows.copy()
    for r in range(len(out)):
        for b in rng.choice(dim, flips, replace=False):
            out[r, b // 64] ^= np.uint64(1) << np.uint64(b % 64)
    return out


def ref_setop_topk(op, qs, codes, k):
    """binary_dot / binary_jaccard top-k of every query over row-major codes (src/binary.rs:178-213): every score,
    stable sort descending (ties -> lower index), take(k); Jaccard as f32 intersection / f32 union, 1.0 for an empty
    union."""
    kk = min(k, len(codes))
    pa = np.bitwise_count(codes).sum(axis=1, dtype=np.int64)
    out_i, out_s = np.zeros((len(qs), kk), np.uint64), np.zeros((len(qs), kk), np.float32)
    for j, q in enumerate(qs):
        inter = np.bitwise_count(codes & q).sum(axis=1, dtype=np.int64)
        if op == "dot":
            sc = inter.astype(np.float32)
        else:
            uni = pa + int(np.bitwise_count(q).sum()) - inter
            with np.errstate(divide="ignore", invalid="ignore"):
                sc = np.where(uni == 0, np.float32(1.0), inter.astype(np.float32) / uni.astype(np.float32)).astype(np.float32)
        order = np.argsort(-sc, kind="stable")[:kk]
        out_i[j], out_s[j] = order, sc[order]
    return out_i, out_s


def hamming(ib, qs, corpus, k, tc):
    ib.set_option("bin_tc", 1 if tc else 0)
    try:
        return ib.hamming_topk_many(qs, corpus, k)
    finally:
        ib.set_option("bin_tc", 1)


def setop_many(ib, op, qs, corpus, k, tc):
    ib.set_option("bin_tc", 1 if tc else 0)
    try:
        return ib.binary_topk_many(op, qs, corpus, k)
    finally:
        ib.set_option("bin_tc", 1)


def check_hamming(ib, qs, corpus, k, n, expect_exact_scan=0):
    gi, gd = hamming(ib, qs, corpus, k, True)
    st = stats()
    assert st["passes"] == len(levels(n, k)), (st, n, k)
    if expect_exact_scan is not None:
        assert st["exact_scan_queries"] == expect_exact_scan, (st, n, k)
    wi, wd = hamming(ib, qs, corpus, k, False)
    assert np.array_equal(gi, wi) and np.array_equal(gd, wd), (len(qs), k)
    return gi, gd


def queries_for(rng, codes, nq, dim):
    """half random codes, half corpus rows with a few bits flipped (their true neighbours are in the corpus)"""
    r = random_codes(rng, nq - nq // 2, dim)
    src = codes[rng.integers(0, len(codes), nq // 2)]
    return np.concatenate([r, near(rng, src, dim, max(1, dim // 64))]) if nq // 2 else r


# ------------------------------------------------------------------------------------------------ 1. Hamming lists
@pytest.mark.parametrize("dim", [64, 100, 128, 1000, 1024, 4096])
def test_hamming_lists(ib, oracle, dim):
    rng = np.random.default_rng(dim)
    n = 150_000
    codes = random_codes(rng, n, dim)
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    qs_all = queries_for(rng, codes, 1025, dim)
    if dim == 1024:
        combos = [(nq, k) for nq in (2, 8, 255, 256, 257, 1024, 1025) for k in (1, 10, 32, 33, 100, 128)]
    else:
        combos = [(nq, k) for nq in (2, 256, 1025) for k in (1, 33, 128)] + [(8, 10), (257, 100)]
    want_i, want_d = oracle.hamming_topk_many(qs_all[:8], codes, 128, n_threads=NT)
    for nq, k in combos:
        qs = qs_all[:nq]
        gi, gd = check_hamming(ib, qs, corpus, k, n)
        m = min(nq, 8)
        assert np.array_equal(gi[:m], want_i[:m, :k]) and np.array_equal(gd[:m], want_d[:m, :k]), (nq, k)
        if nq > 8:  # the queries of the second 1024-query chunk too
            wi, wd = oracle.hamming_topk_many(qs[-2:], codes, k, n_threads=NT)
            assert np.array_equal(gi[-2:], wi) and np.array_equal(gd[-2:], wd), (nq, k)


def test_hamming_c4_size(ib, oracle):
    """C4 size (100M x 1024 bit, generated codes), 1024 queries: the filter against the CUDA-core route."""
    n, dim = 100_000_000, 1024
    corpus = ib.BinaryCorpus.generate(0xC4, 0, n, dim)
    rng = np.random.default_rng(44)
    qs = random_codes(rng, 1024, dim)
    for k in (10, 100):
        check_hamming(ib, qs, corpus, k, n, None)
    del corpus


# ------------------------------------------------------------------------------------------------ 2. dot / Jaccard
@pytest.mark.parametrize("dim,density", [(1000, 0.5), (256, 0.05), (4096, 0.02)])
def test_setop_lists(ib, oracle, dim, density):
    rng = np.random.default_rng(dim + int(density * 100))
    n = 120_000
    codes = random_codes(rng, n, dim, density)
    codes[[5, 4000, 77_777]] = 0                   # empty rows: Jaccard 1.0 against an empty query, 0 otherwise
    qs = random_codes(rng, 40, dim, density)
    qs[3] = 0                                      # an empty query: every Jaccard score 0 except the empty rows (1.0)
    qs[4] = codes[123]                             # a query that equals a row
    qs[5:9] = near(rng, codes[rng.integers(0, n, 4)], dim, 2)
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    for op in ("dot", "jaccard"):
        for k in (1, 10, 100, 128):
            gi, gs = setop_many(ib, op, qs, corpus, k, True)
            st = stats()
            assert st["passes"] == len(levels(n, k)), (st, op, k)
            wi, ws = setop_many(ib, op, qs, corpus, k, False)
            assert np.array_equal(gi, wi) and np.array_equal(bits(gs), bits(ws)), (op, k)
            oi, osc = ref_setop_topk(op, qs, codes, k)
            assert np.array_equal(gi, oi) and np.array_equal(bits(gs), bits(osc)), (op, k)
        for j in (0, 3, 4, 39):  # the single-query entry gives the same rows
            si, ss = ib.binary_topk(op, ib.PackedBinary(qs[j], dim), corpus, 10)
            gi, gs = setop_many(ib, op, qs, corpus, 10, True)
            assert np.array_equal(gi[j], si) and np.array_equal(bits(gs[j]), bits(ss)), (op, j)


def test_jaccard_equal_quotients(ib, oracle):
    """Rows whose quotients are equal as fractions (1/3, 2/6, 3/9, ...) or round to the same f32 from different
    fractions: ties broken by the lower index, exactly as the scan and the oracle."""
    dim, n = 512, 60_000
    rng = np.random.default_rng(9)
    codes = random_codes(rng, n, dim, 0.01)
    q = np.zeros(words_of(dim), np.uint64)
    q[0] = np.uint64(0xFFFF)  # 16 bits set
    rows = []
    for inter, extra in ((1, 2), (2, 4), (3, 6), (4, 8), (5, 10), (8, 16), (16, 32)):
        r = np.zeros(words_of(dim), np.uint64)
        r[0] = np.uint64((1 << inter) - 1)
        r[1] = np.uint64((1 << extra) - 1)  # outside the query's bits: union = 16 + extra
        rows.append(r)
    for j, r in enumerate(rows):
        for pos in (10 + j, 5000 + 7 * j, 50_000 + 3 * j):
            codes[pos] = r
    qs = np.stack([q] + [codes[i] for i in range(1, 8)])
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    for k in (5, 30):
        gi, gs = setop_many(ib, "jaccard", qs, corpus, k, True)
        oi, osc = ref_setop_topk("jaccard", qs, codes, k)
        assert np.array_equal(gi, oi) and np.array_equal(bits(gs), bits(osc)), k


# ------------------------------------------------------------------------------------------------ 3. schedule
def test_schedule_passes(ib, oracle):
    """passes == len(levels(n, k)) at n = 4096, 4097, the first n with an extra prefix (k = 100: k = 10 never takes
    one) and the first n/256 pass (k = 10)."""
    first_extra = next(n for n in range(80_000, 90_000) if levels(n, 100, True)[1] > 0)
    assert levels(first_extra - 1, 100, True)[1] == 0
    first_256 = 4 * 1024 * 256
    assert first_256 // 256 in levels(first_256, 10) and (first_256 - 1) // 256 not in levels(first_256 - 1, 10)
    rng = np.random.default_rng(12)
    dim = 128
    for n, ks in ((4096, (10, 100)), (4097, (10, 100)), (first_extra, (100,)), (first_256, (10,))):
        codes = random_codes(rng, n, dim)
        corpus = ib.BinaryCorpus.from_words(codes, n, dim)
        qs = queries_for(rng, codes, 8, dim)
        for k in ks:
            gi, gd = check_hamming(ib, qs, corpus, k, n, None)
            wi, wd = oracle.hamming_topk_many(qs, codes, k, n_threads=NT)
            assert np.array_equal(gi, wi) and np.array_equal(gd, wd), (n, k)


# ------------------------------------------------------------------------------------------------ 4. ties, overflow
def test_duplicate_tie_groups(ib, oracle):
    """More than CAND_CAP exact copies of the query, inside the dense pass and beyond it: lower indices first, and the
    final lists do not overflow (rows past a prefix tie the threshold distance only with larger indices)."""
    rng = np.random.default_rng(21)
    n, dim, k = 400_000, 256, 10
    codes = random_codes(rng, n, dim)
    qs = random_codes(rng, 4, dim)
    inside = rng.choice(np.arange(0, 1024), 600, replace=False)
    codes[inside] = qs[0]
    codes[rng.choice(np.arange(1024, n), 5000, replace=False)] = qs[0]
    codes[rng.choice(np.arange(5000, n), 6000, replace=False)] = qs[1]  # beyond the dense pass only
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    for kk in (k, 128):
        gi, gd = check_hamming(ib, qs, corpus, kk, n, 0)
        wi, wd = oracle.hamming_topk_many(qs, codes, kk, n_threads=NT)
        assert np.array_equal(gi, wi) and np.array_equal(gd, wd), kk
        assert np.all(gd[:2] == 0) and np.array_equal(gi[0], np.sort(inside)[:kk])
    for op in ("dot", "jaccard"):
        gi, gs = setop_many(ib, op, qs, corpus, k, True)
        oi, osc = ref_setop_topk(op, qs, codes, k)
        assert np.array_equal(gi, oi) and np.array_equal(bits(gs), bits(osc)), op


def _far_then_close(rng, n, dim, qs, lo, hi):
    """rows [lo, hi) close to the queries (a few bits off), every other row far (complements, a few bits off)."""
    codes = np.empty((n, words_of(dim)), np.uint64)
    far = masked(~qs[rng.integers(0, len(qs), n)], dim)
    codes[:] = near(rng, far, dim, 3) if n < 50_000 else far
    close = qs[rng.integers(0, len(qs), hi - lo)]
    codes[lo:hi] = near(rng, close, dim, 2)
    return codes


def test_final_overflow(ib, oracle):
    """The last prefix is far from the queries and the rows after it are strictly closer: every final list overflows,
    the statistics report it, and the exact scan answers those queries with the same results."""
    rng = np.random.default_rng(31)
    n, dim, k = 200_000, 256, 10
    lv = levels(n, k)
    assert len(lv) >= 3
    qs = random_codes(rng, 6, dim)
    codes = _far_then_close(rng, n, dim, qs, lv[-2], n)
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    gi, gd = check_hamming(ib, qs, corpus, k, n, expect_exact_scan=len(qs))
    wi, wd = oracle.hamming_topk_many(qs, codes, k, n_threads=NT)
    assert np.array_equal(gi, wi) and np.array_equal(gd, wd)
    for op in ("dot", "jaccard"):
        gi, gs = setop_many(ib, op, qs, corpus, k, True)
        assert stats()["exact_scan_queries"] == len(qs), op
        oi, osc = ref_setop_topk(op, qs, codes, k)
        assert np.array_equal(gi, oi) and np.array_equal(bits(gs), bits(osc)), op


def test_intermediate_overflow_only(ib, oracle):
    """Rows between the dense pass and the next prefix are close (more than CAND_CAP of them: that pass overflows),
    every other row is far: the final lists do not overflow and the results are exact."""
    rng = np.random.default_rng(41)
    n, dim, k = 200_000, 256, 10
    lv = levels(n, k)
    assert lv[1] - lv[0] > CAND_CAP
    qs = random_codes(rng, 6, dim)
    codes = _far_then_close(rng, n, dim, qs, lv[0], lv[1])
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    gi, gd = check_hamming(ib, qs, corpus, k, n, expect_exact_scan=0)
    wi, wd = oracle.hamming_topk_many(qs, codes, k, n_threads=NT)
    assert np.array_equal(gi, wi) and np.array_equal(gd, wd)


# ------------------------------------------------------------------------------------------------ 5. entries
def _keys_dev(corpus, dq, k, st, op=None):
    import torch
    from innr_b200 import _lib as L
    out = torch.empty(dq.shape[0] * k, dtype=torch.int64, device="cuda")
    st.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(st):
        if op is None:
            L.call("innr_cuda_hamming_topk_keys_dev", corpus.h, C.c_void_p(dq.data_ptr()), dq.shape[0], k,
                   C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))
        else:
            L.call("innr_cuda_binary_topk_keys_dev", corpus.h, {"dot": 0, "jaccard": 1}[op], C.c_void_p(dq.data_ptr()),
                   dq.shape[0], k, C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))
    return out


def _padded(qs):
    """query words padded to whole 128-bit chunks (the device-resident layout)"""
    w = qs.shape[1]
    out = np.zeros((qs.shape[0], (w + 1) // 2 * 2), np.uint64)
    out[:, :w] = qs
    return out


def _decode(keys, k):
    a = keys.cpu().numpy().view(np.uint64).reshape(-1, k)
    return a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)


def test_entries_dev_async(ib, oracle):
    """_keys_dev on two caller streams next to single-query (scan-only) calls, dot / Jaccard _keys_dev, and two
    asynchronous tickets in flight: the bits of the synchronous call."""
    import torch
    from innr_b200 import stream
    n, dim, k = 1_000_000, 1000, 10
    corpus = ib.BinaryCorpus.generate(0xE7, 0, n, dim)
    rng = np.random.default_rng(4)
    qa, qb = random_codes(rng, 64, dim), random_codes(rng, 64, dim)
    wa, wb = hamming(ib, qa, corpus, k, True), hamming(ib, qb, corpus, k, True)
    w1 = hamming(ib, qa[:1], corpus, k, False)
    da, db = (torch.from_numpy(_padded(q).view(np.int64)).cuda() for q in (qa, qb))
    s1, s2, s3 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    outs = [_keys_dev(corpus, da, k, s1), _keys_dev(corpus, da[:1], k, s3), _keys_dev(corpus, db, k, s2),
            _keys_dev(corpus, da[:1], k, s3)]
    torch.cuda.synchronize()
    res = [_decode(o, k) for o in outs]
    assert np.array_equal(res[0][0], wa[0]) and np.array_equal(res[0][1], wa[1])
    assert np.array_equal(res[2][0], wb[0]) and np.array_equal(res[2][1], wb[1])
    assert np.array_equal(res[1][0], w1[0]) and np.array_equal(res[3][0], w1[0])
    for op in ("dot", "jaccard"):
        gi, gs = setop_many(ib, op, qa, corpus, k, True)
        o = _keys_dev(corpus, da, k, s1, op)
        torch.cuda.synchronize()
        idx, hi = _decode(o, k)
        assert np.array_equal(idx, gi), op
        if op == "dot":
            assert np.array_equal((~hi.astype(np.uint32)).astype(np.float32), gs)
    ta = stream.submit_hamming_topk(qa, corpus, k)
    tb = stream.submit_hamming_topk(qb, corpus, k)
    ra, rb = ta.wait(), tb.wait()
    assert np.array_equal(ra[0], wa[0]) and np.array_equal(ra[1], wa[1])
    assert np.array_equal(rb[0], wb[0]) and np.array_equal(rb[1], wb[1])
    assert stats()["passes"] == len(levels(n, k))


def test_no_host_synchronisation(ib, oracle):
    """A qualifying _keys_dev batch queued behind a long sleep on its stream returns while the stream is still busy;
    the keys are right after a synchronise."""
    import torch
    n, dim, k = 2_000_000, 1024, 10
    corpus = ib.BinaryCorpus.generate(0x5EE9, 0, n, dim)
    qs = random_codes(np.random.default_rng(8), 256, dim)
    want = hamming(ib, qs, corpus, k, False)
    dq = torch.from_numpy(_padded(qs).view(np.int64)).cuda()
    st = torch.cuda.Stream()
    _keys_dev(corpus, dq, k, st)  # sizes the buffers and builds the popcounts
    torch.cuda.synchronize()
    with torch.cuda.stream(st):
        torch.cuda._sleep(3_000_000_000)  # about a second or more
    t0 = time.perf_counter()
    out = _keys_dev(corpus, dq, k, st)
    dt = time.perf_counter() - t0
    busy = not st.query()
    torch.cuda.synchronize()
    assert busy and dt < 0.3, (busy, dt)
    idx, dist = _decode(out, k)
    assert np.array_equal(idx, want[0]) and np.array_equal(dist, want[1])
    assert stats()["exact_scan_queries"] == 0


def test_entries_sharded(ib, oracle):
    """Sharded, synchronous and asynchronous, over two devices (skips on one GPU)."""
    import torch
    from innr_b200 import sharded, stream
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n, dim, k = 600_000, 512, 10
    rng = np.random.default_rng(6)
    codes = random_codes(rng, n, dim)
    shards = []
    for dev, (a, b) in enumerate(((0, n // 2), (n // 2, n))):
        ib.init(dev)
        shards.append(ib.BinaryCorpus.from_words(codes[a:b], b - a, dim, index_base=a))
    ib.init(0)
    qs = queries_for(rng, codes, 64, dim)
    wi, wd = oracle.hamming_topk_many(qs, codes, k, n_threads=NT)
    gi, gd = sharded.hamming_topk_sharded(qs, shards, k)
    assert np.array_equal(gi, wi) and np.array_equal(gd, wd)
    ti, td = stream.submit_hamming_topk_sharded(qs, shards, k).wait()
    assert np.array_equal(ti, gi) and np.array_equal(td, gd)
