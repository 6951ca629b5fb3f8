"""The tensor-core filter of batch_knn_u8 (csrc/u8_tc.cu, DESIGN.md section 3.10) against the exact u8 scan and the
oracle.

* The bound: the score interval the filter gives every (query, row) pair of its dense first pass, read through
  innr_cuda_u8_tc_debug_bounds, contains the oracle's score on adversarial rows and queries.
* Whole lists: indices and score bits equal the exact scan's (option u8_tc = 0) and the oracle's, over the batch sizes,
  k and corpus sizes the path serves; which path ran is asserted through u8_tc_last_stats.
* Queries the filter does not answer, overflowing tie groups, the device / asynchronous / sharded entries.
Multi-GPU cases skip on a machine with one GPU."""
import ctypes as C
import os

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NT = max(1, min(os.cpu_count() or 1, 16))
CAND_CAP = 4096


@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    innr_b200.set_option("u8_tc", 1)
    innr_b200.set_option("u8_tc_min_n", 0)
    innr_b200.set_option("u8_tc_min_queries", 2)
    innr_b200.set_option("u8_tc_max_k", 128)   # the kernel serves k <= 128; the default routes k > 32 to the scan
    yield innr_b200
    innr_b200.set_option("u8_tc", 1)
    innr_b200.set_option("u8_tc_min_n", DEFAULT_MIN_N)
    innr_b200.set_option("u8_tc_min_queries", DEFAULT_MIN_Q)
    innr_b200.set_option("u8_tc_max_k", DEFAULT_MAX_K)


DEFAULT_MIN_N, DEFAULT_MIN_Q, DEFAULT_MAX_K = 100_000, 8, 32


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def levels(n, k):
    """tc_filter.cuh: levels(n, k, first_rows(n, k, 0), 0) -- the prefixes of the filter passes."""
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
    while extra and len(out) < 5:
        cur = extra.pop()
        out.append(cur)
    if n > cur:
        out.append(n)
    return out


def scale_exp(q):
    """The filter's power of two: max|q| 2^p in [63.5, 127)."""
    mx = float(np.max(np.abs(q)))
    _, ex = np.frexp(np.float32(mx))
    p = 7 - int(ex)
    if np.float32(mx) * np.float32(2.0 ** p) >= 127:
        p -= 1
    return p


def knn(ib, qs, corpus, k, tc):
    ib.set_option("u8_tc", 1 if tc else 0)
    try:
        return ib.batch_knn_u8_many(qs, corpus, k)
    finally:
        ib.set_option("u8_tc", 1)


def stats(ib):
    from innr_b200 import _lib as L
    return L.u8_tc_last_stats()


def check_lists(ib, qs, corpus, k, n, expect_exact_scan=0):
    """The filter ran (its passes, as tc_filter.cuh schedules them) and answered the queries it should: expect_exact_scan
    = the number the exact scan must answer, or None when overflowing lists are allowed (large k: the interval is wide
    enough that some queries' final lists exceed the 4096 slots)."""
    gi, gs = knn(ib, qs, corpus, k, True)
    st = stats(ib)
    assert st["passes"] == len(levels(n, k)), (st, n, k)
    if expect_exact_scan is None:
        assert st["exact_scan_queries"] < len(qs) or k > 32, (st, n, k)
    else:
        assert st["exact_scan_queries"] == expect_exact_scan, (st, n, k)
    wi, ws = knn(ib, qs, corpus, k, False)
    assert np.array_equal(gi, wi) and np.array_equal(bits(gs), bits(ws)), (len(qs), k)
    return gi, gs


# ------------------------------------------------------------------------------------------------ 1. the bound
def _adversarial_queries(d, rng):
    qs = [rng.uniform(-1, 1, d).astype(np.float32)]
    # elements on rounding half-steps of the i8 grid (max|q| = 1 -> 2^p = 64)
    h = (rng.integers(-126, 126, d) + 0.5).astype(np.float32) / np.float32(64)
    h[0] = 1.0
    qs.append(h)
    # one large element, the rest tiny (they quantise to 0)
    t = (rng.uniform(-1, 1, d) * 1e-4).astype(np.float32)
    t[d // 2] = 3.0
    qs.append(t)
    # subnormal elements and -0
    s = rng.uniform(-1, 1, d).astype(np.float32)
    s[::3] = np.float32(1e-40)
    s[1::3] = np.float32(-0.0)
    s[2::7] = np.float32(-3e-39)
    qs.append(s)
    # max|q| at the power-of-two edges of the scale choice, and at 2^+-100
    for top in (2.0, np.nextafter(np.float32(2.0), np.float32(0)), np.float32(127 / 64), np.float32(127.5 / 64),
                2.0 ** -100, 2.0 ** 100):
        e = rng.uniform(-1, 1, d).astype(np.float32) * np.float32(top)
        e[0] = np.float32(top)
        qs.append(e.astype(np.float32))
    return np.stack(qs).astype(np.float32)


def _flagged_queries(d, rng):
    bad = []
    for v in (np.nan, np.inf, 2.0 ** 101, 2.0 ** -101):
        x = rng.uniform(-1, 1, d).astype(np.float32) * (np.float32(2.0 ** -102) if v == 2.0 ** -101 else 1)
        x[d - 1] = v
        bad.append(x)
    bad.append(np.zeros(d, np.float32))
    return np.stack(bad).astype(np.float32)


@pytest.mark.parametrize("d", [16, 33, 384, 777, 2048])
@pytest.mark.parametrize("alpha,offset", [(2.0, -1.0), (0.37, 0.11), (2.0, -3.0e4)])
def test_bound_adversarial(ib, oracle, d, alpha, offset):
    """lower <= oracle score <= upper for every unflagged pair; (2.0, -3e4): offset * query_sum swamps c * mixed."""
    rng = np.random.default_rng(d * 7 + int(alpha * 100))
    gp, op = ib.QuantizationParams(alpha, offset), oracle.QuantizationParams(alpha, offset)
    qs = _adversarial_queries(d, rng)
    n = 4096
    mat = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    mat[0] = 0
    mat[1] = 255
    mat[2:64] = np.clip(np.rint(128 + rng.normal(0, 6, size=(62, d))), 0, 255).astype(np.uint8)   # near the centre
    # rows of all-0 / all-255 codes aligned with the sign of each query's quantisation residual
    for j, q in enumerate(qs):
        p = scale_exp(q)
        sc = np.float32(2.0 ** p)
        qi = np.rint(q * sc)
        e = q.astype(np.float64) - qi / (2.0 ** p)
        mat[64 + 2 * j] = np.where(e > 0, 255, 0)
        mat[65 + 2 * j] = np.where(e > 0, 0, 255)
    corpus = ib.U8Corpus.from_rows(mat, gp)
    allq = np.concatenate([qs, _flagged_queries(d, rng)])
    lo, hi, flags = ib.scalar.u8_tc_debug_bounds(allq, corpus)
    assert lo.shape == (len(allq), n)
    assert flags.tolist() == [0] * len(qs) + [1] * (len(allq) - len(qs))
    widx, wsc = oracle.batch_knn_u8_many(qs, mat, op, n, n_threads=NT)
    for j in range(len(qs)):
        want = np.empty(n, np.float32)
        want[widx[j].astype(np.int64)] = wsc[j]
        ok = (lo[j] <= want) & (want <= hi[j])
        assert ok.all(), (d, alpha, offset, j, np.flatnonzero(~ok)[:5], lo[j][~ok][:3], want[~ok][:3], hi[j][~ok][:3])


# ------------------------------------------------------------------------------------------------ 2. whole lists
@pytest.fixture(scope="module")
def shard_c5(ib, oracle):
    """An 8-GPU shard of C5: 6.25M x 384 ghash codes (the corpus bench.py's C5 uses, first eighth)."""
    n, d = 6_250_000, 384
    gp = ib.QuantizationParams.from_range(-1.0, 1.0)
    return ib.U8Corpus.generate(0xC5, 0, n, d, gp), n, d


def test_lists_c5_shard(ib, oracle, shard_c5):
    corpus, n, d = shard_c5
    qs_all = oracle.ghash_f32(0x5EED_0C5, 0, 1024 * d).reshape(1024, d)
    for nq in (2, 64, 65, 256, 257, 1024):
        for k in ((1, 10, 32, 33, 100, 128) if nq in (257, 1024) else (10,)):
            check_lists(ib, qs_all[:nq], corpus, k, n, None)
    # the oracle for a subset of queries (host copy of the same ghash codes)
    op = oracle.QuantizationParams.from_range(-1.0, 1.0)
    mat = oracle.ghash_u8_rows(0xC5, 0, n, d, op, NT)
    gi, gs = knn(ib, qs_all[:2], corpus, 100, True)
    wi, ws = oracle.batch_knn_u8_many(qs_all[:2], mat, op, 100, n_threads=NT)
    assert np.array_equal(gi, wi) and np.array_equal(bits(gs), bits(ws))


def test_lists_c5_full(ib, oracle):
    """Once at full C5 size: 50M x 384, 1024 queries, k = 10."""
    n, d = 50_000_000, 384
    corpus = ib.U8Corpus.generate(0xC5, 0, n, d, ib.QuantizationParams.from_range(-1.0, 1.0))
    qs = oracle.ghash_f32(0x5EED_0C5, 0, 1024 * d).reshape(1024, d)
    check_lists(ib, qs, corpus, 10, n, None)
    del corpus


def test_lists_d777_and_schedule_edges(ib, oracle):
    """d = 777 (a K block of 1 chunk past six full ones, a 9-dimension scalar tail) at a smaller n, and n at the edges
    of the schedule: one dense pass only, the 4 x rule of each prefix just met / just missed, a last partial tile."""
    rng = np.random.default_rng(777)
    gp = ib.QuantizationParams.from_range(-1.0, 1.0)
    n, d = 300_001, 777
    corpus = ib.U8Corpus.generate(0x777, 0, n, d, gp)
    qs = rng.uniform(-1, 1, size=(65, d)).astype(np.float32)
    for k in (1, 10, 33, 128):
        check_lists(ib, qs, corpus, k, n, None)
    d = 96
    for n in (1000, 1024, 1025, 4096, 4097, 4 * 1024 * 256 - 1, 4 * 1024 * 256, 4 * 1024 * 256 + 129, 1_048_577):
        corpus = ib.U8Corpus.generate(0x96 + n, 0, n, d, gp)
        qs = rng.uniform(-1, 1, size=(3, d)).astype(np.float32)
        for k in (1, 10, 100):
            check_lists(ib, qs, corpus, min(k, n), n, None)


def test_small_d(ib, oracle):
    """d < 16 (the portable sequential sum) and d = 16, 33 (remainder chains, scalar tail)."""
    rng = np.random.default_rng(5)
    op = oracle.QuantizationParams.from_range(-1.0, 1.0)
    for d in (1, 7, 16, 33):
        n = 20_000
        mat = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
        corpus = ib.U8Corpus.from_rows(mat, ib.QuantizationParams.from_range(-1.0, 1.0))
        qs = rng.uniform(-1, 1, size=(5, d)).astype(np.float32)
        gi, gs = check_lists(ib, qs, corpus, 10, n)
        wi, ws = oracle.batch_knn_u8_many(qs, mat, op, 10, n_threads=NT)
        assert np.array_equal(gi, wi) and np.array_equal(bits(gs), bits(ws)), d


# ------------------------------------------------------------------------------------------------ 3. planted rows
def test_planted_and_ties(ib, oracle):
    """True neighbours planted just past every prefix boundary, decoys whose integer product over-estimates (codes 255
    where the query's residual is negative), and a query whose best rows are 5,000 exact copies (an exact score tie
    group larger than the candidate list: it overflows and is answered by the exact scan)."""
    rng = np.random.default_rng(11)
    n, d, k = 2_000_000, 128, 10
    op = oracle.QuantizationParams.from_range(-1.0, 1.0)
    gp = ib.QuantizationParams.from_range(-1.0, 1.0)
    mat = oracle.ghash_u8_rows(0x9A, 0, n, d, op, NT)
    qs = rng.uniform(-1, 1, size=(3, d)).astype(np.float32)
    lv = levels(n, k)
    for j in range(2):
        q = qs[j]
        best = np.where(q > 0, 255, 0).astype(np.uint8)
        for b in lv[:-1]:
            for off in (0, 1, 127):
                row = best.copy()
                row[np.argsort(-q)[:3 + off % 5]] = 210
                mat[b + off] = row
        p = scale_exp(q)
        e = q.astype(np.float64) - np.rint(q * np.float32(2.0 ** p)) / 2.0 ** p
        decoy = np.where(q > 0, 250, 0).astype(np.uint8)
        decoy[e < 0] = 255
        mat[rng.integers(0, n, 50)] = decoy
    tie = np.where(qs[2] > 0, 255, 0).astype(np.uint8)
    mat[rng.choice(n, 5000, replace=False)] = tie
    corpus = ib.U8Corpus.from_rows(mat, gp)
    gi, gs = check_lists(ib, qs, corpus, k, n, expect_exact_scan=1)
    wi, ws = oracle.batch_knn_u8_many(qs, mat, op, k, n_threads=NT)
    assert np.array_equal(gi, wi) and np.array_equal(bits(gs), bits(ws))


def test_unfiltered_queries(ib, oracle):
    """NaN, inf, all-zero and out-of-range queries go to the exact scan, bit-exact, inside a filtered batch."""
    rng = np.random.default_rng(3)
    n, d = 500_000, 64
    corpus = ib.U8Corpus.generate(0x3, 0, n, d, ib.QuantizationParams.from_range(-1.0, 1.0))
    good = rng.uniform(-1, 1, size=(4, d)).astype(np.float32)
    qs = np.concatenate([good[:2], _flagged_queries(d, rng), good[2:]])
    check_lists(ib, qs, corpus, 10, n, expect_exact_scan=5)


# ------------------------------------------------------------------------------------------------ 4. entries
def test_entries_dev_async(ib, oracle):
    """_keys_dev on two caller streams next to single-query (scan-only) calls; two asynchronous tickets in flight."""
    import torch
    from innr_b200 import _lib as L, stream
    n, d, k = 1_000_000, 384, 10
    corpus = ib.U8Corpus.generate(0xE7, 0, n, d, ib.QuantizationParams.from_range(-1.0, 1.0))
    rng = np.random.default_rng(4)
    qa, qb = (rng.uniform(-1, 1, size=(64, d)).astype(np.float32) for _ in range(2))
    wa, wb = knn(ib, qa, corpus, k, False), knn(ib, qb, corpus, k, False)
    w1 = knn(ib, qa[:1], corpus, k, False)

    def run(q, st):
        dq = torch.from_numpy(q).cuda()
        out = torch.empty(len(q) * k, dtype=torch.int64, device="cuda")
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            L.call("innr_cuda_batch_knn_u8_keys_dev", corpus.h, C.c_void_p(dq.data_ptr()), len(q), k,
                   C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))
        return out, dq

    s1, s2, s3 = torch.cuda.Stream(), torch.cuda.Stream(), torch.cuda.Stream()
    outs = [run(qa, s1), run(qa[:1], s3), run(qb, s2), run(qa[:1], s3)]
    torch.cuda.synchronize()
    idx = [(o.cpu().numpy().view(np.uint64) & np.uint64(0xFFFFFFFF)).reshape(-1, k) for o, _ in outs]
    assert np.array_equal(idx[0], wa[0]) and np.array_equal(idx[2], wb[0])
    assert np.array_equal(idx[1], w1[0]) and np.array_equal(idx[3], w1[0])
    ta = stream.submit_knn_u8(qa, corpus, k)
    tb = stream.submit_knn_u8(qb, corpus, k)
    ra, rb = ta.wait(), tb.wait()
    assert np.array_equal(ra[0], wa[0]) and np.array_equal(bits(ra[1]), bits(wa[1]))
    assert np.array_equal(rb[0], wb[0]) and np.array_equal(bits(rb[1]), bits(wb[1]))
    assert stats(ib)["passes"] == len(levels(n, k))


def test_entries_sharded(ib, oracle):
    """Sharded, synchronous and asynchronous, over two devices (skips on one GPU)."""
    import torch
    from innr_b200 import sharded, stream
    if torch.cuda.device_count() < 2:
        pytest.skip("needs two GPUs")
    n, d, k = 600_000, 128, 10
    op = oracle.QuantizationParams.from_range(-1.0, 1.0)
    gp = ib.QuantizationParams.from_range(-1.0, 1.0)
    mat = oracle.ghash_u8_rows(0x5A, 0, n, d, op, NT)
    shards = []
    for dev, (a, b) in enumerate(((0, n // 2), (n // 2, n))):
        ib.init(dev)
        shards.append(ib.U8Corpus.from_rows(mat[a:b], gp, index_base=a))
    ib.init(0)
    qs = np.random.default_rng(6).uniform(-1, 1, size=(64, d)).astype(np.float32)
    wi, ws = oracle.batch_knn_u8_many(qs[:4], mat, op, k, n_threads=NT)
    gi, gs = sharded.batch_knn_u8_sharded(qs, shards, k)
    assert np.array_equal(gi[:4], wi) and np.array_equal(bits(gs[:4]), bits(ws))
    ta = stream.submit_knn_u8_sharded(qs, shards, k)
    ti, tsc = ta.wait()
    assert np.array_equal(ti, gi) and np.array_equal(bits(tsc), bits(gs))


# ------------------------------------------------------------------------------------------------ 5. pair kernel
def test_pair_kernel_many_tiles_exact_path(ib, oracle):
    """test_gpu_many_tiles.py's 4-query "two pairs" case at 4M x 384 with the filter off: the pair kernel keeps its
    coverage whatever the crossover of the default options is."""
    n, d = 4_000_200, 384
    op = oracle.QuantizationParams.from_range(-1.0, 1.0)
    mat = oracle.ghash_u8_rows(0x4A11_0003, 0, n, d, op, NT)
    qs = oracle.ghash_f32(0x4A11_0004, d, 4 * d).reshape(4, d)
    corpus = ib.U8Corpus.from_rows(mat, ib.QuantizationParams.from_range(-1.0, 1.0))
    widx, wsc = oracle.batch_knn_u8_many(qs, mat, op, 128, n_threads=min(NT, 4))
    for k in (1, 10, 32, 33, 100, 128):
        gi, gs = knn(ib, qs, corpus, k, False)
        assert np.array_equal(gi, widx[:, :k]) and np.array_equal(bits(gs), bits(wsc[:, :k])), k
