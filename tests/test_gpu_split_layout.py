"""Split f32 layout (innr_b200/csrc/pdx.cuh) and the screened single-query kNN (scan_f32.cu, DESIGN.md section 3.1).

Every f32 entry must give on a split corpus exactly what it gives on a plain corpus of the same data (whole keys, score
bits), and the screen's interval must hold the reference's score on adversarial rows. The option f32_split_min_rows
chooses the layout per corpus; the tests set it around each upload."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SPLIT_DEFAULT = 1_000_000


@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    yield innr_b200
    innr_b200.set_option("f32_split_min_rows", SPLIT_DEFAULT)


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def rand_rows(n, d, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, d)) * scale).astype(np.float32)


def both(ib, rows, index_base=0, how="rows"):
    """(plain, split) DeviceBatch of the same n x d rows."""
    n, d = rows.shape
    out = []
    for thr in (2**62, 0):
        ib.set_option("f32_split_min_rows", thr)
        try:
            if how == "rows":
                out.append(ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d, index_base=index_base))
            else:
                out.append(ib.DeviceBatch.from_pdx(np.ascontiguousarray(rows.T).reshape(-1), n, d, index_base=index_base))
        finally:
            ib.set_option("f32_split_min_rows", SPLIT_DEFAULT)
    return out


def same(a, b):
    if isinstance(a, tuple) or isinstance(a, list):
        assert len(a) == len(b)
        for x, y in zip(a, b):
            same(x, y)
        return
    if hasattr(a, "indices"):
        same((np.asarray(a.indices), np.asarray(a.scores, np.float32)), (np.asarray(b.indices), np.asarray(b.scores, np.float32)))
        return
    a, b = np.asarray(a), np.asarray(b)
    if a.dtype == np.float32:
        assert np.array_equal(bits(a), bits(b))
    else:
        assert np.array_equal(a, b)


def knn_keys(ib, db, metric, q, k):
    import torch
    from innr_b200 import _lib as L
    m = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}[metric]
    dq = torch.from_numpy(np.ascontiguousarray(q, np.float32).reshape(-1)).cuda()
    nq = dq.numel() // db.dimension
    out = torch.zeros(nq * k, dtype=torch.int64, device="cuda")
    L.call("innr_cuda_batch_knn_keys_dev", db.h, m, C.c_void_p(dq.data_ptr()), nq, k, C.c_void_p(out.data_ptr()),
           C.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return out.cpu().numpy()


@pytest.mark.parametrize("n,d,base", [(5000, 96, 0), (4097, 33, 7), (300, 1, 0), (70_001, 768, 1000)])
def test_knn_split_equals_plain(ib, n, d, base):
    rows = rand_rows(n, d, n + d)
    plain, split = both(ib, rows, base)
    qs = rand_rows(3, d, 5)
    for metric in ("dot", "cosine", "l2"):
        for k in (1, 10, 32, 100, 128):
            if k > n:
                continue
            for q in qs:
                assert np.array_equal(knn_keys(ib, plain, metric, q, k), knn_keys(ib, split, metric, q, k)), (metric, k)
            same(ib.batch_knn_many(metric, qs, plain, k), ib.batch_knn_many(metric, qs, split, k))


def test_every_f32_entry_split_equals_plain(ib):
    n, d = 6001, 40
    rows = rand_rows(n, d, 11)
    q = rand_rows(1, d, 12)[0]
    for how in ("rows", "pdx"):
        plain, split = both(ib, rows, 5, how)
        assert split.device_bytes() == plain.device_bytes()
        for f in (ib.batch_dot, ib.batch_l2_squared):
            same(f(q, plain), f(q, split))
        same(ib.batch_norms(plain), ib.batch_norms(split))
        nrm = ib.batch_norms(plain)
        same(ib.batch_cosine(q, plain, nrm), ib.batch_cosine(q, split, nrm))
        same(ib.batch_dimension_variance(plain), ib.batch_dimension_variance(split))
        for i in (0, 1, n - 1):
            same(plain.extract_vector(i), split.extract_vector(i))
        assert np.array_equal(bits(split.extract_vector(17)), bits(rows[17]))
        pred = lambda i: i % 3 != 0
        same(ib.batch_knn_filtered(q, plain, 10, pred), ib.batch_knn_filtered(q, split, 10, pred))
        same(ib.batch_l2_squared_pruning(q, plain, 40.0), ib.batch_l2_squared_pruning(q, split, 40.0))
        same(ib.batch_knn_reordered(q, plain, 10), ib.batch_knn_reordered(q, split, 10))
        same(ib.batch_knn_adaptive(q, plain, 10, 8), ib.batch_knn_adaptive(q, split, 10, 8))
        cand = np.arange(5, n + 5, 7, dtype=np.uint64)
        for metric in ("dot", "cosine", "l2"):
            same(ib.batch_knn_subset(metric, q, plain, cand, 10), ib.batch_knn_subset(metric, q, split, cand, 10))
            same(ib.batch_knn_many(metric, q, plain, 300), ib.batch_knn_many(metric, q, split, 300))
        pp, ps = plain.prefix(17), split.prefix(17)
        for metric in ("dot", "cosine", "l2"):
            same(ib.batch_knn_many(metric, q[:17], pp, 10), ib.batch_knn_many(metric, q[:17], ps, 10))
        same(ib.batch_dot(q[:17], pp), ib.batch_dot(q[:17], ps))
        same(ps.extract_vector(3), pp.extract_vector(3))
        from innr_b200 import binary, stream, ternary
        bq = binary.encode_binary(q, 0.1)
        same(binary.hamming_all(bq, binary.BinaryCorpus.from_f32(plain, 0.1)),
             binary.hamming_all(bq, binary.BinaryCorpus.from_f32(split, 0.1)))
        same(ternary.ternary_scores_all("asymmetric_dot", q, ternary.TernaryCorpus.from_f32(plain, 0.3)),
             ternary.ternary_scores_all("asymmetric_dot", q, ternary.TernaryCorpus.from_f32(split, 0.3)))
        prm = ib.QuantizationParams.from_range(-3.0, 3.0)
        same(stream.submit_knn_u8(q, ib.U8Corpus.from_f32(plain, prm), 50).wait(),
             stream.submit_knn_u8(q, ib.U8Corpus.from_f32(split, prm), 50).wait())


def test_generated_and_tensor_core_path(ib):
    from innr_b200 import synth
    n, d = 120_000, 128
    out = []
    for thr in (2**62, 0):
        ib.set_option("f32_split_min_rows", thr)
        out.append(ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d, index_base=3))
    ib.set_option("f32_split_min_rows", SPLIT_DEFAULT)
    plain, split = out
    qs = rand_rows(1024, d, 9)
    for metric in ("dot", "cosine"):   # 1024 queries: the tensor-core filter, which reads the corpus through pdx.cuh
        same(ib.batch_knn_many(metric, qs, plain, 10), ib.batch_knn_many(metric, qs, split, 10))
    for metric in ("dot", "cosine", "l2"):
        for q in qs[:8]:
            assert np.array_equal(knn_keys(ib, plain, metric, q, 10), knn_keys(ib, split, metric, q, 10))


def test_async_entries(ib):
    from innr_b200 import stream
    n, d = 20_000, 64
    rows = rand_rows(n, d, 21)
    plain, split = both(ib, rows)
    qs = rand_rows(4, d, 22)
    for metric in ("dot", "cosine", "l2"):
        for q in qs:
            a, b = stream.submit_knn(metric, q, plain, 10), stream.submit_knn(metric, q, split, 10)
            same(a.wait(), b.wait())


def _oracle_scores(oracle, metric, q, rows):
    n, d = rows.shape
    vb = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    if metric == "dot":
        return np.asarray(oracle.batch_dot(q, vb), np.float32)
    if metric == "l2":
        return np.asarray(oracle.batch_l2_squared(q, vb), np.float32)
    return np.asarray(oracle.batch_cosine(q, vb, oracle.batch_norms(vb)), np.float32)


def adversarial_rows(d, seed):
    """Rows whose low halves are as large as they get (one ulp of the high half short), all of one sign, parallel and
    antiparallel to the query; subnormal rows, zero rows, rows with norms from 1e-30 to 1e18."""
    rng = np.random.default_rng(seed)
    q = np.abs(rng.standard_normal(d)).astype(np.float32) + 0.5
    out = []
    qn = float(np.linalg.norm(q.astype(np.float64)))
    for norm in (1e-30, 1e-20, 1e-10, 1e-3, 1.0, 1e3, 1e10, 1e18):
        scale = norm / qn
        for sign in (1.0, -1.0):
            v = (q * np.float32(scale * sign)).astype(np.float32)
            b = v.view(np.uint32) | np.uint32(0xFFFF)   # lo just below one ulp of hi, same sign as v
            out.append(b.view(np.float32))
            out.append(v)
            out.append(((rng.random(d) * 2 - 1) * scale).astype(np.float32))
    sub = (rng.integers(1, 2**23, size=(4, d)).astype(np.uint32)).view(np.float32)   # subnormals
    out.extend(list(sub))
    out.append(np.zeros(d, np.float32))
    out.extend(list(rng.standard_normal((200, d)).astype(np.float32)))
    return q, np.stack(out).astype(np.float32)


@pytest.mark.parametrize("d", [1, 7, 768])
def test_screen_bound_holds_on_adversarial_rows(ib, oracle, d):
    q, rows = adversarial_rows(d, d)
    _, split = both(ib, rows)
    for metric in ("dot", "cosine", "l2"):
        for qq in (q, -q, q * np.float32(1e-3), q * np.float32(1e4)):
            lower, upper = ib.knn_screen_debug_bounds(metric, qq, split)
            ref = _oracle_scores(oracle, metric, qq, rows)
            ok = np.isfinite(ref)
            assert np.all(lower[ok] <= ref[ok]), (metric, np.nonzero(~(lower <= ref) & ok))
            assert np.all(ref[ok] <= upper[ok]), (metric, np.nonzero(~(ref <= upper) & ok))
            assert np.all(np.isinf(upper[~ok]) | np.isnan(ref[~ok]))
    plain, split = both(ib, rows)
    for metric in ("dot", "cosine", "l2"):
        for k in (1, 10, 100):
            for qq in (q, -q):
                assert np.array_equal(knn_keys(ib, plain, metric, qq, k), knn_keys(ib, split, metric, qq, k))


def test_zero_query_is_not_screened(ib):
    rows = rand_rows(3000, 16, 3)
    plain, split = both(ib, rows)
    with pytest.raises(NotImplementedError):
        ib.knn_screen_debug_bounds("cosine", np.zeros(16, np.float32), split)
    for metric in ("dot", "cosine", "l2"):
        z = np.zeros(16, np.float32)
        assert np.array_equal(knn_keys(ib, plain, metric, z, 10), knn_keys(ib, split, metric, z, 10))


def test_more_candidates_than_capacity_falls_back(ib):
    """Near-duplicates whose intervals all overlap: more than 4096 candidates, the device-side fallback answers."""
    n, d = 9000, 64
    base = rand_rows(1, d, 41)[0]
    rng = np.random.default_rng(42)
    rows = np.tile(base, (n, 1)).view(np.uint32)
    rows = (rows & np.uint32(0xFFFF0000)) | rng.integers(0, 2**16, size=rows.shape, dtype=np.uint32)
    rows = rows.view(np.float32)
    plain, split = both(ib, rows)
    lower, upper = ib.knn_screen_debug_bounds("dot", base, split)
    kth = np.sort(lower)[::-1][9]
    assert np.count_nonzero(upper >= kth) > 4096
    for metric in ("dot", "cosine", "l2"):
        for k in (10, 128):
            assert np.array_equal(knn_keys(ib, plain, metric, base, k), knn_keys(ib, split, metric, base, k))


def test_nonfinite_corpus_is_never_screened(ib):
    rows = rand_rows(3000, 24, 51)
    rows[100, 3] = np.nan
    rows[200, 5] = np.inf
    plain, split = both(ib, rows)
    with pytest.raises(NotImplementedError):
        ib.knn_screen_debug_bounds("dot", rows[0], split)
    for metric in ("dot", "cosine", "l2"):
        assert np.array_equal(knn_keys(ib, plain, metric, rows[1], 10), knn_keys(ib, split, metric, rows[1], 10))


def test_two_lanes_overlap_screened_scans(ib):
    """Screened scans on two caller streams (both workspace lanes) give what each gives alone."""
    import torch
    from innr_b200 import _lib as L
    n, d = 200_000, 96
    rows = rand_rows(n, d, 61)
    _, split = both(ib, rows)
    qs = torch.from_numpy(rand_rows(8, d, 62)).cuda()
    alone = [knn_keys(ib, split, "cosine", qs[j].cpu().numpy(), 10) for j in range(8)]
    streams = [torch.cuda.Stream() for _ in range(3)]
    outs = [torch.zeros(10, dtype=torch.int64, device="cuda") for _ in range(8)]
    for rep in range(3):
        for j in range(8):
            st = streams[j % 3]
            L.call("innr_cuda_batch_knn_keys_dev", split.h, L.METRIC_COSINE, C.c_void_p(qs[j].data_ptr()), 1, 10,
                   C.c_void_p(outs[j].data_ptr()), C.c_void_p(st.cuda_stream))
        torch.cuda.synchronize()
        for j in range(8):
            assert np.array_equal(outs[j].cpu().numpy(), alone[j]), (rep, j)
