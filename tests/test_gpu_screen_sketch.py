"""The 8-bit sketch the screened single-query kNN reads (layout.cu, scan_f32.cu, DESIGN.md sections 2 and 3.1).

What the sketch adds to the split layout: its interval must hold the reference's score on rows that are hard for a
per-row absmax quantiser, queries must be pre-scaled safely or refused, the screen must stay selective on realistic data,
and every writer must build it. Keys are always compared with a plain corpus of the same data."""
import ctypes as C

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SPLIT_DEFAULT = 1_000_000
F32_MAX = np.finfo(np.float32).max


@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    yield innr_b200
    innr_b200.set_option("f32_split_min_rows", SPLIT_DEFAULT)


def rand_rows(n, d, seed):
    return np.random.default_rng(seed).standard_normal((n, d)).astype(np.float32)


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


def oracle_scores(oracle, metric, q, rows):
    n, d = rows.shape
    vb = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    if metric == "dot":
        return np.asarray(oracle.batch_dot(q, vb), np.float32)
    if metric == "l2":
        return np.asarray(oracle.batch_l2_squared(q, vb), np.float32)
    return np.asarray(oracle.batch_cosine(q, vb, oracle.batch_norms(vb)), np.float32)


def check_interval(ib, oracle, split, rows, metric, q):
    """The interval holds the oracle's score, or the query is refused. Returns whether it was screened."""
    try:
        lower, upper = ib.knn_screen_debug_bounds(metric, q, split)
    except NotImplementedError:
        return False
    ref = oracle_scores(oracle, metric, q, rows)
    ok = np.isfinite(ref)
    assert np.all(lower[ok] <= ref[ok]), (metric, np.nonzero(~(lower <= ref) & ok))
    assert np.all(ref[ok] <= upper[ok]), (metric, np.nonzero(~(ref <= upper) & ok))
    assert np.all(np.isinf(upper[~ok]) | np.isnan(ref[~ok]))
    return True


def sketch_adversarial_rows(d, seed):
    """Rows that are hard for a per-row absmax quantiser."""
    rng = np.random.default_rng(seed)
    out = []
    for big in (1.0, 1e3, 1e10, 1.5e19):          # one huge outlier, tiny others (1.5e19: the norm is still finite)
        for tiny in (1e-3, 1e-12, 1e-30):
            v = ((rng.random(d) * 2 - 1) * tiny * big).astype(np.float32)
            v[rng.integers(d)] = np.float32(big * (1 if rng.random() < 0.5 else -1))
            out.append(v)
    s = np.float32(0.125)                          # absmax = 127 s exactly, every other element on a rounding tie
    v = ((rng.integers(-127, 127, size=d) + 0.5) * s).astype(np.float32)
    v[0] = np.float32(127) * s
    out.extend([v, -v])
    for normal in (1e-30, 1e-3, 1.0):             # subnormal and normal elements in one row
        v = (rng.integers(1, 2**23, size=d).astype(np.uint32)).view(np.float32).copy()
        v[rng.random(d) < 0.3] = np.float32(normal)
        out.append(v)
    out.append(np.full(d, -0.0, np.float32))
    out.append(np.zeros(d, np.float32))
    for c in (1.0, -3.5, 1e-20, 1e17):            # all elements equal
        out.append(np.full(d, c, np.float32))
    out.extend(list(rng.standard_normal((200, d)).astype(np.float32)))
    return np.stack(out).astype(np.float32)


@pytest.mark.parametrize("d", [1, 7, 768, 769])
def test_sketch_bound_holds_on_adversarial_rows(ib, oracle, d):
    rows = sketch_adversarial_rows(d, d + 3)
    plain, split = both(ib, rows)
    rng = np.random.default_rng(d)
    q = (np.abs(rng.standard_normal(d)) + 0.5).astype(np.float32)
    for metric in ("dot", "cosine", "l2"):
        for qq in (q, -q, q * np.float32(1e-3), q * np.float32(1e4), rows[0], rows[-1]):
            assert check_interval(ib, oracle, split, rows, metric, qq), metric
        for k in (1, 10, 100):
            for qq in (q, -q, rows[3]):
                assert np.array_equal(knn_keys(ib, plain, metric, qq, k), knn_keys(ib, split, metric, qq, k))


def test_absmax_near_float_max_keeps_the_corpus_off_the_screen(ib):
    rows = rand_rows(3000, 16, 71)
    rows[5, 2] = np.float32(0.99) * F32_MAX          # its reference norm overflows
    plain, split = both(ib, rows)
    with pytest.raises(NotImplementedError):
        ib.knn_screen_debug_bounds("dot", rows[0], split)
    for metric in ("dot", "cosine", "l2"):
        assert np.array_equal(knn_keys(ib, plain, metric, rows[1], 10), knn_keys(ib, split, metric, rows[1], 10))


def test_query_prescale_edges(ib, oracle):
    n, d = 3000, 64
    rows = rand_rows(n, d, 81)
    plain, split = both(ib, rows)
    rng = np.random.default_rng(82)
    queries = []
    wide = (10.0 ** rng.uniform(-30, 30, d) * rng.choice([-1.0, 1.0], d)).astype(np.float32)
    queries.append(wide)                             # elements from 1e-30 to 1e30
    queries.append(np.where(np.arange(d) == 5, np.float32(1), np.float32(0)).astype(np.float32))   # one-hot
    for top in (2.0**100, 2.0**-100, 2.0**99 * (2 - 2**-23), 2.0**-80):
        for nudge in (-1, 0, 1):                     # right at the guard, one ulp inside, one ulp outside
            m = np.nextafter(np.float32(top), np.float32(np.inf if nudge > 0 else 0)) if nudge else np.float32(top)
            qq = (rng.standard_normal(d) * 1e-3 * m).astype(np.float32)
            qq[7] = m
            queries.append(qq)
    screened = 0
    for qq in queries:
        for metric in ("dot", "cosine", "l2"):
            screened += check_interval(ib, oracle, split, rows, metric, qq)
            assert np.array_equal(knn_keys(ib, plain, metric, qq, 10), knn_keys(ib, split, metric, qq, 10)), metric
    assert screened > 0
    with pytest.raises(NotImplementedError):        # max |q_j| past 2^100: refused, answered by the full read
        bad = np.zeros(d, np.float32)
        bad[0] = np.nextafter(np.float32(2.0**100), np.float32(np.inf))
        ib.knn_screen_debug_bounds("dot", bad, split)


def test_screen_stays_selective_on_ghash(ib):
    """Rows whose upper bound reaches the 10th best lower bound: at most 100 of 200K (about 20-35 expected)."""
    from innr_b200 import synth
    n, d, k = 200_000, 768, 10
    ib.set_option("f32_split_min_rows", 0)
    try:
        split = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d)
    finally:
        ib.set_option("f32_split_min_rows", SPLIT_DEFAULT)
    qs = synth.ghash_f32(synth.SALT_QUERY, 0, 8 * d).reshape(8, d)
    for q in qs:
        lower, upper = ib.knn_screen_debug_bounds("cosine", q, split)
        kth = np.partition(lower, n - k)[n - k]
        cand = int(np.count_nonzero(upper >= kth))
        assert k <= cand <= 100, cand


def test_every_writer_builds_the_sketch(ib):
    from innr_b200 import synth
    n, d = 5000, 48
    rows = rand_rows(n, d, 91)
    qs = rand_rows(3, d, 92)
    pairs = [both(ib, rows, 3, "rows"), both(ib, rows, 3, "pdx")]
    gen = []
    for thr in (2**62, 0):
        ib.set_option("f32_split_min_rows", thr)
        try:
            gen.append(ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d, index_base=3))
        finally:
            ib.set_option("f32_split_min_rows", SPLIT_DEFAULT)
    pairs.append(gen)
    for plain, split in pairs:
        lower, upper = ib.knn_screen_debug_bounds("dot", qs[0], split)   # screened: the sketch exists
        assert np.all(lower <= upper)
        for metric in ("dot", "cosine", "l2"):
            for q in qs:
                assert np.array_equal(knn_keys(ib, plain, metric, q, 10), knn_keys(ib, split, metric, q, 10))
    plain, split = pairs[0]
    pp, ps = plain.prefix(17), split.prefix(17)
    with pytest.raises(NotImplementedError):        # a prefix view has no sidecar and is never screened
        ib.knn_screen_debug_bounds("dot", qs[0][:17], ps)
    for metric in ("dot", "cosine", "l2"):
        for q in qs:
            assert np.array_equal(knn_keys(ib, pp, metric, q[:17], 10), knn_keys(ib, ps, metric, q[:17], 10))
