"""The persistent top-k scans against the oracle at sizes where every CTA streams many tiles.

Every persistent scan strides tiles over a grid of at most (resident CTAs per SM) x 148 CTAs (`balanced_grid`), keeps
its warp lists across those tiles and merges them in `block_finish` (finish groups of 32 CTAs, self-resetting
tickets). The single-query Hamming scan also prunes against a launch-wide bound that a CTA refreshes every
SHARED_THR_PERIOD = 4 tiles, and the u8 scans reuse a bulk-copy ring of 6 (12 in the pair kernel) stages. Here every
corpus is sized so that each CTA streams at least 8 tiles, rows are planted where those mechanisms go wrong (the last
partial tile, the final wave, exact tie groups spread over finish groups), and whole results are compared with the
oracle's threaded entries: indices and score bits exactly, MaxSim within the DESIGN section 4 tolerance.

Resident CTAs per SM, from `-Xptxas -v` of the build and each kernel's `__launch_bounds__` (65536 registers, 2048
threads and 228 KB of shared memory per SM, 148 SMs):
  hamming_kernel         256 threads, 32 / 47 registers (R = 1 / 4)  -> <= 8 CTAs / SM (thread limit) -> <= 1184 CTAs
  hamming_multi_kernel   256 threads, 63-86 registers                 -> <= 4 CTAs / SM                -> <=  592 CTAs
  u8_scan_kernel         288 threads, 96 registers, 96 KB ring        -> <= 2 CTAs / SM (registers)    -> <=  296 CTAs
  u8_scan_pair_kernel    288 threads, 164-167 registers, 192 KB ring  -> 1 CTA / SM                    -> <=  148 CTAs
  pdx_screen_kernel      256 threads                                  -> <= 8 CTAs / SM (thread limit) -> <= 1184 CTAs
  pdx_scan_kernel        256 threads                                  -> <= 8 CTAs / SM (thread limit) -> <= 1184 CTAs
  maxsim_tc_kernel       grid = 148 CTAs (one per SM)

Each test prints its wall time and the device memory in use at its peak (run with -rP to see it)."""
import ctypes as C
import os
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SMS = 148
SPLIT_DEFAULT = 1_000_000
KS = (1, 10, 32, 33, 100, 128)
NT = max(1, min(os.cpu_count() or 1, 16))   # oracle threads


@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    yield innr_b200
    innr_b200.set_option("f32_split_min_rows", SPLIT_DEFAULT)


class _Usage:
    def __init__(self):
        import torch
        self.total = torch.cuda.mem_get_info()[1]
        self.peak = self.total - torch.cuda.mem_get_info()[0]
        self.t0 = time.time()

    def note(self):
        import torch
        torch.cuda.synchronize()
        self.peak = max(self.peak, self.total - torch.cuda.mem_get_info()[0])


@pytest.fixture
def usage(request):
    u = _Usage()
    yield u
    u.note()
    print(f"[many-tiles] {request.node.name}: wall {time.time() - u.t0:.1f} s, peak device memory in use {u.peak / 1e9:.1f} GB")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def _free_gb():
    import torch
    return torch.cuda.mem_get_info()[0] / 1e9


def _stream_ptr(st):
    return C.c_void_p(st.cuda_stream)


class Planter:
    """Unused row positions in the places where persistent scans go wrong: the first tile, the tiles 32, 64 and 96
    (first-wave tiles of CTAs in different finish groups), the final wave (the last 64 tiles; every grid here has more
    than 64 CTAs), the last, partial tile, and anywhere in between."""
    CYCLE = ("first", "g1", "last", "g2", "wave", "g3", "mid")

    def __init__(self, n, tile, seed):
        self.n, self.tile = n, tile
        self.rng = np.random.default_rng(seed)
        nt = (n + tile - 1) // tile
        assert nt >= 128
        self.ranges = {"first": (0, tile), "g1": (32 * tile, 33 * tile), "g2": (64 * tile, 65 * tile),
                       "g3": (96 * tile, 97 * tile), "wave": ((nt - 65) * tile, (nt - 1) * tile),
                       "last": ((nt - 1) * tile, n), "mid": (tile, n - tile)}
        self.taken = set()

    def pick(self, region):
        lo, hi = self.ranges[region]
        for _ in range(100_000):
            i = int(self.rng.integers(lo, hi))
            if i not in self.taken:
                self.taken.add(i)
                return i
        raise AssertionError(f"no free row left in {region}")

    def group(self, count, cycle=CYCLE):
        return [self.pick(cycle[j % len(cycle)]) for j in range(count)]


# Copies per level: the levels' running totals straddle every k of KS, so the k-th result of each k falls inside an
# exact tie group of which only the lowest indices may be returned.
LEVELS = (4, 12, 20, 70, 40)   # running totals 4, 16, 36, 106, 146


# ------------------------------------------------------------------------------------------------ 1. Hamming top-k
def test_hamming_1024bit_many_tiles(ib, oracle, usage):
    """8,000,200 codes of 1024 bits (1.02 GB) = 31,251 tiles of 256 codes, the last holding 200 codes.
    hamming_kernel (one query, shared threshold): <= 1184 CTAs -> >= 26 tiles per CTA (8 x 1184 = 9,472 <= 31,251).
    hamming_multi_kernel (2-5 queries): <= 592 CTAs -> >= 52 tiles per CTA.
    Planted rows are copies of a query with m bits flipped (distance exactly m), levels m = 2, 4, 6, 8, 10 of LEVELS
    copies each; the 4 copies at m = 2 and 6 of the 12 at m = 4 sit in one warp of tile 0 (warp j for query j), so the
    shared bound becomes tight early. Queries 0, 2 and 4 also have 3 rows at m = 1 and 2 at m = 3 in the final wave and
    the last tile: found long after the bound has tightened everywhere, they are the top of k = 1 and part of k = 10."""
    n, words = 8_000_200, 16
    codes = oracle.ghash_u64_mt(0x4A11_0001, 0, n * words, NT).reshape(n, words)
    qs = oracle.ghash_u64(0x4A11_0002, 0, 5 * words).reshape(5, words)
    pl = Planter(n, 256, 1)
    rng = np.random.default_rng(2)

    def flipped(q, m):
        b = np.unpackbits(q.view(np.uint8)).copy()
        b[rng.choice(1024, size=m, replace=False)] ^= 1
        return np.packbits(b).view(np.uint64)

    head = ("head",) * 4 + Planter.CYCLE[1:] + ("head",) * 2
    for j, q in enumerate(qs):
        pl.ranges["head"] = (32 * j, 32 * j + 32)   # warp j of tile 0: its 10th key is at distance 4
        for m, count in zip((2, 4, 6, 8, 10), LEVELS):
            for i in pl.group(count, head if m <= 4 else Planter.CYCLE):
                codes[i] = flipped(q, m)
        if j % 2 == 0:
            for m, region in ((1, "wave"), (1, "wave"), (1, "last"), (3, "wave"), (3, "last")):
                codes[pl.pick(region)] = flipped(q, m)
    corpus = ib.BinaryCorpus.from_words(codes.reshape(-1), n, 1024)
    usage.note()
    widx, wd = oracle.hamming_topk_many(qs, codes, 128, n_threads=min(NT, 5))   # stable sort: k < 128 is a prefix
    assert wd[:, 127].max() <= 10
    for k in KS:
        for j in range(5):
            gi, gd = ib.hamming_topk(qs[j], corpus, k)
            assert gi.tolist() == widx[j, :k].tolist() and gd.tolist() == wd[j, :k].tolist(), ("single", j, k)
        for lo, hi in ((0, 2), (1, 4), (0, 4), (0, 5)):
            gi, gd = ib.hamming_topk_many(qs[lo:hi], corpus, k)
            assert np.array_equal(gi, widx[lo:hi, :k]) and np.array_equal(gd, wd[lo:hi, :k]), ("batch", lo, hi, k)

    import torch
    from innr_b200 import _lib as L
    dq = torch.from_numpy(qs.view(np.int64)).cuda()

    def run(j, k, st):
        out = torch.empty(k, dtype=torch.int64, device="cuda")
        L.call("innr_cuda_hamming_topk_keys_dev", corpus.h, C.c_void_p(dq[j].data_ptr()), 1, k, C.c_void_p(out.data_ptr()),
               _stream_ptr(st))
        return out

    for k in (10, 100):
        want = [((wd[j, :k].astype(np.uint64) << np.uint64(32)) | widx[j, :k]) for j in (0, 1)]
        _check_abab(run, k, lambda o, j: np.array_equal(o.view(np.uint64), want[j]))


def _check_abab(run, k, ok):
    """A, B, A on one stream, then A and B on two caller streams (both workspace lanes): every result must be the one
    the query gives alone (tickets and the shared bound were reset by the launch before)."""
    import torch
    main = torch.cuda.current_stream()
    seq = [run(0, k, main), run(1, k, main), run(0, k, main)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    s1.wait_stream(main)
    s2.wait_stream(main)
    par = [run(0, k, s1), run(1, k, s2)]
    torch.cuda.synchronize()
    got = [o.cpu().numpy() for o in seq + par]
    assert np.array_equal(got[0], got[2]) and np.array_equal(got[0], got[3]) and np.array_equal(got[1], got[4]), k
    assert ok(got[0], 0) and ok(got[1], 1), k


# ------------------------------------------------------------------------------------------------ 2. u8
@pytest.mark.parametrize("n,d", [(4_000_200, 384), (1_000_136, 777)])
def test_u8_many_tiles(ib, oracle, usage, n, d):
    """d = 384: 24 chunk rows = 6 ring stages per tile, one tile fills the 6-stage ring exactly; 4,000,200 rows
    (1.54 GB) = 15,626 tiles of 256 rows. d = 777: 49 chunk rows = 13 stages per tile, more than either ring;
    1,000,136 rows (0.78 GB) = 3,907 tiles. The last tile holds 200 rows in both.
    u8_scan_kernel: <= 296 CTAs -> >= 52 (d = 384) / >= 13 (d = 777) tiles per CTA (8 x 296 = 2,368).
    u8_scan_pair_kernel: <= 148 CTAs -> >= 105 / >= 26 tiles per CTA.
    Planted rows: for each query, LEVELS copies of five rows built to score far above the random rows (bytes 255 where
    the query is positive, 0 elsewhere, with 3, 6, ... of the largest positive positions lowered to 200)."""
    gp, op = ib.QuantizationParams.from_range(-1.0, 1.0), oracle.QuantizationParams.from_range(-1.0, 1.0)
    mat = oracle.ghash_u8_rows(0x4A11_0003, 0, n, d, op, NT)
    qs = oracle.ghash_f32(0x4A11_0004, d, 4 * d).reshape(4, d)
    pl = Planter(n, 256, d)
    for q in qs:
        best = np.where(q > 0, 255, 0).astype(np.uint8)
        order = np.argsort(-q)
        for lvl, count in enumerate(LEVELS):
            row = best.copy()
            row[order[:3 * (lvl + 1)]] = 200
            mat[pl.group(count)] = row
    corpus = ib.U8Corpus.from_rows(mat, gp)
    usage.note()
    widx, wsc = oracle.batch_knn_u8_many(qs, mat, op, 128, n_threads=min(NT, 4))   # stable sort: k < 128 is a prefix
    for k in KS:
        for j in (0, 1):
            gi, gs = ib.batch_knn_u8_many(qs[j], corpus, k)
            assert np.array_equal(gi[0], widx[j, :k]) and np.array_equal(bits(gs[0]), bits(wsc[j, :k])), ("single", j, k)
        gi, gs = ib.batch_knn_u8_many(qs, corpus, k)   # two pairs
        assert np.array_equal(gi, widx[:, :k]) and np.array_equal(bits(gs), bits(wsc[:, :k])), ("pairs", k)

    import torch
    from innr_b200 import _lib as L
    dq = torch.from_numpy(qs).cuda()

    def run(j, k, st):
        out = torch.empty(k, dtype=torch.int64, device="cuda")
        L.call("innr_cuda_batch_knn_u8_keys_dev", corpus.h, C.c_void_p(dq[j].data_ptr()), 1, k, C.c_void_p(out.data_ptr()),
               _stream_ptr(st))
        return out

    _check_abab(run, 10, lambda o, j: (o.view(np.uint64) & np.uint64(0xFFFFFFFF)).tolist() == widx[j, :10].tolist())


# ------------------------------------------------------------------------------------------------ 3. screened f32 kNN
def _plant_f32(rows, pdx, qs, pl):
    """Per query, two families of LEVELS exact copies each: q x (4 - 0.01 l) lead dot (and, with every positive
    multiple of q, cosine), q x (1 - 0.001 (l + 1)) lead L2."""
    n, d = rows.shape
    for q in qs:
        for scales in ([4.0 - 0.01 * l for l in range(5)], [1.0 - 0.001 * (l + 1) for l in range(5)]):
            for s, count in zip(scales, LEVELS):
                v = (q * np.float32(s)).astype(np.float32)
                for i in pl.group(count):
                    rows[i] = v
                    if pdx is not None:
                        pdx[:, i] = v


def _want_knn(oracle, metric, qs, ob, k_max):
    """The oracle's top-k_max per query. For L2, whose tie order at the k-th is left open by the reference (DESIGN
    section 4, Ties), the device's order -- the k smallest (distance, index) -- is rebuilt from the oracle's whole
    distance vector, after checking that the oracle's own list agrees with it score for score."""
    widx, wsc = oracle.batch_knn_many(metric, qs, ob, k_max, n_threads=min(NT, len(qs)))
    if metric != "l2":
        return widx, wsc
    out = np.empty_like(widx)
    for j, q in enumerate(qs):
        dist = oracle.batch_l2_squared(q, ob)
        cand = np.flatnonzero(bits(dist) <= bits(wsc[j, -1]))   # non-negative floats order like their bits
        order = cand[np.lexsort((cand, dist[cand]))][:k_max]
        assert np.array_equal(bits(dist[order]), bits(wsc[j])) and np.array_equal(bits(dist[widx[j]]), bits(wsc[j]))
        out[j] = order
    return out, wsc


def _check_knn(ib, db, qs, want, metrics=("dot", "cosine", "l2"), ks=(1, 10, 100, 128)):
    for metric in metrics:
        widx, wsc = want[metric]
        for k in ks:
            for j, q in enumerate(qs):
                gi, gs = ib.batch_knn_many(metric, q, db, k)
                assert np.array_equal(gi[0], widx[j, :k]), (metric, k, j, gi[0][:8], widx[j, :8])
                assert np.array_equal(bits(gs[0]), bits(wsc[j, :k])), (metric, k, j)


def test_screened_knn_tall_split_corpus(ib, oracle, usage):
    """48,000,123 x 16 rows (3.07 GB), uploaded row-major under default options: split (>= f32_split_min_rows) and
    written through the chunked 256 MB staging upload.
    pdx_screen_kernel: 11,719 tiles of 4096 rows, <= 1184 CTAs -> >= 9.9 tiles per CTA (8 x 1184 = 9,472 <= 11,719).
    The same rows as a plain corpus go through pdx_scan_kernel, the full-read scan every screened call can fall back
    to: 46,876 tiles of 1024 rows, <= 1184 CTAs -> >= 39 tiles per CTA.
    Planted exact tie groups (_plant_f32: 146 rows per family and query) stay below the 4096-candidate cap, which is
    checked through the screen's own interval."""
    from innr_b200 import _lib as L
    n, d = 48_000_123, 16
    rows = oracle.ghash_f32_mt(0x4A11_0005, 0, n * d, NT).reshape(n, d)
    ob = oracle.ghash_vertical_batch(0x4A11_0005, 0, n, d, NT)
    qs = oracle.ghash_f32(0x4A11_0006, 0, 3 * d).reshape(3, d)
    _plant_f32(rows, ob.data.reshape(d, n), qs, Planter(n, 4096, 3))
    want = {m: _want_knn(oracle, m, qs, ob, 128) for m in ("dot", "cosine", "l2")}

    split = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    usage.note()
    _check_knn(ib, split, qs, want)
    for metric in ("dot", "cosine", "l2"):   # the screen answered these itself: candidates within the cap
        lower, upper = ib.knn_screen_debug_bounds(metric, qs[0], split)
        if metric == "l2":
            cand = np.count_nonzero(lower <= np.partition(upper, 127)[127])
        else:
            cand = np.count_nonzero(upper >= -np.partition(-lower, 127)[127])
        assert 128 <= cand <= 4096, (metric, cand)
    del lower, upper

    import torch
    dq = torch.from_numpy(qs).cuda()

    def run(j, k, st):
        out = torch.empty(k, dtype=torch.int64, device="cuda")
        L.call("innr_cuda_batch_knn_keys_dev", split.h, L.METRIC_COSINE, C.c_void_p(dq[j].data_ptr()), 1, k,
               C.c_void_p(out.data_ptr()), _stream_ptr(st))
        return out

    _check_abab(run, 10, lambda o, j: (o.view(np.uint64) & np.uint64(0xFFFFFFFF)).tolist() == want["cosine"][0][j, :10].tolist())
    del split
    usage.note()

    ib.set_option("f32_split_min_rows", 2**62)
    try:
        plain = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    finally:
        ib.set_option("f32_split_min_rows", SPLIT_DEFAULT)
    with pytest.raises(NotImplementedError):
        ib.knn_screen_debug_bounds("dot", qs[0], plain)
    _check_knn(ib, plain, qs, want)


def test_screened_knn_c2a_shape_equals_full_read(ib, oracle, usage):
    """C2a's shape: 10M x 768 (30.7 GB split planes + 7.7 GB sketch), generated on the device. Screened keys of 32
    queries x 3 metrics x k in {1, 10, 100, 128} against the full-read scan of `split.prefix(768)` -- the same planes
    without the sidecar -- whole lists of 64-bit keys.
    pdx_screen_kernel: 2,442 tiles of 4096 rows; pdx_scan_kernel: 9,766 tiles of 1024 rows, <= 1184 CTAs -> >= 8.2
    tiles per CTA."""
    from innr_b200 import synth
    from innr_b200 import _lib as L
    if _free_gb() < 50:
        pytest.skip("needs ~40 GB of free HBM")
    import torch
    n, d, nq = 10_000_000, 768, 32
    split = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d)
    full = split.prefix(d)
    usage.note()
    qs = torch.from_numpy(oracle.ghash_f32(0x4A11_0007, 0, nq * d).reshape(nq, d)).cuda()
    st = torch.cuda.current_stream()
    metrics = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}
    for name, m in metrics.items():
        for k in (1, 10, 100, 128):
            a = torch.empty((nq, k), dtype=torch.int64, device="cuda")
            b = torch.empty((nq, k), dtype=torch.int64, device="cuda")
            for j in range(nq):
                for db, out in ((split, a), (full, b)):
                    L.call("innr_cuda_batch_knn_keys_dev", db.h, m, C.c_void_p(qs[j].data_ptr()), 1, k,
                           C.c_void_p(out[j].data_ptr()), _stream_ptr(st))
            torch.cuda.synchronize()
            assert torch.equal(a, b), (name, k, int((a != b).any(1).sum()))


@pytest.mark.parametrize("d", [1536, 1537, 4096, 4097])
def test_screened_knn_dimension_edges(ib, oracle, usage, d):
    """The screen's largest dimensions: the rescoring kernel's shared memory (8 rows of d floats) is 48 KB at d = 1536
    and needs the opt-in above it; SCREEN_MAX_D = 4096 is the last dimension the screen takes, d = 4097 is refused by
    it and answered by the full-read scan. 20,000 rows on a split corpus, with exact tie groups planted; the interval
    must hold the oracle's score of every row, and the keys must equal the oracle's."""
    n = 20_000
    rows = oracle.ghash_f32_mt(0x4A11_0008, 0, n * d, NT).reshape(n, d)
    qs = oracle.ghash_f32(0x4A11_0009, 0, 2 * d).reshape(2, d)
    pos = iter(np.random.default_rng(d).choice(n, size=40, replace=False))
    for q in qs:
        for s, count in ((2.0, 3), (1.5, 12), (1.0, 5)):
            rows[[next(pos) for _ in range(count)]] = (q * np.float32(s)).astype(np.float32)
    ib.set_option("f32_split_min_rows", 0)
    try:
        split = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    finally:
        ib.set_option("f32_split_min_rows", SPLIT_DEFAULT)
    usage.note()
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    want = {m: _want_knn(oracle, m, qs, ob, 128) for m in ("dot", "cosine", "l2")}
    for metric in ("dot", "cosine", "l2"):
        if d > 4096:
            with pytest.raises(NotImplementedError):
                ib.knn_screen_debug_bounds(metric, qs[0], split)
            continue
        ref = (oracle.batch_dot(qs[0], ob) if metric == "dot" else oracle.batch_l2_squared(qs[0], ob) if metric == "l2"
               else oracle.batch_cosine(qs[0], ob, oracle.batch_norms(ob)))
        lower, upper = ib.knn_screen_debug_bounds(metric, qs[0], split)
        assert np.all(lower <= ref) and np.all(ref <= upper), metric
    _check_knn(ib, split, qs, want, ks=(1, 10, 128))


# ------------------------------------------------------------------------------------------------ 4. MaxSim tcgen05
def _maxsim_checks(ib, oracle, corpus, toks, off, qs, cosine, rel):
    """dev (torch's current stream) == host, batch_dev == batch host == singles, bit for bit; all within the DESIGN
    section 4 tolerance, and (rel, the C3 shape) within 1e-5 relative."""
    import torch
    from innr_b200 import _lib as L
    nd = corpus.num_docs
    host = np.stack([ib.maxsim_corpus(q, corpus, cosine=cosine) for q in qs])
    hb = ib.maxsim_corpus_batch(qs, corpus, cosine=cosine)
    dq = torch.from_numpy(np.ascontiguousarray(qs)).cuda()
    one = torch.empty(nd, dtype=torch.float32, device="cuda")
    both = torch.empty((2, nd), dtype=torch.float32, device="cuda")
    st = _stream_ptr(torch.cuda.current_stream())
    L.call("innr_cuda_maxsim_dev", corpus.h, C.c_void_p(dq[0].data_ptr()), qs.shape[1], int(cosine),
           C.c_void_p(one.data_ptr()), st)
    L.call("innr_cuda_maxsim_batch_dev", corpus.h, C.c_void_p(dq.data_ptr()), 2, qs.shape[1], int(cosine),
           C.c_void_p(both.data_ptr()), st)
    torch.cuda.synchronize()
    assert np.array_equal(bits(one.cpu().numpy()), bits(host[0]))
    assert np.array_equal(bits(both.cpu().numpy()), bits(host)) and np.array_equal(bits(hb), bits(host))
    for j, q in enumerate(qs):
        want = oracle.maxsim_corpus(q, toks, off, cosine_flag=cosine, n_threads=NT).astype(np.float64)
        # DESIGN section 4: |got - ref| <= 1e-5 sum_i max_j sum_k |q_ik d_jk| + 1e-6; for cosine every normalised
        # pair's sum is at most 1, so the bound is at most 1e-5 n_q + 1e-6
        cond = (np.full(nd, float(q.shape[0])) if cosine
                else oracle.maxsim_corpus(np.abs(q), np.abs(toks), off, n_threads=NT).astype(np.float64))
        err = np.abs(host[j].astype(np.float64) - want)
        assert np.all(err <= 1e-5 * cond + 1e-6), (cosine, j, float((err - 1e-5 * cond).max()))
        if rel:
            assert float((err / np.maximum(np.abs(want), 1e-30)).max()) < 1e-5, (cosine, j)
    return dq


def test_maxsim_tc_c3_document_shape(ib, oracle, usage):
    """20,000 docs x 180 tokens x 128 (1.84 GB, generated on the device): 28,125 tiles of 128 tokens over a grid of
    148 CTAs -> 190 tiles per CTA (8 x 148 = 1,184). Two 32-token queries."""
    from innr_b200 import synth
    n_docs, nt, dim = 20_000, 180, 128
    corpus = ib.TokenCorpus.generate(synth.SALT_CORPUS, 0, n_docs, nt, dim)
    toks = oracle.ghash_f32_mt(synth.SALT_CORPUS, 0, n_docs * nt * dim, NT).reshape(-1, dim)
    off = np.arange(0, (n_docs + 1) * nt, nt, dtype=np.uint64)
    qs = oracle.ghash_f32(synth.SALT_QUERY, 0, 2 * 32 * dim).reshape(2, 32, dim)
    usage.note()
    for cosine in (True, False):
        dq = _maxsim_checks(ib, oracle, corpus, toks, off, qs, cosine, rel=True)

    import torch
    from innr_b200 import _lib as L
    want = [ib.maxsim_corpus(q, corpus, cosine=True) for q in qs]

    def run(j, k, st):
        out = torch.empty(n_docs, dtype=torch.float32, device="cuda")
        L.call("innr_cuda_maxsim_dev", corpus.h, C.c_void_p(dq[j].data_ptr()), 32, 1, C.c_void_p(out.data_ptr()),
               _stream_ptr(st))
        return out

    _check_abab(run, 0, lambda o, j: np.array_equal(bits(o), bits(want[j])))


def test_maxsim_tc_mixed_lengths(ib, oracle, usage):
    """20,000 uploaded docs of 0-360 tokens (about 3.6M tokens, 1.85 GB): about 28,000 tiles of 128 tokens over 148
    CTAs -> about 190 tiles per CTA; documents straddle tile boundaries everywhere, empty ones score 0."""
    n_docs, dim = 20_000, 128
    lens = np.random.default_rng(5).integers(0, 361, size=n_docs)
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    toks = oracle.ghash_f32_mt(0x4A11_000A, 0, int(off[-1]) * dim, NT).reshape(-1, dim)
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    qs = oracle.ghash_f32(0x4A11_000B, 0, 2 * 32 * dim).reshape(2, 32, dim)
    usage.note()
    assert int(off[-1]) // 128 >= 8 * SMS
    for cosine in (True, False):
        _maxsim_checks(ib, oracle, corpus, toks, off, qs, cosine, rel=False)
