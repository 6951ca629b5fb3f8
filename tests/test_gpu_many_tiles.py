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
    (the masked form of batch_knn_filtered: 38 / 64 registers for R = 1 / 4; the reordered form PDX_L2_PERM)
  ternary_topk_kernel    256 threads, 32-40 registers (all OP, R)     -> <= 8 CTAs / SM (thread limit) -> <= 1184 CTAs
  binary_setops_topk_kernel  256 threads, 32-40 registers             -> <= 8 CTAs / SM (thread limit) -> <= 1184 CTAs
  topk_scores_kernel     256 threads, grid capped at 4 x 148 = 592 CTAs (launch_topk_from_scores); every selection
                         of k > 128, of topk_from_distances and of the filtered / adaptive rounds: <= 592 x 256
                         elements per grid-stride step
  maxsim_tc_kernel       grid = 148 CTAs (one per SM)
Every case asserts its own premise from its sizes (_n_tiles): tiles (or grid-stride steps) >= 8 x the largest grid.
The tests after the MaxSim ones share module-scoped corpora (each built once) and end with launches of different
grids back to back on one workspace.

Each test and each shared corpus prints its wall time, the device memory in use at its peak and the process's
resident host memory at its peak (run with -rP to see it)."""
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
    """Wall time, device memory in use at its peak (sampled by note()), and the process's resident host memory at its
    peak (sampled every 20 ms by a thread)."""

    def __init__(self):
        import threading
        import torch
        self.total = torch.cuda.mem_get_info()[1]
        self.peak = self.total - torch.cuda.mem_get_info()[0]
        self.t0 = time.time()
        self.host_peak = 0
        self._stop = threading.Event()
        self._thread = threading.Thread(target=self._sample_host, daemon=True)
        self._thread.start()

    def _sample_host(self):
        page = os.sysconf("SC_PAGE_SIZE")
        while True:
            with open("/proc/self/statm") as f:
                self.host_peak = max(self.host_peak, int(f.read().split()[1]) * page)
            if self._stop.wait(0.02):
                return

    def note(self):
        import torch
        torch.cuda.synchronize()
        self.peak = max(self.peak, self.total - torch.cuda.mem_get_info()[0])

    def report(self, name):
        self.note()
        self._stop.set()
        self._thread.join()
        print(f"[many-tiles] {name}: wall {time.time() - self.t0:.1f} s, peak device memory in use {self.peak / 1e9:.1f} GB,"
              f" peak host memory resident {self.host_peak / 1e9:.1f} GB")


@pytest.fixture
def usage(request):
    u = _Usage()
    yield u
    u.report(request.node.name)


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
    widx, wd = oracle.hamming_topk_many(qs, codes, 300, n_threads=min(NT, 5))   # stable sort: k < 300 is a prefix
    assert wd[:, 127].max() <= 10
    for k in KS + (129, 300):   # 129 and 300: the scores pass, then selection rounds of kind 2
        for j in range(5):
            gi, gd = ib.hamming_topk(qs[j], corpus, k)
            assert gi.tolist() == widx[j, :k].tolist() and gd.tolist() == wd[j, :k].tolist(), ("single", j, k)
        if k > 128:
            continue
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
    widx, wsc = oracle.batch_knn_u8_many(qs, mat, op, 300, n_threads=min(NT, 4))   # stable sort: k < 300 is a prefix
    for k in KS + (129, 300):   # 129 and 300: the scores pass, then selection rounds of kind 1
        for j in (0, 1):
            gi, gs = ib.batch_knn_u8_many(qs[j], corpus, k)
            assert np.array_equal(gi[0], widx[j, :k]) and np.array_equal(bits(gs[0]), bits(wsc[j, :k])), ("single", j, k)
        if k > 128:
            continue
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


# ------------------------------------------------------------------------------------------------ 5. ternary top-k
KS_ROUNDS = KS + (129, 300)   # k > 128: the scores pass, then selection rounds of topk_scores_kernel
BIG_BASE = 3_000_000_000      # > 2^31: a signed or truncated index shows
TER_N = 2_500_037             # 9,766 tiles of 256 codes, the last holding 197


def _n_tiles(n, tile, max_grid):
    """Tiles (or, for topk_scores_kernel, grid-stride steps of 256 elements) of a launch of n rows, asserted to give each
    CTA of the largest grid the kernel can have at least 8 of them."""
    nt = -(-n // tile)
    assert nt >= 8 * max_grid, (n, tile, nt, max_grid)
    return nt


def _pool_map(fn, items):
    from concurrent.futures import ThreadPoolExecutor
    with ThreadPoolExecutor(NT) as ex:
        return list(ex.map(fn, items))


T_ODD, T_EVEN, ONE = np.uint64(0x5555555555555555), np.uint64(0xAAAAAAAAAAAAAAAA), np.uint64(1)


def _ter_masks(w):
    """innr_ref.cpp ternary_dot / ternary_hamming: +1 and -1 positions (one bit per value) and nonzero positions."""
    hi = (w & T_EVEN) >> ONE
    return w & ~hi & T_ODD, ~w & hi & T_ODD, (w & T_ODD) | hi


def _ter_ref_int(words, qw, block=1 << 16):
    """ternary_dot and ternary_hamming of every row of row-major words against query words qw."""
    n = len(words)
    dot, ham = np.empty(n, np.int32), np.empty(n, np.int32)
    qp, qn, qz = _ter_masks(qw)

    def work(b0):
        w = words[b0:b0 + block]
        p, m, z = _ter_masks(w)
        same = np.bitwise_count((p & qp) | (m & qn)).sum(axis=1, dtype=np.int32)
        diff = np.bitwise_count((p & qn) | (m & qp)).sum(axis=1, dtype=np.int32)
        dot[b0:b0 + block] = same - diff
        x = w ^ qw
        ham[b0:b0 + block] = np.bitwise_count(((x & T_ODD) | ((x & T_EVEN) >> ONE)) & z & qz).sum(axis=1, dtype=np.int32)

    _pool_map(work, range(0, n, block))
    return dot, ham


def _ter_ref_asym(words, q, block=1 << 14):
    """ternary::asymmetric_dot of every row: the sequential f32 sum s = s + q[j] * t[j] (products and sums rounded
    separately, 0b11 reads 0), over dimension-major values unpacked from the words."""
    n, nw = words.shape
    d = len(q)
    out = np.empty(n, np.float32)
    qc = np.asarray(q, np.float32)[:, None]

    def work(b0):
        w = np.ascontiguousarray(words[b0:b0 + block].T)                     # (words, rows)
        by = np.ascontiguousarray(w.view(np.uint8).reshape(nw, -1, 8).transpose(0, 2, 1))   # byte b of word i
        c = np.empty((nw, 8, 4, by.shape[2]), np.uint8)
        for t in range(4):
            c[:, :, t] = (by >> (2 * t)) & 3
        c = c.reshape(nw * 32, -1)[:d]                                          # (d, rows) 2-bit codes
        p = np.multiply((c & 1).astype(np.int8) - (c >> 1).astype(np.int8), qc, dtype=np.float32)
        s = np.zeros(p.shape[1], np.float32)
        for j in range(d):
            np.add(s, p[j], out=s)
        out[b0:b0 + block] = s

    _pool_map(work, range(0, n, block))
    return out


def _stable_order(scores, descending, k):
    """The first k of a stable sort (ties -> lower index) under the order of the keys: f32 by total order."""
    if scores.dtype == np.float32:
        b = scores.view(np.uint32)
        key = np.where(b >> np.uint32(31), ~b, b | np.uint32(0x80000000))
        key = ~key if descending else key
    else:
        key = -scores.astype(np.int64) if descending else scores
    part = np.argpartition(key, k)[:k + 1] if len(key) > k + 1 else np.arange(len(key))
    cut = key[part].max()   # every row with a key <= the (k+1)-th smallest, then sorted stably
    cand = np.flatnonzero(key <= cut)
    return cand[np.argsort(key[cand], kind="stable")][:k]


def _valid_ternary(w, d):
    """pairs 0b11 -> 0b01, padding pairs cleared: what PackedTernary::set can produce"""
    w = w & ~((w & T_ODD) << ONE)
    if d % 32:
        w[..., -1] &= np.uint64((1 << (2 * (d % 32))) - 1)
    return w


@pytest.fixture(scope="module")
def ternary(ib, oracle):
    """For d = 200 (a partial 64-value chunk and a partial word) and d = 1024: 2,500,037 raw random ternary codes (0b11
    pairs and dirty padding bits included, as from_words accepts them) at index_base 3,000,000,000, two ternary queries
    and one f32 query, and the reference top-300 of every (op, query). Planted per ternary query: LEVELS copies of the
    query with m = 1..5 nonzero values negated (dot |q|nz - 2m, Hamming m); per f32 query: LEVELS copies each of five
    rows sign(q) with its 3, 6, ... largest |q| values zeroed (identical rows: identical sums)."""
    u = _Usage()
    out = {}
    for d in (200, 1024):
        words = oracle.ghash_u64_mt(0x4A11_0100 + d, 0, TER_N * ((d + 31) // 32), NT).reshape(TER_N, -1)
        qws = _valid_ternary(oracle.ghash_u64(0x4A11_0101 + d, 0, 2 * words.shape[1]).reshape(2, -1), d)
        qf = oracle.ghash_f32(0x4A11_0102 + d, 0, d)
        qf[d // 3] = -0.0
        pl = Planter(TER_N, 256, d)
        rng = np.random.default_rng(d)
        for qw in qws:
            nzp = np.flatnonzero(np.array([(int(qw[j // 32]) >> (2 * (j % 32))) & 3 for j in range(d)]) != 0)
            for m, count in zip(range(1, 6), LEVELS):
                for i in pl.group(count):
                    row = qw.copy()
                    for j in rng.choice(nzp, size=m, replace=False):
                        row[j // 32] ^= np.uint64(3 << (2 * (j % 32)))
                    words[i] = row
        best = np.where(qf > 0, 1, np.where(qf < 0, 2, 0))
        order = np.argsort(-np.abs(qf), kind="stable")
        for lvl, count in enumerate(LEVELS):
            vals = best.copy()
            vals[order[:3 * (lvl + 1)]] = 0
            row = np.zeros(words.shape[1], np.uint64)
            for j in np.flatnonzero(vals):
                row[j // 32] |= np.uint64(int(vals[j]) << (2 * (j % 32)))
            words[pl.group(count)] = row
        if d % 32:   # dirty padding pairs: the upload masks them, as PackedTernary::new does
            words[::7, -1] |= ~np.uint64((1 << (2 * (d % 32))) - 1)
        corpus = ib.TernaryCorpus.from_words(words.reshape(-1), TER_N, d, index_base=BIG_BASE)
        if d % 32:
            words[:, -1] &= np.uint64((1 << (2 * (d % 32))) - 1)
        want = {}
        for j, qw in enumerate(qws):
            dot, ham = _ter_ref_int(words, qw)
            want["dot", j] = (_stable_order(dot, True, 300), dot)
            want["hamming", j] = (_stable_order(ham, False, 300), ham)
        asym = _ter_ref_asym(words, qf)
        want["asymmetric_dot", 0] = (_stable_order(asym, True, 300), asym)
        # the numpy restatement against the oracle's: planted rows, the last tile, and random rows
        rows = sorted(pl.taken)[::3] + list(range(TER_N - 60, TER_N)) + list(range(0, 40))
        oq = [oracle.PackedTernary(qw, d) for qw in qws]
        for i in rows:
            oc = oracle.PackedTernary(words[i], d)
            for j in range(2):
                assert oracle.ternary_dot(oq[j], oc) == want["dot", j][1][i], (d, i)
                assert oracle.ternary_hamming(oq[j], oc) == want["hamming", j][1][i], (d, i)
            assert bits(np.float32(oracle.ternary_asymmetric_dot(qf, oc))) == bits(asym[i]), (d, i)
        out[d] = {"corpus": corpus,
                  "queries": {"dot": [ib.PackedTernary(qw, d) for qw in qws],
                              "hamming": [ib.PackedTernary(qw, d) for qw in qws], "asymmetric_dot": [qf]},
                  "want": {key: (idx, sc[idx].astype(np.float32)) for key, (idx, sc) in want.items()}}
        del words, dot, ham, asym
    u.report("fixture ternary")
    return out


def test_ternary_topk_many_tiles(ib, ternary, usage):
    """ternary_topk_kernel<OP, R>, all three ops: 9,766 tiles of 256 codes, <= 1184 CTAs (256 threads, 32-40 registers:
    thread limit) -> >= 8.2 tiles per CTA; k = 129 and 300 take the scores kernel and selection rounds of kinds 0 and 1
    over 2,500,037 scores (>= 16 grid-stride steps per thread of topk_scores_kernel's 592 CTAs). Indices carry
    index_base = 3,000,000,000; scores compared bit for bit."""
    _n_tiles(TER_N, 256, 8 * SMS)
    _n_tiles(TER_N, 256, 4 * SMS)
    usage.note()
    for d, t in ternary.items():
        for (op, j), (widx, wsc) in t["want"].items():
            q = t["queries"][op][j]
            for k in KS_ROUNDS:
                gi, gs = ib.ternary_topk(op, q, t["corpus"], k)
                assert gi.tolist() == (widx[:k] + BIG_BASE).tolist(), (d, op, j, k, gi[:6], widx[:6] + BIG_BASE)
                assert np.array_equal(bits(gs), bits(wsc[:k])), (d, op, j, k)


def test_ternary_from_split_corpus(ib, oracle, usage):
    """ternary_from_pdx_kernel over split planes at scale: encode_ternary of a split DeviceBatch of 2,500,037 x 100
    ghash rows (100 values: a partial chunk and a partial word) on the device must give the codes numpy gives: every
    dot and Hamming score of two queries, and the top-k of all three ops, equal those of the uploaded numpy words."""
    n, d, thr = TER_N, 100, 0.25
    rows = oracle.ghash_f32_mt(0x4A11_0103, 0, n * d, NT).reshape(n, d)
    split = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)   # n >= f32_split_min_rows: split planes
    derived = ib.TernaryCorpus.from_f32(split, thr)
    del split
    nw = (d + 31) // 32
    words = np.zeros((n, nw), np.uint64)

    def enc(b0, block=1 << 16):
        v = rows[b0:b0 + block]
        c = np.zeros((len(v), nw * 32), np.uint64)
        c[:, :d] = np.where(v > thr, 1, np.where(v < -thr, 2, 0))
        words[b0:b0 + block] = (c.reshape(len(v), nw, 32) << (2 * np.arange(32, dtype=np.uint64))).sum(axis=2, dtype=np.uint64)

    _pool_map(enc, range(0, n, 1 << 16))
    assert np.count_nonzero(words) > n
    uploaded = ib.TernaryCorpus.from_words(words.reshape(-1), n, d)
    usage.note()
    qws = _valid_ternary(oracle.ghash_u64(0x4A11_0104, 0, 2 * nw).reshape(2, nw), d)
    qf = oracle.ghash_f32(0x4A11_0105, 0, d)
    for qw in qws:
        q = ib.PackedTernary(qw, d)
        for op in ("dot", "hamming"):
            assert np.array_equal(ib.ternary_scores_all(op, q, derived), ib.ternary_scores_all(op, q, uploaded)), op
    dot, ham = _ter_ref_int(words, qws[0])
    assert np.array_equal(ib.ternary_scores_all("dot", ib.PackedTernary(qws[0], d), derived), dot)
    for op, q in (("dot", ib.PackedTernary(qws[0], d)), ("hamming", ib.PackedTernary(qws[1], d)), ("asymmetric_dot", qf)):
        for k in (10, 128, 300):
            gi, gs = ib.ternary_topk(op, q, derived, k)
            wi, ws = ib.ternary_topk(op, q, uploaded, k)
            assert np.array_equal(gi, wi) and np.array_equal(bits(gs), bits(ws)), (op, k)


# ------------------------------------------------------------------------------------------------ 6. binary dot / Jaccard
@pytest.fixture(scope="module")
def setops(ib, oracle):
    """8,000,200 x 1024-bit codes at index_base 0 and 2,500,037 x 200-bit codes at index_base 3,000,000,000, ghash rows
    with planted tie groups for each of two random queries: LEVELS copies of the query with m = 2, 4, .. 10 of its bits
    cleared (dot |q| - m, Jaccard (|q| - m) / |q|), LEVELS copies with m bits set outside it (dot |q|, Jaccard |q| / (|q|
    + m)); and 60 empty rows. Queries: the two, and the empty code. Reference top-300 of both ops (ref_setop_topk)."""
    from test_gpu_bin_tc import ref_setop_topk
    u = _Usage()
    out = {}
    for n, dim, base in ((8_000_200, 1024, 0), (TER_N, 200, BIG_BASE)):
        nw = (dim + 63) // 64
        codes = oracle.ghash_u64_mt(0x4A11_0110 + dim, 0, n * nw, NT).reshape(n, nw)
        if dim % 64:
            codes[:, -1] &= np.uint64((1 << (dim % 64)) - 1)
        qs = oracle.ghash_u64(0x4A11_0111 + dim, 0, 3 * nw).reshape(3, nw)
        if dim % 64:
            qs[:, -1] &= np.uint64((1 << (dim % 64)) - 1)
        qs[2] = 0
        pl = Planter(n, 256, dim)
        rng = np.random.default_rng(dim)
        for q in qs[:2]:
            qb = np.unpackbits(q.view(np.uint8), bitorder="little")
            on, off = np.flatnonzero(qb[:dim]), np.flatnonzero(qb[:dim] == 0)
            for src, sign in ((on, 0), (off, 1)):
                for m, count in zip((2, 4, 6, 8, 10), LEVELS):
                    for i in pl.group(count):
                        b = qb.copy()
                        b[rng.choice(src, size=m, replace=False)] = sign
                        codes[i] = np.packbits(b, bitorder="little").view(np.uint64)
        codes[pl.group(60)] = 0
        corpus = ib.BinaryCorpus.from_words(codes.reshape(-1), n, dim, index_base=base)
        want = {op: ref_setop_topk(op, qs, codes, 300) for op in ("dot", "jaccard")}
        out[dim] = {"corpus": corpus, "qs": qs, "n": n, "base": base, "want": want}
        del codes
    u.report("fixture setops")
    return out


def test_binary_setops_topk_many_tiles(ib, setops, usage):
    """binary_setops_topk_kernel<JACCARD, R> (one query): 31,251 tiles of 256 codes (1024 bits) and 9,766 (200 bits),
    <= 1184 CTAs (256 threads, 32-40 registers: thread limit) -> >= 26 / >= 8.2 tiles per CTA. k = 129 and 300: the
    scores kernels, then selection rounds of kind 4 (dot, u32 descending) and kind 1 (Jaccard) over >= 16 grid-stride
    steps per thread of 592 CTAs. Indices and score bits against ref_setop_topk."""
    usage.note()
    for dim, s in setops.items():
        _n_tiles(s["n"], 256, 8 * SMS)
        for op in ("dot", "jaccard"):
            widx, wsc = s["want"][op]
            for j, q in enumerate(s["qs"]):
                pq = ib.PackedBinary(q, dim)
                for k in KS_ROUNDS:
                    gi, gs = ib.binary_topk(op, pq, s["corpus"], k)
                    assert gi.tolist() == (widx[j, :k] + np.uint64(s["base"])).tolist(), (dim, op, j, k, gi[:6], widx[j, :6])
                    assert np.array_equal(bits(gs), bits(wsc[j, :k])), (dim, op, j, k)

    import torch
    from innr_b200 import _lib as L
    s = setops[1024]
    dq = torch.from_numpy(s["qs"].view(np.int64)).cuda()
    for opi, op in enumerate(("dot", "jaccard")):
        def run(j, k, st):
            out = torch.empty(k, dtype=torch.int64, device="cuda")
            L.call("innr_cuda_binary_topk_keys_dev", s["corpus"].h, opi, C.c_void_p(dq[j].data_ptr()), 1, k,
                   C.c_void_p(out.data_ptr()), _stream_ptr(st))
            return out

        for k in (10, 100):
            _check_abab(run, k, lambda o, j: (o.view(np.uint64) & np.uint64(0xFFFFFFFF)).tolist()
                        == s["want"][op][0][j, :k].tolist())


# ------------------------------------------------------------------------------------------------ 7. selection rounds
def _planted_distances(oracle, n, seed):
    """Integer distances in [0, 2000) (about n / 2000 copies of each), with 100 copies of -3, 60 of -2 and 130 of -1
    planted over the Planter regions: sorted positions 100-159 (127 / 128 inside) and 160-289 (255 / 256 inside) are
    tie groups whose members sit in different regions."""
    d = np.floor(oracle.ghash_f32_mt(seed, 0, n, NT).astype(np.float64) * 1000.0 + 1000.0).astype(np.float32)
    d = np.clip(d, 0, 1999)
    pl = Planter(n, 256, seed)
    for v, count in ((-3.0, 100), (-2.0, 60), (-1.0, 130)):
        d[pl.group(count)] = v
    return d


def test_topk_from_distances_rounds(ib, oracle, usage):
    """topk_scores_kernel<R, 0> in rounds of <= 128, each bounded by the last key of the round before: 5,000,011
    distances, <= 592 CTAs x 256 threads -> >= 33 grid-stride steps per thread; k = 1 .. 5000."""
    n = 5_000_011
    _n_tiles(n, 256, 4 * SMS)
    d = _planted_distances(oracle, n, 0x4A11_0120)
    assert len(np.unique(d)) == 2003
    want = np.lexsort((np.arange(n), d))[:5000]
    ws = d[want]
    assert ws[127] == ws[128] == -2 and ws[255] == ws[256] == -1
    usage.note()
    for k in (1, 127, 128, 129, 255, 256, 257, 1000, 5000):
        got = ib.topk_from_distances(d, k)
        assert [i for i, _ in got] == want[:k].tolist(), k
        assert np.array_equal(bits([v for _, v in got]), bits(ws[:k])), k


# ------------------------------------------------------------------------------------------------ 8. filtered / reordered
FLT_N = 9_700_037   # 9,473 tiles of 1024 rows


@pytest.fixture(scope="module")
def filtered(ib, oracle):
    """9,700,037 x 16 ghash rows with _plant_f32's tie groups for two queries, stored split (default options) and plain;
    every row's squared L2 distance to each query (oracle) and its stable ascending order; four masks."""
    u = _Usage()
    n, d = FLT_N, 16
    rows = oracle.ghash_f32_mt(0x4A11_0130, 0, n * d, NT).reshape(n, d)
    ob = oracle.ghash_vertical_batch(0x4A11_0130, 0, n, d, NT)
    qs = oracle.ghash_f32(0x4A11_0131, 0, 2 * d).reshape(2, d)
    pl = Planter(n, 1024, 5)
    _plant_f32(rows, ob.data.reshape(d, n), qs, pl)
    split = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    ib.set_option("f32_split_min_rows", 2**62)
    try:
        plain = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    finally:
        ib.set_option("f32_split_min_rows", SPLIT_DEFAULT)
    del rows
    dist = [oracle.batch_l2_squared(q, ob) for q in qs]
    order = [np.argsort(x, kind="stable") for x in dist]
    rng = np.random.default_rng(6)
    nt = -(-n // 1024)
    local = np.zeros(n, bool)
    for t in (0, 32, nt - 1):   # tile 0, the first tile of finish group 1, the last partial tile
        local[t * 1024:(t + 1) * 1024] = True
    masks = {"half": rng.random(n) < 0.5, "sparse": rng.random(n) < 0.01, "all": np.ones(n, bool), "tiles": local}
    planted = np.array(sorted(pl.taken))
    assert 0 < np.count_nonzero(masks["half"][planted]) < len(planted)
    u.report("fixture filtered")
    return {"split": split, "plain": plain, "qs": qs, "ob": ob, "dist": dist, "order": order, "masks": masks, "n": n}


def test_filtered_knn_many_tiles(ib, oracle, filtered, usage):
    """pdx_scan_kernel<L2, 1, R, true, MASKED> (k <= 128): 9,473 tiles of 1024 rows, <= 1184 CTAs (256 threads, 38 / 64
    registers for R = 1 / 4) -> >= 8.0 tiles per CTA; k = 129 and 700 take the distance pass and the masked selection
    rounds (>= 64 grid-stride steps per thread of 592 CTAs). Reference: the oracle's distance of every row, the passing
    rows in stable ascending order (ties -> lower index, DESIGN section 4)."""
    f = filtered
    _n_tiles(f["n"], 1024, 8 * SMS)
    _n_tiles(f["n"], 256, 4 * SMS)
    usage.note()
    for mname, mask in f["masks"].items():
        for j, q in enumerate(f["qs"]):
            want = f["order"][j][mask[f["order"][j]]][:700]
            wsc = f["dist"][j][want]
            for store in ("split", "plain"):
                for k in (1, 10, 32, 33, 128, 129, 700):
                    g = ib.batch_knn_filtered(q, f[store], k, mask)
                    assert g.indices == want[:k].tolist(), (mname, j, store, k, g.indices[:6], want[:6])
                    assert np.array_equal(bits(g.scores), bits(wsc[:k])), (mname, j, store, k)
    mask = f["masks"]["sparse"]
    w = oracle.batch_knn_filtered(f["qs"][0], f["ob"], 33, mask.item)
    g = ib.batch_knn_filtered(f["qs"][0], f["split"], 33, mask)
    assert g.indices == w.indices and np.array_equal(bits(g.scores), bits(w.scores))


def test_reordered_knn_many_tiles(ib, oracle, filtered, usage):
    """pdx_scan_kernel<PDX_L2_PERM, ...> (batch_knn_reordered): the corpus of the filtered case, split and plain, 9,473
    tiles of 1024 rows -> >= 8.0 tiles per CTA of <= 1184; against the oracle, indices and score bits."""
    f = filtered
    _n_tiles(f["n"], 1024, 8 * SMS)
    usage.note()
    for q in f["qs"]:
        w = oracle.batch_knn_reordered(q, f["ob"], 128)
        for store in ("split", "plain"):
            for k in (1, 10, 128):
                g = ib.batch_knn_reordered(q, f[store], k)
                assert g.indices == w.indices[:k], (store, k, g.indices[:6], w.indices[:6])
                assert np.array_equal(bits(g.scores), bits(w.scores[:k])), (store, k)


def test_adaptive_knn_many_steps(ib, oracle, usage):
    """batch_knn_adaptive on 1,300,007 x 96 rows (split under default options): its warm-up, masked and kind-3 selection
    rounds stride >= 8 times over 592 CTAs x 256 threads (8 x 592 x 256 = 1,212,416 elements). The "planted" and "ties"
    inputs of test_knn_adaptive_bit_exact, against the oracle."""
    from test_gpu_parity import _adaptive_case
    n, d = 1_300_007, 96
    _n_tiles(n, 256, 4 * SMS)
    for kind in ("planted", "ties"):
        rng = np.random.default_rng(n * 17 + d)
        rows = _adaptive_case(rng, kind, n, d)
        q = _adaptive_case(rng, kind, 1, d)[0] if kind != "planted" else np.zeros(d, np.float32)
        gb = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
        ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
        del rows
        usage.note()
        for k in (10, 150, 1000):
            for w in (8, 33):
                g, want = ib.batch_knn_adaptive(q, gb, k, w), oracle.batch_knn_adaptive(q, ob, k, w)
                assert g.indices == want.indices, (kind, k, w, g.indices[:6], want.indices[:6])
                assert np.array_equal(bits(g.scores), bits(want.scores)), (kind, k, w)
        del gb, ob


# ------------------------------------------------------------------------------------------------ 9. grids in sequence
def test_grids_in_sequence(ib, oracle, ternary, setops, filtered, usage):
    """Launches of different grids back to back on the device's own stream, sharing one workspace: ternary top-k (up to
    1184 CTAs, R = 1 then 4), two topk_from_distances rounds (592), set-operation top-k, filtered kNN, ternary again.
    Each entry returns its own result, so each must equal the same call made alone (here: the reference); a ticket of
    block_finish left set by one grid would corrupt the next launch's merge."""
    t, s, f = ternary[200], setops[1024], filtered
    dist = _planted_distances(oracle, 1_000_003, 0x4A11_0140)
    want_d = np.lexsort((np.arange(len(dist)), dist))[:129]
    mask = f["masks"]["half"]
    want_f = f["order"][0][mask[f["order"][0]]][:10]
    usage.note()
    for _ in range(3):
        for k in (10, 100):
            gi, _s = ib.ternary_topk("dot", t["queries"]["dot"][0], t["corpus"], k)
            assert gi.tolist() == (t["want"]["dot", 0][0][:k] + BIG_BASE).tolist(), k
        assert [i for i, _ in ib.topk_from_distances(dist, 129)] == want_d.tolist()
        gi, _s = ib.binary_topk("jaccard", ib.PackedBinary(s["qs"][0], 1024), s["corpus"], 33)
        assert gi.tolist() == s["want"]["jaccard"][0][0, :33].tolist()
        assert ib.batch_knn_filtered(f["qs"][0], f["split"], 10, mask).indices == want_f.tolist()
        gi, _s = ib.ternary_topk("asymmetric_dot", t["queries"]["asymmetric_dot"][0], t["corpus"], 128)
        assert gi.tolist() == (t["want"]["asymmetric_dot", 0][0][:128] + BIG_BASE).tolist()
