"""The tensor-core batch kNN filter (csrc/knn_tc.cu) against exact references at the shapes where its whole schedule runs.

Query batches of 2 or more f32 queries on a corpus of at least `knn_tc_min_n` rows are answered by `knn_tc_filter_kernel`:
a dense first pass keeps every pair of its rows, every later pass over a longer row prefix keeps the pairs whose upper
bound reaches the k-th largest lower bound the previous pass appended (`knn_tc_select_kernel`), and the final candidates
are rescored exactly (`knn_tc_rescore_kernel`); a query whose list overflows goes to the exact scan, or to the screened
kNN on a split corpus. The result is bit-identical to the reference only if every link of that chain holds, and a link
that is slightly wrong loses a true neighbour only where the later passes run and only on inputs built for it. Here
whole result lists are compared with the multi-query exact scan (`knn_tc = 0`, itself pinned to the oracle elsewhere)
and with the CPU oracle: on a C2b 4-GPU shard, on a corpus with rows planted against the carried thresholds, at the
edges of the prefix schedule, on a split corpus whose lists overflow, and across calls and caller streams.

Every test asserts that `knn_tc_last_stats()["passes"]` equals `len(levels(n, k))`, the schedule restated below, so
each one proves it ran the passes it claims. Each test prints its wall time and the device memory in use at its peak
(run with -rP to see it)."""
import ctypes as C
import os
import time

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

NT = max(1, min(os.cpu_count() or 1, 16))   # oracle threads
METRICS = ("dot", "cosine", "l2")
DEFAULTS = {"knn_tc": 1, "knn_tc_min_n": 100_000, "knn_tc_min_queries": 2, "f32_split_min_rows": 1_000_000}
VT, CAND_CAP = 128, 4096    # rows per filter work unit, slots of a query's candidate list (knn_tc.cu)


def levels(n, k):
    """Row prefixes the filter passes over for an n-row corpus and k results (launch_pdx_knn_tc, default schedule).
    The first is the dense pass (every pair kept), the last is the whole corpus.

    | n                           | k <= 32                      | k in 33..128                            |
    |-----------------------------|------------------------------|-----------------------------------------|
    | 4,096                       | 1024, 4096                   | 4096 (the dense pass is also the last)  |
    | 70,922                      | -                            | k = 128: 4096, 4480 (extra prefix), n   |
    | 133,656                     | 1024, 4224 (n/256), n        | -                                       |
    | 1,250,000 (C2b 8-GPU shard) | 1024, 4992, 39168, n         | 4096, 78208, n                          |
    | 2,500,000 (C2b 4-GPU shard) | 1024, 9856, 78208, n         | 4096, 19584, 156288, n                  |

    k > 32 gets its n/128 pass only from n = 2,097,152 rows on (n/128 >= 4 x 4096)."""
    cur = min(n, 1024 if k <= 32 else CAND_CAP)
    lv = [cur]
    for nx in ((n // 256, n // 32) if k <= 32 else (n // 128, n // 16)):
        if nx >= 4 * cur:                     # a prefix is skipped unless it is 4 x the previous one
            cur = (nx + VT - 1) // VT * VT
            lv.append(cur)
    g = max(4, (CAND_CAP // 2) // k)          # up to 3 extra prefixes, top down, where a step exceeds g
    extra, top = [], n
    while top // cur > g and len(extra) < 3:
        top = ((top + g - 1) // g + VT - 1) // VT * VT
        if top <= cur:
            break
        extra.append(top)
    while extra and len(lv) < 5:
        cur = extra.pop()
        lv.append(cur)
    if n > cur:
        lv.append(n)
    return lv


def test_levels_mirror_matches_its_table():
    n = 2_500_000
    assert levels(4096, 10) == [1024, 4096] and levels(4096, 33) == [4096] and levels(4096, 128) == [4096]
    assert levels(4097, 33) == [4096, 4097]
    assert levels(70_922, 128) == [4096, 4480, 70_922]
    assert levels(133_656, 10) == [1024, 4224, 133_656]
    assert levels(1_250_000, 10) == [1024, 4992, 39_168, 1_250_000]
    assert levels(1_250_000, 100) == [4096, 78_208, 1_250_000]
    assert levels(n, 10) == [1024, 9856, 78_208, n] and levels(n, 128) == [4096, 19_584, 156_288, n]
    assert len(levels(2_097_152, 33)) == 4 and len(levels(2_097_151, 33)) == 3


# ------------------------------------------------------------------------------------------------ fixtures, helpers
@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    yield innr_b200
    for name, v in DEFAULTS.items():
        innr_b200.set_option(name, v)


@pytest.fixture
def opts(ib):
    """set(name=value, ...) for the duration of a test; the library defaults are restored whatever happens."""
    def set_(**kw):
        for name, v in kw.items():
            ib.set_option(name, v)
    try:
        yield set_
    finally:
        for name, v in DEFAULTS.items():
            ib.set_option(name, v)


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
    print(f"[knn-tc-passes] {request.node.name}: wall {time.time() - u.t0:.1f} s, peak device memory in use {u.peak / 1e9:.1f} GB")


def _need(hbm_gb=0.0, ram_gb=0.0):
    import torch
    free = torch.cuda.mem_get_info()[0] / 1e9
    if free < hbm_gb:
        pytest.skip(f"needs {hbm_gb:.0f} GB of free HBM, {free:.0f} GB free")
    avail = None
    try:
        with open("/proc/meminfo") as f:
            for line in f:
                if line.startswith("MemAvailable:"):
                    avail = int(line.split()[1]) * 1024 / 1e9
    except OSError:
        pass
    if avail is not None and avail < ram_gb:
        pytest.skip(f"needs {ram_gb:.0f} GB of available host RAM, {avail:.0f} GB available")


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def same_scores(a, b):
    """Bit equality, except that any NaN matches any NaN (NaN sign and payload are not portable, DESIGN.md)."""
    a, b = np.ascontiguousarray(a, dtype=np.float32), np.ascontiguousarray(b, dtype=np.float32)
    return a.shape == b.shape and bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | (np.isnan(a) & np.isnan(b))))


def _stats(ib, n, d, nq, k, exact_scan_queries=0):
    """The last call ran the filter on this corpus and batch (filter_flops pins n, d and the padded batch), over the
    prefixes levels(n, k), and handed exactly `exact_scan_queries` queries to the exact path."""
    st = ib.knn_tc_last_stats()
    d_pad = (d + 7) // 8 * 8
    flops = 2.0 * ((n + VT - 1) // VT * VT) * ((d_pad + 63) // 64 * 64) * ((nq + 15) // 16 * 16)
    assert st["filter_flops"] == flops, (n, d, nq, k, st)
    assert st["passes"] == len(levels(n, k)), (n, k, levels(n, k), st)
    assert st["exact_scan_queries"] == exact_scan_queries, (n, k, st)
    return st


def _exact(ib, metric, qs, db, k):
    """The same call on the multi-query exact scan."""
    ib.set_option("knn_tc", 0)
    try:
        return ib.batch_knn_many(metric, qs, db, k)
    finally:
        ib.set_option("knn_tc", 1)


def _same(got, want, what):
    assert np.array_equal(got[0], want[0]), (what, np.argwhere(got[0] != want[0])[:5])
    assert np.array_equal(bits(got[1]), bits(want[1])), (what, np.argwhere(bits(got[1]) != bits(want[1]))[:5])


def _want(oracle, metric, qs, ob, k):
    """The oracle's top-k per query, in the device's order. For L2, whose tie order the reference leaves open (DESIGN
    section 4, Ties), the k smallest (distance, index) are rebuilt from the oracle's distance vector after checking
    that the oracle's own list agrees with them score for score."""
    widx, wsc = oracle.batch_knn_many(metric, qs, ob, k, n_threads=min(NT, len(qs)))
    if metric != "l2":
        return widx, wsc
    out = np.empty_like(widx)
    for j, q in enumerate(qs):
        dist = oracle.batch_l2_squared(q, ob)
        cand = np.flatnonzero(bits(dist) <= bits(wsc[j, -1]))   # non-negative floats order like their bits
        order = cand[np.lexsort((cand, dist[cand]))][:k]
        assert np.array_equal(bits(dist[order]), bits(wsc[j])) and np.array_equal(bits(dist[widx[j]]), bits(wsc[j]))
        out[j] = order
    return out, wsc


# ------------------------------------------------------------------------------------------------ 1. a C2b shard
SHARD_FIRST, SHARD_N, SHARD_D = 7_500_000, 2_500_000, 768   # the last shard of C2b on 4 GPUs
NQS = (2, 64, 65, 256, 257, 1024)
KS = (1, 10, 32, 33, 100, 128)


@pytest.fixture(scope="module")
def shard(ib):
    """Generated on the device under default options: stored split, with the screening sketch (>= 1M rows)."""
    from innr_b200 import synth
    _need(hbm_gb=24)
    db = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, SHARD_FIRST, SHARD_N, SHARD_D, index_base=SHARD_FIRST)
    yield db
    del db


@pytest.fixture(scope="module")
def c2b_queries(oracle):
    from innr_b200 import synth
    return oracle.ghash_f32(synth.SALT_QUERY, 0, 1024 * SHARD_D).reshape(1024, SHARD_D)


def test_c2b_shard_whole_results(ib, oracle, opts, usage, shard, c2b_queries):
    """2,500,000 x 768 rows, rows 7.5M-10M of C2b. Batches of 2 and 64 queries take the Q-resident filter (nq_pad <= 64,
    12 K blocks), 65 and 256 the streaming one with one query group (65: a partial 32-column epilogue chunk), 257 a
    second group of 16 columns (one query, 15 padding), 1024 four groups. For every metric, batch and k, the whole (nq, k) index and
    score arrays equal the exact scan's; the first 64 queries' lists also equal the oracle's."""
    from innr_b200 import synth
    _need(ram_gb=12)
    qs = c2b_queries
    n, d = SHARD_N, SHARD_D
    kept = {}
    for metric in METRICS:
        exact = _exact(ib, metric, qs, shard, 128)
        assert exact[0].min() >= SHARD_FIRST and exact[0].max() < SHARD_FIRST + n
        for nq in NQS:
            for k in KS:
                got = ib.batch_knn_many(metric, qs[:nq], shard, k)
                _stats(ib, n, d, nq, k)
                _same(got, (exact[0][:nq, :k], exact[1][:nq, :k]), (metric, nq, k))
        kept[metric] = (exact[0][:64].copy(), exact[1][:64].copy())
        del exact
    usage.note()
    ob = oracle.ghash_vertical_batch(synth.SALT_CORPUS, SHARD_FIRST, n, d, NT)
    for metric in METRICS:
        t0 = time.time()
        widx, wsc = _want(oracle, metric, qs[:64], ob, 128)
        print(f"[knn-tc-passes] oracle {metric}, 64 queries at {n} x {d}: {time.time() - t0:.1f} s")
        _same(kept[metric], (widx + SHARD_FIRST, wsc), (metric, "oracle"))


def test_streaming_variant_with_few_queries(ib, oracle, opts, usage):
    """600,000 x 769: d_pad = 776 is 13 K blocks, one more than the Q-resident variant holds, so 64 queries take the
    streaming filter. Whole lists against the exact scan for every metric and k, 16 queries against the oracle."""
    from innr_b200 import synth
    _need(hbm_gb=8, ram_gb=6)
    n, d, nq = 600_000, 769, 64
    db = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d)
    qs = oracle.ghash_f32(0x4A11_0101, 0, nq * d).reshape(nq, d)
    ob = oracle.ghash_vertical_batch(synth.SALT_CORPUS, 0, n, d, NT)
    usage.note()
    for metric in METRICS:
        exact = _exact(ib, metric, qs, db, 128)
        for k in KS:
            got = ib.batch_knn_many(metric, qs, db, k)
            _stats(ib, n, d, nq, k)
            _same(got, (exact[0][:, :k], exact[1][:, :k]), (metric, k))
        widx, wsc = _want(oracle, metric, qs[:16], ob, 128)
        _same((exact[0][:16], exact[1][:16]), (widx, wsc), (metric, "oracle"))


# ------------------------------------------------------------------------------------------------ 2. carried thresholds
ETA = 2.0 ** -11 - 2.0 ** -16    # a hair inside half an f16 ulp, in units of the component's binade


def _layout(d):
    """The binade levels of test_gpu_parity._half_ulp_unit_vector, largest first: a few components two or three binades
    up, the rest at level J (>= 200 of them, they absorb the remainder with mantissa steps)."""
    J = int(np.ceil(np.log(d) / np.log(4.0))) + 1
    extra = 4.0 ** J / (1.0 + 2.0 ** -11) ** 2 - d
    lev = np.full(d, J)
    k = 0
    for up, gain in ((3, 63), (2, 15), (1, 3)):
        cnt = int(min(d - 200 - k, extra // gain))
        lev[k:k + cnt] = J - up
        k += cnt
        extra -= cnt * gain
    return lev


def _half_ulp_vector(lev, up, lift=None):
    """_half_ulp_unit_vector's construction with the rounding side chosen per component: component k is
    2^-lev_k (m_k + eta_k), m_k = 1 + i_k 2^-10, and f16 rounding of the normalised vector moves it by almost half an
    ulp DOWN in magnitude (eta_k = ETA) or UP (eta_k = -ETA, m_k >= 1 + 2^-10). The mantissa steps i_k of the level-J
    components bring the squared norm to 1 within 2e-6, which keeps x / ||x|| on the intended side of every boundary.
    `lift`: a component that starts one mantissa step higher (the level-J components then take fewer)."""
    eta = np.where(up, -ETA, ETA)
    steps = up.astype(np.int64)
    if lift is not None:
        steps[lift] += 1
    w = 4.0 ** -lev.astype(np.float64)
    free = np.flatnonzero(lev == lev.max())
    tot = float(np.sum(w * (1.0 + steps * 2.0 ** -10 + eta) ** 2))
    i = 0
    while tot < 1.0:
        c = free[i % len(free)]
        old = (1.0 + steps[c] * 2.0 ** -10 + eta[c]) ** 2
        steps[c] += 1
        tot += w[c] * ((1.0 + steps[c] * 2.0 ** -10 + eta[c]) ** 2 - old)
        i += 1
    assert steps.max() <= 12 and tot - 1.0 < 2e-6, (steps.max(), tot)
    return 2.0 ** -lev.astype(np.float64) * (1.0 + steps * 2.0 ** -10 + eta)


def _f16_unit(x):
    """The filter's operand: f16(x / ||x||), normalised in f32 as knn_tc_prep_queries / knn_tc_build_xh do."""
    x = np.asarray(x, np.float32)
    return (x * np.float32(1.0 / np.sqrt(np.sum(x.astype(np.float64) ** 2)))).astype(np.float16).astype(np.float64)


def _cos(q, x):
    q, x = np.asarray(q, np.float32).astype(np.float64), np.asarray(x, np.float32).astype(np.float64)
    return float(q @ x / np.sqrt((q @ q) * (x @ x)))


def _eps_family(d, rng, block):
    """A query q and two rows, target T and decoy D, with cos(q, T) a hair above cos(q, D) (about 0.25) while the f16
    product S = f16(q')·f16(x') UNDER-estimates the cosine for T and OVER-estimates it for D, each by about 0.85 x 2^-10.
    All three share one binade layout whose 12 largest components (3/4 of the squared norm) sit at the dimensions
    `block`. q rounds up on 6 of them and down on the other 6 (and on a random half of the small ones); T flips the sign
    of q's 6 round-up components and rounds up there and down elsewhere, D flips the 6 round-down ones and rounds down
    there and up elsewhere, so that every product of T errs low and every product of D high. Drawn until the
    cosines are ordered and S_D - S_T exceeds 1.3 eps by a margin."""
    lev_sorted = _layout(d)
    nbig = int(np.sum(lev_sorted == lev_sorted.min()))
    assert nbig == len(block) == 12
    eps = 1.05e-3 + 3.5e-7 * d
    for _ in range(200):
        rest = rng.permutation(np.setdiff1d(np.arange(d), block))
        perm = np.concatenate([rng.permutation(block), rest])
        lev = np.empty(d, np.int64)
        lev[perm] = lev_sorted
        big = perm[:nbig]
        up_q = rng.random(d) < 0.5
        up_q[big] = False
        up_q[big[:6]] = True
        sign = rng.choice([-1.0, 1.0], size=d)
        flip_t = np.zeros(d, bool)
        flip_t[big[:6]] = True
        flip_d = np.zeros(d, bool)
        flip_d[big[6:]] = True
        q = (sign * _half_ulp_vector(lev, up_q)).astype(np.float32)
        t = (sign * np.where(flip_t, -1.0, 1.0) * _half_ulp_vector(lev, flip_t)).astype(np.float32)
        dc = (sign * np.where(flip_d, -1.0, 1.0) * _half_ulp_vector(lev, ~flip_d, lift=big[6])).astype(np.float32)
        ct, cd = _cos(q, t), _cos(q, dc)
        st, sd = float(_f16_unit(q) @ _f16_unit(t)), float(_f16_unit(q) @ _f16_unit(dc))
        if 3e-5 < ct - cd and sd - st > 1.36 * eps:
            return q, t, dc
    raise AssertionError("no adversarial triple found")


ADV_N, ADV_D = 2_200_011, 256     # k > 32 gets 4 passes from 2,097,152 rows on; the last unit holds 75 rows
N_EPS = 8                         # queries with decoys and targets
GAP_KS = (10, 33, 128)            # one query each with k - 1 strong rows in the dense pass and the rest late


def _adversarial_corpus(oracle, seed=11):
    """ADV_N x ADV_D rows: background G-hash rows with every planted query direction projected out (cosine ~ 0, norms
    ~ 9, far from every planted list in all three metrics), and planted rows of unit norm:
      * N_EPS threshold queries (_eps_family): 128 copies of the decoy D in the dense passes (10 in rows < 1024, the
        first pass for k <= 32, the rest in rows < 4096), 128 copies of the target T past the dense passes -- two right
        after each later level boundary of k <= 32 and k > 32, four in the last, partial 128-row unit (query 0 also in
        the last row), the rest anywhere after row 4096. The true top-k is T for every k <= 128; the decoys set the
        carried threshold to S_D - eps, which T's upper bound S_T + eps only just reaches.
      * one gap query per k in GAP_KS: k - 1 strong rows (cosine 0.9) inside the dense pass of that k and k + 8 rows of
        cosine 0.5 after it, at the level boundaries and in the last unit. The k-th largest lower bound of the dense pass
        belongs to a background row, the (k - 1)-th to a strong row: a threshold one rank too high prunes the rest of
        the true top-k.
    Returns rows (n, d) f32, queries (N_EPS + 3, d), per threshold query (decoy rows, target rows) and the triples."""
    n, d = ADV_N, ADV_D
    rng = np.random.default_rng(seed)
    triples = [_eps_family(d, rng, np.arange(12 * j, 12 * j + 12)) for j in range(N_EPS)]
    eq = np.stack([q for q, _, _ in triples]).astype(np.float64)
    basis = np.linalg.qr(eq.T)[0]                                   # d x N_EPS, orthonormal
    gq = []
    for _ in GAP_KS:
        g = rng.standard_normal(d)
        g -= basis @ (basis.T @ g)
        g /= np.linalg.norm(g)
        gq.append(g)
    full = np.linalg.qr(np.concatenate([eq, np.stack(gq)]).T)[0]    # every planted query direction
    qs = np.concatenate([eq, np.stack(gq)]).astype(np.float32)

    rows = oracle.ghash_f32_mt(0x4A11_0102, 0, n * d, NT).reshape(n, d)
    fb = full.astype(np.float32)
    for lo in range(0, n, 1 << 18):
        blk = rows[lo:lo + (1 << 18)]
        blk -= (blk @ fb) @ fb.T

    taken = set()

    def take(i):
        assert i not in taken and 0 <= i < n, i
        taken.add(i)
        return i

    def anywhere(lo, hi, count):
        out = []
        while len(out) < count:
            i = int(rng.integers(lo, hi))
            if i not in taken:
                out.append(take(i))
        return out

    bounds = sorted(set(levels(n, 10)[1:-1] + levels(n, 128)[1:-1]))
    last_unit = n - n % VT
    assert n % VT and len(bounds) == 4
    planted = []
    for j, (q, t, dc) in enumerate(triples):
        dec = anywhere(0, 1024, 10) + anywhere(1024, CAND_CAP, 118)
        tgt = [take(b + 2 * j + o) for b in bounds for o in (0, 1)] + [take(last_unit + 4 * j + o) for o in range(4)]
        if j == 0:
            tgt.append(take(n - 1))
        tgt += anywhere(CAND_CAP, n, 128 - len(tgt))
        rows[dec] = dc
        rows[tgt] = t
        planted.append((dec, tgt))

    def near(g, c):   # a unit row at cosine c to g, orthogonal to every other planted query direction
        u = rng.standard_normal(d)
        u -= full @ (full.T @ u)
        u /= np.linalg.norm(u)
        return (c * g + np.sqrt(1.0 - c * c) * u).astype(np.float32)

    for i, (k, g) in enumerate(zip(GAP_KS, gq)):
        for r in anywhere(0, 1024 if k <= 32 else CAND_CAP, k - 1):
            rows[r] = near(g, 0.9)
        late = [take(b + 16 + 2 * i + o) for b in bounds for o in (0, 1)]
        late += [take(last_unit + 32 + 4 * i + o) for o in range(4)]
        late += anywhere(CAND_CAP, n, k + 8 - len(late))
        for r in late:
            rows[r] = near(g, 0.5)
    return rows, qs, planted, triples


def test_thresholds_carried_across_passes_adversarial(ib, oracle, opts, usage):
    """2,200,011 x 256 rows (_adversarial_corpus), where both k <= 32 and k > 32 run 4 passes. With the filter's eps
    every target survives the threshold its decoys carry into each later pass; a bound about 40 % too narrow, a
    rescoring bound of lb + eps, or a threshold taken one rank too high would prune part of the true top-k. Whole lists
    must equal the oracle's for all three metrics and k in {10, 33, 128}, with no query handed to the exact scan."""
    _need(hbm_gb=6, ram_gb=12)
    n, d = ADV_N, ADV_D
    rows, qs, planted, triples = _adversarial_corpus(oracle)
    nq = qs.shape[0]
    eps = 1.05e-3 + 3.5e-7 * d

    db = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    small = rows[:CAND_CAP].copy()
    del rows
    usage.note()
    for metric in METRICS:
        widx, wsc = _want(oracle, metric, qs, ob, 128)
        for j, (dec, tgt) in enumerate(planted):   # the planted targets are the true top-128 of their query
            assert sorted(widx[j].tolist()) == sorted(tgt), (metric, j)
        for k in GAP_KS:
            got = ib.batch_knn_many(metric, qs, db, k)
            _stats(ib, n, d, nq, k)
            _same(got, (widx[:, :k], wsc[:, :k]), (metric, k))

    # the construction really is adversarial, as the device computes the bounds: decoys and targets copied into the
    # rows < 4096 that the debug hook reports
    slots = []
    for j, (q, t, dc) in enumerate(triples):
        dpos = planted[j][0][0]
        tpos = CAND_CAP - 1 - j
        small[tpos] = t
        slots.append((dpos, tpos))
    gb_small = ib.VerticalBatch.from_flat(small.reshape(-1), CAND_CAP, d)
    lower, got_eps, flags = ib.knn_tc_debug_bounds("cosine", qs[:N_EPS], gb_small)
    assert abs(got_eps - eps) < 1e-9 and not flags.any()
    for j, ((q, t, dc), (dpos, tpos)) in enumerate(zip(triples, slots)):
        ref = oracle.batch_cosine(q, oracle.VerticalBatch.from_flat(np.stack([dc, t]).reshape(-1), 2, d),
                                  oracle.batch_norms(oracle.VerticalBatch.from_flat(np.stack([dc, t]).reshape(-1), 2, d)))
        over = float(lower[j, dpos]) + eps - float(ref[0])     # S_D - cos(q, D)
        under = float(ref[1]) - (float(lower[j, tpos]) + eps)  # cos(q, T) - S_T
        assert ref[1] > ref[0] and over + under > 1.3 * eps, (j, over / eps, under / eps)
        # a filter with 0.6 eps would prune T: its upper bound S_T + 0.6 eps stays below S_D - 0.6 eps
        assert float(lower[j, dpos]) - float(lower[j, tpos]) > 1.2 * eps, (j, float(lower[j, dpos] - lower[j, tpos]) / eps)


# ------------------------------------------------------------------------------------------------ 3. schedule edges
@pytest.mark.parametrize("n,ks", [(4096, (10, 33, 128)), (4097, (10, 33, 128)), (70_922, (128,)), (133_656, (10,))])
def test_schedule_edges(ib, oracle, opts, usage, n, ks):
    """With knn_tc_min_n = 4096: n = 4096 at k >= 33 runs the dense pass alone (no threshold is ever selected, the
    rescoring reads the dense list), n = 4097 leaves one row in the last unit, 70,922 at k = 128 runs an extra prefix
    (4480), 133,656 at k = 10 the first n/256 pass (4224). The best row of query 0 is the last row, the best rows of
    query 1 sit at every level boundary. Whole lists against the oracle."""
    opts(knn_tc_min_n=4096)
    d, nq = 96, 40
    rows = oracle.ghash_f32(0x4A11_0103, 0, n * d).reshape(n, d)
    qs = oracle.ghash_f32(0x4A11_0104, 0, nq * d).reshape(nq, d)
    for k in ks:
        for b in levels(n, k)[:-1]:
            if b < n:
                rows[b - 1] = rows[b] = qs[1] * np.float32(0.5)   # the last row of one prefix and the first of the next
    rows[n - 1] = qs[0] * np.float32(4.0)
    db = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    usage.note()
    for metric in METRICS:
        widx, wsc = _want(oracle, metric, qs, ob, max(ks))
        assert widx[0, 0] == n - 1 or metric == "l2"
        for k in ks:
            got = ib.batch_knn_many(metric, qs, db, k)
            _stats(ib, n, d, nq, k)
            _same(got, (widx[:, :k], wsc[:, :k]), (metric, n, k))


def test_c2b_8gpu_shard_schedule(ib, oracle, opts, usage):
    """1,250,000 x 128 G-hash rows (the row count of a C2b shard on 8 GPUs): k = 10 runs 1024, 4992, 39168, n and
    k = 100 runs 4096, 78208, n. 256 queries (a full query group) against the exact scan, 16 against the oracle."""
    from innr_b200 import synth
    _need(hbm_gb=4, ram_gb=3)
    n, d, nq = 1_250_000, 128, 256
    db = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d)
    ob = oracle.ghash_vertical_batch(synth.SALT_CORPUS, 0, n, d, NT)
    qs = oracle.ghash_f32(0x4A11_0105, 0, nq * d).reshape(nq, d)
    usage.note()
    for metric in METRICS:
        widx, wsc = _want(oracle, metric, qs[:16], ob, 100)
        for k in (10, 100):
            got = ib.batch_knn_many(metric, qs, db, k)
            _stats(ib, n, d, nq, k)
            _same(got, _exact(ib, metric, qs, db, k), (metric, k))
            _same((got[0][:16], got[1][:16]), (widx[:, :k], wsc[:, :k]), (metric, k, "oracle"))


# ------------------------------------------------------------------------------------------------ 4. overflow, split corpus
def test_overflow_on_a_split_corpus_goes_to_the_screened_knn(ib, oracle, opts, usage):
    """300,000 x 64 stored split (f32_split_min_rows lowered), 64 queries at k = 128. Queries 5, 20 and 40 each sit in a
    cloud of 6,000 near-duplicates of norm 8 (ahead of every G-hash row in all three metrics), all inside the filter's error band: their final lists overflow the 4096 slots.
    The other queries are orthogonal to the three cloud directions. Query 7 is zero and query 9 holds an inf: the filter does not answer them. These 5 go one by one to the screened
    kNN on lane 0; every list, theirs included, must equal the oracle's."""
    opts(f32_split_min_rows=0)
    n, d, nq, k = 300_000, 64, 64, 128
    rng = np.random.default_rng(78)
    rows = oracle.ghash_f32(0x4A11_0106, 0, n * d).reshape(n, d)
    qs = oracle.ghash_f32(0x4A11_0107, 0, nq * d).reshape(nq, d)
    cloud = rng.permutation(n)[:18_000].reshape(3, -1)
    basis = np.linalg.qr(qs[[5, 20, 40]].T.astype(np.float64))[0]
    others = np.setdiff1d(np.arange(nq), [5, 20, 40])
    qs[others] -= ((qs[others] @ basis) @ basis.T).astype(np.float32)   # the clouds are nobody else's neighbours
    for j, sel in zip((5, 20, 40), cloud):
        u = qs[j] / np.linalg.norm(qs[j])
        rows[sel] = (8.0 * (u[None, :] + 2e-4 * rng.standard_normal((len(sel), d)))).astype(np.float32)
    qs[7] = 0.0
    qs[9, 3] = np.inf
    db = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    usage.note()
    fin = np.ones(nq, bool)
    fin[9] = False
    for metric in METRICS:
        got = ib.batch_knn_many(metric, qs, db, k)
        _stats(ib, n, d, nq, k, exact_scan_queries=5)
        widx, wsc = _want(oracle, metric, qs[fin], ob, k)
        _same((got[0][fin], got[1][fin]), (widx, wsc), metric)
        w9 = oracle.batch_knn_many(metric, qs[9:10], ob, k)
        assert same_scores(got[1][9:10], w9[1]), metric
        if np.isfinite(w9[1]).all():
            assert np.array_equal(got[0][9], w9[0][0]), metric


# ------------------------------------------------------------------------------------------------ 5. state, ordering
def test_same_corpus_varied_calls(ib, opts, usage, shard, c2b_queries):
    """On one corpus, calls that change the query padding, the size of the filter's workspace and the k schedule
    between them: 1024 queries at k = 10, 64 at k = 128 (L2), 1024 at k = 10 (cosine), one screened query, then the
    first call again, which must give the same bits."""
    qs = c2b_queries
    n, d = SHARD_N, SHARD_D
    first = ib.batch_knn_many("dot", qs, shard, 10)
    _stats(ib, n, d, 1024, 10)
    ib.batch_knn_many("l2", qs[:64], shard, 128)
    _stats(ib, n, d, 64, 128)
    ib.batch_knn_many("cosine", qs, shard, 10)
    _stats(ib, n, d, 1024, 10)
    one = ib.batch_knn_many("dot", qs[3], shard, 10)
    _same(one, (first[0][3:4], first[1][3:4]), "screened")
    again = ib.batch_knn_many("dot", qs, shard, 10)
    _stats(ib, n, d, 1024, 10)
    _same(again, first, "repeat")


def test_filter_on_caller_streams(ib, opts, usage, shard, c2b_queries):
    """innr_cuda_batch_knn_keys_dev with 64 queries (the filter: lane 0's Workspace, d_tcws and h_counts) on two caller
    streams, interleaved with single-query screened scans on a third stream and a k = 200 call: every output, as whole
    64-bit keys, equals the call alone."""
    import torch
    from innr_b200 import _lib as L
    dq = torch.from_numpy(c2b_queries[:256]).cuda()
    metrics = {"dot": L.METRIC_DOT, "cosine": L.METRIC_COSINE, "l2": L.METRIC_L2}

    def run(kind, j, st):
        metric, nq, k = kind
        out = torch.empty((nq, k), dtype=torch.int64, device="cuda")
        L.call("innr_cuda_batch_knn_keys_dev", shard.h, metrics[metric], C.c_void_p(dq[j].data_ptr()), nq, k,
               C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))
        return out

    A, B, S, BIG = ("cosine", 64, 10), ("l2", 64, 100), ("dot", 1, 10), ("cosine", 1, 200)
    plan = [(A, 0, 0), (S, 200, 2), (B, 64, 1), (S, 201, 2), (BIG, 202, 1), (A, 128, 0), (S, 203, 2), (B, 0, 1),
            (S, 204, 2), (A, 64, 1), (B, 128, 0), (S, 205, 2)]
    main = torch.cuda.current_stream()
    alone = {}
    for kind, j, _ in plan:
        if (kind, j) not in alone:
            alone[(kind, j)] = run(kind, j, main)
            main.synchronize()
            if kind[1] == 64:
                _stats(ib, SHARD_N, SHARD_D, 64, kind[2])
    streams = [torch.cuda.Stream() for _ in range(3)]
    for s in streams:
        s.wait_stream(main)
    for rep in range(2):
        outs = [(kind, j, run(kind, j, streams[si])) for kind, j, si in plan]
        torch.cuda.synchronize()
        for kind, j, out in outs:
            assert torch.equal(out, alone[(kind, j)]), (rep, kind, j)
