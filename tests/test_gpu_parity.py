"""GPU parity tests proper: the CUDA path (through the C-ABI) against the CPU oracle on the same seeded inputs.

Bar (north_star): integer / byte / index work bit-exact; f32 scan scores bit-exact (sequential unfused sums are
reproduced on the device); MaxSim within 1e-5 relative, condition-aware (|got - ref| <= 1e-5 * sum_i max_j sum_k
|q_ik d_jk| -- the bound the reference's own property tests use, tests/property_tests.rs:56-64).
"""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def ib():
    import innr_b200
    innr_b200.init(0)
    return innr_b200


def bits(a):
    return np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)


def sharded_order_bits(scores):
    """f32::total_cmp order as unsigned integers (the key codec of innr_b200/sharded.py, csrc/common.cuh)."""
    from innr_b200 import sharded
    return sharded.order_bits(np.asarray(scores, dtype=np.float32)).astype(np.int64)


def same_scores(a, b):
    """Bit equality, except that any NaN matches any NaN: NaN sign/payload is not portable across the reference's
    own targets (x86 propagates the operand payload and makes 0*inf a NEGATIVE NaN, aarch64 a positive default
    NaN); the device produces the canonical 0x7FFFFFFF (DESIGN.md, "NaN scores")."""
    a, b = np.ascontiguousarray(a, dtype=np.float32), np.ascontiguousarray(b, dtype=np.float32)
    if a.shape != b.shape:
        return False
    both_nan = np.isnan(a) & np.isnan(b)
    return bool(np.all((a.view(np.uint32) == b.view(np.uint32)) | both_nan))


def rand_rows(n, d, seed, scale=1.0):
    rng = np.random.default_rng(seed)
    return (rng.standard_normal((n, d)) * scale).astype(np.float32)


def assert_knn_equal(got, want, ties_as_sets=False):
    assert np.array_equal(bits(got.scores), bits(want.scores)), (got.scores, want.scores)
    if not ties_as_sets:
        assert got.indices == want.indices
        return
    # SURVEY.md 8a row T (L2/TopK path): exact-tie groups compare as sets
    s = np.asarray(want.scores)
    for v in np.unique(bits(s)):
        sel = bits(s) == v
        g = sorted(np.asarray(got.indices)[sel].tolist())
        w = sorted(np.asarray(want.indices)[sel].tolist())
        if sel.sum() == 1 or g == w:
            assert g == w
    assert len(set(got.indices)) == len(got.indices)


SHAPES = [(1, 1), (5, 3), (63, 7), (1000, 128), (4097, 100), (1024, 8), (20000, 768), (3000, 1)]


@pytest.mark.parametrize("n,d", SHAPES)
def test_scores_bit_exact(ib, oracle, n, d):
    rows = rand_rows(n, d, n * 31 + d)
    q = rand_rows(1, d, 7)[0]
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    assert np.array_equal(gb.data, ob.data)
    for fn in ("batch_dot", "batch_l2_squared"):
        assert np.array_equal(bits(getattr(ib, fn)(q, gb)), bits(getattr(oracle, fn)(q, ob))), fn
    gn, on = ib.batch_norms(gb), oracle.batch_norms(ob)
    assert np.array_equal(bits(gn), bits(on))
    assert np.array_equal(bits(ib.batch_cosine(q, gb, gn)), bits(oracle.batch_cosine(q, ob, on)))
    # caller-supplied (arbitrary) norms, incl. zero / tiny / negative entries
    weird = on.copy()
    weird[:: max(1, n // 7)] = 0.0
    weird[1:: max(2, n // 5)] = 1e-10
    assert np.array_equal(bits(ib.batch_cosine(q, gb, weird)), bits(oracle.batch_cosine(q, ob, weird)))


@pytest.mark.parametrize("n,d", SHAPES)
@pytest.mark.parametrize("k", [1, 10, 33, 128])
def test_knn_bit_exact(ib, oracle, n, d, k):
    rows = rand_rows(n, d, n * 17 + d + k)
    q = rand_rows(1, d, 11)[0]
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    assert_knn_equal(ib.batch_knn_dot(q, gb, k), oracle.batch_knn_dot(q, ob, k))
    assert_knn_equal(ib.batch_knn_cosine(q, gb, k), oracle.batch_knn_cosine(q, ob, k))
    assert_knn_equal(ib.batch_knn(q, gb, k), oracle.batch_knn(q, ob, k), ties_as_sets=True)


def test_knn_ties_lower_index_first(ib, oracle):
    # heavy exact ties: integer-valued rows, many duplicates
    rng = np.random.default_rng(5)
    rows = rng.integers(-2, 3, size=(5000, 16)).astype(np.float32)
    q = rng.integers(-2, 3, size=16).astype(np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), 5000, 16), oracle.VerticalBatch.from_flat(rows.reshape(-1), 5000, 16)
    for k in (1, 10, 100):
        assert_knn_equal(ib.batch_knn_dot(q, gb, k), oracle.batch_knn_dot(q, ob, k))
        assert_knn_equal(ib.batch_knn_cosine(q, gb, k), oracle.batch_knn_cosine(q, ob, k))
        assert_knn_equal(ib.batch_knn(q, gb, k), oracle.batch_knn(q, ob, k), ties_as_sets=True)


def test_knn_special_values(ib, oracle):
    # propagated NaN / inf / -0.0 ordering follows f32::total_cmp (SURVEY.md 8b edge contracts)
    rows = rand_rows(300, 4, 3)
    rows[5, 0] = np.nan       # positive quiet NaN input: propagates (x86 keeps the operand's sign)
    rows[9, 1] = np.inf       # dot -> -inf; L2 -> +inf
    rows[30] = 0.0
    rows[31] = -0.0
    q = np.array([1.0, -2.0, 0.5, 0.0], np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), 300, 4), oracle.VerticalBatch.from_flat(rows.reshape(-1), 300, 4)
    for k in (3, 100):
        g, w = ib.batch_knn_dot(q, gb, k), oracle.batch_knn_dot(q, ob, k)
        assert g.indices == w.indices and same_scores(g.scores, w.scores)
        g, w = ib.batch_knn(q, gb, k), oracle.batch_knn(q, ob, k)
        assert g.indices == w.indices and same_scores(g.scores, w.scores)
    assert ib.batch_knn_dot(q, gb, 300 if False else 128).indices[0] == 5      # NaN sorts greatest (total_cmp)
    zq = np.zeros(4, np.float32)  # zero query: all cosines 0.0 -> first k indices
    g, w = ib.batch_knn_cosine(zq, gb, 10), oracle.batch_knn_cosine(zq, ob, 10)
    assert g.indices == w.indices == list(range(10))
    # -0.0 < +0.0 under total_cmp: descending dot puts +0.0 (row 30) before -0.0 rows
    z = np.zeros((40, 2), np.float32)
    z[::2] = -0.0
    g = ib.batch_knn_dot(np.array([1.0, 1.0], np.float32), ib.VerticalBatch.from_flat(z.reshape(-1), 40, 2), 40)
    w = oracle.batch_knn_dot(np.array([1.0, 1.0], np.float32), oracle.VerticalBatch.from_flat(z.reshape(-1), 40, 2), 40)
    assert g.indices == w.indices and np.array_equal(bits(g.scores), bits(w.scores))


def test_generated_nan_is_canonical_positive_on_device(ib):
    """Documented divergence (DESIGN.md "NaN scores"): a NaN *generated* on the device (inf/inf, inf-inf, 0*inf) is
    the canonical positive 0x7FFFFFFF and sorts greatest under total_cmp; the x86 reference generates the NEGATIVE
    default NaN (sorts least), its aarch64 build the positive one. NaN sign is not portable across the reference's
    own targets, so index parity is only claimed for finite scores and propagated input NaNs."""
    rows = rand_rows(50, 3, 1)
    rows[7, 0] = np.inf  # cosine: -inf / (qn * inf) -> NaN generated on the device
    q = np.array([-1.0, 0.5, 0.25], np.float32)
    g = ib.batch_knn_cosine(q, ib.VerticalBatch.from_flat(rows.reshape(-1), 50, 3), 5)
    assert g.indices[0] == 7 and np.isnan(g.scores[0]) and bits(g.scores)[0] == 0x7FFFFFFF


def test_multi_query_equals_single(ib, oracle):
    n, d, nq, k = 6000, 64, 19, 10
    rows = rand_rows(n, d, 1)
    qs = rand_rows(nq, d, 2)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for metric, single in (("dot", "batch_knn_dot"), ("cosine", "batch_knn_cosine"), ("l2", "batch_knn")):
        idx, sc = ib.batch_knn_many(metric, qs, gb, k)
        for j in range(nq):
            w = getattr(oracle, single)(qs[j], ob, k)
            assert idx[j].tolist() == w.indices, (metric, j)
            assert np.array_equal(bits(sc[j]), bits(w.scores))


def test_config1_batch_demo_gref(ib, oracle):
    """BASELINE config 1: 10K x 128 G-ref lattice (examples/batch_demo.rs:159-170), 100 queries, batch_knn_dot k=10.
    The lattice is an adversarial near-tie fixture (SURVEY.md F11); corpus generated on the device."""
    n, d, nq, k = 10_000, 128, 100, 10
    dev = ib.DeviceBatch.generate("gref", 0, 0, n, d)
    rows = np.stack([oracle.generate_embedding(d, i) for i in range(n)])
    for i in (0, 1, 4097, n - 1):
        assert np.array_equal(bits(dev.extract_vector(i)), bits(rows[i]))
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    qs = np.stack([oracle.generate_embedding(d, 50_000 + j) for j in range(nq)])
    idx, sc = ib.batch_knn_many("dot", qs, dev, k)
    widx, wsc = oracle.batch_knn_many("dot", qs, ob, k, n_threads=8)
    assert np.array_equal(idx, widx) and np.array_equal(bits(sc), bits(wsc))
    assert np.array_equal(bits(ib.batch_l2_squared(qs[0], dev)), bits(oracle.batch_l2_squared(qs[0], ob)))


def test_device_generators_match_oracle(ib, oracle):
    n, d = 777, 48
    dev = ib.DeviceBatch.generate("ghash", 0x5EED0000, 1000, n, d, index_base=1000)
    want = oracle.ghash_f32(0x5EED0000, 1000 * d, n * d).reshape(n, d)
    for i in (0, 1, 500, n - 1):
        assert np.array_equal(bits(dev.extract_vector(i)), bits(want[i]))
    q = oracle.ghash_f32(0x5EED0001, 0, d)
    g = ib.batch_knn_cosine(q, dev, 10)
    w = oracle.batch_knn_cosine(q, oracle.VerticalBatch.from_flat(want.reshape(-1), n, d), 10)
    assert g.indices == [i + 1000 for i in w.indices]          # global indices = index_base + local
    assert np.array_equal(bits(g.scores), bits(w.scores))


def test_rows_upload_transposes_on_device(ib):
    n, d = 1234, 37
    rows = rand_rows(n, d, 9)
    a = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    b = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d).device()
    q = rand_rows(1, d, 10)[0]
    assert np.array_equal(bits(ib.batch_dot(q, a)), bits(ib.batch_dot(q, b)))
    assert np.array_equal(bits(a.extract_vector(n - 1)), bits(rows[n - 1]))


def test_rows_upload_in_chunks(ib):
    """A row-major corpus larger than the 256 MB staging chunk is ingested chunk by chunk (VerticalBatch::from_flat,
    src/batch.rs:167, on the device): every column lands where the PDX layout says, the pitch padding stays zero."""
    n, d = 700_001, 200            # 560 MB of rows -> 3 chunks, ragged last chunk
    rng = np.random.default_rng(12)
    rows = rng.standard_normal((n, d)).astype(np.float32)
    a = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    for i in (0, 1, 335_543, 335_544, 671_087, 671_088, n - 2, n - 1):
        assert np.array_equal(bits(a.extract_vector(i)), bits(rows[i])), i
    q = rng.standard_normal(d).astype(np.float32)
    got = ib.batch_dot(q, a)
    idx = rng.integers(0, n, size=2000)
    want = np.array([np.float32(0)] * len(idx))
    for j, i in enumerate(idx):
        acc = np.float32(0)
        for dd in range(d):
            acc = np.float32(acc + np.float32(q[dd] * rows[i, dd]))
        want[j] = acc
    assert np.array_equal(bits(got[idx]), bits(want))
    g = ib.batch_knn_dot(q, a, 10)
    assert max(g.indices) < n


def test_topk_from_distances_random(ib, oracle):
    rng = np.random.default_rng(3)
    for n, k in ((1, 1), (31, 5), (1000, 10), (100_000, 100), (5000, 128)):
        d = rng.standard_normal(n).astype(np.float32)
        got = ib.topk_from_distances(d, k)
        order = np.lexsort((np.arange(n), d))[:k]
        assert [i for i, _ in got] == order.tolist()
        assert np.array_equal(bits([s for _, s in got]), bits(d[order]))


# ------------------------------------------------------------------------------------------------ Hamming
@pytest.mark.parametrize("dim", [64, 100, 128, 1000, 1024, 2048 + 17])
def test_hamming_bit_exact(ib, oracle, dim):
    words = (dim + 63) // 64
    n = 5000
    rng = np.random.default_rng(dim)
    codes = rng.integers(0, 2**64, size=(n, words), dtype=np.uint64)
    q = rng.integers(0, 2**64, size=words, dtype=np.uint64)
    # dirty padding bits must be masked like PackedBinary::new does
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    qpb = ib.PackedBinary(q, dim)
    opb = [oracle.PackedBinary(c, dim) for c in codes[:50]]
    oq = oracle.PackedBinary(q, dim)
    allg = ib.hamming_all(qpb, corpus)
    for i in range(50):
        assert int(allg[i]) == oracle.binary_hamming(oq, opb[i])
    masked = np.stack([oracle.PackedBinary(c, dim).data for c in codes])
    for k in (1, 100, 128):
        gi, gd = ib.hamming_topk(qpb.data, corpus, k)
        wi, wd = oracle.hamming_topk(oq.data, masked, k)
        assert gi.tolist() == wi.tolist() and gd.tolist() == wd.tolist()


def test_hamming_generator_and_multi_query(ib, oracle):
    n, dim, k = 20_000, 1024, 100
    corpus = ib.BinaryCorpus.generate(0x5EED0002, 0, n, dim)
    codes = oracle.ghash_u64(0x5EED0002, 0, n * 16).reshape(n, 16)
    qs = oracle.ghash_u64(0x5EED0001, 0, 3 * 16).reshape(3, 16)
    gi, gd = ib.hamming_topk_many(qs, corpus, k)
    wi, wd = oracle.hamming_topk_many(qs, codes, k, n_threads=3)
    assert np.array_equal(gi, wi) and np.array_equal(gd, wd)


@pytest.mark.parametrize("dim", [1, 63, 64, 65, 200, 768, 1024])
def test_binary_dot_jaccard_scans_exact(ib, oracle, dim):
    """binary_dot / binary_jaccard (src/binary.rs:178-213) of one query against a corpus: integer-exact intersection,
    bit-exact f32 quotient, empty-union convention 1.0."""
    n = 3001
    rng = np.random.default_rng(dim)
    words = (dim + 63) // 64
    codes = rng.integers(0, 2**63, size=(n, words), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, words), dtype=np.uint64)
    codes[5] = 0                       # empty code
    q = rng.integers(0, 2**63, size=words, dtype=np.uint64) * np.uint64(2) + np.uint64(1)
    gq, oq = ib.PackedBinary(q.copy(), dim), oracle.PackedBinary(q.copy(), dim)
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    got_dot, got_j = ib.binary_dot_all(gq, corpus), ib.binary_jaccard_all(gq, corpus)
    for i in range(0, n, 13):
        oc = oracle.PackedBinary(codes[i].copy(), dim)
        assert int(got_dot[i]) == oracle.binary_dot(oq, oc), (dim, i)
        assert np.float32(got_j[i]).tobytes() == np.float32(oracle.binary_jaccard(oq, oc)).tobytes(), (dim, i)
    z = ib.PackedBinary.zeros(dim)
    assert float(ib.binary_jaccard_all(z, corpus)[5]) == 1.0 and int(ib.binary_dot_all(z, corpus)[5]) == 0
    # top-k by similarity == stable descending sort of the full score vectors (ties -> lower index), any k
    for k in (1, 10, 100, 400, n + 1):
        for op, full in (("dot", got_dot.astype(np.float32)), ("jaccard", got_j)):
            idx, sc = ib.binary_topk(op, gq, corpus, k)
            order = np.lexsort((np.arange(n), -full.astype(np.float64)))[:k]
            assert idx.tolist() == order.tolist(), (dim, op, k)
            assert np.array_equal(bits(sc), bits(full[order])), (dim, op, k)


# ------------------------------------------------------------------------------------------------ host threads
def test_concurrent_host_threads(ib, oracle):
    """SURVEY 8b 'Threading': handles are immutable after upload and calls from several host threads must be safe
    (a per-device mutex serialises them; ctypes drops the GIL during the call). Every thread must get its own exact
    answer."""
    import threading
    n, d, k = 20000, 64, 10
    rows = rand_rows(n, d, 99)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    codes = np.random.default_rng(5).integers(0, 2**62, size=(n, 4), dtype=np.uint64)
    bc = ib.BinaryCorpus.from_words(codes, n, 256)
    qs = rand_rows(16, d, 123)
    qcs = np.random.default_rng(6).integers(0, 2**62, size=(16, 4), dtype=np.uint64)
    want = [oracle.batch_knn_cosine(qs[i], ob, k) for i in range(16)]
    want_h = [oracle.hamming_topk(qcs[i], codes, k) for i in range(16)]
    errors = []

    def worker(t):
        try:
            for rep in range(6):
                i = (t * 5 + rep) % 16
                if (t + rep) % 2 == 0:
                    got = ib.batch_knn_cosine(qs[i], gb, k)
                    assert list(got.indices) == list(want[i].indices)
                    assert np.array_equal(bits(got.scores), bits(want[i].scores))
                else:
                    gi, gd = ib.hamming_topk_many(qcs[i].reshape(1, -1), bc, k)
                    assert np.array_equal(gi[0], want_h[i][0]) and np.array_equal(gd[0], want_h[i][1])
        except Exception as e:  # noqa: BLE001
            errors.append((t, repr(e)))

    ts = [threading.Thread(target=worker, args=(t,)) for t in range(8)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    assert not errors, errors[:3]


def test_c_abi_sharded_entries(ib, oracle):
    """innr_cuda_*_sharded: row shards (here three on one device; test_one_process_two_devices spreads them over two),
    one host thread per shard inside the library, host merge in the device's key order == the unsharded result,
    with heavy ties across shard boundaries."""
    from innr_b200 import sharded
    n, d, nq = 9001, 40, 5
    rng = np.random.default_rng(14)
    rows = rng.integers(-3, 4, size=(n, d)).astype(np.float32)
    qs = rng.integers(-3, 4, size=(nq, d)).astype(np.float32)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    cuts = [0, 2500, 2500, 7003, n]          # one empty shard
    shards = [ib.DeviceBatch.from_rows_flat(rows[a:b].reshape(-1), b - a, d, index_base=a) for a, b in zip(cuts, cuts[1:])]
    for metric in ("dot", "cosine", "l2"):
        for k in (1, 10, 100, 300):
            idx, sc = sharded.batch_knn_sharded(metric, qs, shards, k)
            widx, wsc = oracle.batch_knn_many(metric, qs, ob, k, n_threads=4)
            assert np.array_equal(bits(sc), bits(wsc)), (metric, k)
            if metric != "l2":
                assert np.array_equal(idx, widx), (metric, k)
    codes = rng.integers(0, 2**62, size=(n, 3), dtype=np.uint64)
    qc = rng.integers(0, 2**62, size=(2, 3), dtype=np.uint64)
    bsh = [ib.BinaryCorpus.from_words(codes[a:b], b - a, 192, index_base=a) for a, b in zip(cuts, cuts[1:])]
    gi, gd = sharded.hamming_topk_sharded(qc, bsh, 100)
    wi, wd = oracle.hamming_topk_many(qc, codes, 100, n_threads=2)
    assert np.array_equal(gi, wi) and np.array_equal(gd, wd)
    mat = rng.integers(0, 256, size=(n, 48), dtype=np.uint8)
    q8 = rng.uniform(-1, 1, size=(3, 48)).astype(np.float32)
    gp, op = ib.QuantizationParams.from_range(-1.0, 1.0), oracle.QuantizationParams.from_range(-1.0, 1.0)
    ush = [ib.U8Corpus.from_rows(mat[a:b], gp, index_base=a, dimension=48) for a, b in zip(cuts, cuts[1:])]
    ui, us = sharded.batch_knn_u8_sharded(q8, ush, 10)
    wi, ws = oracle.batch_knn_u8_many(q8, mat, op, 10, n_threads=2)
    assert np.array_equal(ui, wi) and np.array_equal(bits(us), bits(ws))


def test_one_process_two_devices(ib, oracle):
    """INTEGRATION.md section 4: one host process driving several GPUs, one thread and one row shard per device
    (per-device mutexes, per-device function attributes): local top-k per shard, merged on the host by key order."""
    import threading
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs (run with gpurun --gpus 2)")
    n, d, k = 50000, 96, 10
    rows = rand_rows(n, d, 7)
    q = rand_rows(1, d, 8)[0]
    want = oracle.batch_knn_cosine(q, oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d), k)
    half = n // 2
    out, errors = {}, []

    def worker(dev):
        try:
            ib.init(dev)
            lo, hi = (0, half) if dev == 0 else (half, n)
            shard = ib.DeviceBatch.from_rows_flat(rows[lo:hi].reshape(-1), hi - lo, d, index_base=lo)
            for _ in range(5):
                idx, sc = ib.batch_knn_many("cosine", q.reshape(1, -1), shard, k)
            toks = rand_rows(40 * 30, 128, 9 + dev)
            off = np.arange(0, 40 * 30 + 1, 30, dtype=np.uint64)
            ms = ib.maxsim_corpus(rand_rows(32, 128, 11), ib.TokenCorpus.from_tokens(toks, off, 128), cosine=True)
            ref = oracle.maxsim_corpus(rand_rows(32, 128, 11), toks, off, cosine_flag=True)
            assert np.allclose(ms, ref, rtol=1e-5, atol=1e-5)
            out[dev] = (idx[0], sc[0])
        except Exception as e:  # noqa: BLE001
            errors.append((dev, repr(e)))

    ts = [threading.Thread(target=worker, args=(dv,)) for dv in (0, 1)]
    for t in ts:
        t.start()
    for t in ts:
        t.join()
    ib.init(0)
    assert not errors, errors
    pairs = sorted(((-float(s), int(i)) for dv in (0, 1) for i, s in zip(*out[dv])))[:k]
    assert [i for _, i in pairs] == [int(i) for i in want.indices]
    # the library's own sharded entry over shards on both devices
    from innr_b200 import sharded
    shards = []
    for dev, (lo, hi) in enumerate(((0, half), (half, n))):
        ib.init(dev)
        shards.append(ib.DeviceBatch.from_rows_flat(rows[lo:hi].reshape(-1), hi - lo, d, index_base=lo))
    ib.init(0)
    qs = rand_rows(6, d, 31)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for metric in ("cosine", "dot"):
        idx, sc = sharded.batch_knn_sharded(metric, qs, shards, k)
        widx, wsc = oracle.batch_knn_many(metric, qs, ob, k, n_threads=4)
        assert np.array_equal(idx, widx) and np.array_equal(bits(sc), bits(wsc)), metric


# ------------------------------------------------------------------------------------------------ two-stage retrieval
@pytest.mark.parametrize("n,d", [(3000, 96), (5000, 200), (1500, 7)])
def test_derived_encodings_and_rerank(ib, oracle, n, d):
    """SURVEY 8f row 2: one f32 ingest, binary and u8 encodings derived on the device (bit-identical to encode_binary /
    quantize_u8 of every row), first pass on the codes, exact re-rank of the candidates (= the reference's function on
    the gathered sub-batch, original indices)."""
    rng = np.random.default_rng(n + d)
    rows = rng.standard_normal((n, d)).astype(np.float32)
    rows[3] = 0.0
    q = rng.standard_normal(d).astype(np.float32)
    base = 1000
    gb = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d, index_base=base)
    # binary: Hamming distances of the derived codes == oracle on encode_binary of each row
    bc = ib.BinaryCorpus.from_f32(gb, 0.0)
    qb_g, qb_o = ib.encode_binary(q, 0.0), oracle.encode_binary(q, 0.0)
    got = ib.hamming_all(qb_g, bc)
    want = np.array([oracle.binary_hamming(qb_o, oracle.encode_binary(rows[i], 0.0)) for i in range(n)], np.uint32)
    assert np.array_equal(got, want)
    # u8: derived codes == quantize_u8 of each row (checked through exact mixed dots against the oracle's codes)
    gp, op = ib.QuantizationParams.from_range(-3.0, 3.0), oracle.QuantizationParams.from_range(-3.0, 3.0)
    uc = ib.U8Corpus.from_f32(gb, gp)
    mat = oracle.quantize_u8(rows.reshape(-1), op).data.reshape(n, d)
    gm = ib.mixed_dot_u8_all(q, uc)
    for i in range(0, n, 37):
        assert np.float32(gm[i]).tobytes() == np.float32(oracle.mixed_dot_u8_f32(q, mat[i])).tobytes()
    # two-stage: Hamming top-300 (k > 128) -> exact re-rank top-10, all three metrics
    cand, _ = ib.hamming_topk_many(np.asarray(qb_g.data, np.uint64).reshape(1, -1), bc, 300)
    cand = cand[0]
    assert cand.min() >= base
    local = (cand - base).astype(np.int64)
    order = np.argsort(local, kind="stable")
    sub = oracle.VerticalBatch.from_flat(rows[local[order]].reshape(-1), len(local), d)
    for metric, fn in (("dot", "batch_knn_dot"), ("cosine", "batch_knn_cosine"), ("l2", "batch_knn")):
        got = ib.batch_knn_subset(metric, q, gb, cand, 10)
        want = getattr(oracle, fn)(q, sub, 10)
        want_idx = [int(local[order][int(j)]) + base for j in want.indices]
        assert np.array_equal(bits(got.scores), bits(want.scores)), metric
        if metric != "l2":
            assert [int(i) for i in got.indices] == want_idx, metric
        else:
            assert sorted(int(i) for i in got.indices) == sorted(want_idx)


def test_matryoshka_prefix_view(ib, oracle):
    """A prefix view (first D' rows of the PDX corpus, zero-copy) answers exactly like the reference's batch functions
    on the truncated vectors -- single queries (scan) and query batches (tensor-core filter on the view's own operands)."""
    n, d = 120_000, 96
    rows = rand_rows(n, d, 21)
    full = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    qs = rand_rows(12, d, 22)
    for dp in (32, 80, 96, 200):
        view = full.prefix(dp)
        de = min(dp, d)
        ob = oracle.VerticalBatch.from_flat(np.ascontiguousarray(rows[:, :de]).reshape(-1), n, de)
        for metric in ("cosine", "dot", "l2"):
            idx, sc = ib.batch_knn_many(metric, qs[:1, :de], view, 10)
            widx, wsc = oracle.batch_knn_many(metric, np.ascontiguousarray(qs[:1, :de]), ob, 10)
            assert np.array_equal(bits(sc), bits(wsc)) and (metric == "l2" or np.array_equal(idx, widx)), (dp, metric)
            idx, sc = ib.batch_knn_many(metric, np.ascontiguousarray(qs[:, :de]), view, 10)
            widx, wsc = oracle.batch_knn_many(metric, np.ascontiguousarray(qs[:, :de]), ob, 10, n_threads=8)
            assert np.array_equal(bits(sc), bits(wsc)) and (metric == "l2" or np.array_equal(idx, widx)), (dp, metric)
        assert np.array_equal(bits(ib.batch_dot(qs[0, :de], view)), bits(oracle.batch_dot(qs[0, :de], ob)))


# ------------------------------------------------------------------------------------------------ k > 128
@pytest.mark.parametrize("k", [129, 300, 1000, 5000])
def test_big_k_all_paths_exact(ib, oracle, k):
    """k > 128 leaves the fused register lists: one scores pass, then rounds of <= 128 keys over the score vector,
    each round bounded below by the last key of the round before. Same bits and order as the reference's full sort,
    with heavy ties (integer-valued rows) and k > N."""
    n, d = 4000, 24
    rng = np.random.default_rng(k)
    rows = rng.integers(-3, 4, size=(n, d)).astype(np.float32)
    q = rng.integers(-3, 4, size=d).astype(np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for name in ("batch_knn_dot", "batch_knn_cosine"):
        got, want = getattr(ib, name)(q, gb, k), getattr(oracle, name)(q, ob, k)
        assert len(got.indices) == min(k, n)
        assert list(got.indices) == list(want.indices), name
        assert np.array_equal(bits(got.scores), bits(want.scores)), name
    assert_knn_equal(ib.batch_knn(q, gb, k), oracle.batch_knn(q, ob, k), ties_as_sets=True)
    # Hamming
    codes = rng.integers(0, 2**62, size=(n, 2), dtype=np.uint64)
    qc = rng.integers(0, 2**62, size=2, dtype=np.uint64)
    gi, gd = ib.hamming_topk(qc, codes, k)
    wi, wd = oracle.hamming_topk(qc, codes, k)
    assert np.array_equal(gi, wi) and np.array_equal(gd, wd)
    # u8
    mat = rng.integers(0, 256, size=(n, 48), dtype=np.uint8)
    q8 = rng.uniform(-1, 1, 48).astype(np.float32)
    gp, op = ib.QuantizationParams.from_range(-1.0, 1.0), oracle.QuantizationParams.from_range(-1.0, 1.0)
    got = ib.batch_knn_u8(q8, ib.U8Corpus.from_rows(mat, gp), gp, k)
    want = oracle.batch_knn_u8(q8, mat, op, k)
    assert [i for i, _ in got] == [i for i, _ in want]
    assert np.array_equal(bits([s for _, s in got]), bits([s for _, s in want]))
    # TopK analogue
    dist = rng.integers(0, 50, size=n).astype(np.float32)
    got = ib.topk_from_distances(dist, k)
    order = sorted(range(n), key=lambda i: (dist[i], i))[:k]
    assert [i for i, _ in got] == order and [s for _, s in got] == [float(dist[i]) for i in order]


# ------------------------------------------------------------------------------------------------ filtered / pruning
@pytest.mark.parametrize("n,d,sel", [(5000, 33, 0.5), (70001, 16, 0.01), (4097, 128, 0.9), (300, 7, 0.0), (2049, 5, 1.0)])
def test_knn_filtered_bit_exact(ib, oracle, n, d, sel):
    """batch_knn_filtered (src/batch.rs:820-882) with the predicate as a bitmask: passing set, L2 bits, stable order."""
    rng = np.random.default_rng(n + d)
    rows = rng.integers(-4, 5, size=(n, d)).astype(np.float32) if d < 10 else rng.standard_normal((n, d)).astype(np.float32)
    q = rng.standard_normal(d).astype(np.float32)
    mask = rng.random(n) < sel
    if sel == 0.0:
        mask[:] = False
        mask[n // 2] = True          # exactly one passing vector
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for k in (1, 10, 100, 129, 700):   # > 128: a scores pass plus masked selection rounds
        got = ib.batch_knn_filtered(q, gb, k, mask)
        want = oracle.batch_knn_filtered(q, ob, k, lambda i: bool(mask[i]))
        assert list(got.indices) == list(want.indices), (k, got.indices[:5], want.indices[:5])
        assert np.array_equal(bits(got.scores), bits(want.scores))
        assert all(mask[int(i)] for i in got.indices)


@pytest.mark.parametrize("n,d", [(5000, 33), (70001, 16), (1025, 128), (300, 1)])
def test_l2_pruning_bit_exact(ib, oracle, n, d):
    """batch_l2_squared_pruning (src/batch.rs:320-365): survivor set, order and distance bits, over thresholds from
    'nothing survives' to 'everything survives', with NaN / inf rows (a NaN partial never exceeds the threshold)."""
    rng = np.random.default_rng(n * 3 + d)
    rows = rng.standard_normal((n, d)).astype(np.float32)
    rows[7, 0] = np.nan
    rows[9, d - 1] = np.inf
    if d > 2:
        rows[11, 0] = 1e20           # overflows to inf in the first dimension, then inf - ... stays inf
        rows[13, 1] = np.nan         # NaN after a finite first partial
    q = rng.standard_normal(d).astype(np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    full = oracle.batch_l2_squared(q, ob)
    finite = full[np.isfinite(full)]
    for thr in (-1.0, 0.0, float(np.quantile(finite, 0.001)), float(np.quantile(finite, 0.3)), float(finite.max()),
                float("inf"), float("nan")):
        got = ib.batch_l2_squared_pruning(q, gb, thr)
        want = oracle.batch_l2_squared_pruning(q, ob, thr)
        assert [i for i, _ in got] == [i for i, _ in want], (thr, len(got), len(want))
        assert same_scores([s for _, s in got], [s for _, s in want]), thr


@pytest.mark.parametrize("dim,nq", [(1024, 2), (1024, 4), (1024, 9), (200, 5), (64, 7)])
def test_hamming_query_batches_share_a_pass(ib, oracle, dim, nq):
    """Batches of Hamming queries run four per pass over the codes; each must equal the single-query result
    (distance, then lower index: stable sort_by_key), with the heavy ties of near-uniform codes."""
    n = 30_011
    rng = np.random.default_rng(dim + nq)
    words = (dim + 63) // 64
    codes = rng.integers(0, 2**63, size=(n, words), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, size=(n, words), dtype=np.uint64)
    if dim % 64:
        codes[:, -1] &= np.uint64((1 << (dim % 64)) - 1)
    qs = codes[rng.integers(0, n, size=nq)] ^ np.uint64(0x5)
    if dim % 64:
        qs[:, -1] &= np.uint64((1 << (dim % 64)) - 1)
    corpus = ib.BinaryCorpus.from_words(codes, n, dim)
    for k in (1, 10, 100):
        gi, gd = ib.hamming_topk_many(qs, corpus, k)
        wi, wd = oracle.hamming_topk_many(qs, codes, k, n_threads=4)
        assert np.array_equal(gi, wi) and np.array_equal(gd, wd), (dim, nq, k)


# ------------------------------------------------------------------------------------------------ ternary
@pytest.mark.parametrize("dim", [1, 31, 32, 33, 63, 64, 65, 128, 200, 768, 13000])
def test_ternary_scans_exact(ib, oracle, dim):
    """ternary_dot / ternary_hamming (integer-exact) and ternary::asymmetric_dot (sequential unfused f32 sum, bit-exact)
    of one query against a corpus; top-k in the reference's stable order; encodings derived on the device."""
    n = 3001
    rng = np.random.default_rng(dim)
    rows = rng.standard_normal((n, dim)).astype(np.float32)
    rows[7] = 0.0
    codes_o = [oracle.encode_ternary(rows[i], 0.4) for i in range(n)]
    words = np.stack([c.data for c in codes_o])
    corpus = ib.TernaryCorpus.from_words(words, n, dim)
    derived = ib.TernaryCorpus.from_f32(ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, dim), 0.4)
    qf = rng.standard_normal(dim).astype(np.float32)
    if dim > 2:
        qf[1] = -0.0
    qg, qo = ib.encode_ternary(qf, 0.4), oracle.encode_ternary(qf, 0.4)
    assert np.array_equal(qg.data, qo.data)
    for corp in (corpus, derived):
        d = ib.ternary_scores_all("dot", qg, corp)
        h = ib.ternary_scores_all("hamming", qg, corp)
        a = ib.ternary_scores_all("asymmetric_dot", qf, corp)
        for i in range(0, n, 7):
            assert int(d[i]) == oracle.ternary_dot(qo, codes_o[i]), (dim, i)
            assert int(h[i]) == oracle.ternary_hamming(qo, codes_o[i]), (dim, i)
            assert np.float32(a[i]).tobytes() == np.float32(oracle.ternary_asymmetric_dot(qf, codes_o[i])).tobytes(), (dim, i)
    want_d = np.array([oracle.ternary_dot(qo, c) for c in codes_o])
    want_h = np.array([oracle.ternary_hamming(qo, c) for c in codes_o])
    for k in (1, 10, 300):
        idx, sc = ib.ternary_topk("dot", qg, corpus, k)
        order = sorted(range(n), key=lambda i: (-want_d[i], i))[:k]
        assert [int(i) for i in idx] == order and [int(s) for s in sc] == [int(want_d[i]) for i in order]
        idx, sc = ib.ternary_topk("hamming", qg, corpus, k)
        order = sorted(range(n), key=lambda i: (want_h[i], i))[:k]
        assert [int(i) for i in idx] == order and [int(s) for s in sc] == [int(want_h[i]) for i in order]
    # asymmetric dot top-k (fused single pass for k <= 128, score vector + selection rounds above): descending under
    # total_cmp, ties -> lower index, scores bit-identical to the full scan's
    a_full = ib.ternary_scores_all("asymmetric_dot", qf, corpus)
    okey = sharded_order_bits(a_full)
    for k in (1, 10, 100, 300):
        idx, sc = ib.ternary_topk("asymmetric_dot", qf, corpus, k)
        order = sorted(range(n), key=lambda i: (-int(okey[i]), i))[:k]
        assert [int(i) for i in idx] == order, (dim, k)
        assert np.array_equal(bits(sc), bits(a_full[order])), (dim, k)


# ------------------------------------------------------------------------------------------------ u8
@pytest.mark.parametrize("d", [1, 8, 15, 16, 17, 31, 32, 33, 40, 63, 64, 65, 100, 128, 384, 777])
def test_u8_bit_exact(ib, oracle, d):
    n = 3000
    rng = np.random.default_rng(d)
    mat = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    q = (rng.standard_normal(d) * 3).astype(np.float32)
    gp, op = ib.QuantizationParams.from_range(-1.5, 2.0), oracle.QuantizationParams.from_range(-1.5, 2.0)
    corpus = ib.U8Corpus.from_rows(mat, gp)
    mixed = ib.mixed_dot_u8_all(q, corpus)
    asym = ib.asymmetric_dot_u8_all(q, corpus)
    for i in range(0, n, 97):
        assert np.float32(mixed[i]).tobytes() == np.float32(oracle.mixed_dot_u8_f32(q, mat[i])).tobytes(), (d, i)
        assert np.float32(asym[i]).tobytes() == np.float32(
            oracle.asymmetric_dot_u8(q, oracle.QuantizedU8(mat[i], d), op)).tobytes(), (d, i)
    for k in (1, 10, 100):
        got = ib.batch_knn_u8(q, corpus, gp, k)
        want = oracle.batch_knn_u8(q, mat, op, k)
        assert [i for i, _ in got] == [i for i, _ in want]
        assert np.array_equal(bits([s for _, s in got]), bits([s for _, s in want]))


@pytest.mark.parametrize("d", [32, 64, 96, 384, 400, 777])
@pytest.mark.parametrize("qkind", ["unit", "zeros", "wide_range", "cancel", "below_range", "denormal", "ge4", "nan"])
def test_u8_scaled_chains_bit_exact(ib, oracle, d, qkind):
    """The u8 scan runs its 32 FMA chains scaled by 2^-23 (byte bits as the f32 b*2^-149, query * 2^126) when every
    main-loop query element is 0 or in [2^-80, 4), else with the de-biasing FADD. Both must reproduce dot_u8_f32_avx2
    (src/arch/x86_64.rs:928-1020) bit for bit; queries at and beyond the edges of the admissible range are the cases."""
    n = 2048 + 7
    rng = np.random.default_rng(d * 31 + len(qkind))
    mat = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    mat[0] = 0
    mat[1] = 255
    q = rng.uniform(-1, 1, d).astype(np.float32)
    if qkind == "zeros":
        q[::3] = 0.0
        q[1::7] = -0.0
    elif qkind == "wide_range":      # exponents spread over the whole admissible range
        q = (np.ldexp(rng.uniform(0.5, 1.0, d), rng.integers(-79, 2, d)) * rng.choice([-1, 1], d)).astype(np.float32)
        q[0], q[1] = np.float32(2.0 ** -80), np.float32(np.nextafter(np.float32(4.0), np.float32(0.0)))
    elif qkind == "cancel":          # chains that cancel to tiny / zero partial sums
        q[32:64] = -q[0:32] if d >= 64 else q[32:64]
        mat[:, 32:64] = mat[:, 0:32] if d >= 64 else mat[:, 32:64]
        q[5] = np.float32(2.0 ** -80)
    elif qkind == "below_range":
        q[3] = np.float32(2.0 ** -81)
    elif qkind == "denormal":
        q[3] = np.float32(1e-40)
    elif qkind == "ge4":
        q[7] = np.float32(4.0)
        q[9] = np.float32(-3.0e20)
    elif qkind == "nan":
        q[11] = np.nan
    gp, op = ib.QuantizationParams.from_range(-1.0, 1.0), oracle.QuantizationParams.from_range(-1.0, 1.0)
    corpus = ib.U8Corpus.from_rows(mat, gp)
    want = np.array([oracle.mixed_dot_u8_f32(q, mat[i]) for i in range(n)], dtype=np.float32)
    try:
        for mode in (1, 0):
            ib.set_option("u8_scaled_chains", mode)
            got = ib.mixed_dot_u8_all(q, corpus)
            assert np.array_equal(bits(got), bits(want)) or (
                qkind == "nan" and np.array_equal(np.isnan(got), np.isnan(want))), (mode, qkind, d)
    finally:
        ib.set_option("u8_scaled_chains", 1)
    if qkind != "nan":
        got = ib.batch_knn_u8(q, corpus, gp, 10)
        want_k = oracle.batch_knn_u8(q, mat, op, 10)
        assert [i for i, _ in got] == [i for i, _ in want_k]
        assert np.array_equal(bits([s for _, s in got]), bits([s for _, s in want_k]))


@pytest.mark.parametrize("d,nq", [(384, 2), (384, 5), (100, 4), (33, 3), (8, 2), (777, 7)])
def test_u8_query_batches_share_a_pass(ib, oracle, d, nq):
    """batch_knn_u8 for several queries: two queries share each pass over the codes (the byte -> f32 conversion is
    shared); every list must be bit-identical to the single-query result, incl. a query that forces the de-biasing
    path for its pair (|q| >= 4) and every tail shape."""
    n = 5000
    rng = np.random.default_rng(d * 7 + nq)
    mat = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    qs = rng.uniform(-1, 1, size=(nq, d)).astype(np.float32)
    qs[-1, 0] = 7.5                                  # outside the scaled-chain range
    gp, op = ib.QuantizationParams.from_range(-2.0, 1.0), oracle.QuantizationParams.from_range(-2.0, 1.0)
    corpus = ib.U8Corpus.from_rows(mat, gp)
    for k in (1, 10, 100):
        gi, gs = ib.batch_knn_u8_many(qs, corpus, k)
        wi, ws = oracle.batch_knn_u8_many(qs, mat, op, k, n_threads=4)
        assert np.array_equal(gi, wi), (d, nq, k)
        assert np.array_equal(bits(gs), bits(ws)), (d, nq, k)


def test_u8_generator_and_quantize(ib, oracle):
    n, d = 4000, 384
    gp, op = ib.QuantizationParams.from_range(-1.0, 1.0), oracle.QuantizationParams.from_range(-1.0, 1.0)
    vals = oracle.ghash_f32(0x5EED0000, 0, n * d)
    assert np.array_equal(ib.quantize_u8(vals, gp).data, oracle.quantize_u8(vals, op).data)
    corpus = ib.U8Corpus.generate(0x5EED0000, 0, n, d, gp)
    mat = oracle.quantize_u8(vals, op).data.reshape(n, d)
    q = oracle.ghash_f32(0x5EED0001, 0, d)
    got = ib.batch_knn_u8(q, corpus, gp, 10)
    want = oracle.batch_knn_u8(q, mat, op, 10)
    assert [i for i, _ in got] == [i for i, _ in want]
    assert np.array_equal(bits([s for _, s in got]), bits([s for _, s in want]))


# ------------------------------------------------------------------------------------------------ MaxSim
def _maxsim_scale(q, toks, off):
    out = np.zeros(len(off) - 1)
    aq = np.abs(q.astype(np.float64))
    for j in range(len(off) - 1):
        t = np.abs(toks[off[j]:off[j + 1]].astype(np.float64))
        out[j] = float(np.sum(np.max(aq @ t.T, axis=1))) if t.shape[0] else 0.0
    return out


@pytest.mark.parametrize("nq,dim", [(1, 4), (3, 30), (32, 128), (40, 64), (32, 16), (7, 129),
                                    # wide rows: the contraction runs over 256-column chunks, queries re-staged per chunk
                                    (5, 300), (32, 768), (40, 1001), (300, 132), (33, 256), (2, 2050),
                                    (300, 128), (700, 64)])  # many query tokens on the tcgen05 path: passes of 64
def test_maxsim_within_tolerance(ib, oracle, nq, dim):
    rng = np.random.default_rng(nq * 100 + dim)
    lens = rng.integers(0, 200, size=60)
    lens[3] = 0                                   # empty doc -> 0.0
    lens[10] = 180
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    toks = rng.standard_normal((int(off[-1]), dim)).astype(np.float32)
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    for cos in (False, True):
        got = ib.maxsim_corpus(q, corpus, cosine=cos)
        want = oracle.maxsim_corpus(q, toks, off, cosine_flag=cos)
        scale = _maxsim_scale(q, toks, off) if not cos else np.full(len(lens), float(nq))
        assert np.all(np.abs(got.astype(np.float64) - want) <= 1e-5 * scale + 1e-6), (
            cos, float(np.max(np.abs(got - want))))
        assert got[3] == 0.0


def test_maxsim_colbert_shape_generated(ib, oracle):
    """C3 shape at reduced doc count: 32 x 128 query tokens vs docs of 180 x 128 tokens, generated on the device."""
    n_docs, nt, dim, nq = 500, 180, 128, 32
    corpus = ib.TokenCorpus.generate(0x5EED0000, 0, n_docs, nt, dim)
    toks = oracle.ghash_f32(0x5EED0000, 0, n_docs * nt * dim).reshape(n_docs * nt, dim)
    q = oracle.ghash_f32(0x5EED0001, 0, nq * dim).reshape(nq, dim)
    off = np.arange(0, n_docs * nt + 1, nt, dtype=np.uint64)
    for cos in (False, True):
        got = ib.maxsim_corpus(q, corpus, cosine=cos)
        want = oracle.maxsim_corpus(q, toks, off, cosine_flag=cos, n_threads=8)
        scale = _maxsim_scale(q, toks, off) if not cos else np.full(n_docs, float(nq))
        assert np.all(np.abs(got.astype(np.float64) - want) <= 1e-5 * scale + 1e-6)
        rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-30)
        assert float(np.max(rel)) < 1e-5, float(np.max(rel))   # north_star: f32 scores within 1e-5 relative


@pytest.mark.parametrize("shape", ["tiny_docs", "one_huge", "mixed", "few_docs", "single_token"])
@pytest.mark.parametrize("nq", [32, 5, 64, 47])
def test_maxsim_tc_stream_edges(ib, oracle, shape, nq):
    """The tcgen05 path (dim 128, <= 32 query tokens) cuts every CTA's range into four document-aligned streams and
    handles document boundaries inside a 32-token chunk as masked segments: documents shorter than a chunk (many per
    chunk, with empty ones between), one document longer than many tiles, fewer documents than streams."""
    dim = 128
    rng = np.random.default_rng({"tiny_docs": 1, "one_huge": 2, "mixed": 3, "few_docs": 4, "single_token": 5}[shape] + nq)
    if shape == "tiny_docs":
        lens = rng.integers(0, 6, size=3000)
    elif shape == "one_huge":
        lens = np.array([3, 0, 7001, 2, 0, 0, 45])
    elif shape == "mixed":
        lens = np.concatenate([rng.integers(0, 40, size=500), [1500], rng.integers(100, 400, size=40), [0, 0, 1]])
    elif shape == "few_docs":
        lens = np.array([200, 31])
    else:
        lens = np.array([1])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    toks = rng.standard_normal((int(off[-1]), dim)).astype(np.float32)
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    for cos in (False, True):
        got = ib.maxsim_corpus(q, corpus, cosine=cos)
        want = oracle.maxsim_corpus(q, toks, off, cosine_flag=cos)
        scale = _maxsim_scale(q, toks, off) if not cos else np.full(len(lens), float(nq))
        err = np.abs(got.astype(np.float64) - want)
        assert np.all(err <= 1e-5 * scale + 1e-6), (shape, cos, int(np.argmax(err - 1e-5 * scale)), float(err.max()))
        assert np.all(got[lens == 0] == 0.0)


@pytest.mark.parametrize("dim", [32, 64, 96, 128, 4, 20, 36, 48, 100, 124,   # not a multiple of 32: TMA zero-fills the last panel
                                 132, 160, 192, 200, 256])                  # 129..256: two K halves of 128 columns per tile
@pytest.mark.parametrize("nq", [1, 33, 64, 100])
def test_maxsim_tc_dims_and_query_groups(ib, oracle, dim, nq):
    """tcgen05 path at every supported token dimension, and with more than 32 query tokens (one corpus pass per group
    of 32, partial sums accumulated per document) -- the reference's own bench shapes use 32 and 64 query tokens
    (benches/maxsim.rs:21,44)."""
    rng = np.random.default_rng(dim * 7 + nq)
    lens = np.concatenate([rng.integers(0, 300, size=120), [0, 1, 700]])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    toks = rng.standard_normal((int(off[-1]), dim)).astype(np.float32)
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    for cos in (False, True):
        got = ib.maxsim_corpus(q, corpus, cosine=cos)
        want = oracle.maxsim_corpus(q, toks, off, cosine_flag=cos)
        scale = _maxsim_scale(q, toks, off) if not cos else np.full(len(lens), float(nq))
        err = np.abs(got.astype(np.float64) - want)
        assert np.all(err <= 1e-5 * scale + 1e-6), (dim, nq, cos, float(err.max()))
        assert np.all(got[lens == 0] == 0.0)


@pytest.mark.parametrize("n_queries,nq,dim", [(2, 32, 128), (5, 17, 128), (3, 32, 64), (1, 8, 96), (4, 40, 128), (3, 6, 48),
                                              (3, 20, 256), (2, 40, 160)])
def test_maxsim_query_batches(ib, oracle, n_queries, nq, dim):
    """Batches of queries: on the tcgen05 path two queries of <= 32 tokens share each corpus pass (their tokens are the two
    column groups of one accumulator, sums kept apart); every row must equal the single-query result."""
    rng = np.random.default_rng(n_queries * 1000 + nq + dim)
    lens = np.concatenate([rng.integers(0, 120, size=150), [0, 900, 1]])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    toks = rng.standard_normal((int(off[-1]), dim)).astype(np.float32)
    qs = rng.standard_normal((n_queries, nq, dim)).astype(np.float32)
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    for cos in (False, True):
        got = ib.maxsim_corpus_batch(qs, corpus, cosine=cos)
        for i in range(n_queries):
            single = ib.maxsim_corpus(qs[i], corpus, cosine=cos)
            want = oracle.maxsim_corpus(qs[i], toks, off, cosine_flag=cos)
            scale = _maxsim_scale(qs[i], toks, off) if not cos else np.full(len(lens), float(nq))
            assert np.all(np.abs(got[i].astype(np.float64) - want) <= 1e-5 * scale + 1e-6), (i, cos)
            if nq <= 32 and dim % 32 == 0 and dim <= 128:
                assert np.array_equal(bits(got[i]), bits(single)), (i, cos)   # same arithmetic, same bits
            assert np.all(got[i][lens == 0] == 0.0)


def test_maxsim_tc_nan_and_zero_tokens(ib, oracle):
    """NaN scores never replace the running max (`>` compare, x86_64.rs:135); a document whose every score is NaN sums
    -inf; zero-norm tokens and zero-norm query tokens give cosine 0.0 (x86_64.rs:781-785)."""
    dim, nq = 128, 8
    rng = np.random.default_rng(77)
    lens = np.array([40, 3, 64, 2])
    off = np.concatenate([[0], np.cumsum(lens)]).astype(np.uint64)
    toks = rng.standard_normal((int(off[-1]), dim)).astype(np.float32)
    toks[5, 17] = np.nan            # one NaN token inside doc 0
    toks[40:43, 0] = np.nan         # doc 1: every token NaN
    toks[50] = 0.0                  # zero-norm token in doc 2
    q = rng.standard_normal((nq, dim)).astype(np.float32)
    q[3] = 0.0                      # zero-norm query token
    corpus = ib.TokenCorpus.from_tokens(toks, off, dim)
    for cos in (False, True):
        got = ib.maxsim_corpus(q, corpus, cosine=cos)
        want = oracle.maxsim_corpus(q, toks, off, cosine_flag=cos)
        for j in (0, 2, 3):
            assert abs(float(got[j]) - float(want[j])) <= 1e-4 * max(1.0, abs(float(want[j]))), (cos, j, got[j], want[j])
        if cos:   # cosine of NaN vectors: aa/bb comparisons with NaN are false -> 0.0 per pair
            assert np.isnan(want[1]) == np.isnan(got[1]) and (np.isnan(want[1]) or got[1] == want[1]), (got[1], want[1])
        else:
            assert got[1] == want[1] == -np.inf, (got[1], want[1])


# ------------------------------------------------------------------------------------------------ sharding (K10)
@pytest.mark.parametrize("k", [10, 300])
def test_sharded_merge_on_one_gpu(ib, oracle, k):
    """The multi-rank path emulated as one process over all ranks' data (B200_PROFILING.md: never run ranks that wait
    on one another on one GPU): 3 contiguous row shards with index_base, local keys via *_keys_dev on torch's
    stream, concatenated as an allgather would, merged by merge_keys_kernel (k > 128: selection rounds over the
    gathered keys)."""
    import ctypes as C
    import torch
    from innr_b200 import _lib as L, sharded
    n, d, nq = 9001, 40, 5
    rng = np.random.default_rng(4)
    rows = rng.integers(-3, 4, size=(n, d)).astype(np.float32)   # heavy ties
    qs = rng.integers(-3, 4, size=(nq, d)).astype(np.float32)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    world = 3
    shards = []
    for r in range(world):
        lo, hi = sharded.shard_range(n, r, world)
        pdx = np.ascontiguousarray(rows[lo:hi].T).reshape(-1)
        shards.append(ib.DeviceBatch.from_pdx(pdx, hi - lo, d, index_base=lo))
    dq = torch.from_numpy(qs).cuda()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for metric, mid, single in (("dot", L.METRIC_DOT, "batch_knn_dot"), ("cosine", L.METRIC_COSINE, "batch_knn_cosine"),
                                ("l2", L.METRIC_L2, "batch_knn")):
        gathered = torch.empty(world * nq * k, dtype=torch.int64, device="cuda")
        for r, sh in enumerate(shards):
            L.call("innr_cuda_batch_knn_keys_dev", sh.h, mid, C.c_void_p(dq.data_ptr()), nq, k,
                   C.c_void_p(gathered[r * nq * k:].data_ptr()), stream)
        idx = torch.empty(nq * k, dtype=torch.int64, device="cuda")
        sc = torch.empty(nq * k, dtype=torch.float32, device="cuda")
        L.call("innr_cuda_merge_keys_dev", C.c_void_p(gathered.data_ptr()), world, nq, k, mid, None,
               C.c_void_p(idx.data_ptr()), C.c_void_p(sc.data_ptr()), stream)
        torch.cuda.synchronize()
        idx, sc = idx.cpu().numpy().reshape(nq, k), sc.cpu().numpy().reshape(nq, k)
        for j in range(nq):
            if metric == "l2":
                dist_all = oracle.batch_l2_squared(qs[j], ob)
                order = np.lexsort((np.arange(n), dist_all))[:k]
                assert idx[j].tolist() == order.tolist() and np.array_equal(bits(sc[j]), bits(dist_all[order]))
            else:
                w = getattr(oracle, single)(qs[j], ob, k)
                assert idx[j].tolist() == w.indices and np.array_equal(bits(sc[j]), bits(w.scores))
    # ShardedKnn (world size 1 when torch.distributed is not initialised) == the plain call
    sk = sharded.ShardedKnn(shards[0], "f32", "cosine")
    i1, s1 = sk.knn(qs, k)
    i2, s2 = ib.batch_knn_many("cosine", qs, shards[0], k)
    assert np.array_equal(i1, i2) and np.array_equal(bits(s1), bits(s2))


@pytest.mark.parametrize("k,nq", [(10, 5), (100, 2), (10, 70)])
def test_peer_exchange_emulated_on_one_gpu(ib, oracle, k, nq):
    """The peer-mapped exchange (csrc/exchange.cu) with all three ranks emulated on ONE device: ranks that are not the
    target publish only (ranks that wait on one another must not share a GPU), the target publishes, finds every flag
    raised, merges and decodes in the same launch. Every rank takes the target role, over several calls (both mailbox
    parities, slot reuse); nq = 70 spreads the queries over several CTAs."""
    import ctypes as C
    import torch
    from innr_b200 import _lib as L, sharded
    n, d, world = 6000, 32, 3
    rng = np.random.default_rng(5)
    rows = rng.integers(-3, 4, size=(n, d)).astype(np.float32)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    shards = []
    for r in range(world):
        lo, hi = sharded.shard_range(n, r, world)
        shards.append(ib.DeviceBatch.from_pdx(np.ascontiguousarray(rows[lo:hi].T).reshape(-1), hi - lo, d, index_base=lo))
    exs = [sharded.PeerExchange(world, r) for r in range(world)]
    sharded.PeerExchange.connect_local(exs)
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    for call, target in enumerate([2, 0, 1, 1, 0]):
        qs = rng.integers(-3, 4, size=(nq, d)).astype(np.float32)
        dq = torch.from_numpy(qs).cuda()
        loc = [torch.empty(nq * k, dtype=torch.int64, device="cuda") for _ in range(world)]
        for r in range(world):
            L.call("innr_cuda_batch_knn_keys_dev", shards[r].h, L.METRIC_COSINE, C.c_void_p(dq.data_ptr()), nq, k,
                   C.c_void_p(loc[r].data_ptr()), stream)
        idx = torch.empty(nq * k, dtype=torch.int64, device="cuda")
        sc = torch.empty(nq * k, dtype=torch.float32, device="cuda")
        for r in [x for x in range(world) if x != target] + [target]:
            exs[r].merge_dev(loc[r].data_ptr(), nq, k, L.METRIC_DOT, stream, idx=idx if r == target else None,
                             score=sc if r == target else None, publish_only=(r != target))
        torch.cuda.synchronize()
        assert exs[target].status() == 0
        idx_h, sc_h = idx.cpu().numpy().reshape(nq, k), sc.cpu().numpy().reshape(nq, k)
        for j in range(nq):
            w = oracle.batch_knn_cosine(qs[j], ob, k)
            assert idx_h[j].tolist() == w.indices and np.array_equal(bits(sc_h[j]), bits(w.scores)), (call, target, j)


def test_peer_exchange_times_out_instead_of_hanging(ib):
    """A rank whose peers never publish gives up after the timeout and reports it; nothing spins forever."""
    import ctypes as C
    import torch
    from innr_b200 import _lib as L, sharded
    exs = [sharded.PeerExchange(2, r) for r in range(2)]
    sharded.PeerExchange.connect_local(exs)
    exs[0].set_timeout_ms(50.0)
    loc = torch.zeros(10, dtype=torch.int64, device="cuda")
    idx = torch.empty(10, dtype=torch.int64, device="cuda")
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    exs[0].merge_dev(loc.data_ptr(), 1, 10, L.METRIC_DOT, stream, idx=idx)   # rank 1 never calls
    torch.cuda.synchronize()
    assert exs[0].status() == 1
    with pytest.raises(NotImplementedError):   # k > 128 and oversized requests are refused, not truncated
        exs[0].merge_dev(loc.data_ptr(), 1, 200, L.METRIC_DOT, stream, idx=idx)


@pytest.mark.parametrize("k", [10, 100, 300])
def test_keys_dev_shard_smaller_than_k(ib, oracle, k):
    """A shard that holds fewer rows than k (the last ranks of a small corpus): the `_dev` entries must still write
    n_queries x k rows, sentinel-padded (include/innr_cuda.h), so the gathered lists merge to the unsharded result --
    also for several queries at once and for k > 128 (selection rounds)."""
    import ctypes as C
    import torch
    from innr_b200 import _lib as L
    d, nq = 24, 3
    sizes = [7, 400, 3]   # two shards smaller than every k tested, one larger than k = 10 / 100 / 300
    n = sum(sizes)
    rng = np.random.default_rng(11)
    rows = rng.integers(-2, 3, size=(n, d)).astype(np.float32)
    qs = rng.integers(-2, 3, size=(nq, d)).astype(np.float32)
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    dq = torch.from_numpy(qs).cuda()
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    base, shards = 0, []
    for m in sizes:
        shards.append(ib.DeviceBatch.from_pdx(np.ascontiguousarray(rows[base:base + m].T).reshape(-1), m, d, index_base=base))
        base += m
    kk = min(k, n)
    for metric, mid, single in (("dot", L.METRIC_DOT, "batch_knn_dot"), ("cosine", L.METRIC_COSINE, "batch_knn_cosine")):
        gathered = torch.full((len(sizes) * nq * k,), 12345, dtype=torch.int64, device="cuda")  # poison: rows must be overwritten
        for r, sh in enumerate(shards):
            L.call("innr_cuda_batch_knn_keys_dev", sh.h, mid, C.c_void_p(dq.data_ptr()), nq, k,
                   C.c_void_p(gathered[r * nq * k:].data_ptr()), stream)
        idx = torch.empty(nq * k, dtype=torch.int64, device="cuda")
        sc = torch.empty(nq * k, dtype=torch.float32, device="cuda")
        L.call("innr_cuda_merge_keys_dev", C.c_void_p(gathered.data_ptr()), len(sizes), nq, k, mid, None,
               C.c_void_p(idx.data_ptr()), C.c_void_p(sc.data_ptr()), stream)
        torch.cuda.synchronize()
        g = gathered.cpu().numpy().view(np.uint64).reshape(len(sizes), nq, k)
        for r, m in enumerate(sizes):   # every row: min(k, m) keys then sentinels
            assert np.all(g[r, :, min(k, m):] == np.uint64(0xFFFFFFFFFFFFFFFF)), (metric, r)
            assert np.all(g[r, :, :min(k, m)] != np.uint64(0xFFFFFFFFFFFFFFFF)), (metric, r)
        idx, sc = idx.cpu().numpy().reshape(nq, k), sc.cpu().numpy().reshape(nq, k)
        for j in range(nq):
            w = getattr(oracle, single)(qs[j], ob, k)
            assert idx[j, :kk].tolist() == w.indices and np.array_equal(bits(sc[j, :kk]), bits(w.scores)), (metric, j)
    # the same contract on the Hamming and u8 entries
    codes = rng.integers(0, 2**63, size=(n, 4), dtype=np.uint64)
    qc = rng.integers(0, 2**63, size=(nq, 4), dtype=np.uint64)
    base, gathered = 0, torch.full((len(sizes) * nq * k,), 12345, dtype=torch.int64, device="cuda")
    dqc = torch.from_numpy(qc.view(np.int64)).cuda()
    keep = []
    for r, m in enumerate(sizes):
        sh = ib.BinaryCorpus.from_words(codes[base:base + m], m, 256, index_base=base)
        keep.append(sh)
        L.call("innr_cuda_hamming_topk_keys_dev", sh.h, C.c_void_p(dqc.data_ptr()), nq, k,
               C.c_void_p(gathered[r * nq * k:].data_ptr()), stream)
        base += m
    keys = torch.empty(nq * k, dtype=torch.int64, device="cuda")
    idx = torch.empty(nq * k, dtype=torch.int64, device="cuda")
    L.call("innr_cuda_merge_keys_dev", C.c_void_p(gathered.data_ptr()), len(sizes), nq, k, L.METRIC_L2,
           C.c_void_p(keys.data_ptr()), C.c_void_p(idx.data_ptr()), None, stream)
    torch.cuda.synchronize()
    idx = idx.cpu().numpy().reshape(nq, k)
    for j in range(nq):
        wi, wd = oracle.hamming_topk(qc[j], codes, k)
        assert idx[j, :kk].tolist() == wi.tolist(), j


def test_dev_entries_on_different_streams_do_not_share_the_workspace_unordered(ib, oracle):
    """`_dev` entries return while their kernels are still in flight on the CALLER's stream; the per-device workspace
    (partial lists, tickets) is ordered between streams by an event, so back-to-back calls on two streams, and a
    host-facing call right behind them, all give the single-call results."""
    import ctypes as C
    import torch
    from innr_b200 import _lib as L
    n, d, k, nq = 300_000, 64, 10, 1
    rows = rand_rows(n, d, 21)
    qs = rand_rows(4, d, 22)
    db = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    want = [ib.batch_knn_many("dot", qs[j], db, k) for j in range(4)]
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    dq = torch.from_numpy(qs).cuda()
    outs = [torch.empty(k, dtype=torch.int64, device="cuda") for _ in range(4)]
    torch.cuda.synchronize()
    for rep in range(20):
        for j, st in enumerate((s1, s2, s1, s2)):
            L.call("innr_cuda_batch_knn_keys_dev", db.h, L.METRIC_DOT, C.c_void_p(dq[j].data_ptr()), nq, k,
                   C.c_void_p(outs[j].data_ptr()), C.c_void_p(st.cuda_stream))
        host = ib.batch_knn_many("dot", qs[rep % 4], db, k)   # internal stream, right behind the asynchronous calls
        torch.cuda.synchronize()
        assert np.array_equal(host[0], want[rep % 4][0]) and np.array_equal(bits(host[1]), bits(want[rep % 4][1]))
        for j in range(4):
            keys = outs[j].cpu().numpy().view(np.uint64)
            assert (keys & np.uint64(0xFFFFFFFF)).tolist() == want[j][0][0].tolist(), (rep, j)


def test_two_lanes_overlapping_scans_of_every_kind(ib, oracle):
    """The fused k <= 128 scans of `_dev` entries may take either of the device's two workspaces (api.cu lanes), so
    independent scans on two caller streams really run concurrently. Every overlapped result must equal the one the
    same call gives alone -- whole 64-bit keys, every kind, 3 streams (more streams than lanes), a host-facing call and a
    lane-0-only call (k > 128) in between."""
    import ctypes as C
    import torch
    from innr_b200 import _lib as L
    n, d = 400_000, 96
    rows = rand_rows(n, d, 31)
    qs = rand_rows(6, d, 32)
    db = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    rng = np.random.default_rng(33)
    codes = rng.integers(0, 2**63, size=(n, 4), dtype=np.int64).view(np.uint64)
    bc = ib.BinaryCorpus.from_words(codes.reshape(-1), n, 256)
    qw = rng.integers(0, 2**63, size=(6, 4), dtype=np.int64)
    u8rows = rng.integers(0, 256, size=(n, d), dtype=np.uint8)
    uc = ib.U8Corpus.from_rows(u8rows, ib.QuantizationParams(0.01, -1.0))
    dq, dqw = torch.from_numpy(qs).cuda(), torch.from_numpy(qw).cuda()

    def f32(j, out, st, k=10):
        L.call("innr_cuda_batch_knn_keys_dev", db.h, L.METRIC_COSINE, C.c_void_p(dq[j].data_ptr()), 1, k,
               C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))

    def ham(j, out, st, k=100):
        L.call("innr_cuda_hamming_topk_keys_dev", bc.h, C.c_void_p(dqw[j].data_ptr()), 1, k,
               C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))

    def u8(j, out, st, k=10):
        L.call("innr_cuda_batch_knn_u8_keys_dev", uc.h, C.c_void_p(dq[j].data_ptr()), 1, k,
               C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))

    def f32_pair(j, out, st, k=10):   # two queries per call: the query-blocked scan / pair kernels on either lane
        L.call("innr_cuda_batch_knn_keys_dev", db.h, L.METRIC_DOT, C.c_void_p(dq[j % 5].data_ptr()), 2, k,
               C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))

    def ham_pair(j, out, st, k=100):
        L.call("innr_cuda_hamming_topk_keys_dev", bc.h, C.c_void_p(dqw[j % 5].data_ptr()), 2, k,
               C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))

    def u8_pair(j, out, st, k=10):
        L.call("innr_cuda_batch_knn_u8_keys_dev", uc.h, C.c_void_p(dq[j % 5].data_ptr()), 2, k,
               C.c_void_p(out.data_ptr()), C.c_void_p(st.cuda_stream))

    ib.set_option("knn_tc", 0)   # two f32 queries on 400 K rows would take the tensor-core filter (lane 0 only)
    try:
        kinds = [(f32, 10), (ham, 100), (u8, 10), (f32_pair, 20), (ham_pair, 200), (u8_pair, 20)]
        main = torch.cuda.current_stream()
        alone = {}
        for fn, k in kinds:
            for j in range(6):
                out = torch.empty(k, dtype=torch.int64, device="cuda")
                fn(j, out, main)
                torch.cuda.synchronize()
                alone[(fn, j)] = out.cpu().numpy().copy()
        big_alone = torch.empty(200, dtype=torch.int64, device="cuda")
        f32(0, big_alone, main, k=200)
        torch.cuda.synchronize()
        streams = [torch.cuda.Stream() for _ in range(3)]
        for rep in range(15):
            outs = []
            for i in range(18):
                fn, k = kinds[i % len(kinds)]
                j = (i + rep) % 6
                out = torch.empty(k, dtype=torch.int64, device="cuda")
                fn(j, out, streams[i % 3])
                outs.append((fn, j, out))
                if i == 7:   # k > 128 takes the scores pass + selection: lane 0 and the scratch buffers
                    big = torch.empty(200, dtype=torch.int64, device="cuda")
                    f32(0, big, streams[1], k=200)
                if i == 11:  # a host-facing call right in the middle
                    host = ib.batch_knn_many("cosine", qs[2], db, 10)
            torch.cuda.synchronize()
            for fn, j, out in outs:
                assert np.array_equal(out.cpu().numpy(), alone[(fn, j)]), (rep, fn.__name__, j)
            assert np.array_equal(big.cpu().numpy(), big_alone.cpu().numpy())
            assert (alone[(f32, 2)].view(np.uint64) & np.uint64(0xFFFFFFFF)).tolist() == host[0][0].tolist()
    finally:
        ib.set_option("knn_tc", 1)


def test_pipelined_single_rank_matches_knn_dev(ib):
    """ShardedKnn.knn_dev_pipelined on one rank (no exchange): scans alternate between two streams and the decode runs
    behind each; a run of different queries gives what knn_dev gives for each."""
    import torch
    from innr_b200 import sharded
    n, d = 300_000, 64
    rows = rand_rows(n, d, 41)
    qs = rand_rows(8, d, 42)
    db = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    rng = np.random.default_rng(43)
    bc = ib.BinaryCorpus.from_words(rng.integers(0, 2**63, size=n * 4, dtype=np.int64).view(np.uint64), n, 256)
    qw = torch.from_numpy(rng.integers(0, 2**63, size=(8, 4), dtype=np.int64)).cuda()
    dq = torch.from_numpy(qs).cuda()
    for sk, q, k in ((sharded.ShardedKnn(db, "f32", "cosine"), dq, 10), (sharded.ShardedKnn(db, "f32", "l2"), dq, 10),
                     (sharded.ShardedKnn(bc, "binary"), qw, 100)):
        want = []
        for j in range(8):
            idx, sc = sk.knn_dev(q[j], 1, k)
            want.append((idx.cpu().numpy().copy(), sc.cpu().numpy().copy()))
        got = []
        for j in range(8):
            idx, sc, ev = sk.knn_dev_pipelined(q[j], 1, k)
            assert ev is not None
            ev.synchronize()   # results are reused by the call after next: read them now
            got.append((idx.cpu().numpy().copy(), sc.cpu().numpy().copy()))
        for j in range(8):
            assert np.array_equal(got[j][0], want[j][0]) and np.array_equal(bits(got[j][1]), bits(want[j][1])), (sk.kind, j)
        # and without reading in between (the steady state of a throughput loop): the last two results are intact
        for j in range(8):
            last = sk.knn_dev_pipelined(q[j], 1, k)
        sk.drain()
        torch.cuda.synchronize()
        assert np.array_equal(last[0].cpu().numpy(), want[7][0])
        # host-buffer streaming: pinned queries in, pinned results out
        hq = q.cpu().pin_memory()
        pending, got = None, []
        for j in range(8):
            cur = sk.knn_dev_pipelined(None, 1, k, host_queries=hq[j], host_out=True)
            if pending is not None:
                pending[2].synchronize()
                got.append((pending[0].numpy().copy(), pending[1].numpy().copy()))
            pending = cur
        pending[2].synchronize()
        got.append((pending[0].numpy().copy(), pending[1].numpy().copy()))
        for j in range(8):
            assert np.array_equal(got[j][0], want[j][0]) and np.array_equal(bits(got[j][1]), bits(want[j][1])), (sk.kind, "host", j)


def test_async_host_calls_match_the_synchronous_ones(ib):
    """innr_cuda_*_async + innr_cuda_ticket_wait: two calls in flight per device, results bit-identical to the
    synchronous entries for every corpus kind (fused scans, the k > 128 path and the tensor-core filter path), a third
    submit is refused, empty results keep the reference's shape, a ticket is good for one wait."""
    from innr_b200 import stream
    n, d = 150_000, 64
    rows = rand_rows(n, d, 51)
    qs = rand_rows(6, d, 52)
    db = ib.DeviceBatch.from_rows_flat(rows.reshape(-1), n, d)
    rng = np.random.default_rng(53)
    bc = ib.BinaryCorpus.from_words(rng.integers(0, 2**63, size=n * 4, dtype=np.int64).view(np.uint64), n, 256)
    qw = rng.integers(0, 2**63, size=(6, 4), dtype=np.int64).view(np.uint64)
    uc = ib.U8Corpus.from_rows(rng.integers(0, 256, size=(n, d), dtype=np.uint8), ib.QuantizationParams(0.01, -1.0))

    def same(a, b):
        return np.array_equal(a[0], b[0]) and a[1].tobytes() == b[1].tobytes()

    calls = []
    for j in range(6):
        for metric in ("cosine", "dot", "l2"):
            calls.append((lambda j=j, m=metric: stream.submit_knn(m, qs[j], db, 10), lambda j=j, m=metric: ib.batch_knn_many(m, qs[j], db, 10)))
        calls.append((lambda j=j: stream.submit_hamming_topk(qw[j], bc, 100), lambda j=j: ib.hamming_topk_many(qw[j], bc, 100)))
        calls.append((lambda j=j: stream.submit_knn_u8(qs[j], uc, 10), lambda j=j: ib.batch_knn_u8_many(qs[j], uc, 10)))
    calls.append((lambda: stream.submit_knn("cosine", qs[0], db, 200), lambda: ib.batch_knn_many("cosine", qs[0], db, 200)))   # k > 128
    calls.append((lambda: stream.submit_knn("dot", qs[:4], db, 10), lambda: ib.batch_knn_many("dot", qs[:4], db, 10)))        # filter path
    calls.append((lambda: stream.submit_hamming_topk(qw[:2], bc, 100), lambda: ib.hamming_topk_many(qw[:2], bc, 100)))
    want = [sync() for _, sync in calls]
    pending, got = None, []
    for submit, _ in calls:
        t = submit()
        if pending is not None:
            got.append(pending.wait())
        pending = t
    got.append(pending.wait())
    for i, (g, w) in enumerate(zip(got, want)):
        assert same(g, w), i
    # two in flight, the third is refused until one of them has been collected
    t1 = stream.submit_knn("cosine", qs[0], db, 10)
    t2 = stream.submit_knn_u8(qs[1], uc, 10)
    with pytest.raises(ib.InnrCudaError):
        stream.submit_knn("cosine", qs[2], db, 10)
    assert same(t2.wait(), ib.batch_knn_u8_many(qs[1], uc, 10))   # any order
    t3 = stream.submit_knn("l2", qs[2], db, 10)
    assert same(t1.wait(), ib.batch_knn_many("cosine", qs[0], db, 10))
    assert same(t3.wait(), ib.batch_knn_many("l2", qs[2], db, 10))
    with pytest.raises(ib.InnrCudaError):
        t3.wait()
    # tickets dropped without a wait free their slots (two more submits go through)
    stream.submit_knn("cosine", qs[0], db, 10)
    stream.submit_knn("cosine", qs[1], db, 10)
    assert same(stream.submit_knn("cosine", qs[3], db, 10).wait(), ib.batch_knn_many("cosine", qs[3], db, 10))
    # k == 0 and an empty corpus: empty result, like the reference
    idx, sc = stream.submit_knn("dot", qs[0], db, 0).wait()
    assert idx.shape == (1, 0) and sc.shape == (1, 0)
    empty = ib.DeviceBatch.from_rows_flat(np.zeros(0, np.float32), 0, d)
    idx, sc = stream.submit_knn("dot", qs[0], empty, 5).wait()
    assert idx.shape == (1, 0)
    # a wrong query length is refused at submit, with the reference's message
    with pytest.raises(AssertionError):
        stream.submit_knn("dot", qs[0][:5], db, 3)


def test_kernel_timing_is_opt_in(ib):
    """innr_cuda_last_kernel_ms reports only after set_option("kernel_timing", 1): the timed event records are kept out
    of short calls by default (include/innr_cuda.h)."""
    from innr_b200 import _lib as L
    vb = ib.VerticalBatch.from_flat(rand_rows(2000, 32, 5).reshape(-1), 2000, 32)
    q = rand_rows(1, 32, 6)[0]
    L.set_option("kernel_timing", 0)
    ib.batch_knn_dot(q, vb, 5)
    before = ib.last_kernel_ms()
    L.set_option("kernel_timing", 1)
    try:
        ib.batch_knn_dot(q, vb, 5)
        assert ib.last_kernel_ms() > 0.0
        assert ib.last_kernel_ms() != before or before > 0.0
    finally:
        L.set_option("kernel_timing", 0)


def test_entries_leave_the_current_device_alone(ib):
    import torch
    before = torch.cuda.current_device()
    ib.batch_knn_dot(np.ones(4, np.float32), ib.VerticalBatch.from_flat(np.ones(8, np.float32), 2, 4), 1)
    assert torch.cuda.current_device() == before
    x = torch.ones(4, device="cuda") * 2   # torch still works on its own device after library calls
    assert float(x.sum()) == 8.0


# ------------------------------------------------------------------------------------------------ full BASELINE sizes
def _free_gb():
    import torch
    return torch.cuda.mem_get_info()[0] / 1e9


def test_full_size_c2a_properties(ib, oracle):
    """BASELINE C2a at full size (10M x 768, G-hash, generated on the device) through size-independent properties:
    every returned (index, score) is re-derived bit-exactly on the CPU from the stateless generator; results are
    sorted by (score desc, index asc); no sampled row outside the result beats the k-th score; and
    top-k(whole) == merge(top-k(first half), top-k(second half))."""
    from innr_b200 import synth, sharded
    if _free_gb() < 70:
        pytest.skip("needs ~62 GB of free HBM")
    n, d, k = 10_000_000, 768, 10
    whole = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d)
    q = oracle.ghash_f32(synth.SALT_QUERY, 0, d)
    for metric, single, desc in (("cosine", "batch_knn_cosine", True), ("l2", "batch_knn", False)):
        idx, sc = ib.batch_knn_many(metric, q, whole, k)
        idx, sc = idx[0], sc[0]
        rows = np.stack([oracle.ghash_f32(synth.SALT_CORPUS, int(i) * d, d) for i in idx])
        small = oracle.VerticalBatch.from_flat(rows.reshape(-1), k, d)
        want = oracle.batch_cosine(q, small, oracle.batch_norms(small)) if metric == "cosine" else oracle.batch_l2_squared(q, small)
        assert np.array_equal(bits(sc), bits(want)), metric
        keys = sharded.encode_keys(sc, idx, desc)
        assert np.all(keys[:-1] < keys[1:])
        rng = np.random.default_rng(1)
        sample = rng.integers(0, n, size=3000)
        srows = np.stack([oracle.ghash_f32(synth.SALT_CORPUS, int(i) * d, d) for i in sample])
        sb = oracle.VerticalBatch.from_flat(srows.reshape(-1), len(sample), d)
        ssc = oracle.batch_cosine(q, sb, oracle.batch_norms(sb)) if metric == "cosine" else oracle.batch_l2_squared(q, sb)
        skeys = sharded.encode_keys(ssc, sample, desc)
        inside = set(int(i) for i in idx)
        assert all(int(i) in inside for i, kk in zip(sample, skeys) if kk < keys[-1])
    halves = [ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, lo, n // 2, d, index_base=lo) for lo in (0, n // 2)]
    parts = [ib.batch_knn_many("cosine", q, h, k) for h in halves]
    merged = sharded.merge_keys_host(np.stack([sharded.encode_keys(p[1][0], p[0][0], True) for p in parts]), k)
    idx, sc = ib.batch_knn_many("cosine", q, whole, k)
    assert np.array_equal(merged, sharded.encode_keys(sc[0], idx[0], True))


def test_full_size_c2b_filter_properties(ib, oracle):
    """BASELINE C2b at full size (10M x 768, 1024 queries through the tcgen05 filter + exact rescoring): every list is
    sorted by (score desc, index asc); sampled entries are re-derived bit-exactly on the CPU; and for a handful of
    queries the whole list equals the bit-exact single-query scan (scores AND indices)."""
    from innr_b200 import synth, sharded
    if _free_gb() < 70:
        pytest.skip("needs ~50 GB of free HBM")
    n, d, k, nq = 10_000_000, 768, 10, 1024
    whole = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d)
    qs = oracle.ghash_f32(synth.SALT_QUERY, 0, nq * d).reshape(nq, d)
    rng = np.random.default_rng(3)
    for metric, desc in (("cosine", True), ("l2", False)):
        idx, sc = ib.batch_knn_many(metric, qs, whole, k)
        st = ib.knn_tc_last_stats()
        assert st["passes"] >= 2 and st["exact_scan_queries"] == 0, st
        assert idx.shape == (nq, k)
        for j in range(nq):
            keys = sharded.encode_keys(sc[j], idx[j], desc)
            assert np.all(keys[:-1] < keys[1:]), (metric, j)
        for j in rng.integers(0, nq, size=12):
            r = int(rng.integers(0, k))
            row = oracle.ghash_f32(synth.SALT_CORPUS, int(idx[j, r]) * d, d)
            one = oracle.VerticalBatch.from_flat(row, 1, d)
            want = (oracle.batch_cosine(qs[j], one, oracle.batch_norms(one)) if metric == "cosine"
                    else oracle.batch_l2_squared(qs[j], one))
            assert np.float32(sc[j, r]).tobytes() == np.float32(want[0]).tobytes(), (metric, j, r)
        ib.set_option("knn_tc", 0)
        try:
            for j in rng.integers(0, nq, size=4):
                si, ss = ib.batch_knn_many(metric, qs[j], whole, k)      # the bit-exact scan
                assert np.array_equal(si[0], idx[j]) and np.array_equal(bits(ss[0]), bits(sc[j])), (metric, j)
        finally:
            ib.set_option("knn_tc", 1)


def test_full_size_c3_maxsim_properties(ib, oracle):
    """BASELINE C3 at full size (1M docs x 180 tokens x 128d, 32 query tokens, generated on the device): a random sample
    of documents is re-scored by the oracle from the stateless generator (<= 1e-5 relative, the north-star tolerance),
    for maxsim_cosine and maxsim; two queries scored as a batch equal the single-query calls bit for bit."""
    from innr_b200 import synth
    if _free_gb() < 110:
        pytest.skip("needs ~94 GB of free HBM")
    n_docs, nt, dim, nq = 1_000_000, 180, 128, 32
    corpus = ib.TokenCorpus.generate(synth.SALT_CORPUS, 0, n_docs, nt, dim)
    qs = oracle.ghash_f32(synth.SALT_QUERY, 0, 2 * nq * dim).reshape(2, nq, dim)
    rng = np.random.default_rng(4)
    sample = np.concatenate([[0, n_docs - 1], rng.integers(0, n_docs, size=150)])
    off = np.arange(0, (len(sample) + 1) * nt, nt, dtype=np.uint64)
    toks = np.concatenate([oracle.ghash_f32(synth.SALT_CORPUS, int(dd) * nt * dim, nt * dim).reshape(nt, dim) for dd in sample])
    singles = {}
    for cos in (True, False):
        got = ib.maxsim_corpus(qs[0], corpus, cosine=cos)
        singles[cos] = got
        want = oracle.maxsim_corpus(qs[0], toks, off, cosine_flag=cos, n_threads=8)
        rel = np.abs(got[sample].astype(np.float64) - want) / np.maximum(np.abs(want), 1e-30)
        assert float(rel.max()) < 1e-5, (cos, float(rel.max()))
    both = ib.maxsim_corpus_batch(qs, corpus, cosine=True)
    assert np.array_equal(bits(both[0]), bits(singles[True]))
    assert np.array_equal(bits(both[1]), bits(ib.maxsim_corpus(qs[1], corpus, cosine=True)))


def test_full_size_c4_c5_properties(ib, oracle):
    """BASELINE C4 (100M x 1024-bit, top-100) and C5 (50M x 384 u8, top-10) at full size: every returned entry is
    re-derived bit-exactly on the CPU; order is (distance asc | score desc, index asc); a random sample holds no
    better candidate."""
    from innr_b200 import synth
    if _free_gb() < 40:
        pytest.skip("needs ~35 GB of free HBM")
    n, k = 100_000_000, 100
    corpus = ib.BinaryCorpus.generate(synth.SALT_CODES, 0, n, 1024)
    qc = oracle.ghash_u64(synth.SALT_QUERY, 0, 16)
    idx, ds = ib.hamming_topk(qc, corpus, k)
    want = [oracle.binary_hamming(oracle.PackedBinary(qc, 1024),
                                  oracle.PackedBinary(oracle.ghash_u64(synth.SALT_CODES, int(i) * 16, 16), 1024)) for i in idx]
    assert ds.tolist() == want
    keys = (ds.astype(np.uint64) << np.uint64(32)) | idx
    assert np.all(keys[:-1] < keys[1:])
    rng = np.random.default_rng(2)
    sample = rng.integers(0, n, size=20000)
    scodes = np.stack([oracle.ghash_u64(synth.SALT_CODES, int(i) * 16, 16) for i in sample])
    sd = np.array([bin(int(x)).count("1") for x in np.bitwise_xor(scodes, qc).reshape(-1)]).reshape(-1, 16).sum(1)
    skeys = (sd.astype(np.uint64) << np.uint64(32)) | sample.astype(np.uint64)
    inside = set(int(i) for i in idx)
    assert all(int(i) in inside for i, kk in zip(sample, skeys) if kk < keys[-1])
    del corpus

    n, d, k = 50_000_000, 384, 10
    gp, op = ib.QuantizationParams.from_range(-1.0, 1.0), oracle.QuantizationParams.from_range(-1.0, 1.0)
    c8 = ib.U8Corpus.generate(synth.SALT_CORPUS, 0, n, d, gp)
    q = oracle.ghash_f32(synth.SALT_QUERY, 0, d)
    got = ib.batch_knn_u8(q, c8, gp, k)
    for i, s in got:
        row = oracle.quantize_u8(oracle.ghash_f32(synth.SALT_CORPUS, i * d, d), op)
        assert np.float32(s).tobytes() == np.float32(oracle.asymmetric_dot_u8(q, row, op)).tobytes()
    assert all((got[j][1], -got[j][0]) > (got[j + 1][1], -got[j + 1][0]) for j in range(k - 1))


# ------------------------------------------------------------------------------------------------ tensor-core filter path
@pytest.fixture
def tc_small(ib):
    ib.set_option("knn_tc_min_n", 4096)       # exercise the tensor-core path at test sizes
    ib.set_option("knn_tc_min_queries", 1)
    yield ib
    ib.set_option("knn_tc_min_n", 100000)
    ib.set_option("knn_tc_min_queries", 2)


@pytest.mark.parametrize("n,d,nq", [(20_000, 768, 64), (50_000, 100, 40), (8_192, 32, 130), (33_000, 8, 33),
                                    (300_000, 64, 272), (120_000, 96, 9), (40_000, 200, 17), (70_000, 768, 1), (9_000, 48, 2),
                                    (25_000, 1000, 5)])
def test_knn_tc_filter_path_is_exact(tc_small, oracle, n, d, nq):
    """Large query batches go through tcgen05 as a pruning filter (csrc/knn_tc.cu); the exact rescoring must make the
    result bit-identical to the reference (indices AND scores), including zero / tiny / huge vectors and queries,
    duplicates (ties -> lower index first) and queries the filter hands to the exact scan. At these sizes (<= 300 K
    rows) the prefix schedule is short: the n/256 pass and, for k > 32, the n/128 pass never run. The schedule itself
    is covered at product shape by tests/test_gpu_knn_tc_passes.py."""
    ib = tc_small
    rows = rand_rows(n, d, n + d)
    rows[17] = 0.0                      # zero-norm vector -> cosine 0.0
    rows[100] = rows[200] = rows[300]   # exact duplicates -> ties -> lower index first
    rows[400:420] *= np.float32(1e-6)   # norms spread over many orders of magnitude (dot ranking != cosine ranking)
    rows[420:440] *= np.float32(1e5)
    rows[440] *= np.float32(1e-12)      # below the reference's 1e-9 cosine guard -> cosine 0.0, dot tiny
    rows[441] *= np.float32(1e-30)      # denormal range
    qs = rand_rows(nq, d, 99)
    if nq > 8:
        qs[3] = 0.0                     # zero-norm query -> every cosine 0.0 -> first k indices (exact-scan fallback)
        qs[5] = rows[300] * 2.0         # query parallel to the duplicates
        qs[6] *= np.float32(1e-12)      # below the cosine guard
        qs[7] *= np.float32(1e6)
        qs[8] = -rows[421]              # antiparallel to a huge vector
    elif nq > 1:
        qs[1] = rows[300] * 2.0
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for metric in ("cosine", "dot"):
        for k in (1, 10, 32, 100):
            idx, sc = ib.batch_knn_many(metric, qs, gb, k)
            st = ib.knn_tc_last_stats()
            assert st["passes"] >= 2 and (k > 32 or st["exact_scan_queries"] <= 4), st   # the filter really answered the batch
            widx, wsc = oracle.batch_knn_many(metric, qs, ob, k, n_threads=8)
            assert np.array_equal(idx, widx), (metric, k, np.argwhere(idx != widx)[:5])
            assert np.array_equal(bits(sc), bits(wsc)), (metric, k)
    # squared L2 (batch_knn, the TopK path: exact-tie groups compare as sets, SURVEY 8a row T)
    for k in (1, 10, 32, 100):
        idx, sc = ib.batch_knn_many("l2", qs, gb, k)
        st = ib.knn_tc_last_stats()
        assert st["passes"] >= 2 and (k > 32 or st["exact_scan_queries"] <= 4), st
        widx, wsc = oracle.batch_knn_many("l2", qs, ob, k, n_threads=8)
        assert np.array_equal(bits(sc), bits(wsc)), ("l2", k, np.argwhere(bits(sc) != bits(wsc))[:5])
        for j in range(nq):
            got_r = type("R", (), {"indices": [int(i) for i in idx[j]], "scores": sc[j]})
            want_r = type("R", (), {"indices": [int(i) for i in widx[j]], "scores": wsc[j]})
            assert_knn_equal(got_r, want_r, ties_as_sets=True)


def _half_ulp_unit_vector(d, rng, eta):
    """A UNIT vector of dimension d whose every component sits `eta` (in units of its binade, |eta| a hair off 2^-11 = half
    an f16 ulp) away from an f16-representable value, all on the same side: t_k = 2^-j (m_k + eta) with m_k = 1 + i_k 2^-10,
    i_k small -- mantissas near 1.0, where a half-ulp is the largest RELATIVE error f16 rounding can make. The i_k are
    chosen so that sum t_k^2 = 1 to ~1e-6, which keeps x / ||x|| (computed in f32 on the device) on the intended side of
    the rounding boundary. Returns the vector in float64 (random signs are the caller's business)."""
    J = int(np.ceil(np.log(d) / np.log(4.0))) + 1
    i0 = 0 if eta > 0 else 1                      # eta < 0: stay clear of the binade's lower edge (the ulp halves below it)
    unit = (1.0 + i0 * 2.0 ** -10 + eta) ** 2
    # every component starts at level J (one unit of 4^-J each); promoting a component 1 / 2 / 3 levels up adds 3 / 15 /
    # 63 units. Greedy change-making brings the squared norm to just below 1; >= 200 components stay at level J and
    # absorb the remainder (< 3 units) with a few mantissa steps each.
    extra = 4.0 ** J / unit - d
    lev = np.full(d, J)
    k = 0
    for up, gain in ((3, 63), (2, 15), (1, 3)):
        cnt = int(min(d - 200 - k, extra // gain))
        lev[k:k + cnt] = J - up
        k += cnt
        extra -= cnt * gain
    assert 0.0 <= extra < 3.0, (d, extra)
    a = k
    steps = np.full(d, i0, np.int64)

    def total():
        return float(np.sum(4.0 ** -lev * (1.0 + steps * 2.0 ** -10 + eta) ** 2))
    k = a  # bump the mantissas of the small components round-robin until the squared norm reaches 1
    while total() < 1.0:
        steps[k] += 1
        k = k + 1 if k + 1 < d else a
    assert steps.max() <= 12 and abs(total() - 1.0) < 8e-3 / d, (steps.max(), total())
    t = 2.0 ** -lev * (1.0 + steps * 2.0 ** -10 + eta)
    return t[rng.permutation(d)]


@pytest.mark.parametrize("d", [768, 4096, 12288])
def test_knn_tc_bound_holds_on_adversarial_inputs(ib, oracle, d):
    """The f16 tensor-core filter may only prune what its bound allows: for every (query, row) pair the reference's score
    must lie inside [lower, lower + 2 e] as the filter computes it (csrc/knn_tc.cu; eps = 1.05e-3 + 3.5e-7 d). Driven
    with inputs built to maximise the f16 rounding error -- every normalised component a hair off a half-ulp boundary
    with aligned signs, parallel and antiparallel to the query (where Cauchy-Schwarz is tight) -- plus f16-subnormal
    components, norms from 1e-30 to 1e18 and random rows, for all three metrics. Reports the worst |S r - ref| / e."""
    rng = np.random.default_rng(d)
    n = 4096
    rows = np.zeros((n, d), np.float64)
    half_ulp = 2.0 ** -11
    etas = [half_ulp - 2.0 ** -15, half_ulp + 2.0 ** -15, -(half_ulp - 2.0 ** -15), 3 * half_ulp - 2.0 ** -15]
    qvecs = []
    for e_i, eta in enumerate(etas):
        x = _half_ulp_unit_vector(d, rng, eta)
        qvecs.append(x.copy())
        base = e_i * 64
        for r in range(64):
            y = x.copy()
            if r % 4 == 1:
                y = -y                                     # antiparallel: cos = -1
            if r % 4 == 2:
                sgn = rng.choice([-1.0, 1.0], size=d)      # same magnitudes, random signs: the errors partly cancel
                y = y * sgn
            if r % 4 == 3:
                y[rng.permutation(d)[: d // 2]] *= 2.0 ** -9   # half of the components become f16-subnormal after normalisation
            rows[base + r] = y * 10.0 ** rng.uniform(-3, 3)
    # norms spanning 1e-30 .. 1e30, heavy-tailed components, and plain Gaussian rows
    k0 = 64 * len(etas)
    # (1e18 is as far up as f32 goes here: the squared norm must stay finite, or the reference's own score is NaN and
    # the corpus never takes the filter path)
    rows[k0:k0 + 512] = rng.standard_normal((512, d)) * (10.0 ** rng.uniform(-30, 18, size=(512, 1)) / np.sqrt(d))
    rows[k0 + 512:k0 + 1024] = rng.standard_normal((512, d)) * np.exp(rng.standard_normal((512, d)) * 4.0)
    rows[k0 + 1024:] = rng.standard_normal((n - k0 - 1024, d))
    rows[k0 + 1030] = 0.0
    rows32 = rows.astype(np.float32)
    qs = np.stack(qvecs + [-qvecs[0], rows[k0 + 1500], rows[k0 + 1501] * 1e15, rows[k0 + 700] * 1e-3]).astype(np.float32)
    nq = qs.shape[0]
    gb = ib.VerticalBatch.from_flat(rows32.reshape(-1), n, d)
    ob = oracle.VerticalBatch.from_flat(rows32.reshape(-1), n, d)
    norms = oracle.batch_norms(ob)
    assert np.isfinite(norms).all()
    f32 = np.float32
    worst = {}
    for metric in ("cosine", "dot", "l2"):
        lower, eps, flags = ib.knn_tc_debug_bounds(metric, qs, gb)
        assert lower.shape == (nq, n) and abs(eps - (1.05e-3 + 3.5e-7 * d)) < 1e-9 and not flags.any()
        for j in range(nq):
            q = qs[j]
            qn = f32(np.sqrt(f32(oracle.batch_dot(q, oracle.VerticalBatch.from_flat(q, 1, d))[0])))
            if metric == "cosine":
                ref = oracle.batch_cosine(q, ob, norms).astype(np.float64)
                e = np.where(norms > 1e-9, eps, 0.0)
                lo, hi = lower[j].astype(np.float64), lower[j].astype(np.float64) + 2 * e
            elif metric == "dot":
                ref = oracle.batch_dot(q, ob).astype(np.float64) / float(qn)        # the filter's units: score / ||q||
                r = np.where(norms >= 1e-30, norms, 0.0).astype(np.float64)
                e = eps * r + 1e-18
                lo, hi = lower[j].astype(np.float64), lower[j].astype(np.float64) + 2 * e
            else:
                dist = oracle.batch_l2_squared(q, ob).astype(np.float64)
                ref = (float(qn) ** 2 - dist) / (2 * float(qn))                       # u = (||q||^2 - d) / (2 ||q||)
                r = np.where(norms >= 1e-30, norms, 0.0).astype(np.float64)
                e = eps * r + 1e-18
                delta = (4.0 * d + 32.0) * 2.0 ** -24
                cq = 2.0 * (d + 2.0) * 2.0 ** -24 * float(qn)
                xx = norms.astype(np.float64) ** 2
                h = 0.5 / float(qn)
                lo = lower[j].astype(np.float64)
                hi = lo + 2 * e + xx * h * 2 * delta + 2 * cq                         # upper(j) + cq in the kernel's terms
            slack = 1e-6 * (np.abs(lo) + np.abs(hi)) + 1e-30                          # f32 rounding of the bounds themselves
            bad = (ref < lo - slack) | (ref > hi + slack)
            assert not bad.any(), (metric, j, int(np.argmax(bad)), ref[bad][:3], lo[bad][:3], hi[bad][:3])
            mid, half = 0.5 * (lo + hi), 0.5 * (hi - lo)
            ratio = np.where(half > 0, np.abs(ref - mid) / np.maximum(half, 1e-300), 0.0)
            worst[metric] = max(worst.get(metric, 0.0), float(ratio.max()))
            if metric == "cosine":
                worst["cosine_abs"] = max(worst.get("cosine_abs", 0.0), float(np.abs(ref - mid).max()))
    print(f"d={d}: eps = {eps:.3e}; worst |S r - ref| / e = {worst}")
    # the construction really is adversarial: the half-ulp rows reach (almost) the whole f16 budget of 2^-10 = 9.77e-4
    assert worst["cosine_abs"] > 8.5e-4, worst
    assert max(worst["cosine"], worst["dot"], worst["l2"]) <= 1.0


def test_knn_tc_candidate_overflow_falls_back_to_the_exact_scan(tc_small, oracle):
    """300 000 rows that all lie inside the filter's error band of the best score (a cloud of near-duplicates around the
    query direction) at k = 128: every row is a candidate, the per-query list (4096 slots) overflows, and the query must
    be answered by the exact scan -- still bit for bit."""
    ib = tc_small
    n, d, k = 300_000, 64, 128
    rng = np.random.default_rng(77)
    u = rng.standard_normal(d)
    u /= np.linalg.norm(u)
    rows = (u[None, :] + 2e-4 * rng.standard_normal((n, d))).astype(np.float32)   # cos(u, row) = 1 - O(1e-6): all within eps
    qs = np.stack([u, 3.0 * u, u + 1e-3 * rng.standard_normal(d)]).astype(np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for metric in ("cosine", "dot", "l2"):
        idx, sc = ib.batch_knn_many(metric, qs, gb, k)
        st = ib.knn_tc_last_stats()
        assert st["passes"] >= 2 and st["exact_scan_queries"] == qs.shape[0], (metric, st)   # every list overflowed
        widx, wsc = oracle.batch_knn_many(metric, qs, ob, k, n_threads=8)
        assert np.array_equal(bits(sc), bits(wsc)), metric
        if metric != "l2":
            assert np.array_equal(idx, widx), metric


def test_knn_tc_on_the_reference_lattice(tc_small, oracle):
    """The G-ref lattice (SURVEY.md F11) has near-ties below f32 resolution: the adversarial case for a low-precision
    filter (many pairs inside the error band -> long candidate lists or the exact-scan fallback; never a wrong answer)."""
    ib = tc_small
    n, d, nq, k = 30_000, 128, 64, 10
    dev = ib.DeviceBatch.generate("gref", 0, 0, n, d)
    rows = np.stack([oracle.generate_embedding(d, i) for i in range(n)])
    ob = oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    qs = np.stack([oracle.generate_embedding(d, 50_000 + j) for j in range(nq)])
    for metric in ("dot", "cosine"):
        idx, sc = ib.batch_knn_many(metric, qs, dev, k)
        widx, wsc = oracle.batch_knn_many(metric, qs, ob, k, n_threads=8)
        assert np.array_equal(idx, widx) and np.array_equal(bits(sc), bits(wsc)), metric


def test_knn_tc_non_finite_inputs_fall_back_to_the_exact_scan(tc_small, oracle):
    """A corpus with a non-finite norm never takes the filter path; a non-finite query is answered by the exact scan.
    Scores compare with same_scores (NaN sign is not portable, DESIGN.md)."""
    ib = tc_small
    n, d, nq, k = 9_000, 48, 40, 10
    rows = rand_rows(n, d, 5)
    qs = rand_rows(nq, d, 6)
    qs[2, 7] = np.inf
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    idx, sc = ib.batch_knn_many("dot", qs, gb, k)
    assert ib.knn_tc_last_stats()["exact_scan_queries"] == 1
    widx, wsc = oracle.batch_knn_many("dot", qs, ob, k, n_threads=8)
    fin = np.isfinite(wsc).all(axis=1)
    assert np.array_equal(idx[fin], widx[fin]) and same_scores(sc, wsc)
    rows[123, 4] = np.inf               # corpus with a non-finite vector: exact scan for everything
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    qs = rand_rows(nq, d, 7)
    idx, sc = ib.batch_knn_many("dot", qs, gb, k)   # +-inf scores order identically everywhere (cosine would be NaN)
    widx, wsc = oracle.batch_knn_many("dot", qs, ob, k, n_threads=8)
    assert np.array_equal(idx, widx) and same_scores(sc, wsc)


# ---------------------------------------------------------------------------------------------------------
# batch_dimension_variance / batch_knn_reordered (src/batch.rs:572-659): bit-exact variances (two sequential f32 sums
# per dimension row), the same variance order, and distances summed in that order; ties -> lower index
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("n,d", [(2, 1), (3, 5), (127, 8), (128, 9), (129, 16), (511, 33), (512, 7), (513, 64), (3000, 40),
                                 (20000, 24)])
def test_dimension_variance_bit_exact(ib, oracle, n, d):
    rng = np.random.default_rng(n * 131 + d)
    rows = (rng.standard_normal((n, d)) * rng.uniform(0.1, 3.0, size=d) + rng.uniform(-2, 2, size=d)).astype(np.float32)
    if d > 2:
        rows[:, 1] = 0.25          # constant row: variance exactly 0
        rows[:, 2] = rows[:, 0]    # duplicate row: equal variances -> the stable order keeps the lower dimension first
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    g, w = ib.batch_dimension_variance(gb), oracle.batch_dimension_variance(ob)
    assert np.array_equal(bits(g), bits(w)), (n, d)


def test_dimension_variance_non_finite(ib, oracle):
    rng = np.random.default_rng(5)
    rows = rng.standard_normal((700, 6)).astype(np.float32)
    rows[13, 0] = np.inf      # mean inf -> x - mean = NaN for that row
    rows[600, 1] = np.nan
    rows[:, 2] = 3.0e38       # the sum overflows to +inf
    rows[5, 3] = -0.0
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), 700, 6), oracle.VerticalBatch.from_flat(rows.reshape(-1), 700, 6)
    assert same_scores(ib.batch_dimension_variance(gb), oracle.batch_dimension_variance(ob))


@pytest.mark.parametrize("n,d", [(1, 3), (5, 2), (1000, 16), (1025, 37), (4097, 128), (30000, 48)])
def test_knn_reordered_bit_exact(ib, oracle, n, d):
    rng = np.random.default_rng(n + 7 * d)
    rows = (rng.standard_normal((n, d)) * rng.uniform(0.05, 4.0, size=d)).astype(np.float32)
    q = rng.standard_normal(d).astype(np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for k in (1, 10, 33, 128, 200, n + 3):
        g, w = ib.batch_knn_reordered(q, gb, k), oracle.batch_knn_reordered(q, ob, k)
        assert g.indices == w.indices, (n, d, k)
        assert np.array_equal(bits(g.scores), bits(w.scores)), (n, d, k)
    # summed in another order than batch_knn: same neighbours, scores equal up to rounding (reference's own check)
    g, e = ib.batch_knn_reordered(q, gb, 5), ib.batch_knn(q, gb, 5)
    assert np.allclose(g.scores, e.scores, rtol=1e-5)


def test_knn_reordered_ties_and_equal_variances(ib, oracle):
    rng = np.random.default_rng(17)
    n, d = 5000, 12
    rows = rng.integers(-1, 2, size=(n, d)).astype(np.float32)   # few distinct distances: ties everywhere
    rows[:, 5] = rows[:, 4]                                       # equal variances
    q = rng.integers(-1, 2, size=d).astype(np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for k in (7, 100, 300):
        g, w = ib.batch_knn_reordered(q, gb, k), oracle.batch_knn_reordered(q, ob, k)
        assert g.indices == w.indices and np.array_equal(bits(g.scores), bits(w.scores)), k
    assert ib.batch_knn_reordered(q, gb, 0).indices == []
    with pytest.raises(AssertionError):
        ib.batch_knn_reordered(q[:-1], gb, 3)


# ---------------------------------------------------------------------------------------------------------
# batch_knn_adaptive (src/batch.rs:441-564): the approximate heuristic reproduced exactly -- survivors, complete
# distances and order -- in every regime: thresholds that prune nothing, that prune most candidates, and that would
# prune below k (the reference's `alive_count > k` guard then depends on the (dimension, index) visiting order)
# ---------------------------------------------------------------------------------------------------------
def _adaptive_case(rng, kind, n, d):
    if kind == "gauss":            # flat spectrum: the extrapolated threshold is too tight, the guard binds
        rows = rng.standard_normal((n, d))
    elif kind == "mrl":            # decaying spectrum (Matryoshka-like): early dimensions carry the distance
        rows = rng.standard_normal((n, d)) * (0.97 ** np.arange(d))
    elif kind == "rising":         # later dimensions carry more than the warm-up suggests
        rows = rng.standard_normal((n, d)) * np.linspace(0.2, 2.0, d)
    elif kind == "planted":        # ten uniform-offset neighbours of the origin among far vectors: pruning is benign
        rows = rng.integers(50, 100, size=(n, d)) * rng.choice([-1, 1], size=(n, d))
        for j in range(min(10, n)):
            rows[(j * 37) % n] = j + 1
    else:                          # integer lattice: exact ties in partial and complete distances
        rows = rng.integers(-2, 3, size=(n, d))
    return rows.astype(np.float32)


@pytest.mark.parametrize("kind", ["gauss", "mrl", "rising", "ties", "planted"])
@pytest.mark.parametrize("n,d", [(1, 5), (7, 3), (300, 40), (5000, 96), (4097, 130), (20000, 64)])
def test_knn_adaptive_bit_exact(ib, oracle, kind, n, d):
    rng = np.random.default_rng(n * 17 + d)
    rows = _adaptive_case(rng, kind, n, d)
    q = _adaptive_case(rng, kind, 1, d)[0] if kind != "planted" else np.zeros(d, np.float32)
    gb, ob = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d), oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d)
    for k in (1, 10, 100, 150, n, n + 5):
        for w in (1, 8, 31, 32, 33, d, d + 9):
            g, want = ib.batch_knn_adaptive(q, gb, k, w), oracle.batch_knn_adaptive(q, ob, k, w)
            assert g.indices == want.indices, (kind, n, d, k, w, g.indices[:6], want.indices[:6])
            assert np.array_equal(bits(g.scores), bits(want.scores)), (kind, n, d, k, w)


def test_knn_adaptive_regimes_are_exercised(ib, oracle):
    """The cases above must cover both outcomes: adaptive == exact kNN (benign pruning) and adaptive != exact kNN (true
    neighbours pruned, the documented failure mode) -- otherwise the parity test proves less than it claims."""
    rng = np.random.default_rng(3)
    n, d, k = 5000, 96, 10
    same = differ = 0
    for kind in ("gauss", "planted"):
        rows = _adaptive_case(rng, kind, n, d)
        q = _adaptive_case(rng, kind, 1, d)[0] if kind != "planted" else np.zeros(d, np.float32)
        gb = ib.VerticalBatch.from_flat(rows.reshape(-1), n, d)
        a, e = ib.batch_knn_adaptive(q, gb, k, 8), ib.batch_knn(q, gb, k)
        same += a.indices == e.indices
        differ += a.indices != e.indices
    assert same >= 1 and differ >= 1, (same, differ)
    with pytest.raises(AssertionError):
        ib.batch_knn_adaptive(np.zeros(d, np.float32), gb, k, 0)
    with pytest.raises(AssertionError):
        ib.batch_knn_adaptive(np.zeros(d - 1, np.float32), gb, k, 4)
