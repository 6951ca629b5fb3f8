"""bench.py --dump-outputs: what the last timed step returned, written as .npy files that two builds can compare."""
import os
import subprocess
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_dump_outputs_dtypes_and_seeded_sample(tmp_path):
    n = bench.DUMP_SAMPLE + 12345
    scores = np.arange(n, dtype=np.float32)
    bench.dump_outputs(str(tmp_path), "w", {"indices": np.array([[3, 1 << 40]], np.int64), "scores": scores,
                                            "dist": np.array([7, 9], np.int32)})
    idx = np.load(tmp_path / "w_indices.npy")
    assert idx.dtype == np.float64 and idx.tolist() == [[3.0, float(1 << 40)]]
    dist = np.load(tmp_path / "w_dist.npy")
    assert dist.dtype == np.float64 and dist.tolist() == [7.0, 9.0]
    got, pos = np.load(tmp_path / "w_scores.npy"), np.load(tmp_path / "w_scores_positions.npy")
    assert got.dtype == np.float32 and got.size == bench.DUMP_SAMPLE and np.all(np.diff(pos) > 0)
    assert np.array_equal(got, scores[pos.astype(np.int64)])
    bench.dump_outputs(str(tmp_path / "again"), "w", {"scores": scores})   # same positions on every run
    assert np.array_equal(np.load(tmp_path / "again" / "w_scores_positions.npy"), pos)
    assert not os.path.exists(tmp_path / "w_indices_positions.npy")


def test_dump_outputs_is_refused_where_it_would_write_nothing():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--dump-outputs", "x"],
                       capture_output=True, text=True, timeout=120)
    assert r.returncode != 0 and "--dump-outputs" in r.stderr
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"], capture_output=True, text=True,
                       timeout=120)
    assert r.returncode != 0 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_of_the_timed_path(tmp_path, oracle):
    """C1 (batch_demo) at 1000 rows: the dumped last step is the oracle's top-10 of the bench's own inputs, bit for bit."""
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--workload", "batch_demo", "--scale", "0.1",
                        "--steps", "4", "--warmup", "3", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert sorted(os.listdir(tmp_path)) == ["batch_demo_indices.npy", "batch_demo_scores.npy"]
    n, d = 1000, 128
    rows = np.stack([oracle.generate_embedding(d, i) for i in range(n)])
    qs = np.stack([oracle.generate_embedding(d, 50_000 + j) for j in range(100)])
    want_idx, want_sc = oracle.batch_knn_many("dot", qs, oracle.VerticalBatch.from_flat(rows.reshape(-1), n, d), 10)
    idx, sc = np.load(tmp_path / "batch_demo_indices.npy"), np.load(tmp_path / "batch_demo_scores.npy")
    assert idx.shape == (100, 10) and np.array_equal(idx, want_idx.astype(np.float64))
    assert sc.dtype == np.float32 and sc.tobytes() == np.ascontiguousarray(want_sc, np.float32).tobytes()
