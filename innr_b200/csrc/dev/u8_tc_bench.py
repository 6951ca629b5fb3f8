"""dev: batch_knn_u8 at C5 size (50M x 384, ghash codes), the tensor-core filter (u8_tc.cu) against the exact scan
(single-query / pair kernels), alternated in one process, outputs asserted equal. k = 10 and 100, nq = 1 .. 1024.

Per (k, nq): ms per synchronous call (median of the rounds, host clock around a call that ends in a device sync), and for
the filter its statistics (u8_tc_last_stats): candidates per query, final-pass ms and integer ops/s of that pass against
the data sheet's dense INT8 rate. Writes a JSON file (default profiles/r06a_u8_tc.json) with the card's name and power
limit.

    python innr_b200/csrc/dev/u8_tc_bench.py [--out FILE] [--rounds R]
"""
import argparse
import json
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, ".")
import innr_b200 as ib  # noqa: E402
from innr_b200 import _lib as L, synth  # noqa: E402

DENSE_INT8_TOPS = 4500.0  # HGX B200 data sheet, one GPU, dense (a sixteenth of the 8-GPU sparse figure), 1000 W card


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r06a_u8_tc.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--n", type=int, default=50_000_000)
    args = ap.parse_args()
    ib.init(0)
    ib.set_option("u8_tc_min_n", 0)
    ib.set_option("u8_tc_min_queries", 2)
    ib.set_option("u8_tc_max_k", 128)  # measure the filter at k = 100 too (the default sends k > 32 to the scan)
    n, d = args.n, 384
    corpus = ib.U8Corpus.generate(synth.SALT_CORPUS, 0, n, d, ib.QuantizationParams.from_range(-1.0, 1.0))
    qs_all = synth.ghash_f32(synth.SALT_QUERY, 0, 1024 * d).reshape(1024, d)
    rows = []
    for k in (10, 100):
        for nq in (1, 2, 8, 64, 256, 1024):
            qs = qs_all[:nq]
            paths = ("scan",) if nq == 1 else ("scan", "tc")
            times = {p: [] for p in paths}
            res, st = {}, None
            for r in range(args.rounds + 1):  # round 0 warms up (radius sidecar, module load, workspace growth)
                for p in paths:
                    ib.set_option("u8_tc", 1 if p == "tc" else 0)
                    t0 = time.perf_counter()
                    out = ib.batch_knn_u8_many(qs, corpus, k)
                    dt = (time.perf_counter() - t0) * 1e3
                    if r:
                        times[p].append(dt)
                    if p == "tc":
                        st = L.u8_tc_last_stats()
                    if p in res:
                        assert np.array_equal(out[0], res[p][0]) and out[1].tobytes() == res[p][1].tobytes()
                    res[p] = out
            if "tc" in res:
                assert np.array_equal(res["tc"][0], res["scan"][0]) and res["tc"][1].tobytes() == res["scan"][1].tobytes(), (k, nq)
            row = {"k": k, "nq": nq, **{f"{p}_ms": float(np.median(t)) for p, t in times.items()}}
            if st:
                row.update({"candidates_per_query": st["candidates"] / nq, "exact_scan_queries": st["exact_scan_queries"],
                            "passes": st["passes"], "final_pass_ms": st["filter_ms"], "filter_call_ms": st["total_ms"],
                            "final_pass_int_tops": st["filter_ops"] / (st["filter_ms"] * 1e-3) / 1e12})
                row["final_pass_share_of_dense_int8"] = row["final_pass_int_tops"] / DENSE_INT8_TOPS
            print(json.dumps(row), flush=True)
            rows.append(row)
    ib.set_option("u8_tc", 1)
    doc = {"card": card(), "corpus": f"{n} x {d} u8 (ghash, from_range(-1, 1))", "rounds": args.rounds,
           "timing": "median host wall time of a synchronous batch_knn_u8 call (queries up, keys down included)",
           "dense_int8_tops_datasheet": DENSE_INT8_TOPS, "rows": rows}
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("card:", doc["card"])


if __name__ == "__main__":
    main()
