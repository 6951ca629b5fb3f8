"""dev: binary top-k query batches at C4 size (100M x 1024 bit, generated codes), the tensor-core filter (bin_tc.cu)
against the CUDA-core route (option bin_tc = 0: the 4-query / 2-query Hamming kernels, one scan per query for dot and
Jaccard), alternated in one process, outputs asserted equal. Hamming at nq = 2 .. 1024 and k = 10, 100; dot and Jaccard
at a few points.

Per (op, k, nq): device ms of a `_keys_dev` call on device-resident queries (CUDA events around the call on its stream,
median of the rounds), and for the filter its statistics (bin_tc_last_stats): candidates per query, overflowed queries,
passes, final-pass ms and the integer ops/s of that pass against the data sheet's dense INT8 rate. Writes a JSON file
(default profiles/r07a_bin_tc.json) with the card's name and power limit, read in the same run.

    python innr_b200/csrc/dev/bin_tc_bench.py [--out FILE] [--rounds R] [--n N]
"""
import argparse
import ctypes as C
import json
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import innr_b200 as ib  # noqa: E402
from innr_b200 import _lib as L  # noqa: E402

DENSE_INT8_TOPS = 4500.0  # HGX B200 data sheet, one GPU, dense (a sixteenth of the 8-GPU sparse figure), 1000 W card
OPS = {"hamming": None, "dot": 0, "jaccard": 1}


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[0] if out else "unknown"


def keys_dev(corpus, op, dq, k, out):
    s = torch.cuda.current_stream().cuda_stream
    if OPS[op] is None:
        L.call("innr_cuda_hamming_topk_keys_dev", corpus.h, C.c_void_p(dq.data_ptr()), dq.shape[0], k,
               C.c_void_p(out.data_ptr()), C.c_void_p(s))
    else:
        L.call("innr_cuda_binary_topk_keys_dev", corpus.h, OPS[op], C.c_void_p(dq.data_ptr()), dq.shape[0], k,
               C.c_void_p(out.data_ptr()), C.c_void_p(s))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="profiles/r07a_bin_tc.json")
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--n", type=int, default=100_000_000)
    args = ap.parse_args()
    ib.init(0)
    ib.set_option("bin_tc_min_n", 0)
    ib.set_option("bin_tc_min_queries", 2)
    ib.set_option("bin_tc_max_k", 128)
    n, dim = args.n, 1024
    corpus = ib.BinaryCorpus.generate(0xC4C4, 0, n, dim)
    rng = np.random.default_rng(0xC4)
    words = rng.integers(0, 2**64, size=(1024, dim // 64), dtype=np.uint64).view(np.int64)
    dq_all = torch.from_numpy(words).cuda()
    plan = [("hamming", k, nq) for k in (10, 100) for nq in (2, 8, 16, 32, 64, 256, 1024)]
    plan += [(op, 10, nq) for op in ("dot", "jaccard") for nq in (8, 64, 1024)]
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    rows = []
    for op, k, nq in plan:
        dq = dq_all[:nq]
        times = {"cuda_cores": [], "tc": []}
        res, st = {}, None
        for r in range(args.rounds + 1):  # round 0 warms up (popcounts, module load, workspace growth)
            for p in times:
                ib.set_option("bin_tc", 1 if p == "tc" else 0)
                out = torch.empty(nq * k, dtype=torch.int64, device="cuda")
                ev0.record()
                keys_dev(corpus, op, dq, k, out)
                ev1.record()
                torch.cuda.synchronize()
                if r:
                    times[p].append(ev0.elapsed_time(ev1))
                if p == "tc":
                    st = L.bin_tc_last_stats()
                got = out.cpu().numpy()
                if p in res:
                    assert np.array_equal(got, res[p])
                res[p] = got
        ib.set_option("bin_tc", 1)
        equal = bool(np.array_equal(res["tc"], res["cuda_cores"]))
        assert equal, (op, k, nq)
        row = {"op": op, "k": k, "nq": nq, **{f"{p}_ms": float(np.median(t)) for p, t in times.items()},
               "outputs_equal": equal}
        row["speedup"] = row["cuda_cores_ms"] / row["tc_ms"]
        row.update({"candidates_per_query": st["candidates"] / nq, "exact_scan_queries": st["exact_scan_queries"],
                    "passes": st["passes"], "final_pass_ms": st["filter_ms"], "filter_call_ms": st["total_ms"],
                    "final_pass_int_tops": st["filter_ops"] / (st["filter_ms"] * 1e-3) / 1e12})
        row["final_pass_share_of_dense_int8"] = row["final_pass_int_tops"] / DENSE_INT8_TOPS
        print(json.dumps(row), flush=True)
        rows.append(row)
    doc = {"card": card(), "corpus": f"{n} x {dim} bit (innr_cuda_generate_binary)", "rounds": args.rounds,
           "timing": "median device time (CUDA events on the calling stream) of a _keys_dev call on device-resident "
                     "queries; the first round of each point is a warm-up",
           "dense_int8_tops_datasheet": DENSE_INT8_TOPS, "rows": rows}
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)
    print("card:", doc["card"])


if __name__ == "__main__":
    main()
