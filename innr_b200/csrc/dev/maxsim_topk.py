"""dev: what MaxSim top-k costs over the score vector it ranks, at the C3 document shape (180 tokens x 128, cosine,
32 query tokens, G-hash tokens generated on the device).

* 1,000,000 documents (the whole C3 corpus, 92 GB) and 125,000 documents (one 8-GPU shard): innr_cuda_maxsim_dev
  against innr_cuda_maxsim_topk_keys_dev for k = 10, 100, 1000, interleaved over several rounds (CUDA events over many
  launches after warm-up); the selection's device time per call from torch.profiler in a run of its own (kernel
  topk_scores_kernel, one launch per 128 results), and its share of the top-k call;
* a batch of 64 queries: innr_cuda_maxsim_batch_dev against innr_cuda_maxsim_topk_keys_dev (k = 10, 100);
* the host entries end to end (host clock, each call synchronises): innr_cuda_maxsim (n_docs floats to the host) plus
  a stable descending sort there, against innr_cuda_maxsim_topk (k = 10);
* the in-process sharded entry over every GPU of the box (one shard of 1M / n_gpus documents per device): ms per call
  and bit-equality with the unsharded call.
The GPU's name, power limit and max SM clock are read in the same run. Writes one JSON.
Usage: python innr_b200/csrc/dev/maxsim_topk.py [out.json]"""
import ctypes as C
import json
import re
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, ".")
import innr_b200 as ib
from innr_b200 import _lib as L, sharded, synth

out_path = sys.argv[1] if len(sys.argv) > 1 else None
ib.init(0)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()
print("gpu:", gpu)
NT, DIM, NQ_TOK, KS = 180, 128, 32, (10, 100, 1000)
report = {"gpu": gpu, "shape": {"tokens_per_doc": NT, "dim": DIM, "query_tokens": NQ_TOK, "metric": "cosine"}, "sizes": {}}
stream = torch.cuda.current_stream()
sp = C.c_void_p(stream.cuda_stream)
q1 = torch.from_numpy(synth.ghash_f32(synth.SALT_QUERY, 0, NQ_TOK * DIM).reshape(1, NQ_TOK, DIM)).cuda()
q64 = torch.from_numpy(synth.ghash_f32(synth.SALT_QUERY, 0, 64 * NQ_TOK * DIM).reshape(64, NQ_TOK, DIM)).cuda()


def scores_call(corpus, q, nq, out):
    if nq == 1:
        L.call("innr_cuda_maxsim_dev", corpus.h, C.c_void_p(q.data_ptr()), NQ_TOK, 1, C.c_void_p(out.data_ptr()), sp)
    else:
        L.call("innr_cuda_maxsim_batch_dev", corpus.h, C.c_void_p(q.data_ptr()), nq, NQ_TOK, 1, C.c_void_p(out.data_ptr()), sp)


def topk_call(corpus, q, nq, k, keys):
    L.call("innr_cuda_maxsim_topk_keys_dev", corpus.h, C.c_void_p(q.data_ptr()), nq, NQ_TOK, 1, k, C.c_void_p(keys.data_ptr()), sp)


def event_ms(fn, calls):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(calls):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / calls


def kernel_name(key):
    key = key.replace("(anonymous namespace)::", "")
    m = re.match(r"(?:void\s+)?([\w:]+)", key)
    return m.group(1).split("::")[-1] if m else key


def profile_kernels(fn, calls):
    """device ms per call of each kernel name, in a profiler run of its own"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(calls):
            fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        if t and ev.count:
            name = kernel_name(ev.key)
            out[name] = out.get(name, 0.0) + t / 1000.0 / calls
    return {k: round(v, 4) for k, v in out.items()}


def measure_size(corpus, n_docs, rounds, calls, batch_calls):
    res = {"n_docs": n_docs}
    out1 = torch.empty(n_docs, dtype=torch.float32, device="cuda")
    keys = {k: torch.empty(64 * k, dtype=torch.int64, device="cuda") for k in KS}
    fns = {"maxsim_dev": lambda: scores_call(corpus, q1, 1, out1)}
    for k in KS:
        fns[f"topk_keys_dev_k{k}"] = (lambda k=k: topk_call(corpus, q1, 1, k, keys[k]))
    for fn in fns.values():
        for _ in range(3):
            fn()
    torch.cuda.synchronize()
    times = {name: [] for name in fns}
    for _ in range(rounds):           # interleaved: every variant once per round
        for name, fn in fns.items():
            times[name].append(round(event_ms(fn, calls), 4))
    res["single_query_ms"] = {name: {"median": float(np.median(v)), "rounds": v} for name, v in times.items()}
    base = res["single_query_ms"]["maxsim_dev"]["median"]
    res["profile_ms_per_call"] = {}
    for k in KS:
        prof = profile_kernels(fns[f"topk_keys_dev_k{k}"], max(3, calls // 4))
        sel = prof.get("topk_scores_kernel", 0.0)
        tot = res["single_query_ms"][f"topk_keys_dev_k{k}"]["median"]
        res["profile_ms_per_call"][f"k{k}"] = prof
        res[f"selection_k{k}"] = {"kernel_ms": sel, "share_of_topk_call": round(sel / tot, 5),
                                  "topk_minus_scores_ms": round(tot - base, 4)}
    # the keys equal the stable sort of the score vector
    torch.cuda.synchronize()
    sc = out1.cpu().numpy()
    order = np.argsort(~sharded.order_bits(sc), kind="stable")
    for k in KS:
        idx, val = sharded.decode_keys(keys[k][:k].cpu().numpy().view(np.uint64), descending=True)
        res[f"keys_equal_sorted_scores_k{k}"] = bool(np.array_equal(idx, order[:k].astype(np.uint64))
                                                     and val.tobytes() == sc[order[:k]].tobytes())
    # a batch of 64 queries
    out64 = torch.empty(64 * n_docs, dtype=torch.float32, device="cuda")
    bfns = {"maxsim_batch_dev": lambda: scores_call(corpus, q64, 64, out64)}
    for k in (10, 100):
        bfns[f"topk_keys_dev_k{k}"] = (lambda k=k: topk_call(corpus, q64, 64, k, keys[k]))
    for fn in bfns.values():
        fn()
    torch.cuda.synchronize()
    res["batch64_ms"] = {name: round(event_ms(fn, batch_calls), 3) for name, fn in bfns.items()}
    del out64
    # host entries end to end
    qh = q1[0].cpu().numpy()
    host_sc = np.zeros(n_docs, np.float32)
    ib.maxsim_corpus(qh, corpus, cosine=True, out=host_sc)
    ib.maxsim_topk(qh, corpus, 10, cosine=True)
    t0 = time.perf_counter()
    for _ in range(calls):
        ib.maxsim_corpus(qh, corpus, cosine=True, out=host_sc)
    t1 = time.perf_counter()
    for _ in range(calls):
        np.argsort(~sharded.order_bits(host_sc), kind="stable")[:10]
    t2 = time.perf_counter()
    for _ in range(calls):
        hi, hs = ib.maxsim_topk(qh, corpus, 10, cosine=True)
    t3 = time.perf_counter()
    res["host_entries_ms"] = {"maxsim": round((t1 - t0) * 1e3 / calls, 3),
                              "host_stable_sort_of_scores": round((t2 - t1) * 1e3 / calls, 3),
                              "maxsim_topk_k10": round((t3 - t2) * 1e3 / calls, 3)}
    res["host_topk_equals_sorted_host_scores"] = bool(np.array_equal(hi, order[:10].astype(np.uint64)))
    return res


n_gpus = torch.cuda.device_count()
report["n_gpus"] = n_gpus
for n_docs, rounds, calls, batch_calls in ((125_000, 5, 40, 3), (1_000_000, 3, 10, 2)):
    corpus = ib.TokenCorpus.generate(synth.SALT_CORPUS, 0, n_docs, NT, DIM)
    report["sizes"][str(n_docs)] = measure_size(corpus, n_docs, rounds, calls, batch_calls)
    print(json.dumps(report["sizes"][str(n_docs)]), flush=True)
    if n_docs == 1_000_000:
        # in-process sharded over every GPU of the box (shard d on device d, index_base = its first document)
        if n_gpus == 1:
            shards = [corpus]
        else:
            del corpus
            shards = []
            for dev in range(n_gpus):
                lo, hi = sharded.shard_range(n_docs, dev, n_gpus)
                ib.init(dev)
                shards.append(ib.TokenCorpus.generate(synth.SALT_CORPUS, lo, hi - lo, NT, DIM, index_base=lo))
            ib.init(0)
            corpus = ib.TokenCorpus.generate(synth.SALT_CORPUS, 0, n_docs, NT, DIM)
        qh = q1.cpu().numpy()
        sh = {}
        for k in (10, 100, 200):
            want = ib.maxsim_topk_batch(qh, corpus, k, cosine=True)
            got = sharded.maxsim_topk_sharded(qh, shards, k, cosine=True)
            t0 = time.perf_counter()
            for _ in range(5):
                sharded.maxsim_topk_sharded(qh, shards, k, cosine=True)
            ms = (time.perf_counter() - t0) * 1e3 / 5
            sh[f"k{k}"] = {"ms_per_call": round(ms, 3), "equals_unsharded": bool(
                np.array_equal(got[0], want[0]) and got[1].tobytes() == want[1].tobytes())}
        report["sharded_inprocess"] = {"n_shards": len(shards), "route": "exchange" if len(shards) > 1 else "single shard",
                                       **sh}
        print(json.dumps(report["sharded_inprocess"]), flush=True)
    del corpus
    torch.cuda.empty_cache()
report["gpu_after"] = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                                     capture_output=True, text=True).stdout.strip().splitlines()
if out_path:
    with open(out_path, "w") as f:
        json.dump(report, f, indent=1)
print("done")
