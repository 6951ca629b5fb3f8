"""dev: A/B of the single-query f32 kNN on the plain layout (full read) against the split layout (screen on the 8-bit
sketch + exact rescoring), at C2a (10M x 768, G-hash, cosine top-10) and at one 8-GPU shard (1.25M rows). Both corpora
are generated on the device; the calls alternate back to back for several rounds. Prints per-call CUDA-event times, the
per-phase kernel times of the split path (torch.profiler, in a run of its own: screen, compaction, rescoring, selection,
the fallback full-read launch that returns at once) with the bytes the screen moves and its rate, candidates per query
(from the screen's bounds), bit-equality of the keys over 16 queries, and a full-read scores-mode (batch_dot) A/B.
Usage: python innr_b200/csrc/dev/split_scan_ab.py [out_dir]"""
import ctypes as C
import json
import os
import re
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, ".")
import innr_b200 as ib
from innr_b200 import _lib as L, synth

out_dir = sys.argv[1] if len(sys.argv) > 1 else None
ib.init(0)
gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                     capture_output=True, text=True).stdout.strip().splitlines()[0]
print("gpu:", gpu)
D, K, ROUNDS, CALLS = 768, 10, 6, 40
q = torch.from_numpy(synth.ghash_f32(synth.SALT_QUERY, 0, 16 * D).reshape(16, D)).cuda()
stream = torch.cuda.current_stream()
report = {"gpu": gpu, "sizes": {}}
# kernel name (profiler keys look like "void innr::(anonymous namespace)::pdx_screen_kernel<1, 1>(...)") -> phase
PHASES = {"pdx_screen_kernel": "screen", "screen_compact_kernel": "compaction", "screen_rescore_kernel": "rescoring",
          "topk_scores_kernel": "selection", "pdx_scan_kernel": "fallback_full_read_noop"}


def kernel_name(key):
    key = key.replace("(anonymous namespace)::", "")
    m = re.match(r"(?:void\s+)?([\w:]+)", key)
    return m.group(1).split("::")[-1] if m else key


def call(db, i, out):
    L.call("innr_cuda_batch_knn_keys_dev", db.h, L.METRIC_COSINE, C.c_void_p(q[i % 16].data_ptr()), 1, K,
           C.c_void_p(out.data_ptr()), C.c_void_p(stream.cuda_stream))


def time_calls(db, out):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(CALLS):
        call(db, i, out)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / CALLS


for n in (10_000_000, 1_250_000):
    ib.set_option("f32_split_min_rows", 2**62)
    plain = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, D)
    ib.set_option("f32_split_min_rows", 0)
    split = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, D)
    ib.set_option("f32_split_min_rows", 1_000_000)
    outs = {name: torch.empty(16 * K, dtype=torch.int64, device="cuda") for name in ("plain", "split")}
    for name, db in (("plain", plain), ("split", split)):   # warm-up + the 16 queries' keys
        for i in range(16):
            call(db, i, outs[name][i * K:(i + 1) * K])
    torch.cuda.synchronize()
    equal = bool(torch.equal(outs["plain"], outs["split"]))
    one = torch.empty(K, dtype=torch.int64, device="cuda")
    rounds = {"plain": [], "split": []}
    for r in range(ROUNDS):
        for name, db in (("plain", plain), ("split", split)):
            rounds[name].append(time_calls(db, one))
    # candidates per query: rows whose optimistic bound reaches the k-th best pessimistic bound
    cands = []
    for i in range(16):
        lo, up = ib.knn_screen_debug_bounds("cosine", q[i].cpu().numpy(), split)
        kth = np.partition(lo, n - K)[n - K]
        cands.append(int(np.count_nonzero(up >= kth)))
    # per-kernel times of the split path, a run of its own
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for i in range(20):
            call(split, i, one)
        torch.cuda.synchronize()
    phases = {}
    for ev in prof.key_averages():
        if ev.device_type.name == "CUDA" and ev.count:
            name = kernel_name(ev.key)
            name = PHASES.get(name, name)
            t = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
            phases[name] = phases.get(name, 0.0) + t / 20 / 1000.0   # ms per call
    # full-read scores mode (both planes through the load helper against the f32 loads)
    ib.set_option("kernel_timing", 1)
    scores = {"plain": [], "split": []}
    qh = q[0].cpu().numpy()
    ms = C.c_float(0)
    for r in range(ROUNDS):
        for name, db in (("plain", plain), ("split", split)):
            ib.batch_dot(qh, db)
            L.call("innr_cuda_last_kernel_ms", C.byref(ms))
            scores[name].append(ms.value)
    ib.set_option("kernel_timing", 0)
    f32_bytes = n * D * 4
    # the screen reads the sketch (1 B per element) and 16 B per row: scale, residual bound, reference norm, and writes
    # the 4 B optimistic bound
    screen_bytes = n * D + n * 16
    med = {k: float(np.median(v)) for k, v in rounds.items()}
    res = {"n": n, "keys_bit_equal_16_queries": equal, "ms_per_call": rounds, "median_ms": med,
           "speedup": med["plain"] / med["split"], "candidates_per_query": cands,
           "split_kernels_ms_per_call": phases,
           "screen_bytes": screen_bytes,
           "screen_tb_per_s": screen_bytes / (phases.get("screen", float("nan")) / 1e3) / 1e12,
           "split_call_tb_per_s": screen_bytes / (med["split"] / 1e3) / 1e12,
           "plain_tb_per_s": f32_bytes / (med["plain"] / 1e3) / 1e12,
           "bytes_moved_split": screen_bytes, "bytes_moved_plain": f32_bytes,
           "scores_mode_kernel_ms": scores}
    report["sizes"][str(n)] = res
    print(json.dumps(res, indent=1))
    del plain, split
    torch.cuda.empty_cache()

if out_dir:
    os.makedirs(out_dir, exist_ok=True)
    with open(os.path.join(out_dir, "split_scan_ab.json"), "w") as f:
        json.dump(report, f, indent=1)
