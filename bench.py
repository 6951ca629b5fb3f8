#!/usr/bin/env python
"""bench.py -- benchmark of the innr batch similarity-search hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME|all] [--impl reference] [--sharding nccl|inproc]
                  [--dump-outputs DIR]
  (N > 1: python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...)

A "step" is one pass of the hot path over one batch of synthetic input. Prints ONE JSON line on rank 0.

The headline (top-level keys) is the configuration BASELINE.json's metric is quoted on -- C2a: batch_knn_cosine top-10
over a 10M x 768 f32 corpus, one query per step, row-sharded over the N GPUs. With the default `--workload all` the same
line also carries `workloads`: one entry per BASELINE.json config (C1 batch_demo, C2a, C2b 1024-query batches, C3 MaxSim
docs/s, C4 Hamming top-100, C5 u8 kNN), each measured back to back in this process with the same K / W and with its own
value / ms_per_step / e2e / roofline / clocks (and cpu_baseline at N == 1). `--workload NAME` measures that one only.

  value     queries/s (docs/s for maxsim) of the whole job, inputs resident in HBM, CUDA events, max over ranks
  e2e       the same metric through the public API with HOST buffers (pinned H2D of the query, D2H of the result)
  roofline  dominant kernel: algorithmic bytes (or flops) per launch / its CUDA-event time, against MEASURED_PEAKS.json
  cpu_baseline  the oracle (C++ restatement of innr 0.6.3, "port") timed on this box's host cores: one query per thread
            over ALL rows of the config when host RAM allows (else the largest prefix that fits, flagged `extrapolated`)

`--impl reference` times that CPU implementation as its own arm (rank 0 only), one step = one query per host thread over
the whole config. `--scale f` shrinks every corpus (quick checks; reported in config).
"""
import argparse
import ctypes as C
import gc
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (config id, description, metric name, unit)
    "knn_cosine_1q": ("C2a", "batch_knn_cosine 10M x 768 f32, 1 query/step, k=10", "batch_knn_cosine_top10_queries_per_s", "queries/s"),
    "knn_cosine_multi": ("C2b", "batch_knn_cosine 10M x 768 f32, Q queries/step, k=10", "batch_knn_cosine_top10_queries_per_s", "queries/s"),
    "knn_cosine_1q_filter": ("C2a-filter", "batch_knn_cosine 10M x 768 f32, 1 query/step, k=10, through the f16 tensor-core filter + exact rescoring (option knn_tc_min_queries=1; same bits as the scan)", "batch_knn_cosine_top10_queries_per_s", "queries/s"),
    "batch_demo": ("C1", "batch_knn_dot 10K x 128 f32 G-ref lattice, 100 queries/step, k=10", "batch_knn_dot_top10_queries_per_s", "queries/s"),
    "maxsim": ("C3", "maxsim_cosine 32 x 128 query tokens vs 1M docs x 180 tokens x 128d", "maxsim_cosine_docs_per_s", "docs/s"),
    "hamming": ("C4", "binary_hamming top-100 over 100M 1024-bit codes, 1 query/step", "hamming_top100_queries_per_s", "queries/s"),
    "u8": ("C5", "batch_knn_u8 50M x 384 u8 corpus, f32 query, k=10, 1 query/step", "batch_knn_u8_top10_queries_per_s", "queries/s"),
}
HEADLINE = "knn_cosine_1q"
ALL_ORDER = ["knn_cosine_1q", "knn_cosine_multi", "hamming", "u8", "batch_demo", "maxsim"]  # C3 last: it needs 93 GB
PORT_NOTE = " (C++ restatement of innr 0.6.3, not the Rust crate)"


def corpus_shape(workload, scale):
    """(rows, bytes per row) of the config at `scale`."""
    if workload == "batch_demo":
        return int(10_000 * scale), 128 * 4
    if workload in ("knn_cosine_1q", "knn_cosine_multi", "knn_cosine_1q_filter"):
        return int(10_000_000 * scale), 768 * 4
    if workload == "maxsim":
        return int(1_000_000 * scale), 180 * 128 * 4
    if workload == "hamming":
        return int(100_000_000 * scale), 128
    return int(50_000_000 * scale), 384


def config_of(workload, scale, n_gpus, queries=1024):
    """The `config` object -- identical in the b200 and reference arms (it names the workload, not the implementation)."""
    n, row_bytes = corpus_shape(workload, scale)
    gb = n * row_bytes / 1e9
    desc = WORKLOADS[workload][1].replace("Q queries/step", f"{queries} queries/step")
    return {"workload": desc, "id": WORKLOADS[workload][0], "scale": scale, "corpus_gb": round(gb, 3), "sharding": f"rows/{n_gpus}",
            "l2": "inputs larger than L2 (corpus >> 126 MB), no flush" if gb / n_gpus > 0.5
            else ("corpus is L2-resident by design of this config (latency-bound); no flush" if workload == "batch_demo"
                  else "scaled-down corpus (quick check): may be L2-resident; no flush"),
            "generator": "G-ref lattice" if workload == "batch_demo" else "G-hash (splitmix64)"}


def host_mem_available():
    """Bytes of host RAM this process may still take: min(system available, cgroup limit - usage)."""
    avail = None
    try:
        import psutil
        avail = int(psutil.virtual_memory().available)
    except Exception:
        pass
    for lim, cur in (("/sys/fs/cgroup/memory.max", "/sys/fs/cgroup/memory.current"),
                     ("/sys/fs/cgroup/memory/memory.limit_in_bytes", "/sys/fs/cgroup/memory/memory.usage_in_bytes")):
        try:
            a, b = open(lim).read().strip(), open(cur).read().strip()
            if a != "max" and int(a) < (1 << 60):
                left = int(a) - int(b)
                avail = left if avail is None else min(avail, left)
        except Exception:
            pass
    return avail if avail is not None else 32 << 30


def plan_cpu_sample(n_rows, row_bytes, per_thread_bytes_per_row, cores, full=True, max_rows=None):
    """How many rows and threads the CPU leg can use: all rows and all cores when they fit in 80 % of the free host
    RAM (corpus + one query's working set per thread), else fewer threads, else a prefix of the rows."""
    budget = int(host_mem_available() * 0.8)
    rows = n_rows if max_rows is None else min(n_rows, max_rows)
    if not full:
        return rows, cores  # small samples always fit
    threads = cores
    while threads > 1 and rows * (row_bytes + threads * per_thread_bytes_per_row) > budget:
        threads -= 1
    if rows * (row_bytes + threads * per_thread_bytes_per_row) > budget:
        rows = max(1, budget // (row_bytes + threads * per_thread_bytes_per_row))
    return rows, threads


def load_traffic(workload, scale, world):
    """Per-launch DRAM traffic of the dominant kernel from the committed ncu --set full capture (profiles/), only
    meaningful for the exact captured configuration (scale 1.0, 1 GPU); else null."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if scale != 1.0 or world != 1 or not os.path.exists(p):
        return None
    return json.load(open(p)).get(workload, {}).get("bytes")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_tensor_peak():
    """Dense 16-bit tensor peak (TFLOP/s) for a kernel timed inside a long step: the sustained cuBLAS bf16 figure of
    MEASURED_PEAKS.json (f16 and bf16 issue at the same rate), else the profiling guide's fallback."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if "bf16_tflops_sustained" in d:
            return float(d["bf16_tflops_sustained"]), "measured sustained cuBLAS bf16 (MEASURED_PEAKS.json)"
        if "bf16_tflops" in d:
            return float(d["bf16_tflops"]), "measured burst cuBLAS bf16 (MEASURED_PEAKS.json)"
    return 1500.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock + clocks-event (throttle) reasons sampled DURING the timed region. NVML in a thread every ~2 ms
    (a 4 ms step needs a faster sampler than `nvidia-smi -lms 100`); nvidia-smi (the B200_PROFILING.md clocks line)
    is the fallback when NVML cannot be loaded. Only samples taken between mark_begin() and mark_end() are reported."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.samples, self.stop_flag, self.t = gpu_index, [], False, None
        self.t_begin = self.t_end = None
        self.mode, self.proc, self.max_mhz = None, None, None

    def _nvml_index(self):
        vis = os.environ.get("CUDA_VISIBLE_DEVICES")
        if vis:
            ids = [x.strip() for x in vis.split(",") if x.strip()]
            if self.gpu < len(ids) and ids[self.gpu].isdigit():
                return int(ids[self.gpu])
        return self.gpu

    def start(self):
        try:
            import pynvml as nv
            nv.nvmlInit()
            self.nv, self.h = nv, nv.nvmlDeviceGetHandleByIndex(self._nvml_index())
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(self.h, nv.NVML_CLOCK_SM))
            self.mode = "nvml"
            self.t = threading.Thread(target=self._poll_nvml, daemon=True)
            self.t.start()
            return
        except Exception:
            self.mode = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20", "-i", str(self._nvml_index())], stdout=subprocess.PIPE, text=True)
            self.mode = "nvidia-smi"
            self.t = threading.Thread(target=self._read_smi, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _poll_nvml(self):
        nv = self.nv
        names = (("hw_slowdown", nv.nvmlClocksEventReasonHwSlowdown),
                 ("hw_thermal_slowdown", nv.nvmlClocksEventReasonHwThermalSlowdown),
                 ("sw_thermal_slowdown", nv.nvmlClocksEventReasonSwThermalSlowdown),
                 ("sw_power_cap", nv.nvmlClocksEventReasonSwPowerCap),
                 ("hw_power_brake", nv.nvmlClocksEventReasonHwPowerBrakeSlowdown))
        while not self.stop_flag:
            try:
                mhz = float(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                mask = int(nv.nvmlDeviceGetCurrentClocksEventReasons(self.h))
                try:
                    watts = nv.nvmlDeviceGetPowerUsage(self.h) / 1e3
                except Exception:
                    watts = None
                self.samples.append((time.perf_counter(), mhz, tuple(n for n, bit in names if mask & bit), watts))
            except Exception:
                pass
            time.sleep(0.002)

    def _read_smi(self):
        for line in self.proc.stdout:
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                mhz, self.max_mhz = float(f[1]), float(f[2])
            except ValueError:
                continue
            rs = tuple(n for n, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9])
                       if v.lower().startswith("active"))
            try:
                watts = float(f[3])
            except ValueError:
                watts = None
            self.samples.append((time.perf_counter(), mhz, rs, watts))

    def mark_begin(self):
        self.t_begin = time.perf_counter()

    def mark_end(self):
        self.t_end = time.perf_counter()

    def stop(self):
        if self.mode is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["clock sampler unavailable"]}
        self.stop_flag = True
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()
        if self.t:
            self.t.join(timeout=2)
        lo, hi = self.t_begin or 0.0, self.t_end or float("inf")
        inside = [s for s in self.samples if lo <= s[0] <= hi]
        nearest = False
        if not inside and self.samples:  # a timed region shorter than the sampling period (C1: < 1 ms): nearest samples
            mid = 0.5 * (lo + min(hi, self.samples[-1][0]))
            inside = sorted(self.samples, key=lambda s: abs(s[0] - mid))[:3]
            nearest = True
        sm = [s[1] for s in inside]
        reasons = sorted({r for s in inside for r in s[2]})
        watts = [s[3] for s in inside if s[3] is not None]
        return {"power_w_max": max(watts) if watts else None,
                "sm_mhz": statistics.median(sm) if sm else None, "sm_min_mhz": min(sm) if sm else None,
                "sm_max_mhz": self.max_mhz, "samples": len(sm), "reasons": reasons, "sampler": self.mode,
                "nearest_samples_outside_window": nearest,
                "window_ms": (hi - lo) * 1e3 if self.t_end else None}


# ------------------------------------------------------------------------------------------------ workloads
class Workload:
    """One config of BASELINE.json on this rank's shard. __init__ fixes the shape and the host-side queries (no device
    needed: the reference arm uses only that and the cpu_* methods); setup() builds the device shard.
    Subclasses fill: step_dev(i), step_e2e(i), units_per_step, kernel_bytes (algorithmic bytes of the dominant kernel per
    launch on THIS rank), cpu_prepare(cores, full) / cpu_step()."""
    kernel_timed_by_keys_entry = False

    def __init__(self, args, workload, rank, world):
        self.args, self.workload, self.rank, self.world = args, workload, rank, world
        self.torch = None
        self._cpu = None
        self.exchange = None  # PeerExchange of this rank (N > 1, --sharding peer)

    @property
    def dev(self):
        return self.torch.device(f"cuda:{self.torch.cuda.current_device()}")

    def pinned(self, arr):
        t = self.torch.from_numpy(np.ascontiguousarray(arr)).pin_memory()
        return t, t.numpy()

    def fetch(self, idx, score):
        """D2H of a result pair into pinned host tensors with ONE stream synchronisation."""
        key = (tuple(idx.shape), idx.dtype, score.dtype)
        if getattr(self, "_fetch_key", None) != key:
            self._fetch_key = key
            self._h_idx = self.torch.empty(idx.shape, dtype=idx.dtype).pin_memory()
            self._h_sc = self.torch.empty(score.shape, dtype=score.dtype).pin_memory()
        self._h_idx.copy_(idx, non_blocking=True)
        self._h_sc.copy_(score, non_blocking=True)
        self.torch.cuda.current_stream().synchronize()
        return self._h_idx, self._h_sc

    _pending = None

    def e2e_collect(self, ticket):
        """Keeps one asynchronous call in flight behind the one just submitted; returns the previous call's result."""
        prev, self._pending = self._pending, ticket
        return prev.wait() if prev is not None else None

    def e2e_drain(self):
        prev, self._pending = self._pending, None
        return prev.wait() if prev is not None else None

    def drain(self):
        """Queue a wait for everything step_dev left on side streams (the pipelined exchanges at N > 1)."""
        sk = getattr(self, "sk", None)
        if sk is not None:
            sk.drain()

    def outputs(self, result):
        """Host copies of what a caller of step_dev receives from one step (the top-k workloads' result pair)."""
        return {"indices": result[0].cpu().numpy(), "scores": result[1].cpu().numpy()}

    def close(self):
        """Drop the device shard (and the CPU sample) before the next workload is built."""
        for name in ("sk", "shard", "q_dev", "out", "out_b", "_cpu", "_h_idx", "_h_sc"):
            if hasattr(self, name):
                setattr(self, name, None)
        gc.collect()
        if self.torch is not None:
            self.torch.cuda.empty_cache()

    # ---- CPU leg (oracle): one step = one query per host thread over the planned rows -------------------------------
    def cpu_measure(self, cores, full=True, steps=1, warmup=0, budget_s=None):
        """Returns (value in the workload's unit for the FULL config, info dict, seconds per step). When fewer rows than
        the config's are used the rate is scaled by rows/N and `extrapolated` is true. budget_s bounds the whole run: if
        the first warm-up step over all rows shows that W + K such steps would not fit, the remaining steps use the
        prefix of the rows that does (the full-rows step time is reported beside the value)."""
        t_start = time.perf_counter()
        self.cpu_prepare(cores, full)
        full_rows_step_s = None
        for i in range(warmup):
            _, dt = self.cpu_step()
            left = steps + warmup - 1 - i
            if i == 0 and budget_s and self._cpu["scales_with_rows"]:
                remaining = max(budget_s - (time.perf_counter() - t_start), 0.05 * budget_s)
                if dt * left > remaining:
                    full_rows_step_s = dt
                    self.cpu_prepare(cores, full, max_rows=max(1000, int(self._cpu["rows"] * remaining / (dt * left))))
        dts, units = [], 0
        for _ in range(steps):
            u, dt = self.cpu_step()
            units += u
            dts.append(dt)
        c = self._cpu
        scale = c["rows"] / c["n"] if c["scales_with_rows"] else 1.0
        value = units / sum(dts) * scale
        info = {"cores": c["threads"], "rows": c["rows"], "rows_of_config": c["n"], "extrapolated": c["rows"] < c["n"] and c["scales_with_rows"],
                "sample": c["sample"] + PORT_NOTE, "build_s": round(c["build_s"], 2)}
        if full_rows_step_s is not None:
            info["full_rows_step_s"] = round(full_rows_step_s, 3)
            info["full_rows_value"] = c["threads"] / full_rows_step_s
        return value, info, sum(dts) / len(dts)


class KnnF32(Workload):
    def __init__(self, args, workload, rank, world):
        super().__init__(args, workload, rank, world)
        from innr_b200 import synth
        demo = workload == "batch_demo"
        self.demo = demo
        self.n, self.d, self.k = corpus_shape(workload, args.scale)[0], (128 if demo else 768), 10
        self.metric = "dot" if demo else "cosine"
        self.nq = 100 if demo else (args.queries if workload == "knn_cosine_multi" else 1)
        n_distinct = 16
        if demo:
            qs = np.stack([self._gref(self.d, 50_000 + j) for j in range(self.nq)])[None].repeat(n_distinct, 0)
        else:
            qs = synth.ghash_f32(synth.SALT_QUERY, 0, n_distinct * self.nq * self.d).reshape(n_distinct, self.nq, self.d)
        self.q_np = np.ascontiguousarray(qs)
        self.units_per_step = self.nq
        self.h2d, self.d2h = self.nq * self.d * 4, self.nq * self.k * 12

    def setup(self, torch):
        import innr_b200 as ib
        from innr_b200 import sharded, synth
        self.torch = torch
        lo, hi = sharded.shard_range(self.n, self.rank, self.world)
        self.n_local = hi - lo
        gen, salt = ("gref", 0) if self.demo else ("ghash", synth.SALT_CORPUS)
        self.shard = ib.DeviceBatch.generate(gen, salt, lo, self.n_local, self.d, index_base=lo)
        self.sk = sharded.ShardedKnn(self.shard, "f32", self.metric, exchange=self.exchange)
        self.q_host_t, self.q_host = self.pinned(self.q_np)
        self.q_dev = torch.from_numpy(self.q_np).to(self.dev)
        passes = (self.nq + 7) // 8 if self.nq > 1 else 1
        self.kernel_bytes = self.n_local * self.d * 4 * passes
        self.kernel_name = "pdx_scan_kernel"
        ib.set_option("knn_tc_min_queries", 2)
        if self.workload == "knn_cosine_1q_filter":
            # the bytes the filter actually streams: the f16 unit-vector copy (the f32 corpus is only touched by the
            # ~200 rescored rows); reported against HBM like the scan
            ib.set_option("knn_tc_min_queries", 1)
            self.kernel_bytes = self.n_local * self.d * 2
            self.kernel_name = "knn_tc_filter_kernel<QRES> (4 passes + exact rescoring: whole call)"
        self.kernel_timed_by_keys_entry = True

    @staticmethod
    def _gref(dim, seed):
        i = np.arange(dim, dtype=np.uint64)
        with np.errstate(over="ignore"):
            x = np.uint64(seed) * np.uint64(6364136223846793005) + i * np.uint64(1442695040888963407)
        return ((x >> np.uint64(33)).astype(np.float32) / np.float32(2**31) * np.float32(2.0) - np.float32(1.0)).astype(np.float32)

    def step_dev(self, i):
        # C1's step is bound by the host's launch rate (one 30 us launch): keep its scans on one stream
        return self.sk.knn_dev_pipelined(self.q_dev[i % self.q_dev.shape[0]], self.nq, self.k,
                                         overlap_scans=self.workload != "batch_demo")

    def step_e2e(self, i):
        if self.world == 1:
            # the C-ABI with host buffers, asynchronous form: submit call i, then collect call i - 1 (two in flight)
            from innr_b200 import stream
            return self.e2e_collect(stream.submit_knn(self.metric, self.q_host[i % self.q_host.shape[0]], self.shard, self.k))
        # N > 1: pinned query in, pinned result out, streamed (results one call late, one host sync per batch of calls)
        q = self.q_host_t[i % self.q_host_t.shape[0]]
        return self.sk.knn_dev_pipelined(None, self.nq, self.k, overlap_scans=self.workload != "batch_demo",
                                         host_queries=q, host_out=True)

    def keys_entry(self, L, q, b, stream):
        L.call("innr_cuda_batch_knn_keys_dev", self.shard.h, self.sk._metric_id, C.c_void_p(q.data_ptr()), self.nq, self.k,
               C.c_void_p(b["local"].data_ptr()), stream)

    def cpu_prepare(self, cores, full, max_rows=None):
        from oracle import innr_oracle as orc
        from innr_b200 import synth
        # per query and thread the reference holds norms + scores (8 B/row) and the (usize, f32) pairs it sorts plus the
        # stable sort's scratch (32 B/row)
        rows, threads = plan_cpu_sample(self.n, self.d * 4, 40, cores, full, max_rows or (None if full else 200_000))
        if self._cpu and self._cpu["rows"] == rows:
            self._cpu["threads"] = threads
            return
        t0 = time.perf_counter()
        if self.demo:
            ob = orc.VerticalBatch.from_flat(np.stack([orc.generate_embedding(self.d, i) for i in range(rows)]).reshape(-1), rows, self.d)
        else:
            ob = orc.ghash_vertical_batch(synth.SALT_CORPUS, 0, rows, self.d, cores)
        what = "all" if rows == self.n else "the first"
        self._cpu = {"rows": rows, "n": self.n, "threads": threads, "batch": ob, "scales_with_rows": True, "build_s": time.perf_counter() - t0,
                     "sample": (f"one step = {self.nq} queries (the config's batch) spread over {threads} threads" if self.demo
                                else f"one step = {threads} queries, one per thread,") + f" over {what} {rows} of {self.n} rows x {self.d}"}

    def cpu_step(self):
        from oracle import innr_oracle as orc
        c = self._cpu
        nq = self.nq if self.demo else c["threads"]
        flat = self.q_np.reshape(-1, self.d)
        qs = np.ascontiguousarray(flat[np.arange(nq) % flat.shape[0]])
        t0 = time.perf_counter()
        orc.batch_knn_many(self.metric, qs, c["batch"], self.k, n_threads=c["threads"])
        return nq, time.perf_counter() - t0


class Hamming(Workload):
    def __init__(self, args, workload, rank, world):
        super().__init__(args, workload, rank, world)
        from innr_b200 import synth
        self.n, self.dim, self.k, self.nq = corpus_shape(workload, args.scale)[0], 1024, 100, 1
        self.q_np = synth.ghash_u64(synth.SALT_QUERY, 0, 16 * 16).reshape(16, 16).view(np.int64)
        self.units_per_step = 1
        self.h2d, self.d2h = 128, self.k * 16

    def setup(self, torch):
        import innr_b200 as ib
        from innr_b200 import sharded, synth
        self.torch = torch
        lo, hi = sharded.shard_range(self.n, self.rank, self.world)
        self.n_local = hi - lo
        self.shard = ib.BinaryCorpus.generate(synth.SALT_CODES, lo, self.n_local, self.dim, index_base=lo)
        self.sk = sharded.ShardedKnn(self.shard, "binary", exchange=self.exchange)
        self.q_host_t, self.q_host = self.pinned(self.q_np)
        self.q_dev = torch.from_numpy(self.q_np).to(self.dev)
        self.kernel_bytes = self.n_local * 128
        self.kernel_name = "hamming_kernel"
        self.kernel_timed_by_keys_entry = True

    def step_dev(self, i):
        return self.sk.knn_dev_pipelined(self.q_dev[i % 16], 1, self.k)

    def step_e2e(self, i):
        if self.world == 1:
            from innr_b200 import stream
            return self.e2e_collect(stream.submit_hamming_topk(self.q_host[i % 16].view(np.uint64).reshape(1, -1), self.shard, self.k))
        return self.sk.knn_dev_pipelined(None, 1, self.k, host_queries=self.q_host_t[i % 16], host_out=True)

    def keys_entry(self, L, q, b, stream):
        L.call("innr_cuda_hamming_topk_keys_dev", self.shard.h, C.c_void_p(q.data_ptr()), self.nq, self.k,
               C.c_void_p(b["local"].data_ptr()), stream)

    batch_queries = 2  # k = 100 lists: two queries share every pass over the codes (hamming_multi_kernel)

    def step_batch(self, i):
        j = (2 * i) % 14
        return self.sk.knn_dev(self.q_dev[j:j + 2], 2, self.k)

    def cpu_prepare(self, cores, full, max_rows=None):
        from oracle import innr_oracle as orc
        from innr_b200 import synth
        # per query and thread: the (usize, u32) pairs the caller sorts + the stable sort's scratch (32 B/code)
        rows, threads = plan_cpu_sample(self.n, 128, 32, cores, full, max_rows or (None if full else 2_000_000))
        if self._cpu and self._cpu["rows"] == rows:
            self._cpu["threads"] = threads
            return
        t0 = time.perf_counter()
        codes = orc.ghash_u64_mt(synth.SALT_CODES, 0, rows * 16, cores).reshape(rows, 16)
        what = "all" if rows == self.n else "the first"
        self._cpu = {"rows": rows, "n": self.n, "threads": threads, "codes": codes, "scales_with_rows": True, "build_s": time.perf_counter() - t0,
                     "sample": f"one step = {threads} queries, one per thread, over {what} {rows} of {self.n} codes x 1024 bit"}

    def cpu_step(self):
        from oracle import innr_oracle as orc
        c = self._cpu
        nq = c["threads"]
        qs = np.ascontiguousarray(self.q_np.view(np.uint64)[np.arange(nq) % 16])
        t0 = time.perf_counter()
        orc.hamming_topk_many(qs, c["codes"], self.k, n_threads=c["threads"])
        return nq, time.perf_counter() - t0


class U8(Workload):
    def __init__(self, args, workload, rank, world):
        super().__init__(args, workload, rank, world)
        from innr_b200 import synth
        self.n, self.d, self.k, self.nq = corpus_shape(workload, args.scale)[0], 384, 10, 1
        self.q_np = synth.ghash_f32(synth.SALT_QUERY, 0, 16 * self.d).reshape(16, self.d)
        self.units_per_step = 1
        self.h2d, self.d2h = self.d * 4, self.k * 12

    def setup(self, torch):
        import innr_b200 as ib
        from innr_b200 import sharded, synth
        self.torch = torch
        lo, hi = sharded.shard_range(self.n, self.rank, self.world)
        self.n_local = hi - lo
        self.params = ib.QuantizationParams.from_range(-1.0, 1.0)
        self.shard = ib.U8Corpus.generate(synth.SALT_CORPUS, lo, self.n_local, self.d, self.params, index_base=lo)
        self.sk = sharded.ShardedKnn(self.shard, "u8", exchange=self.exchange)
        self.q_host_t, self.q_host = self.pinned(self.q_np)
        self.q_dev = torch.from_numpy(self.q_np).to(self.dev)
        self.kernel_bytes = self.n_local * self.d
        self.kernel_name = "u8_scan_kernel"
        self.kernel_timed_by_keys_entry = True

    def step_dev(self, i):
        return self.sk.knn_dev_pipelined(self.q_dev[i % 16], 1, self.k)

    def step_e2e(self, i):
        if self.world == 1:
            from innr_b200 import stream
            return self.e2e_collect(stream.submit_knn_u8(self.q_host[i % 16].reshape(1, -1), self.shard, self.k))
        return self.sk.knn_dev_pipelined(None, 1, self.k, host_queries=self.q_host_t[i % 16], host_out=True)

    def keys_entry(self, L, q, b, stream):
        L.call("innr_cuda_batch_knn_u8_keys_dev", self.shard.h, C.c_void_p(q.data_ptr()), self.nq, self.k,
               C.c_void_p(b["local"].data_ptr()), stream)

    batch_queries = 2  # two queries share every pass over the codes (u8_scan_pair_kernel)

    def step_batch(self, i):
        j = (2 * i) % 14
        return self.sk.knn_dev(self.q_dev[j:j + 2], 2, self.k)

    def cpu_prepare(self, cores, full, max_rows=None):
        from oracle import innr_oracle as orc
        from innr_b200 import synth
        # per query and thread: scores (4 B/row), the (usize, f32) pairs + the stable sort's scratch (32 B/row)
        rows, threads = plan_cpu_sample(self.n, self.d, 36, cores, full, max_rows or (None if full else 500_000))
        if self._cpu and self._cpu["rows"] == rows:
            self._cpu["threads"] = threads
            return
        t0 = time.perf_counter()
        p = orc.QuantizationParams.from_range(-1.0, 1.0)
        mat = orc.ghash_u8_rows(synth.SALT_CORPUS, 0, rows, self.d, p, cores)
        what = "all" if rows == self.n else "the first"
        self._cpu = {"rows": rows, "n": self.n, "threads": threads, "mat": mat, "params": p, "scales_with_rows": True,
                     "build_s": time.perf_counter() - t0,
                     "sample": f"one step = {threads} queries, one per thread, over {what} {rows} of {self.n} rows x {self.d}"}

    def cpu_step(self):
        from oracle import innr_oracle as orc
        c = self._cpu
        nq = c["threads"]
        qs = np.ascontiguousarray(self.q_np[np.arange(nq) % 16])
        t0 = time.perf_counter()
        orc.batch_knn_u8_many(qs, c["mat"], c["params"], self.k, n_threads=c["threads"])
        return nq, time.perf_counter() - t0


class MaxSim(Workload):
    def __init__(self, args, workload, rank, world):
        super().__init__(args, workload, rank, world)
        from innr_b200 import synth
        self.n, self.nt, self.dim, self.nq = corpus_shape(workload, args.scale)[0], 180, 128, 32
        self.q_np = synth.ghash_f32(synth.SALT_QUERY, 0, 4 * self.nq * self.dim).reshape(4, self.nq, self.dim)
        self.units_per_step = self.n  # docs scored per step by the whole job

    def setup(self, torch):
        import innr_b200 as ib
        from innr_b200 import sharded, synth
        self.torch = torch
        lo, hi = sharded.shard_range(self.n, self.rank, self.world)
        self.n_local = hi - lo
        self.shard = ib.TokenCorpus.generate(synth.SALT_CORPUS, lo, self.n_local, self.nt, self.dim, index_base=lo)
        self.q_host_t, self.q_host = self.pinned(self.q_np)
        self.q_dev = torch.from_numpy(self.q_np).to(self.dev)
        self.out = torch.empty(self.n_local, dtype=torch.float32, device=self.dev)
        self.out_host_t = torch.empty(self.n_local, dtype=torch.float32).pin_memory()  # caller-owned result buffer
        self.out_host = self.out_host_t.numpy()
        self.kernel_bytes = self.n_local * self.nt * self.dim * 4
        self.kernel_name = "maxsim_tc_kernel"
        self.h2d, self.d2h = self.nq * self.dim * 4, self.n_local * 4

    def step_dev(self, i):
        from innr_b200 import _lib as L
        s = C.c_void_p(self.torch.cuda.current_stream().cuda_stream)
        L.call("innr_cuda_maxsim_dev", self.shard.h, C.c_void_p(self.q_dev[i % 4].data_ptr()), self.nq, 1,
               C.c_void_p(self.out.data_ptr()), s)
        return self.out

    def outputs(self, result):
        return {"scores": result.cpu().numpy()}

    def step_e2e(self, i):
        import innr_b200 as ib
        return ib.maxsim_corpus(self.q_host[i % 4], self.shard, cosine=True, out=self.out_host)

    batch_queries = 2  # two queries of 32 tokens share every pass over the token matrix

    def step_batch(self, i):
        from innr_b200 import _lib as L
        if getattr(self, "out_b", None) is None:
            self.out_b = self.torch.empty(2 * self.n_local, dtype=self.torch.float32, device=self.dev)
        s = C.c_void_p(self.torch.cuda.current_stream().cuda_stream)
        L.call("innr_cuda_maxsim_batch_dev", self.shard.h, C.c_void_p(self.q_dev[2 * (i % 2)].data_ptr()), 2, self.nq, 1,
               C.c_void_p(self.out_b.data_ptr()), s)
        return self.out_b

    def cpu_prepare(self, cores, full, max_rows=None):
        from oracle import innr_oracle as orc
        from innr_b200 import synth
        # documents are independent and identical in shape: the rate does not depend on how many are scored, so a prefix
        # is an exact sample of the config (no extrapolation involved); all docs when they fit in host RAM
        rows, threads = plan_cpu_sample(self.n, self.nt * self.dim * 4, 0, cores, full, max_rows or (None if full else 250 * cores))
        if self._cpu and self._cpu["rows"] == rows:
            return
        t0 = time.perf_counter()
        toks = orc.ghash_f32_mt(synth.SALT_CORPUS, 0, rows * self.nt * self.dim, cores).reshape(rows * self.nt, self.dim)
        off = np.arange(0, rows * self.nt + 1, self.nt, dtype=np.uint64)
        what = "all" if rows == self.n else "the first"
        self._cpu = {"rows": rows, "n": self.n, "threads": cores, "toks": toks, "off": off, "scales_with_rows": False, "i": 0,
                     "build_s": time.perf_counter() - t0,
                     "sample": f"one step = {what} {rows} of {self.n} docs x {self.nt} tokens x {self.dim}d scored once, docs split over {cores} threads"}

    def cpu_step(self):
        from oracle import innr_oracle as orc
        c = self._cpu
        q = self.q_np[c["i"] % 4]
        c["i"] += 1
        t0 = time.perf_counter()
        orc.maxsim_corpus(q, c["toks"], c["off"], cosine_flag=True, n_threads=c["threads"])
        return c["rows"], time.perf_counter() - t0


def make_workload(args, workload, rank, world):
    cls = {"knn_cosine_1q": KnnF32, "knn_cosine_1q_filter": KnnF32, "knn_cosine_multi": KnnF32, "batch_demo": KnnF32,
           "maxsim": MaxSim, "hamming": Hamming, "u8": U8}[workload]
    return cls(args, workload, rank, world)


def dtype_of(workload):
    return {"hamming": "u64", "u8": "f32xu8"}.get(workload, "f32")


# ------------------------------------------------------------------------------------------------ reference arm
def run_reference(args, rank):
    """The reference's own CPU implementation of the path (oracle port: the Rust crate cannot be built here) on this
    box's host cores: one step = one query per host thread over ALL rows of the config (the largest prefix that fits in
    host RAM otherwise, flagged `extrapolated`)."""
    if rank != 0:
        return
    workload = HEADLINE if args.workload == "all" else args.workload
    _, _, metric, unit = WORKLOADS[workload]
    cores = os.cpu_count() or 1
    w = make_workload(args, workload, 0, 1)
    value, info, s_per_step = w.cpu_measure(cores, full=not args.ref_small_sample, steps=args.steps, warmup=args.warmup,
                                            budget_s=args.ref_budget_s)
    line = {"impl": "reference", "metric": metric, "value": value, "unit": unit, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype_of(workload),
            "data": "synthetic", "config": config_of(workload, args.scale, args.gpus, args.queries),
            "cpu_baseline": {"value": value, "unit": unit, "kind": "port", **info},
            "e2e": {"value": value, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------ b200 arm
def measure(w, args, env):
    """Builds the workload's shard, times K steps device-resident (CUDA events, barrier + synchronize on both sides, max
    over ranks), the dominant kernel alone, and K steps end to end with host buffers. Returns the workload's entry."""
    torch, dist, ib = env["torch"], env["dist"], env["ib"]
    rank, world, local_rank = env["rank"], env["world"], env["local_rank"]
    from innr_b200 import _lib as L
    steps, warmup = args.steps, args.warmup
    cid, _, metric, unit = WORKLOADS[w.workload]
    w.exchange = env.get("exchange")
    w.setup(torch)
    torch.cuda.synchronize()

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---- N > 1: the peer-mapped exchange must give what the NCCL allgather + merge path gives (same bits, every rank)
    exchange_check = None
    if world > 1 and getattr(w, "sk", None) is not None and w.exchange is not None and w.exchange.fits(w.nq, w.k):
        from innr_b200 import sharded
        ref_sk = sharded.ShardedKnn(w.shard, w.sk.kind, w.sk.metric)
        bad = 0
        for i in range(4):
            q = w.q_dev[i % w.q_dev.shape[0]]
            a = [t.clone() for t in w.sk.knn_dev(q, w.nq, w.k)]
            b = [t.clone() for t in ref_sk.knn_dev(q, w.nq, w.k)]
            torch.cuda.synchronize()
            bad += int(not (torch.equal(a[0], b[0]) and torch.equal(a[1].double(), b[1].double())))
        bad = int(max_over_ranks(float(bad)))
        exchange_check = "peer exchange == nccl allgather + merge on 4 steps, all ranks" if bad == 0 else f"MISMATCH on {bad} steps"
        if bad or w.exchange.status() != 0:
            raise RuntimeError(f"{w.workload}: {exchange_check}; exchange status {w.exchange.status()}")
        del ref_sk

    # ---- device-resident timed region ---------------------------------------------------------------
    for i in range(warmup):
        w.step_dev(i)
    w.drain()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    l0 = ib.launch_count()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    kev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    barrier()
    sampler.mark_begin()
    ev[0].record()
    for i in range(steps):
        kev[i][0].record()
        last = w.step_dev(i)
        kev[i][1].record()
    w.drain()  # N > 1: the exchanges run on a side stream under the next scan; the region ends when the last one has
    ev[1].record()
    barrier()
    sampler.mark_end()
    # copied before anything else runs: the result buffers are reused by the measurements below
    w.last_outputs = w.outputs(last) if args.dump_outputs and rank == 0 else None
    total_ms = max_over_ranks(ev[0].elapsed_time(ev[1]))
    launches = ib.launch_count() - l0
    step_ms = [a.elapsed_time(b) for a, b in kev]
    clocks = sampler.stop() if rank == 0 else None

    # ---- dominant kernel alone: CUDA events around the library's scan launch only, on the launching stream ----------
    stream = C.c_void_p(torch.cuda.current_stream().cuda_stream)
    if w.kernel_timed_by_keys_entry:
        b = w.sk._buffers(w.nq, w.k, w.dev)
        # back to back on the launching stream, like the timed region above (a launch that starts from an idle GPU pays
        # for clock and power-state ramps that a step in a stream of steps does not)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = min(steps, 20)
        w.keys_entry(L, w.q_dev[0], b, stream)
        torch.cuda.synchronize()
        e0.record()
        for i in range(reps):
            w.keys_entry(L, w.q_dev[i % w.q_dev.shape[0]], b, stream)
        e1.record()
        torch.cuda.synchronize()
        kern_ms = e0.elapsed_time(e1) / reps
    else:
        kern_ms = sum(step_ms) / len(step_ms)
    tc = ib.knn_tc_last_stats() if w.workload == "knn_cosine_multi" else None
    barrier()

    # ---- query batches of the single-query configs: several queries share every pass over the corpus ------------------
    batch = None
    if hasattr(w, "step_batch") and args.scale >= 0.01:
        nb, reps = w.batch_queries, min(steps, 20)
        for i in range(2):
            w.step_batch(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(reps):
            w.step_batch(i)
        e1.record()
        barrier()
        bms = max_over_ranks(e0.elapsed_time(e1)) / reps
        per_q_units = w.units_per_step  # queries (1) or docs per query
        batch = {"queries_per_call": nb, "ms_per_call": bms, "ms_per_query": bms / nb, "value": per_q_units * nb / (bms / 1e3),
                 "unit": unit, "note": f"{nb} queries share every pass over the corpus; same results as {nb} single calls"}

    # ---- end-to-end through the public API with host buffers ---------------------------------------------
    for i in range(min(warmup, 3)):
        w.step_e2e(i)
    w.e2e_drain()
    barrier()
    t0 = time.perf_counter()
    for i in range(steps):
        w.step_e2e(i)
    w.e2e_drain()  # the last asynchronous call's result is read inside the timed region too
    torch.cuda.synchronize()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    barrier()

    value = w.units_per_step * steps / (total_ms / 1e3)
    e2e_value = w.units_per_step * steps / e2e_s
    peak, peak_src = load_peaks()
    achieved = w.kernel_bytes / (kern_ms / 1e3) / 1e9
    if w.workload == "batch_demo":
        # the 5 MB corpus is L2-resident by construction: no HBM roofline applies; the launch is latency-bound
        roofline = {"bound": "latency", "kernel": w.kernel_name, "achieved": achieved, "peak": None, "unit": "GB/s (from L2)",
                    "frac": None, "traffic": load_traffic(w.workload, args.scale, world),
                    "algorithmic_bytes_per_launch": int(w.kernel_bytes), "kernel_ms": kern_ms,
                    "note": "corpus (5.12 MB) is L2-resident: one launch scores 100 queries; HBM fraction is not meaningful"}
    else:
        roofline = {"bound": "hbm", "kernel": w.kernel_name, "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "traffic": load_traffic(w.workload, args.scale, world),
                    "peak_source": peak_src, "algorithmic_bytes_per_launch": int(w.kernel_bytes), "kernel_ms": kern_ms}
    if tc and tc["passes"] > 0 and tc["filter_ms"] > 0:
        # large query batches: the dominant kernel is the tcgen05 filter (csrc/knn_tc.cu); algorithmic flops per launch =
        # 2 * rows * d * queries of THIS rank, time = CUDA events around that launch inside the library
        tpeak, tsrc = load_tensor_peak()
        flops = 2.0 * w.n_local * w.d * w.nq
        tf = flops / (tc["filter_ms"] / 1e3) / 1e12
        roofline = {"bound": "tensor", "kernel": "knn_tc_filter_kernel (kind::f16, exact rescoring after it)",
                    "achieved": tf, "peak": tpeak, "unit": "TFLOP/s", "frac": tf / tpeak, "traffic": None,
                    "peak_source": tsrc, "algorithmic_flops_per_launch": flops, "kernel_ms": tc["filter_ms"],
                    "call_ms": tc["total_ms"], "filter_passes": tc["passes"], "rescored_pairs": tc["candidates"],
                    "exact_scan_queries": tc["exact_scan_queries"]}
    if w.workload == "maxsim":
        # secondary view (north_star asks for tensor-pipe utilisation): MMA flops the kernel issues per launch -- per
        # 128-token tile one kind::tf32 MMA of N = 64 ([Qhi;Qlo]) and one of N = 32 (Xlo x Qhi), K = 128 -- against the
        # TF32 dense peak, taken as half the measured bf16 figure (not measured separately: stated assumption)
        tpeak, tsrc = load_tensor_peak()
        issued = 2.0 * w.n_local * w.nt * w.dim * (64 + 32)
        roofline["tensor"] = {"issued_tflops": issued / (kern_ms / 1e3) / 1e12, "tf32_peak_assumed": tpeak / 2,
                              "frac": issued / (kern_ms / 1e3) / 1e12 / (tpeak / 2), "peak_source": tsrc + " / 2",
                              "logical_flops_per_launch": 2.0 * w.n_local * w.nt * w.dim * w.nq}
    entry = None
    if rank == 0:
        entry = {
            "metric": metric, "value": value, "unit": unit, "n_gpus": world, "steps": steps, "warmup": warmup,
            "ms_per_step": total_ms / steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": dtype_of(w.workload), "data": "synthetic",
            "config": config_of(w.workload, args.scale, world, args.queries),
            "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": w.h2d, "d2h_bytes_per_step": w.d2h,
                    "mode": ("host-buffer C-ABI calls, asynchronous form (innr_cuda_*_async + innr_cuda_ticket_wait): call i is "
                             "submitted before the result of call i - 1 is collected" if world == 1 and getattr(w, "sk", None) is not None
                             else "one synchronous host-buffer C-ABI call per step" if world == 1
                             else "streamed per rank: pinned query H2D -> shard scan -> peer exchange -> D2H into pinned "
                                  "buffers, double-buffered, one host synchronisation after the last step")},
            "gpu_launches": int(launches),
            "roofline": roofline,
            "clocks": clocks,
        }
        if batch:
            entry["query_batch"] = batch
        if getattr(w, "sk", None) is not None and w.workload not in ("knn_cosine_multi", "batch_demo"):
            entry["step_overlap"] = ("device-resident steps are independent queries: their scans alternate between two streams "
                                     "(two workspaces per device), so the head of scan i+1 fills the SMs under the tail and the "
                                     "merge of scan i; roofline.kernel_ms is the same launch back to back on ONE stream")
        if world > 1:
            entry["exchange"] = env["exchange_desc"] if getattr(w, "sk", None) is not None else "none (documents are independent)"
            if exchange_check:
                entry["exchange_check"] = exchange_check
    return entry


DUMP_SAMPLE = 1 << 20  # elements; a longer output is written as a seeded sample of this many


def dump_outputs(out_dir, workload, arrays):
    """Writes the arrays of one workload's last timed step as <out_dir>/<workload>_<name>.npy: float32 scores as they
    are, indices and integer distances as float64 (exact). An output of more than DUMP_SAMPLE elements is written as the
    values at a fixed, seeded set of flat positions, stored beside it as <workload>_<name>_positions.npy, so that the
    dumps of two builds compare element for element and the whole dump stays under 64 MB."""
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        a = np.asarray(a)
        a = a.astype(np.float32 if a.dtype == np.float32 else np.float64)
        base = os.path.join(out_dir, f"{workload}_{name}")
        if a.size > DUMP_SAMPLE:
            pos = np.sort(np.random.default_rng(0).choice(a.size, DUMP_SAMPLE, replace=False))
            np.save(base + "_positions.npy", pos.astype(np.float64))
            a = a.reshape(-1)[pos]
        np.save(base + ".npy", a)


def run_inproc(args):
    """One process, N GPUs, no torch.distributed: row shards on every device, queries and results in HOST buffers, the
    C-ABI's own sharded entries (persistent worker thread per device + peer-mapped exchange inside the library). Every
    number here is end to end by construction (wall clock around the host-facing call)."""
    import torch
    import innr_b200 as ib
    from innr_b200 import sharded, stream, synth
    n_dev = args.gpus
    if torch.cuda.device_count() < n_dev:
        raise SystemExit(f"--gpus {n_dev} but only {torch.cuda.device_count()} devices are visible")
    peak, peak_src = load_peaks()
    names = ["knn_cosine_1q", "hamming", "u8"] if args.workload == "all" else [args.workload]
    entries = {}
    for name in names:
        cid, _, metric, unit = WORKLOADS[name]
        n, row_bytes = corpus_shape(name, args.scale)
        shards = []
        for dev in range(n_dev):
            ib.init(dev)
            lo, hi = sharded.shard_range(n, dev, n_dev)
            if name == "knn_cosine_1q":
                shards.append(ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, lo, hi - lo, 768, index_base=lo))
            elif name == "hamming":
                shards.append(ib.BinaryCorpus.generate(synth.SALT_CODES, lo, hi - lo, 1024, index_base=lo))
            elif name == "u8":
                shards.append(ib.U8Corpus.generate(synth.SALT_CORPUS, lo, hi - lo, 384, ib.QuantizationParams.from_range(-1.0, 1.0), index_base=lo))
            else:
                raise SystemExit(f"--sharding inproc covers knn_cosine_1q, hamming and u8, not {name}")
        ib.init(0)
        if name == "knn_cosine_1q":
            qs = synth.ghash_f32(synth.SALT_QUERY, 0, 16 * 768).reshape(16, 768)
            call = lambda i: sharded.batch_knn_sharded("cosine", qs[i % 16], shards, 10)  # noqa: E731
            submit = lambda i: stream.submit_knn_sharded("cosine", qs[i % 16], shards, 10)  # noqa: E731
        elif name == "hamming":
            qs = synth.ghash_u64(synth.SALT_QUERY, 0, 16 * 16).reshape(16, 16)
            call = lambda i: sharded.hamming_topk_sharded(qs[i % 16], shards, 100)  # noqa: E731
            submit = lambda i: stream.submit_hamming_topk_sharded(qs[i % 16], shards, 100)  # noqa: E731
        else:
            qs = synth.ghash_f32(synth.SALT_QUERY, 0, 16 * 384).reshape(16, 384)
            call = lambda i: sharded.batch_knn_u8_sharded(qs[i % 16], shards, 10)  # noqa: E731
            submit = lambda i: stream.submit_knn_u8_sharded(qs[i % 16], shards, 10)  # noqa: E731
        for i in range(max(args.warmup, 3)):
            call(i)
        t0 = time.perf_counter()
        for i in range(args.steps):
            call(i)
        dt_sync = time.perf_counter() - t0
        # asynchronous form: call i is submitted before the result of call i - 1 is collected (two in flight)
        pending = None
        for i in range(max(args.warmup, 3)):
            t = submit(i)
            if pending is not None:
                pending.wait()
            pending = t
        pending.wait()
        pending = None
        l0 = ib.launch_count()
        t0 = time.perf_counter()
        for i in range(args.steps):
            t = submit(i)
            if pending is not None:
                pending.wait()
            pending = t
        pending.wait()
        dt = time.perf_counter() - t0
        entries[cid] = {"metric": metric, "value": args.steps / dt, "unit": unit, "n_gpus": n_dev, "steps": args.steps,
                        "warmup": max(args.warmup, 3), "ms_per_step": dt / args.steps * 1e3, "higher_is_better": True,
                        "scaling": "strong", "vs_baseline": None, "dtype": dtype_of(name), "data": "synthetic",
                        "config": config_of(name, args.scale, n_dev, args.queries),
                        "e2e": {"value": args.steps / dt, "unit": unit, "h2d_bytes_per_step": int(qs[0].nbytes) * n_dev,
                                "d2h_bytes_per_step": (100 if name == "hamming" else 10) * 12},
                        "gpu_launches": int(ib.launch_count() - l0),
                        "roofline": {"bound": "hbm", "kernel": "whole host-facing call (wall clock), all devices", "achieved": n * row_bytes / dt * args.steps / 1e9,
                                     "peak": peak * n_dev, "unit": "GB/s", "frac": n * row_bytes / dt * args.steps / 1e9 / (peak * n_dev),
                                     "traffic": None, "peak_source": peak_src + f" x {n_dev}"},
                        "synchronous_ms_per_call": dt_sync / args.steps * 1e3,
                        "exchange": "one process: worker thread per device + peer-mapped mailbox merge on device 0 "
                                    "(innr_cuda_*_sharded_async + innr_cuda_ticket_wait, two calls in flight; "
                                    "synchronous_ms_per_call = innr_cuda_*_sharded)"}
        del shards
        gc.collect()
    first = entries[WORKLOADS[names[0]][0]]
    line = dict(first)
    line["workloads"] = entries
    print(json.dumps(line), flush=True)


def inproc_selfcheck(n_dev, steps):
    """Runs on rank 0 of an N-process job while the other ranks wait on the host: the C-ABI's own sharded entries (ONE
    process driving all N devices: worker thread per device + peer-mapped mailbox merge, what a Rust host would call) on
    a 2M x 768 corpus sharded over the N devices, compared bit for bit with the unsharded call on one device, and timed.
    This is the one place the driver's multi-GPU lease exercises the in-process path."""
    import innr_b200 as ib
    from innr_b200 import sharded, synth
    n, d, k = 2_000_000, 768, 10
    shards = []
    for dev in range(n_dev):
        ib.init(dev)
        lo, hi = sharded.shard_range(n, dev, n_dev)
        shards.append(ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, lo, hi - lo, d, index_base=lo))
    ib.init(0)
    whole = ib.DeviceBatch.generate("ghash", synth.SALT_CORPUS, 0, n, d)
    qs = synth.ghash_f32(synth.SALT_QUERY, 0, 8 * d).reshape(8, d)
    bad = 0
    for j in range(8):
        gi, gs = sharded.batch_knn_sharded("cosine", qs[j], shards, k)
        wi, ws = ib.batch_knn_many("cosine", qs[j], whole, k)
        bad += int(not (np.array_equal(gi, wi) and gs.tobytes() == ws.tobytes()))
    t0 = time.perf_counter()
    for i in range(steps):
        sharded.batch_knn_sharded("cosine", qs[i % 8], shards, k)
    ms = (time.perf_counter() - t0) / steps * 1e3
    t0 = time.perf_counter()
    for i in range(steps):
        ib.batch_knn_many("cosine", qs[i % 8], whole, k)
    ms1 = (time.perf_counter() - t0) / steps * 1e3
    return {"check": "innr_cuda_batch_knn_sharded over %d devices == unsharded call on 8 queries" % n_dev if bad == 0
            else f"MISMATCH on {bad} of 8 queries", "rows": n, "ms_per_call_sharded": ms, "ms_per_call_one_device": ms1,
            "speedup": ms1 / ms, "note": "host buffers in and out, wall clock; one process, worker thread per device"}


def cpu_baseline_entry(w, unit, cache):
    """The oracle on this box's host cores for workload w (rank 0, N == 1 only): one step over the full config."""
    cores = os.cpu_count() or 1
    key = (type(w).__name__, w.n, getattr(w, "d", 0), getattr(w, "metric", ""))
    if key in cache:  # C2b scores the same corpus with the same per-query function as C2a: one query per thread either way
        out = dict(cache[key])
        out["sample"] = "same measurement as C2a (a 1024-query batch is 1024 independent single-query calls on the CPU): " + out["sample"]
        return out
    value, info, s_per_step = w.cpu_measure(cores, full=True, steps=1, warmup=0)
    out = {"value": value, "unit": unit, "kind": "port", "step_s": round(s_per_step, 3), **info}
    if not getattr(w, "demo", False) and w.workload != "maxsim":
        # the small cache-resident sample the round-1 figures were extrapolated from, for comparison
        w._cpu = None
        v2, info2, _ = w.cpu_measure(cores, full=False, steps=1, warmup=0)
        out["small_sample"] = {"value": v2, "rows": info2["rows"], "extrapolated": True}
    cache[key] = out
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=50)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--workload", default="all", choices=sorted(WORKLOADS) + ["all"])
    ap.add_argument("--queries", type=int, default=1024, help="queries per step for knn_cosine_multi")
    ap.add_argument("--scale", type=float, default=1.0, help="corpus size multiplier (1.0 = BASELINE.json size)")
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-inproc-check", action="store_true", help="N > 1: skip rank 0's one-process-all-devices self-check")
    ap.add_argument("--sharding", default="peer", choices=["peer", "nccl", "inproc"],
                    help="N > 1: how the per-shard top-k lists meet -- peer-mapped mailboxes (one launch, default), one "
                         "NCCL allgather + merge launch (the comparison), or `inproc`: ONE process (no torchrun) drives "
                         "all N GPUs through the C-ABI's innr_cuda_*_sharded entries (what a Rust host would call)")
    ap.add_argument("--ref-small-sample", action="store_true",
                    help="reference arm: score a small prefix of the rows and scale (the round-1 behaviour)")
    ap.add_argument("--ref-budget-s", type=float, default=420.0,
                    help="reference arm: wall-clock bound of the whole run; if W + K full-size steps would exceed it, the "
                         "steps after the first use the prefix of the rows that fits (flagged extrapolated)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what each workload's last device-resident timed step returned as DIR/<workload>_<name>.npy "
                         "(rank 0's results at N > 1); the inputs depend only on the arguments")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.sharding == "inproc"):
        ap.error("--dump-outputs covers the device-resident steps of the b200 arm (not --impl reference or --sharding inproc)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    if args.impl == "reference":
        run_reference(args, rank)
        return
    if args.sharding == "inproc":
        if world > 1:
            raise SystemExit("--sharding inproc runs in ONE process: start it with plain `python bench.py --gpus N --sharding inproc`")
        run_inproc(args)
        return

    import torch
    import torch.distributed as dist
    import innr_b200 as ib

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: innr_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device(f"cuda:{local_rank}"))
    ib.init(local_rank)
    env = {"torch": torch, "dist": dist, "ib": ib, "rank": rank, "world": world, "local_rank": local_rank,
           "exchange": None, "exchange_desc": "nccl all_gather_into_tensor of k keys per rank + merge launch"}
    if world > 1 and args.sharding == "peer":
        # mailboxes mapped between the ranks with CUDA IPC; every rank must succeed or all use the NCCL path
        from innr_b200 import sharded
        ex, why = None, ""
        try:
            ex = sharded.PeerExchange.for_process_group(dist)
        except Exception as e:  # e.g. no peer access between the GPUs, IPC not permitted in this container
            why = f"{type(e).__name__}: {e}"[:200]
        ok = torch.tensor([1 if ex is not None else 0], device="cuda")
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        if int(ok.item()) == 1:
            env["exchange"] = ex
            env["exchange_desc"] = ("peer-mapped mailboxes over NVLink (CUDA IPC): publish + wait + merge in one launch, no NCCL on "
                                    "the data path; device-resident steps pipeline it on a side stream under the next scan")
        else:
            env["exchange_desc"] += f" (peer exchange unavailable on some rank: {why or 'see other ranks'})"

    names = ALL_ORDER if args.workload == "all" else [args.workload]
    entries, cpu_cache = {}, {}
    t_all = time.perf_counter()
    for name in names:
        t0 = time.perf_counter()
        w = make_workload(args, name, rank, world)
        try:
            entry = measure(w, args, env)
            if w.last_outputs is not None:
                dump_outputs(args.dump_outputs, name, w.last_outputs)
            if rank == 0 and world == 1 and not args.no_cpu_baseline:
                w.close()  # device memory first: the CPU leg needs the host RAM, not the GPU
                entry["cpu_baseline"] = cpu_baseline_entry(w, WORKLOADS[name][3], cpu_cache)
        except Exception as e:  # one workload must not take the headline down with it
            if name == names[0]:
                raise
            entry = {"error": f"{type(e).__name__}: {e}"[:400]} if rank == 0 else None
        finally:
            w.close()
        if rank == 0:
            entry["wall_s"] = round(time.perf_counter() - t0, 1)
            entries[name] = entry
    inproc = None
    if world > 1 and args.workload == "all" and not args.no_inproc_check:
        # rank 0 drives every device from this one process through the C-ABI's sharded entries; the other ranks wait on
        # the HOST (store key), not in a device-side barrier, so their GPUs are idle for rank 0's kernels
        from torch.distributed.distributed_c10d import _get_default_store
        store = _get_default_store()
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()
        if rank == 0:
            try:
                inproc = inproc_selfcheck(world, min(args.steps, 50))
            except Exception as e:  # never takes the measured line down
                inproc = {"error": f"{type(e).__name__}: {e}"[:300]}
            store.set("innr_inproc_done", "1")
        else:
            store.wait(["innr_inproc_done"])
    if rank == 0:
        line = dict(entries[names[0]])
        if args.workload == "all":
            line["workloads"] = {WORKLOADS[n][0]: entries[n] for n in names}
            line["wall_s"] = round(time.perf_counter() - t_all, 1)
        if inproc:
            line["inproc_check"] = inproc
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
