"""ctypes binding of libinnr_cuda.so (include/innr_cuda.h).

The library is the product; this module only loads it and turns status codes into the exceptions the
reference raises as panics (AssertionError for INNR_EINVAL, so parity tests read like the Rust tests).
There is no fallback: if the shared library is missing or no CUDA device is present, every compute call fails
loudly (RuntimeError).
"""
from __future__ import annotations

import ctypes as C
import os
import subprocess

_HERE = os.path.dirname(os.path.abspath(__file__))
SO_PATH = os.path.join(_HERE, "libinnr_cuda.so")
HEADER_PATH = os.path.join(os.path.dirname(_HERE), "include", "innr_cuda.h")

INNR_OK, INNR_EINVAL, INNR_ECUDA, INNR_ENOMEM, INNR_EUNSUPPORTED, INNR_EBUSY = 0, 1, 2, 3, 4, 5
METRIC_DOT, METRIC_COSINE, METRIC_L2 = 0, 1, 2

f32p = C.POINTER(C.c_float)
u64p = C.POINTER(C.c_uint64)
u32p = C.POINTER(C.c_uint32)
u8p = C.POINTER(C.c_uint8)
szp = C.POINTER(C.c_size_t)
vp = C.c_void_p
sz = C.c_size_t
u64 = C.c_uint64
f32 = C.c_float
ci = C.c_int
handle_p = C.POINTER(vp)

# name -> argtypes (restype is int for all but the two string getters)
SIGNATURES = {
    "innr_cuda_device_count": [C.POINTER(ci)],
    "innr_cuda_init": [ci],
    "innr_cuda_shutdown": [],
    "innr_cuda_dense_backend": [sz, C.POINTER(ci)],
    "innr_cuda_set_option": [C.c_char_p, C.c_double],
    "innr_cuda_knn_tc_last_stats": [f32p, f32p, C.POINTER(C.c_double), u64p, C.POINTER(C.c_uint32), C.POINTER(ci)],
    "innr_cuda_knn_tc_debug_bounds": [vp, ci, f32p, sz, sz, f32p, szp, f32p, u32p],
    "innr_cuda_knn_screen_debug_bounds": [vp, ci, f32p, sz, f32p, f32p],
    "innr_cuda_u8_tc_last_stats": [f32p, f32p, C.POINTER(C.c_double), u64p, C.POINTER(C.c_uint32), C.POINTER(ci)],
    "innr_cuda_bin_tc_last_stats": [f32p, f32p, C.POINTER(C.c_double), u64p, C.POINTER(C.c_uint32), C.POINTER(ci)],
    "innr_cuda_u8_tc_debug_bounds": [vp, f32p, sz, sz, f32p, f32p, szp, u32p],
    "innr_cuda_launch_count": [u64p],
    "innr_cuda_last_kernel_ms": [f32p],
    "innr_cuda_upload_f32_pdx": [f32p, sz, sz, u64, handle_p],
    "innr_cuda_upload_f32_rows": [f32p, sz, sz, u64, handle_p],
    "innr_cuda_wrap_f32_pdx_dev": [vp, sz, sz, sz, u64, handle_p],
    "innr_cuda_prefix_view": [vp, sz, handle_p],
    "innr_cuda_generate_f32_pdx": [ci, u64, u64, sz, sz, u64, handle_p],
    "innr_cuda_free": [vp],
    "innr_cuda_corpus_info": [vp, C.POINTER(ci), szp, szp, szp, u64p, szp],
    "innr_cuda_extract_vector": [vp, sz, f32p],
    "innr_cuda_batch_dot": [vp, f32p, sz, f32p],
    "innr_cuda_batch_l2_squared": [vp, f32p, sz, f32p],
    "innr_cuda_batch_norms": [vp, f32p],
    "innr_cuda_batch_cosine": [vp, f32p, sz, f32p, sz, f32p],
    "innr_cuda_batch_knn": [vp, ci, f32p, sz, sz, sz, u64p, f32p, szp],
    "innr_cuda_batch_knn_subset": [vp, ci, f32p, sz, u64p, sz, sz, u64p, f32p, szp],
    "innr_cuda_binary_from_f32": [vp, f32, handle_p],
    "innr_cuda_u8_from_f32": [vp, f32, f32, handle_p],
    "innr_cuda_batch_knn_filtered": [vp, f32p, sz, sz, u64p, sz, u64p, f32p, szp],
    "innr_cuda_batch_l2_squared_pruning": [vp, f32p, sz, f32, u64p, f32p, sz, szp],
    "innr_cuda_batch_knn_adaptive": [vp, f32p, sz, sz, sz, u64p, f32p, szp],
    "innr_cuda_binary_topk": [vp, ci, u64p, sz, sz, u64p, f32p, szp],
    "innr_cuda_binary_topk_batch": [vp, ci, u64p, sz, sz, sz, u64p, f32p, szp],
    "innr_cuda_binary_topk_keys_dev": [vp, ci, vp, sz, sz, vp, vp],
    "innr_cuda_batch_dimension_variance": [vp, f32p, sz],
    "innr_cuda_batch_knn_reordered": [vp, f32p, sz, sz, u64p, f32p, szp],
    "innr_cuda_batch_knn_keys_dev": [vp, ci, vp, sz, sz, vp, vp],
    "innr_cuda_merge_keys_dev": [vp, sz, sz, sz, ci, vp, vp, vp, vp],
    "innr_cuda_topk_from_distances": [f32p, sz, sz, u32p, f32p, szp],
    "innr_cuda_upload_binary": [u64p, sz, sz, u64, handle_p],
    "innr_cuda_generate_binary": [u64, u64, sz, sz, u64, handle_p],
    "innr_cuda_hamming_all": [vp, u64p, sz, u32p],
    "innr_cuda_binary_dot_all": [vp, u64p, sz, u32p],
    "innr_cuda_binary_jaccard_all": [vp, u64p, sz, f32p],
    "innr_cuda_hamming_topk": [vp, u64p, sz, sz, sz, u64p, u32p, szp],
    "innr_cuda_hamming_topk_keys_dev": [vp, vp, sz, sz, vp, vp],
    "innr_cuda_encode_binary": [f32p, sz, f32, u64p],
    "innr_cuda_upload_ternary": [u64p, sz, sz, u64, handle_p],
    "innr_cuda_ternary_from_f32": [vp, f32, handle_p],
    "innr_cuda_encode_ternary": [f32p, sz, f32, u64p],
    "innr_cuda_ternary_scores_all": [vp, ci, vp, sz, f32p, C.POINTER(C.c_int32)],
    "innr_cuda_ternary_topk": [vp, ci, vp, sz, sz, u64p, f32p, szp],
    "innr_cuda_upload_u8": [u8p, sz, sz, f32, f32, u64, handle_p],
    "innr_cuda_generate_u8": [u64, u64, sz, sz, f32, f32, u64, handle_p],
    "innr_cuda_quantize_u8": [f32p, sz, f32, f32, u8p],
    "innr_cuda_mixed_dot_u8_all": [vp, f32p, sz, f32p],
    "innr_cuda_asymmetric_dot_u8_all": [vp, f32p, sz, f32p],
    "innr_cuda_batch_knn_u8": [vp, f32p, sz, sz, sz, u64p, f32p, szp],
    "innr_cuda_batch_knn_u8_keys_dev": [vp, vp, sz, sz, vp, vp],
    "innr_cuda_upload_tokens": [f32p, u64p, sz, sz, u64, handle_p],
    "innr_cuda_generate_tokens": [u64, u64, sz, sz, sz, u64, handle_p],
    "innr_cuda_maxsim": [vp, f32p, sz, sz, ci, f32p],
    "innr_cuda_batch_knn_sharded": [vp, sz, ci, f32p, sz, sz, sz, u64p, f32p, szp],
    "innr_cuda_hamming_topk_sharded": [vp, sz, u64p, sz, sz, sz, u64p, u32p, szp],
    "innr_cuda_batch_knn_u8_sharded": [vp, sz, f32p, sz, sz, sz, u64p, f32p, szp],
    "innr_cuda_batch_knn_async": [vp, ci, f32p, sz, sz, sz, handle_p],
    "innr_cuda_hamming_topk_async": [vp, u64p, sz, sz, sz, handle_p],
    "innr_cuda_batch_knn_u8_async": [vp, f32p, sz, sz, sz, handle_p],
    "innr_cuda_ticket_wait": [vp, u64p, f32p, u32p, szp],
    "innr_cuda_batch_knn_sharded_async": [vp, sz, ci, f32p, sz, sz, sz, handle_p],
    "innr_cuda_hamming_topk_sharded_async": [vp, sz, u64p, sz, sz, sz, handle_p],
    "innr_cuda_batch_knn_u8_sharded_async": [vp, sz, f32p, sz, sz, sz, handle_p],
    "innr_cuda_exchange_create": [ci, ci, sz, handle_p],
    "innr_cuda_exchange_ipc_handle": [vp, vp],
    "innr_cuda_exchange_connect_ipc": [vp, vp],
    "innr_cuda_exchange_connect_local": [vp, ci],
    "innr_cuda_exchange_free": [vp],
    "innr_cuda_exchange_set_timeout_ms": [vp, C.c_double],
    "innr_cuda_exchange_status": [vp, C.POINTER(ci)],
    "innr_cuda_exchange_merge_dev": [vp, vp, sz, sz, ci, ci, vp, vp, vp, vp, vp],
    "innr_cuda_maxsim_batch": [vp, f32p, sz, sz, sz, ci, f32p],
    "innr_cuda_maxsim_batch_dev": [vp, vp, sz, sz, ci, vp, vp],
    "innr_cuda_maxsim_dev": [vp, vp, sz, ci, vp, vp],
    "innr_cuda_maxsim_topk": [vp, f32p, sz, sz, sz, ci, sz, u64p, f32p, szp],
    "innr_cuda_maxsim_topk_keys_dev": [vp, vp, sz, sz, ci, sz, vp, vp],
    "innr_cuda_maxsim_topk_async": [vp, f32p, sz, sz, sz, ci, sz, handle_p],
    "innr_cuda_maxsim_topk_sharded": [vp, sz, f32p, sz, sz, sz, ci, sz, u64p, f32p, szp],
    "innr_cuda_maxsim_topk_sharded_async": [vp, sz, f32p, sz, sz, sz, ci, sz, handle_p],
}
STRING_GETTERS = ("innr_cuda_last_error", "innr_cuda_backend_name")

_lib = None


def build(verbose: bool = False) -> str:
    """Compile libinnr_cuda.so with nvcc for sm_100a (csrc/Makefile). Cross-compiles without a GPU."""
    subprocess.check_call(["make", "-C", os.path.join(_HERE, "csrc"), "-j8"] + ([] if verbose else ["-s"]))
    return SO_PATH


def lib() -> C.CDLL:
    global _lib
    if _lib is None:
        if not os.path.exists(SO_PATH):
            raise RuntimeError(
                f"{SO_PATH} is missing: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
                "(innr_b200 has no CPU fallback)")
        L = C.CDLL(SO_PATH)
        for name, args in SIGNATURES.items():
            fn = getattr(L, name)
            fn.restype = ci
            fn.argtypes = args
        for name in STRING_GETTERS:
            getattr(L, name).restype = C.c_char_p
            getattr(L, name).argtypes = []
        _lib = L
    return _lib


class InnrCudaError(RuntimeError):
    pass


def check(rc: int) -> None:
    if rc == INNR_OK:
        return
    msg = lib().innr_cuda_last_error().decode()
    if rc == INNR_EINVAL:
        raise AssertionError(msg)  # the reference panics (assert_eq!) on these
    if rc == INNR_EUNSUPPORTED:
        raise NotImplementedError(msg)
    if rc == INNR_ENOMEM:
        raise MemoryError(msg)
    raise InnrCudaError(msg)


def call(name: str, *args) -> None:
    check(getattr(lib(), name)(*args))


def backend_name() -> str:
    return lib().innr_cuda_backend_name().decode()


def launch_count() -> int:
    v = C.c_uint64(0)
    call("innr_cuda_launch_count", C.byref(v))
    return int(v.value)


def last_kernel_ms() -> float:
    """Device time of the last host-facing call's kernels; recorded only after set_option("kernel_timing", 1)."""
    v = C.c_float(0)
    call("innr_cuda_last_kernel_ms", C.byref(v))
    return float(v.value)


def knn_tc_last_stats() -> dict:
    """Statistics of the most recent batch_knn call that used the tensor-core filter (include/innr_cuda.h)."""
    f, t, fl, cand, ex, p = C.c_float(), C.c_float(), C.c_double(), C.c_uint64(), C.c_uint32(), C.c_int()
    call("innr_cuda_knn_tc_last_stats", C.byref(f), C.byref(t), C.byref(fl), C.byref(cand), C.byref(ex), C.byref(p))
    return {"filter_ms": f.value, "total_ms": t.value, "filter_flops": fl.value, "candidates": cand.value,
            "exact_scan_queries": ex.value, "passes": p.value}


def u8_tc_last_stats() -> dict:
    """Statistics of the most recent batch_knn_u8 call that used the tensor-core filter (include/innr_cuda.h)."""
    f, t, ops, cand, ex, p = C.c_float(), C.c_float(), C.c_double(), C.c_uint64(), C.c_uint32(), C.c_int()
    call("innr_cuda_u8_tc_last_stats", C.byref(f), C.byref(t), C.byref(ops), C.byref(cand), C.byref(ex), C.byref(p))
    return {"filter_ms": f.value, "total_ms": t.value, "filter_ops": ops.value, "candidates": cand.value,
            "exact_scan_queries": ex.value, "passes": p.value}


def bin_tc_last_stats() -> dict:
    """Statistics of the most recent binary top-k call that used the tensor-core filter (include/innr_cuda.h). Waits for
    that call to finish on the device."""
    f, t, ops, cand, ex, p = C.c_float(), C.c_float(), C.c_double(), C.c_uint64(), C.c_uint32(), C.c_int()
    call("innr_cuda_bin_tc_last_stats", C.byref(f), C.byref(t), C.byref(ops), C.byref(cand), C.byref(ex), C.byref(p))
    return {"filter_ms": f.value, "total_ms": t.value, "filter_ops": ops.value, "candidates": cand.value,
            "exact_scan_queries": ex.value, "passes": p.value}


def set_option(name: str, value: float) -> None:
    """Tuning knobs of the library (see include/innr_cuda.h); results never depend on them."""
    call("innr_cuda_set_option", name.encode(), float(value))


def init(device: int = 0) -> None:
    call("innr_cuda_init", device)
