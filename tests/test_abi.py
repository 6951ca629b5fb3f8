"""CPU-side checks of the drop-in boundary: libinnr_cuda.so loads, exports every symbol include/innr_cuda.h
declares (and nothing is bound that the header lacks), and the product fails loudly without a CUDA device."""
import ctypes
import os
import re

import numpy as np
import pytest

import innr_b200
from innr_b200 import _lib as L

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _header_symbols():
    text = open(os.path.join(ROOT, "include", "innr_cuda.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(innr_cuda_[a-z0-9_]+)\s*\(", text)))


def test_library_exports_every_header_symbol():
    if not os.path.exists(L.SO_PATH):
        innr_b200.build()
    lib = ctypes.CDLL(L.SO_PATH)
    syms = _header_symbols()
    assert len(syms) >= 35
    for s in syms:
        assert hasattr(lib, s), f"{s} declared in include/innr_cuda.h but not exported"


def test_python_binding_covers_the_header():
    declared = set(_header_symbols())
    bound = set(L.SIGNATURES) | set(L.STRING_GETTERS)
    assert declared == bound, (sorted(declared - bound), sorted(bound - declared))
    L.lib()  # binds argtypes for every symbol


def test_backend_string_and_enum():
    assert innr_b200.backend_name() == "cuda"                       # new Backend::Cuda Display string
    assert str(innr_b200.Backend.Avx512) == "avx512" and str(innr_b200.Backend.Portable) == "portable"  # src/backend.rs:114-120
    assert str(innr_b200.Backend.Cuda) == "cuda"


def test_no_cpu_fallback_without_device():
    import torch
    if torch.cuda.is_available():
        pytest.skip("a CUDA device is present")
    b = innr_b200.VerticalBatch.from_rows([[1.0, 2.0], [3.0, 4.0]])   # host-side layout only
    assert b.get(1, 0) == 2.0
    with pytest.raises(innr_b200.InnrCudaError, match="no CPU fallback"):
        innr_b200.batch_dot([1.0, 1.0], b)
    with pytest.raises(innr_b200.InnrCudaError):
        innr_b200.encode_binary([1.0, -1.0], 0.0)
    with pytest.raises(innr_b200.InnrCudaError):
        innr_b200.quantize_u8([0.5], innr_b200.QuantizationParams.from_range(0.0, 1.0))
    from innr_b200 import stream
    with pytest.raises(innr_b200.InnrCudaError):   # the asynchronous forms upload lazily like the synchronous ones
        stream.submit_knn("dot", [1.0, 1.0], b, 1)


def test_host_side_types_match_reference_contracts():
    pb = innr_b200.PackedBinary([0xFFFFFFFFFFFFFFFF], 8)              # src/binary.rs:59-66 padding mask
    assert int(pb.data[0]) == 0xFF
    with pytest.raises(AssertionError):
        innr_b200.PackedBinary([0, 0], 8)
    p = innr_b200.QuantizationParams.from_range(1.0, 1.0)             # alpha <= 0 -> 1.0 (src/scalar.rs:54-60)
    assert p.alpha == 1.0 and p.offset == 1.0
    with pytest.raises(AssertionError):
        innr_b200.QuantizedU8([1, 2, 3], 2)
    vb = innr_b200.VerticalBatch.from_rows([[1.0, 2.0, 3.0], [4.0, 5.0, 6.0]])
    assert list(vb.dimension_slice(1)) == [2.0, 5.0] and list(vb.data) == [1.0, 4.0, 2.0, 5.0, 3.0, 6.0]
    with pytest.raises(AssertionError):
        innr_b200.VerticalBatch.from_rows([[1.0], [1.0, 2.0]])


def _strip_rust(text):
    """Rust source without comments and string literals (enough for the structural checks below)."""
    text = re.sub(r"//[^\n]*", "", text)
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return re.sub(r'"(?:\\.|[^"\\])*"', '""', text)


RUST_STD_NAMES = {"Self", "Vec", "Result", "Option", "Ok", "Err", "Some", "None", "String", "CStr", "CString", "Send", "Sync",
                  "Drop", "Fn", "F", "T", "Default", "Clone", "Debug", "PartialEq", "Eq", "Copy", "Arc", "OnceLock",
                  "PhantomData", "Deref", "Target", "Display", "Formatter", "INNR_OK", "INNR_EINVAL", "INNR_METRIC_DOT",
                  "INNR_METRIC_COSINE", "INNR_METRIC_L2", "INNR_TERNARY_DOT", "INNR_TERNARY_HAMMING",
                  "INNR_TERNARY_ASYMMETRIC_DOT", "AVAILABLE", "MIN_DEVICE_ELEMENTS"}


def _rust_fn_bodies(text):
    """(name, body) of every fn item with a body, by brace matching on comment- and string-free source."""
    out = []
    for m in re.finditer(r"\bfn\s+([a-z_][a-z0-9_]*)\s*(?:<[^{;]*?>)?\s*\(", text):
        j = text.find("{", m.end())
        semi = text.find(";", m.end())
        if j < 0 or (0 <= semi < j):
            continue  # a declaration (extern block / trait), not a definition
        depth, k = 0, j
        while k < len(text):
            depth += text[k] == "{"
            depth -= text[k] == "}"
            if depth == 0:
                break
            k += 1
        out.append((m.group(1), text[j + 1:k]))
    return out


def _check_rust_source(path, extra_defined=()):
    text = _strip_rust(open(path).read())
    bodies = _rust_fn_bodies(text)
    assert len(bodies) >= 10, path
    for name, body in bodies:
        assert body.strip(), f"{path}: fn {name} has an empty (comment-only) body"
    defined = set(re.findall(r"\b(?:struct|enum|type|trait|union)\s+([A-Z][A-Za-z0-9]*)", text)) | set(extra_defined)
    defined |= set(re.findall(r"\b([A-Z][A-Za-z0-9]*)\s*(?:\(|=>|,|\})", "".join(re.findall(r"enum\s+\w+\s*\{([^}]*)\}", text))))
    used = set(re.findall(r"\b([A-Z][A-Za-z0-9_]*)\b", text))
    unknown = sorted(u for u in used if u not in defined and u not in RUST_STD_NAMES)
    assert not unknown, f"{path}: type names used but not defined anywhere: {unknown}"
    return text, {n for n, _ in bodies}


def test_rust_shim_is_complete_source():
    """innr-cuda/ (the reference-side binding; no Rust toolchain exists here, so it cannot be compiled) must at least be
    structurally whole: sys.rs is exactly what gen_sys.py derives from include/innr_cuda.h (every symbol, right arity);
    every function of the safe layer has a body; no type name is used that is not defined; every FFI symbol the safe
    layer calls is declared; every reference function of SURVEY 8a has a wrapper; build.rs compiles the real csrc/."""
    import subprocess
    import sys
    shim = os.path.join(ROOT, "innr-cuda")
    assert subprocess.run([sys.executable, os.path.join(shim, "gen_sys.py"), "--check"]).returncode == 0, \
        "innr-cuda/src/sys.rs is stale: run python innr-cuda/gen_sys.py"
    sys_text = open(os.path.join(shim, "src", "sys.rs")).read()
    declared = set(re.findall(r"pub fn (innr_cuda_[a-z0-9_]+)\s*\(", sys_text))
    assert declared == set(_header_symbols())
    header = re.sub(r"/\*.*?\*/", "", open(os.path.join(ROOT, "include", "innr_cuda.h")).read(), flags=re.S)
    for name in declared:  # arity of every declaration
        c_params = re.search(rf"\b{name}\s*\(([^)]*)\)", header).group(1).strip()
        n_c = 0 if c_params in ("", "void") else c_params.count(",") + 1
        r_params = re.search(rf"pub fn {name}\(([^)]*)\)", sys_text).group(1).strip()
        n_r = 0 if not r_params else r_params.count(",") + 1
        assert n_c == n_r, (name, n_c, n_r)
    text, fns = _check_rust_source(os.path.join(shim, "src", "lib.rs"), extra_defined={"innr_cuda_corpus", "innr_cuda_exchange", "innr_cuda_ticket"})
    called = set(re.findall(r"\b(innr_cuda_[a-z0-9_]+)\s*\(", text))
    assert called <= declared, sorted(called - declared)
    # SURVEY 8a: one wrapper per reference function of the path
    for need in ("from_pdx", "from_rows", "extract_vector", "dot_into", "l2_squared_into", "norms_into", "cosine_into", "knn",
                 "knn_many", "knn_filtered", "l2_squared_pruning", "topk_from_distances", "from_words", "hamming_all",
                 "hamming_top_k", "encode_binary", "quantize_u8", "mixed_dot_all", "asymmetric_dot_all", "from_tokens", "maxsim",
                 "maxsim_batch", "knn_sharded", "hamming_top_k_sharded", "knn_u8_sharded", "backend_name"):
        assert need in fns, f"innr-cuda/src/lib.rs lacks a wrapper `{need}`"
    build = open(os.path.join(shim, "build.rs")).read()
    assert '"innr_b200"' in build and '"csrc"' in build and "compute_100a" in build and "-ffp-contract=off" in build
    cargo = open(os.path.join(shim, "Cargo.toml")).read()
    assert not re.search(r"^innr\s*=", cargo, flags=re.M), "innr-cuda must not depend on innr (innr's cuda feature depends on it)"


PATCH = os.path.join(ROOT, "integration", "innr-cuda.patch")
CUDA_RS_DEFINED_ELSEWHERE = {"VerticalBatch", "BatchKnnResult", "PackedBinary", "QuantizedU8", "QuantizationParams", "Error",
                             "Metric", "F32Corpus", "BinaryCorpus", "U8Corpus", "TokenCorpus", "L2", "Dot", "Cosine"}
CUDA_FEATURE_GATE = '#[cfg(feature = "cuda")]'


def _patch_sections(ptxt):
    """{path in the patched tree: (lines added, lines removed)} of a unified diff."""
    out, cur = {}, None
    for line in ptxt.splitlines():
        if line.startswith("+++ b/"):
            cur = out.setdefault(line[len("+++ b/"):].split("\t")[0], ([], []))
        elif line.startswith(("--- ", "diff ")):
            continue
        elif cur is not None and line[:1] in ("+", "-"):
            cur[line[0] == "-"].append(line[1:])
    return out


def _check_cuda_rs(path):
    """src/cuda.rs of the patched reference: whole, every adapter of the feature present, and every call into innr-cuda
    defined by innr-cuda/src/lib.rs."""
    text, fns = _check_rust_source(path, extra_defined=CUDA_RS_DEFINED_ELSEWHERE)
    for need in ("from_batch", "knn_l2", "knn_dot", "knn_cosine", "l2_squared_into", "dot_into", "norms_into", "cosine_into",
                 "from_codes", "hamming_top_k", "from_quantized", "batch_knn_u8", "from_docs", "maxsim", "maxsim_cosine",
                 "get_or_upload", "device_available"):
        assert need in fns, f"src/cuda.rs lacks `{need}`"
    lib_methods = _check_rust_source(os.path.join(ROOT, "innr-cuda", "src", "lib.rs"),
                                     extra_defined={"innr_cuda_corpus", "innr_cuda_exchange", "innr_cuda_ticket"})[1]
    for m in set(re.findall(r"self\.inner\.([a-z_0-9]+)\(", text)):   # every call into innr-cuda exists there
        assert m in lib_methods, f"src/cuda.rs calls innr_cuda::*::{m}, which innr-cuda/src/lib.rs does not define"


def test_integration_patch_is_whole(tmp_path):
    """integration/innr-cuda.patch (Backend::Cuda, the `cuda` feature, feature-gated branches, src/cuda.rs) is
    structurally whole, read from the patch alone: src/cuda.rs is a new file, so its whole text is in the patch, and the
    feature-gated branches it adds to src/batch.rs are counted on the added lines."""
    ptxt = open(PATCH).read()
    for needle in ('+    Cuda,', '+            Backend::Cuda => "cuda",', '+cuda = ["dep:innr-cuda"]', '+pub mod cuda;',
                   '+    if let Some(dev) = batch.device() {', '+++ b/src/cuda.rs'):
        assert needle in ptxt, needle
    sections = _patch_sections(ptxt)
    added, removed = sections["src/cuda.rs"]
    assert added and not removed
    (tmp_path / "cuda.rs").write_text("\n".join(added) + "\n")
    _check_cuda_rs(str(tmp_path / "cuda.rs"))
    assert "\n".join(sections["src/batch.rs"][0]).count(CUDA_FEATURE_GATE) >= 13


def test_integration_patch_applies_to_the_reference():
    """integration/innr-cuda.patch applies cleanly to the reference tree, and the patched tree passes the checks of
    test_integration_patch_is_whole. The reference (innr 0.6.3, a Rust crate) is not part of this repository: point
    INNR_REFERENCE_DIR at a checkout of it to run this test."""
    import shutil
    import subprocess
    import tempfile
    ref = os.environ.get("INNR_REFERENCE_DIR", "")
    if not os.path.isdir(ref):
        pytest.skip("INNR_REFERENCE_DIR does not name a checkout of innr 0.6.3")
    with tempfile.TemporaryDirectory() as tmp:
        shutil.copy(os.path.join(ref, "Cargo.toml"), tmp)
        shutil.copytree(os.path.join(ref, "src"), os.path.join(tmp, "src"))
        r = subprocess.run(["patch", "-p1", "--batch", "-i", PATCH], cwd=tmp, capture_output=True, text=True)
        assert r.returncode == 0, r.stdout + r.stderr
        _check_cuda_rs(os.path.join(tmp, "src", "cuda.rs"))
        batch = open(os.path.join(tmp, "src", "batch.rs")).read()
        assert batch.count(CUDA_FEATURE_GATE) >= 13
