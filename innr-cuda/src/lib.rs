//! innr-cuda: B200 (sm_100a) device path for innr's batch similarity-search hot path.
//!
//! * [`sys`] -- the `extern "C"` block, generated from `include/innr_cuda.h` (`gen_sys.py`).
//! * this module -- a safe layer in terms of plain slices: RAII corpus handles (`F32Corpus`, `BinaryCorpus`,
//!   `U8Corpus`, `TokenCorpus`, `TernaryCorpus`) and one method per reference function of the path. It deliberately
//!   does NOT depend on `innr` (innr's `cuda` feature depends on this crate; the glue that speaks innr's own types --
//!   `VerticalBatch`, `BatchKnnResult`, `PackedBinary`, `QuantizedU8` -- is `src/cuda.rs` inside innr, added by
//!   `integration/innr-cuda.patch`).
//!
//! Every wrapper panics where the reference panics (`assert_eq!` on length / dimension mismatches, with the reference's
//! message) BEFORE crossing the FFI boundary, and turns any other non-zero status into `Err(Error)`.
//!
//! NOT COMPILED IN THE AUTHORING ENVIRONMENT (no cargo/rustc there). The C-ABI underneath is built and tested through
//! Python ctypes bindings of the same symbols; `tests/test_abi.py` keeps `sys.rs` in sync with the header and checks that
//! every function here has a body and only uses types that are defined.

pub mod sys;

use core::ffi::{c_int, c_void};
use std::ffi::{CStr, CString};
use sys::*;

// ------------------------------------------------------------------------------------------------ errors
/// A non-zero status of the C-ABI with the library's thread-local message.
#[derive(Debug, Clone, PartialEq, Eq)]
pub struct Error {
    /// `INNR_EINVAL` (1), `INNR_ECUDA` (2), `INNR_ENOMEM` (3), `INNR_EUNSUPPORTED` (4) or `INNR_EBUSY` (5).
    pub code: i32,
    /// `innr_cuda_last_error()` at the time of the failure.
    pub message: String,
}

impl core::fmt::Display for Error {
    fn fmt(&self, f: &mut core::fmt::Formatter<'_>) -> core::fmt::Result {
        write!(f, "innr-cuda error {}: {}", self.code, self.message)
    }
}

impl std::error::Error for Error {}

/// Result alias of this crate.
pub type Result<T> = core::result::Result<T, Error>;

fn check(rc: c_int) -> Result<()> {
    if rc == INNR_OK {
        return Ok(());
    }
    let message = unsafe { CStr::from_ptr(innr_cuda_last_error()) }.to_string_lossy().into_owned();
    Err(Error { code: rc as i32, message })
}

// ------------------------------------------------------------------------------------------------ library / device
/// Number of CUDA devices the library can see (0 without a driver: there is no CPU fallback).
pub fn device_count() -> usize {
    let mut n: c_int = 0;
    let _ = unsafe { innr_cuda_device_count(&mut n) };
    n.max(0) as usize
}

/// Binds the calling thread's subsequent uploads to `device` and creates its stream and workspace.
pub fn init(device: usize) -> Result<()> {
    check(unsafe { innr_cuda_init(device as c_int) })
}

/// Display string of `Backend::Cuda` (src/backend.rs:31-41 keeps these strings stable): `"cuda"`.
pub fn backend_name() -> &'static str {
    unsafe { CStr::from_ptr(innr_cuda_backend_name()) }.to_str().unwrap_or("cuda")
}

/// Tuning knob of the library (see the header); results never depend on them.
pub fn set_option(name: &str, value: f64) -> Result<()> {
    let c = CString::new(name).map_err(|_| Error { code: INNR_EINVAL as i32, message: "option name contains NUL".into() })?;
    check(unsafe { innr_cuda_set_option(c.as_ptr(), value) })
}

/// Metric selector of the f32 scans.
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
pub enum Metric {
    /// `batch_dot` / `batch_knn_dot` (src/batch.rs:270, :742): descending.
    Dot,
    /// `batch_cosine` / `batch_knn_cosine` (src/batch.rs:690, :777): descending.
    Cosine,
    /// `batch_l2_squared` / `batch_knn` (src/batch.rs:236, :385): ascending.
    L2,
}

impl Metric {
    fn id(self) -> c_int {
        match self {
            Metric::Dot => INNR_METRIC_DOT,
            Metric::Cosine => INNR_METRIC_COSINE,
            Metric::L2 => INNR_METRIC_L2,
        }
    }
}

/// Owns one `innr_cuda_corpus*`. Immutable after upload, hence `Send + Sync` (calls are serialised per device inside
/// the library).
struct Handle(*mut innr_cuda_corpus);
unsafe impl Send for Handle {}
unsafe impl Sync for Handle {}
impl Drop for Handle {
    fn drop(&mut self) {
        if !self.0.is_null() {
            unsafe { innr_cuda_free(self.0) };
        }
    }
}

fn knn_buffers(n_queries: usize, k: usize) -> (Vec<u64>, Vec<f32>) {
    let len = (n_queries * k).max(1);
    (vec![0u64; len], vec![0f32; len])
}

fn split_results(idx: Vec<u64>, sc: Vec<f32>, n_queries: usize, k: usize, count: usize) -> Vec<(Vec<usize>, Vec<f32>)> {
    (0..n_queries)
        .map(|q| {
            let lo = q * k;
            (idx[lo..lo + count].iter().map(|&i| i as usize).collect(), sc[lo..lo + count].to_vec())
        })
        .collect()
}

// ------------------------------------------------------------------------------------------------ f32 PDX corpus
/// Device-resident `VerticalBatch` (src/batch.rs:88-220): dimension-major `data[d * n + i]`.
pub struct F32Corpus {
    h: Handle,
    n: usize,
    d: usize,
    index_base: u64,
}

impl F32Corpus {
    /// `pdx` is exactly what `VerticalBatch::data()` returns (src/batch.rs:212). `index_base` is added to reported
    /// indices (row shards report global indices).
    pub fn from_pdx(pdx: &[f32], n: usize, d: usize, index_base: u64) -> Result<Self> {
        assert_eq!(pdx.len(), n * d, "Data length must equal num_vectors * dimension"); // src/batch.rs:168-172
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_upload_f32_pdx(pdx.as_ptr(), n, d, index_base, &mut h) })?;
        Ok(Self { h: Handle(h), n, d, index_base })
    }

    /// Row-major `n x d` input of `VerticalBatch::from_flat` (src/batch.rs:167); transposed on the device.
    pub fn from_rows(rows: &[f32], n: usize, d: usize, index_base: u64) -> Result<Self> {
        assert_eq!(rows.len(), n * d, "Data length must equal num_vectors * dimension");
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_upload_f32_rows(rows.as_ptr(), n, d, index_base, &mut h) })?;
        Ok(Self { h: Handle(h), n, d, index_base })
    }

    /// `VerticalBatch::num_vectors` (src/batch.rs:199).
    pub fn num_vectors(&self) -> usize {
        self.n
    }

    /// `VerticalBatch::dimension` (src/batch.rs:204).
    pub fn dimension(&self) -> usize {
        self.d
    }

    /// First global index of this shard.
    pub fn index_base(&self) -> u64 {
        self.index_base
    }

    /// Raw handle for the `_dev` / sharded entries of [`sys`].
    pub fn as_ptr(&self) -> *const innr_cuda_corpus {
        self.h.0
    }

    /// `VerticalBatch::extract_vector` (src/batch.rs:217).
    pub fn extract_vector(&self, vec_idx: usize) -> Result<Vec<f32>> {
        assert!(vec_idx < self.n, "index out of bounds");
        let mut out = vec![0f32; self.d];
        check(unsafe { innr_cuda_extract_vector(self.h.0, vec_idx, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// Matryoshka prefix (pairwise forms: src/dense.rs:436-462): a zero-copy view of the first `prefix_dim` dimensions.
    /// The view borrows `self`, so it cannot outlive the corpus whose memory it shares.
    pub fn prefix(&self, prefix_dim: usize) -> Result<F32View<'_>> {
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_prefix_view(self.h.0, prefix_dim, &mut h) })?;
        Ok(F32View {
            inner: F32Corpus { h: Handle(h), n: self.n, d: prefix_dim.min(self.d), index_base: self.index_base },
            _parent: core::marker::PhantomData,
        })
    }

    /// `batch_dot_into` (src/batch.rs:284-297).
    pub fn dot_into(&self, query: &[f32], products: &mut Vec<f32>) -> Result<()> {
        assert_eq!(query.len(), self.d); // src/batch.rs:285
        products.clear();
        products.resize(self.n, 0.0);
        check(unsafe { innr_cuda_batch_dot(self.h.0, query.as_ptr(), query.len(), products.as_mut_ptr()) })
    }

    /// `batch_l2_squared_into` (src/batch.rs:250-266).
    pub fn l2_squared_into(&self, query: &[f32], distances: &mut Vec<f32>) -> Result<()> {
        assert_eq!(query.len(), self.d); // src/batch.rs:251
        distances.clear();
        distances.resize(self.n, 0.0);
        check(unsafe { innr_cuda_batch_l2_squared(self.h.0, query.as_ptr(), query.len(), distances.as_mut_ptr()) })
    }

    /// `batch_norms_into` (src/batch.rs:672-686).
    pub fn norms_into(&self, norms: &mut Vec<f32>) -> Result<()> {
        norms.clear();
        norms.resize(self.n, 0.0);
        check(unsafe { innr_cuda_batch_norms(self.h.0, norms.as_mut_ptr()) })
    }

    /// `batch_cosine_into` (src/batch.rs:705-728) with caller-supplied norms.
    pub fn cosine_into(&self, query: &[f32], norms: &[f32], similarities: &mut Vec<f32>) -> Result<()> {
        assert_eq!(query.len(), self.d); // src/batch.rs:710
        assert_eq!(norms.len(), self.n); // src/batch.rs:711
        similarities.clear();
        similarities.resize(self.n, 0.0);
        check(unsafe {
            innr_cuda_batch_cosine(self.h.0, query.as_ptr(), query.len(), norms.as_ptr(), norms.len(), similarities.as_mut_ptr())
        })
    }

    /// `batch_knn` / `batch_knn_dot` / `batch_knn_cosine` (src/batch.rs:385, :742, :777): `(indices, scores)`, k clamped
    /// to N, empty when N == 0 or k == 0, ties -> lower index.
    pub fn knn(&self, metric: Metric, query: &[f32], k: usize) -> Result<(Vec<usize>, Vec<f32>)> {
        Ok(self.knn_many(metric, query, 1, k)?.pop().unwrap_or_default())
    }

    /// `n_queries x d` row-major queries in ONE call (corpus passes are shared between queries; from two queries on a
    /// large corpus the tensor-core filter + exact rescoring path runs). Same results as `n_queries` single calls.
    pub fn knn_many(&self, metric: Metric, queries: &[f32], n_queries: usize, k: usize) -> Result<Vec<(Vec<usize>, Vec<f32>)>> {
        assert_eq!(queries.len(), n_queries * self.d); // src/batch.rs:386 / :743 / :778, per query
        let (mut idx, mut sc) = knn_buffers(n_queries, k);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_batch_knn(self.h.0, metric.id(), queries.as_ptr(), n_queries, self.d, k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        Ok(split_results(idx, sc, n_queries, k, count))
    }

    /// Asynchronous `knn_many`: queues the call and returns at once; `Ticket::wait` blocks on this call only and gives
    /// what `knn_many` gives. Two tickets per device may be in flight -- submitting call i + 1 before waiting for call i
    /// keeps two scans overlapping on the device.
    pub fn knn_submit(&self, metric: Metric, queries: &[f32], n_queries: usize, k: usize) -> Result<Ticket> {
        assert_eq!(queries.len(), n_queries * self.d); // src/batch.rs:386 / :743 / :778, per query
        let mut t: *mut innr_cuda_ticket = std::ptr::null_mut();
        check(unsafe { innr_cuda_batch_knn_async(self.h.0, metric.id(), queries.as_ptr(), n_queries, self.d, k, &mut t) })?;
        Ok(Ticket { t, n_queries, k, binary: false })
    }

    /// `batch_knn_filtered` (src/batch.rs:820-882). The closure is evaluated into a bitmask here (the reference builds
    /// `mask: Vec<bool>` itself, :839); rows of rejected vectors are never read on the device.
    pub fn knn_filtered<F: Fn(usize) -> bool>(&self, query: &[f32], k: usize, predicate: F) -> Result<(Vec<usize>, Vec<f32>)> {
        assert_eq!(query.len(), self.d); // src/batch.rs:829
        let mut mask = vec![0u64; (self.n + 63) / 64];
        for i in 0..self.n {
            if predicate(i) {
                mask[i / 64] |= 1u64 << (i % 64);
            }
        }
        let (mut idx, mut sc) = knn_buffers(1, k.min(self.n));
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_batch_knn_filtered(self.h.0, query.as_ptr(), query.len(), k, mask.as_ptr(), mask.len(), idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        idx.truncate(count);
        sc.truncate(count);
        Ok((idx.into_iter().map(|i| i as usize).collect(), sc))
    }

    /// `batch_l2_squared_pruning` (src/batch.rs:320-365): survivors in ascending index order.
    pub fn l2_squared_pruning(&self, query: &[f32], threshold: f32) -> Result<Vec<(usize, f32)>> {
        assert_eq!(query.len(), self.d); // src/batch.rs:325
        let cap = self.n.max(1);
        let (mut idx, mut dist) = (vec![0u64; cap], vec![0f32; cap]);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_batch_l2_squared_pruning(self.h.0, query.as_ptr(), query.len(), threshold, idx.as_mut_ptr(), dist.as_mut_ptr(), self.n, &mut count)
        })?;
        Ok(idx.into_iter().zip(dist).take(count).map(|(i, d)| (i as usize, d)).collect())
    }

    /// `batch_dimension_variance` (src/batch.rs:572-592).
    pub fn dimension_variance(&self) -> Result<Vec<f32>> {
        let mut out = vec![0f32; self.d];
        check(unsafe { innr_cuda_batch_dimension_variance(self.h.0, out.as_mut_ptr(), out.len()) })?;
        Ok(out)
    }

    /// `batch_knn_reordered` (src/batch.rs:621-659).
    pub fn knn_reordered(&self, query: &[f32], k: usize) -> Result<(Vec<usize>, Vec<f32>)> {
        assert_eq!(query.len(), self.d); // src/batch.rs:622
        let (mut idx, mut sc) = knn_buffers(1, k.min(self.n));
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_batch_knn_reordered(self.h.0, query.as_ptr(), query.len(), k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        idx.truncate(count);
        sc.truncate(count);
        Ok((idx.into_iter().map(|i| i as usize).collect(), sc))
    }

    /// `batch_knn_adaptive` (src/batch.rs:441-564), reproduced exactly (same survivors, same order).
    pub fn knn_adaptive(&self, query: &[f32], k: usize, warmup_dims: usize) -> Result<(Vec<usize>, Vec<f32>)> {
        assert_eq!(query.len(), self.d); // src/batch.rs:447
        assert!(warmup_dims > 0, "warmup_dims must be > 0"); // src/batch.rs:448
        let (mut idx, mut sc) = knn_buffers(1, k.min(self.n));
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_batch_knn_adaptive(self.h.0, query.as_ptr(), query.len(), k, warmup_dims, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        idx.truncate(count);
        sc.truncate(count);
        Ok((idx.into_iter().map(|i| i as usize).collect(), sc))
    }

    /// Re-rank stage of the documented two-stage retrieval (src/scalar.rs:366-368, examples/binary_demo.rs:235-237): the
    /// exact kNN restricted to `candidates` (distinct global indices), original indices reported.
    pub fn knn_subset(&self, metric: Metric, query: &[f32], candidates: &[usize], k: usize) -> Result<(Vec<usize>, Vec<f32>)> {
        assert_eq!(query.len(), self.d);
        let cand: Vec<u64> = candidates.iter().map(|&c| c as u64).collect();
        let (mut idx, mut sc) = knn_buffers(1, k.min(cand.len()));
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_batch_knn_subset(self.h.0, metric.id(), query.as_ptr(), query.len(), cand.as_ptr(), cand.len(), k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        idx.truncate(count);
        sc.truncate(count);
        Ok((idx.into_iter().map(|i| i as usize).collect(), sc))
    }

    /// `encode_binary` (src/binary.rs:133-141) of every vector, on the device; the code set inherits `index_base`.
    pub fn to_binary(&self, threshold: f32) -> Result<BinaryCorpus> {
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_binary_from_f32(self.h.0, threshold, &mut h) })?;
        Ok(BinaryCorpus { h: Handle(h), n: self.n, dim_bits: self.d })
    }

    /// `quantize_u8` (src/scalar.rs:212-225) of every vector, on the device.
    pub fn to_u8(&self, alpha: f32, offset: f32) -> Result<U8Corpus> {
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_u8_from_f32(self.h.0, alpha, offset, &mut h) })?;
        Ok(U8Corpus { h: Handle(h), n: self.n, d: self.d, alpha, offset })
    }

    /// `encode_ternary` (src/ternary.rs:163-173) of every vector, on the device.
    pub fn to_ternary(&self, threshold: f32) -> Result<TernaryCorpus> {
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_ternary_from_f32(self.h.0, threshold, &mut h) })?;
        Ok(TernaryCorpus { h: Handle(h), n: self.n, dimension: self.d })
    }
}

/// A prefix view of an [`F32Corpus`]; derefs to it.
pub struct F32View<'a> {
    inner: F32Corpus,
    _parent: core::marker::PhantomData<&'a F32Corpus>,
}

impl<'a> core::ops::Deref for F32View<'a> {
    type Target = F32Corpus;
    fn deref(&self) -> &F32Corpus {
        &self.inner
    }
}

/// `TopK` (src/topk.rs:47-187) over a whole distance array at once: the k smallest by `(total_cmp(distance), id)`,
/// i.e. what inserting `(i, distances[i])` for every i and calling `into_sorted()` yields (exact ties: DESIGN.md row T).
pub fn topk_from_distances(distances: &[f32], k: usize) -> Result<Vec<(u32, f32)>> {
    assert!(k > 0, "k must be > 0"); // src/topk.rs:65
    let kk = k.min(distances.len()).max(1);
    let (mut id, mut dist) = (vec![0u32; kk], vec![0f32; kk]);
    let mut count = 0usize;
    check(unsafe { innr_cuda_topk_from_distances(distances.as_ptr(), distances.len(), k, id.as_mut_ptr(), dist.as_mut_ptr(), &mut count) })?;
    Ok(id.into_iter().zip(dist).take(count).collect())
}

// ------------------------------------------------------------------------------------------------ binary codes
/// Device-resident set of `PackedBinary` codes (src/binary.rs:37-117), packed contiguously at upload.
pub struct BinaryCorpus {
    h: Handle,
    n: usize,
    dim_bits: usize,
}

impl BinaryCorpus {
    /// `words`: `n x ceil(dim_bits / 64)` u64, each code's `PackedBinary::data()` in order.
    pub fn from_words(words: &[u64], n: usize, dim_bits: usize, index_base: u64) -> Result<Self> {
        assert_eq!(words.len(), n * ((dim_bits + 63) / 64), "data length must match ceil(dimension / 64)"); // src/binary.rs:51-57
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_upload_binary(words.as_ptr(), n, dim_bits, index_base, &mut h) })?;
        Ok(Self { h: Handle(h), n, dim_bits })
    }

    /// Number of codes.
    pub fn len(&self) -> usize {
        self.n
    }

    /// True when the set holds no code.
    pub fn is_empty(&self) -> bool {
        self.n == 0
    }

    /// Bits per code (`PackedBinary::dimension`).
    pub fn dimension(&self) -> usize {
        self.dim_bits
    }

    /// Raw handle for the `_dev` / sharded entries of [`sys`].
    pub fn as_ptr(&self) -> *const innr_cuda_corpus {
        self.h.0
    }

    fn check_query(&self, query_words: &[u64], query_dim_bits: usize, who: &str) {
        assert_eq!(query_dim_bits, self.dim_bits, "innr::{who}: dimension mismatch ({query_dim_bits} vs {})", self.dim_bits); // src/binary.rs:155-159
        assert_eq!(query_words.len(), (self.dim_bits + 63) / 64);
    }

    /// `binary_hamming` (src/binary.rs:154) of the query against every code.
    pub fn hamming_all(&self, query_words: &[u64], query_dim_bits: usize) -> Result<Vec<u32>> {
        self.check_query(query_words, query_dim_bits, "binary_hamming");
        let mut out = vec![0u32; self.n];
        check(unsafe { innr_cuda_hamming_all(self.h.0, query_words.as_ptr(), query_dim_bits, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// `binary_dot` (src/binary.rs:178) of the query against every code.
    pub fn dot_all(&self, query_words: &[u64], query_dim_bits: usize) -> Result<Vec<u32>> {
        self.check_query(query_words, query_dim_bits, "binary_dot");
        let mut out = vec![0u32; self.n];
        check(unsafe { innr_cuda_binary_dot_all(self.h.0, query_words.as_ptr(), query_dim_bits, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// `binary_jaccard` (src/binary.rs:198) of the query against every code.
    pub fn jaccard_all(&self, query_words: &[u64], query_dim_bits: usize) -> Result<Vec<f32>> {
        self.check_query(query_words, query_dim_bits, "binary_jaccard");
        let mut out = vec![0f32; self.n];
        check(unsafe { innr_cuda_binary_jaccard_all(self.h.0, query_words.as_ptr(), query_dim_bits, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// The caller composition of examples/binary_demo.rs:174-180 (all distances, stable `sort_by_key`, `take(k)`) as one
    /// fused scan: `(index, distance)` ascending, ties -> lower index.
    pub fn hamming_top_k(&self, query_words: &[u64], query_dim_bits: usize, k: usize) -> Result<Vec<(usize, u32)>> {
        self.check_query(query_words, query_dim_bits, "binary_hamming");
        let kk = k.min(self.n).max(1);
        let (mut idx, mut dist) = (vec![0u64; kk], vec![0u32; kk]);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_hamming_topk(self.h.0, query_words.as_ptr(), 1, query_dim_bits, k, idx.as_mut_ptr(), dist.as_mut_ptr(), &mut count)
        })?;
        Ok(idx.into_iter().zip(dist).take(count).map(|(i, d)| (i as usize, d)).collect())
    }

    /// Asynchronous `hamming_top_k` (see `F32Corpus::knn_submit`); `Ticket::wait_hamming` returns `(index, distance)`.
    pub fn hamming_top_k_submit(&self, query_words: &[u64], query_dim_bits: usize, k: usize) -> Result<Ticket> {
        self.check_query(query_words, query_dim_bits, "binary_hamming");
        let mut t: *mut innr_cuda_ticket = std::ptr::null_mut();
        check(unsafe { innr_cuda_hamming_topk_async(self.h.0, query_words.as_ptr(), 1, query_dim_bits, k, &mut t) })?;
        Ok(Ticket { t, n_queries: 1, k, binary: true })
    }

    /// Top-k by `binary_dot` (`jaccard == false`) or `binary_jaccard` (`true`): descending, ties -> lower index.
    pub fn similarity_top_k(&self, jaccard: bool, query_words: &[u64], query_dim_bits: usize, k: usize) -> Result<Vec<(usize, f32)>> {
        self.check_query(query_words, query_dim_bits, if jaccard { "binary_jaccard" } else { "binary_dot" });
        let kk = k.min(self.n).max(1);
        let (mut idx, mut sc) = (vec![0u64; kk], vec![0f32; kk]);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_binary_topk(self.h.0, jaccard as c_int, query_words.as_ptr(), query_dim_bits, k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        Ok(idx.into_iter().zip(sc).take(count).map(|(i, s)| (i as usize, s)).collect())
    }

    /// `hamming_top_k` for a batch of queries (`query_words`: `n_queries` codes back to back) in one call, one list per
    /// query; batches run on the tensor cores when they qualify, with the same results.
    pub fn hamming_top_k_many(&self, query_words: &[u64], n_queries: usize, query_dim_bits: usize, k: usize) -> Result<Vec<Vec<(usize, u32)>>> {
        assert_eq!(query_dim_bits, self.dim_bits, "innr::binary_hamming: dimension mismatch ({query_dim_bits} vs {})", self.dim_bits);
        let words = (self.dim_bits + 63) / 64;
        assert_eq!(query_words.len(), n_queries * words);
        if n_queries == 0 {
            return Ok(Vec::new());
        }
        let kk = k.max(1);
        let (mut idx, mut dist) = (vec![0u64; n_queries * kk], vec![0u32; n_queries * kk]);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_hamming_topk(self.h.0, query_words.as_ptr(), n_queries, query_dim_bits, k, idx.as_mut_ptr(), dist.as_mut_ptr(), &mut count)
        })?;
        Ok((0..n_queries)
            .map(|q| (0..count).map(|j| (idx[q * kk + j] as usize, dist[q * kk + j])).collect())
            .collect())
    }

    /// `similarity_top_k` for a batch of queries (`query_words`: `n_queries` codes back to back) in one call, one list
    /// per query, the same results as one call per query.
    pub fn binary_top_k_many(&self, jaccard: bool, query_words: &[u64], n_queries: usize, query_dim_bits: usize, k: usize) -> Result<Vec<Vec<(usize, f32)>>> {
        assert_eq!(query_dim_bits, self.dim_bits, "dimension mismatch ({query_dim_bits} vs {})", self.dim_bits);
        let words = (self.dim_bits + 63) / 64;
        assert_eq!(query_words.len(), n_queries * words);
        if n_queries == 0 {
            return Ok(Vec::new());
        }
        let kk = k.max(1);
        let (mut idx, mut sc) = (vec![0u64; n_queries * kk], vec![0f32; n_queries * kk]);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_binary_topk_batch(self.h.0, jaccard as c_int, query_words.as_ptr(), n_queries, query_dim_bits, k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        Ok((0..n_queries)
            .map(|q| (0..count).map(|j| (idx[q * kk + j] as usize, sc[q * kk + j])).collect())
            .collect())
    }
}

/// `encode_binary` (src/binary.rs:133-141): the words of the resulting `PackedBinary`.
pub fn encode_binary(values: &[f32], threshold: f32) -> Result<Vec<u64>> {
    let mut out = vec![0u64; (values.len() + 63) / 64];
    check(unsafe { innr_cuda_encode_binary(values.as_ptr(), values.len(), threshold, out.as_mut_ptr()) })?;
    Ok(out)
}

// ------------------------------------------------------------------------------------------------ u8 codes
/// Device-resident `&[QuantizedU8]` (src/scalar.rs:171-208) with the collection's `QuantizationParams`.
pub struct U8Corpus {
    h: Handle,
    n: usize,
    d: usize,
    alpha: f32,
    offset: f32,
}

impl U8Corpus {
    /// `rows`: `n x d` bytes, each vector's `QuantizedU8::data()` in order.
    pub fn from_rows(rows: &[u8], n: usize, d: usize, alpha: f32, offset: f32, index_base: u64) -> Result<Self> {
        assert_eq!(rows.len(), n * d, "data length must match dimension"); // src/scalar.rs:183-188, per vector
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_upload_u8(rows.as_ptr(), n, d, alpha, offset, index_base, &mut h) })?;
        Ok(Self { h: Handle(h), n, d, alpha, offset })
    }

    /// Number of vectors.
    pub fn len(&self) -> usize {
        self.n
    }

    /// True when the set holds no vector.
    pub fn is_empty(&self) -> bool {
        self.n == 0
    }

    /// Dimension of every vector.
    pub fn dimension(&self) -> usize {
        self.d
    }

    /// `(alpha, offset)` the codes were quantised with.
    pub fn params(&self) -> (f32, f32) {
        (self.alpha, self.offset)
    }

    /// Raw handle for the `_dev` / sharded entries of [`sys`].
    pub fn as_ptr(&self) -> *const innr_cuda_corpus {
        self.h.0
    }

    /// `mixed_dot_u8_f32` (src/scalar.rs:314) of the query against every row.
    pub fn mixed_dot_all(&self, query: &[f32]) -> Result<Vec<f32>> {
        assert_eq!(query.len(), self.d, "mixed_dot_u8_f32: slice length mismatch ({} vs {})", query.len(), self.d); // src/scalar.rs:315-321
        let mut out = vec![0f32; self.n];
        check(unsafe { innr_cuda_mixed_dot_u8_all(self.h.0, query.as_ptr(), query.len(), out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// `asymmetric_dot_u8` (src/scalar.rs:261-300) of the query against every row.
    pub fn asymmetric_dot_all(&self, query: &[f32]) -> Result<Vec<f32>> {
        assert_eq!(query.len(), self.d, "asymmetric_dot_u8: dimension mismatch ({} vs {})", query.len(), self.d); // src/scalar.rs:266-272
        let mut out = vec![0f32; self.n];
        check(unsafe { innr_cuda_asymmetric_dot_u8_all(self.h.0, query.as_ptr(), query.len(), out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// `batch_knn_u8` (src/scalar.rs:370-393): `(index, score)` descending, ties -> lower index.
    pub fn knn(&self, query: &[f32], k: usize) -> Result<Vec<(usize, f32)>> {
        if self.n == 0 || k == 0 {
            return Ok(Vec::new()); // src/scalar.rs:376-378, before any length check
        }
        assert_eq!(query.len(), self.d, "asymmetric_dot_u8_precomputed: dimension mismatch ({} vs {})", query.len(), self.d); // src/scalar.rs:290-296
        let (mut idx, mut sc) = knn_buffers(1, k.min(self.n));
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_batch_knn_u8(self.h.0, query.as_ptr(), 1, query.len(), k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        Ok(idx.into_iter().zip(sc).take(count).map(|(i, s)| (i as usize, s)).collect())
    }
}

impl U8Corpus {
    /// Asynchronous `knn` (see `F32Corpus::knn_submit`).
    pub fn knn_submit(&self, query: &[f32], k: usize) -> Result<Ticket> {
        if self.n != 0 && k != 0 {
            assert_eq!(query.len(), self.d, "asymmetric_dot_u8_precomputed: dimension mismatch ({} vs {})", query.len(), self.d); // src/scalar.rs:290-296
        }
        let mut t: *mut innr_cuda_ticket = std::ptr::null_mut();
        check(unsafe { innr_cuda_batch_knn_u8_async(self.h.0, query.as_ptr(), 1, query.len(), k, &mut t) })?;
        Ok(Ticket { t, n_queries: 1, k, binary: false })
    }
}

/// One asynchronous top-k call in flight. The library owns the ticket; waiting consumes it. A ticket that is dropped
/// without a wait is waited for in `drop` (its slot must be free before the device accepts a third call).
pub struct Ticket {
    t: *mut innr_cuda_ticket,
    n_queries: usize,
    k: usize,
    binary: bool,
}

impl Ticket {
    /// f32 and u8 corpora: per query `(indices, scores)`, exactly what the synchronous call returns.
    pub fn wait(mut self) -> Result<Vec<(Vec<usize>, Vec<f32>)>> {
        assert!(!self.binary, "a Hamming ticket is read with wait_hamming");
        let (mut idx, mut sc) = knn_buffers(self.n_queries, self.k);
        let mut count = 0usize;
        let t = std::mem::replace(&mut self.t, std::ptr::null_mut());
        check(unsafe { innr_cuda_ticket_wait(t, idx.as_mut_ptr(), sc.as_mut_ptr(), std::ptr::null_mut(), &mut count) })?;
        Ok(split_results(idx, sc, self.n_queries, self.k, count))
    }

    /// Binary corpora: `(index, distance)` of the single query, ascending distance, ties -> lower index.
    pub fn wait_hamming(mut self) -> Result<Vec<(usize, u32)>> {
        assert!(self.binary, "not a Hamming ticket");
        let kk = self.k.max(1) * self.n_queries.max(1);
        let (mut idx, mut dist) = (vec![0u64; kk], vec![0u32; kk]);
        let mut count = 0usize;
        let t = std::mem::replace(&mut self.t, std::ptr::null_mut());
        check(unsafe { innr_cuda_ticket_wait(t, idx.as_mut_ptr(), std::ptr::null_mut(), dist.as_mut_ptr(), &mut count) })?;
        Ok(idx.into_iter().zip(dist).take(count).map(|(i, d)| (i as usize, d)).collect())
    }
}

impl Drop for Ticket {
    fn drop(&mut self) {
        if !self.t.is_null() {
            let kk = self.k.max(1) * self.n_queries.max(1);
            let (mut idx, mut sc, mut dist) = (vec![0u64; kk], vec![0f32; kk], vec![0u32; kk]);
            let mut count = 0usize;
            let _ = unsafe { innr_cuda_ticket_wait(self.t, idx.as_mut_ptr(), sc.as_mut_ptr(), dist.as_mut_ptr(), &mut count) };
        }
    }
}

/// `quantize_u8` (src/scalar.rs:212-225): the bytes of the resulting `QuantizedU8`.
pub fn quantize_u8(values: &[f32], alpha: f32, offset: f32) -> Result<Vec<u8>> {
    let mut out = vec![0u8; values.len()];
    check(unsafe { innr_cuda_quantize_u8(values.as_ptr(), values.len(), alpha, offset, out.as_mut_ptr()) })?;
    Ok(out)
}

// ------------------------------------------------------------------------------------------------ token matrix (MaxSim)
/// Device-resident document set for ColBERT MaxSim: all token rows contiguous, `doc_offsets` delimiting documents.
pub struct TokenCorpus {
    h: Handle,
    n_docs: usize,
    dim: usize,
}

impl TokenCorpus {
    /// `tokens`: `total_tokens x dim` row-major; document j owns rows `doc_offsets[j] .. doc_offsets[j + 1]`.
    pub fn from_tokens(tokens: &[f32], doc_offsets: &[u64], dim: usize, index_base: u64) -> Result<Self> {
        assert!(!doc_offsets.is_empty(), "doc_offsets must hold n_docs + 1 entries");
        let n_docs = doc_offsets.len() - 1;
        assert_eq!(tokens.len(), doc_offsets[n_docs] as usize * dim, "dimension mismatch (doc)"); // src/maxsim.rs:107-110
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_upload_tokens(tokens.as_ptr(), doc_offsets.as_ptr(), n_docs, dim, index_base, &mut h) })?;
        Ok(Self { h: Handle(h), n_docs, dim })
    }

    /// Number of documents.
    pub fn num_docs(&self) -> usize {
        self.n_docs
    }

    /// Token dimension.
    pub fn dimension(&self) -> usize {
        self.dim
    }

    /// Raw handle for the `_dev` entries of [`sys`].
    pub fn as_ptr(&self) -> *const innr_cuda_corpus {
        self.h.0
    }

    /// `maxsim` (`cosine == false`, src/maxsim.rs:96) or `maxsim_cosine` (`true`, :168) of one query token set
    /// (`n_q x dim` row-major) against every document: the caller loop of examples/maxsim_colbert.rs:171-174.
    pub fn maxsim(&self, q_tokens: &[f32], n_q: usize, cosine: bool) -> Result<Vec<f32>> {
        assert_eq!(q_tokens.len(), n_q * self.dim, "dimension mismatch (query)"); // src/maxsim.rs:103-106
        let mut out = vec![0f32; self.n_docs];
        check(unsafe { innr_cuda_maxsim(self.h.0, q_tokens.as_ptr(), n_q, self.dim, cosine as c_int, out.as_mut_ptr()) })?;
        Ok(out)
    }

    /// Several queries of `n_q` tokens each (`n_queries x n_q x dim`): scores are query-major `n_queries x n_docs`; queries
    /// of <= 32 tokens share corpus passes on the tensor-core path. Same values as one `maxsim` call per query.
    pub fn maxsim_batch(&self, q_tokens: &[f32], n_queries: usize, n_q: usize, cosine: bool) -> Result<Vec<f32>> {
        assert_eq!(q_tokens.len(), n_queries * n_q * self.dim, "dimension mismatch (query)");
        let mut out = vec![0f32; n_queries * self.n_docs];
        check(unsafe {
            innr_cuda_maxsim_batch(self.h.0, q_tokens.as_ptr(), n_queries, n_q, self.dim, cosine as c_int, out.as_mut_ptr())
        })?;
        Ok(out)
    }

    /// The `k` best documents for one query token set: `(index, score)` descending under `f32::total_cmp`, exact ties ->
    /// lower index (`index_base + doc`). The scores are `maxsim`'s bit for bit, so this is a stable descending
    /// `total_cmp` sort of `maxsim`'s output truncated to `k`, without copying `num_docs` floats to the host.
    pub fn maxsim_topk(&self, q_tokens: &[f32], n_q: usize, cosine: bool, k: usize) -> Result<Vec<(usize, f32)>> {
        assert_eq!(q_tokens.len(), n_q * self.dim, "dimension mismatch (query)"); // src/maxsim.rs:103-106
        let (mut idx, mut sc) = knn_buffers(1, k);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_maxsim_topk(self.h.0, q_tokens.as_ptr(), 1, n_q, self.dim, cosine as c_int, k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        Ok(idx.into_iter().zip(sc).take(count).map(|(i, s)| (i as usize, s)).collect())
    }

    /// `maxsim_topk` of several queries of `n_q` tokens each (`n_queries x n_q x dim`): per query `(indices, scores)`,
    /// the same as one `maxsim_topk` call per query.
    pub fn maxsim_topk_batch(&self, q_tokens: &[f32], n_queries: usize, n_q: usize, cosine: bool, k: usize) -> Result<Vec<(Vec<usize>, Vec<f32>)>> {
        assert_eq!(q_tokens.len(), n_queries * n_q * self.dim, "dimension mismatch (query)");
        let (mut idx, mut sc) = knn_buffers(n_queries, k);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_maxsim_topk(self.h.0, q_tokens.as_ptr(), n_queries, n_q, self.dim, cosine as c_int, k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        Ok(split_results(idx, sc, n_queries, k, count))
    }
}

// ------------------------------------------------------------------------------------------------ ternary codes
/// Ternary score selector (src/ternary.rs).
#[derive(Debug, Clone, Copy, PartialEq, Eq)]
pub enum TernaryOp {
    /// `ternary_dot` (src/ternary.rs:191): packed query, descending.
    Dot,
    /// `ternary_hamming` (src/ternary.rs:301): packed query, ascending.
    Hamming,
}

/// Device-resident set of `PackedTernary` codes (src/ternary.rs:50-157).
pub struct TernaryCorpus {
    h: Handle,
    n: usize,
    dimension: usize,
}

impl TernaryCorpus {
    /// `words`: `n x ceil(dimension / 32)` u64, each code's `PackedTernary::data()` in order.
    pub fn from_words(words: &[u64], n: usize, dimension: usize, index_base: u64) -> Result<Self> {
        assert_eq!(words.len(), n * ((dimension + 31) / 32), "data length must match ceil(dimension / 32)"); // src/ternary.rs:64-70
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_upload_ternary(words.as_ptr(), n, dimension, index_base, &mut h) })?;
        Ok(Self { h: Handle(h), n, dimension })
    }

    /// Number of codes.
    pub fn len(&self) -> usize {
        self.n
    }

    /// True when the set holds no code.
    pub fn is_empty(&self) -> bool {
        self.n == 0
    }

    /// `ternary_dot` / `ternary_hamming` of a packed query against every code (exact integers).
    pub fn scores_all(&self, op: TernaryOp, query_words: &[u64], query_dimension: usize) -> Result<Vec<i32>> {
        assert_eq!(query_dimension, self.dimension, "innr::ternary_dot: dimension mismatch ({query_dimension} vs {})", self.dimension); // src/ternary.rs:192-196
        assert_eq!(query_words.len(), (self.dimension + 31) / 32);
        let id = if op == TernaryOp::Dot { INNR_TERNARY_DOT } else { INNR_TERNARY_HAMMING };
        let mut out = vec![0i32; self.n];
        check(unsafe {
            innr_cuda_ternary_scores_all(self.h.0, id, query_words.as_ptr() as *const c_void, query_dimension, core::ptr::null_mut(), out.as_mut_ptr())
        })?;
        Ok(out)
    }

    /// `ternary::asymmetric_dot` (src/ternary.rs:286-296) of an f32 query against every code (bit-exact sequential sum).
    pub fn asymmetric_dot_all(&self, query: &[f32]) -> Result<Vec<f32>> {
        assert_eq!(query.len(), self.dimension); // src/ternary.rs:287
        let mut out = vec![0f32; self.n];
        check(unsafe {
            innr_cuda_ternary_scores_all(self.h.0, INNR_TERNARY_ASYMMETRIC_DOT, query.as_ptr() as *const c_void, query.len(), out.as_mut_ptr(), core::ptr::null_mut())
        })?;
        Ok(out)
    }

    /// Top-k of the asymmetric dot product: descending, ties -> lower index.
    pub fn asymmetric_top_k(&self, query: &[f32], k: usize) -> Result<Vec<(usize, f32)>> {
        assert_eq!(query.len(), self.dimension); // src/ternary.rs:287
        let kk = k.min(self.n).max(1);
        let (mut idx, mut sc) = (vec![0u64; kk], vec![0f32; kk]);
        let mut count = 0usize;
        check(unsafe {
            innr_cuda_ternary_topk(self.h.0, INNR_TERNARY_ASYMMETRIC_DOT, query.as_ptr() as *const c_void, query.len(), k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
        })?;
        Ok(idx.into_iter().zip(sc).take(count).map(|(i, s)| (i as usize, s)).collect())
    }
}

/// `encode_ternary` (src/ternary.rs:163-173): the words of the resulting `PackedTernary`.
pub fn encode_ternary(values: &[f32], threshold: f32) -> Result<Vec<u64>> {
    let mut out = vec![0u64; (values.len() + 31) / 32];
    check(unsafe { innr_cuda_encode_ternary(values.as_ptr(), values.len(), threshold, out.as_mut_ptr()) })?;
    Ok(out)
}

// ------------------------------------------------------------------------------------------------ one process, several GPUs
/// Row shards on different devices (each created after `init(device)` on the creating thread, with `index_base` = its
/// first global row): the unsharded `knn_many` result, merged inside the library -- no collective library involved.
pub fn knn_sharded(shards: &[&F32Corpus], metric: Metric, queries: &[f32], n_queries: usize, k: usize) -> Result<Vec<(Vec<usize>, Vec<f32>)>> {
    assert!(!shards.is_empty(), "no shards");
    let d = shards[0].d;
    assert_eq!(queries.len(), n_queries * d);
    let ptrs: Vec<*const innr_cuda_corpus> = shards.iter().map(|s| s.as_ptr()).collect();
    let (mut idx, mut sc) = knn_buffers(n_queries, k);
    let mut count = 0usize;
    check(unsafe {
        innr_cuda_batch_knn_sharded(ptrs.as_ptr(), ptrs.len(), metric.id(), queries.as_ptr(), n_queries, d, k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
    })?;
    Ok(split_results(idx, sc, n_queries, k, count))
}

/// Hamming top-k over row shards of codes on different devices.
pub fn hamming_top_k_sharded(shards: &[&BinaryCorpus], query_words: &[u64], query_dim_bits: usize, k: usize) -> Result<Vec<(usize, u32)>> {
    assert!(!shards.is_empty(), "no shards");
    let ptrs: Vec<*const innr_cuda_corpus> = shards.iter().map(|s| s.as_ptr()).collect();
    let (mut idx, mut dist) = (vec![0u64; k.max(1)], vec![0u32; k.max(1)]);
    let mut count = 0usize;
    check(unsafe {
        innr_cuda_hamming_topk_sharded(ptrs.as_ptr(), ptrs.len(), query_words.as_ptr(), 1, query_dim_bits, k, idx.as_mut_ptr(), dist.as_mut_ptr(), &mut count)
    })?;
    Ok(idx.into_iter().zip(dist).take(count).map(|(i, d)| (i as usize, d)).collect())
}

/// Asynchronous `knn_sharded` (shards on pairwise distinct devices): one `Ticket` for the whole call, two calls in flight
/// per device group, no device synchronised until the wait. `Ok(None)`: the result is empty (no rows, k == 0).
pub fn knn_sharded_submit(shards: &[&F32Corpus], metric: Metric, query: &[f32], k: usize) -> Result<Option<Ticket>> {
    assert!(!shards.is_empty(), "no shards");
    let ptrs: Vec<*const innr_cuda_corpus> = shards.iter().map(|s| s.as_ptr()).collect();
    let mut t: *mut innr_cuda_ticket = std::ptr::null_mut();
    check(unsafe { innr_cuda_batch_knn_sharded_async(ptrs.as_ptr(), ptrs.len(), metric.id(), query.as_ptr(), 1, query.len(), k, &mut t) })?;
    Ok(if t.is_null() { None } else { Some(Ticket { t, n_queries: 1, k, binary: false }) })
}

/// Asynchronous `hamming_top_k_sharded`; read the ticket with `Ticket::wait_hamming`.
pub fn hamming_top_k_sharded_submit(shards: &[&BinaryCorpus], query_words: &[u64], query_dim_bits: usize, k: usize) -> Result<Option<Ticket>> {
    assert!(!shards.is_empty(), "no shards");
    let ptrs: Vec<*const innr_cuda_corpus> = shards.iter().map(|s| s.as_ptr()).collect();
    let mut t: *mut innr_cuda_ticket = std::ptr::null_mut();
    check(unsafe { innr_cuda_hamming_topk_sharded_async(ptrs.as_ptr(), ptrs.len(), query_words.as_ptr(), 1, query_dim_bits, k, &mut t) })?;
    Ok(if t.is_null() { None } else { Some(Ticket { t, n_queries: 1, k, binary: true }) })
}

/// Asynchronous `knn_u8_sharded`.
pub fn knn_u8_sharded_submit(shards: &[&U8Corpus], query: &[f32], k: usize) -> Result<Option<Ticket>> {
    assert!(!shards.is_empty(), "no shards");
    let ptrs: Vec<*const innr_cuda_corpus> = shards.iter().map(|s| s.as_ptr()).collect();
    let mut t: *mut innr_cuda_ticket = std::ptr::null_mut();
    check(unsafe { innr_cuda_batch_knn_u8_sharded_async(ptrs.as_ptr(), ptrs.len(), query.as_ptr(), 1, query.len(), k, &mut t) })?;
    Ok(if t.is_null() { None } else { Some(Ticket { t, n_queries: 1, k, binary: false }) })
}

/// `batch_knn_u8` over row shards on different devices.
pub fn knn_u8_sharded(shards: &[&U8Corpus], query: &[f32], k: usize) -> Result<Vec<(usize, f32)>> {
    assert!(!shards.is_empty(), "no shards");
    let ptrs: Vec<*const innr_cuda_corpus> = shards.iter().map(|s| s.as_ptr()).collect();
    let (mut idx, mut sc) = knn_buffers(1, k);
    let mut count = 0usize;
    check(unsafe {
        innr_cuda_batch_knn_u8_sharded(ptrs.as_ptr(), ptrs.len(), query.as_ptr(), 1, query.len(), k, idx.as_mut_ptr(), sc.as_mut_ptr(), &mut count)
    })?;
    Ok(idx.into_iter().zip(sc).take(count).map(|(i, s)| (i as usize, s)).collect())
}

/// One rank's end of the peer-mapped key exchange between GPUs (the header's `innr_cuda_exchange_*` section): for hosts
/// that run one process per GPU and own their device buffers and streams. The merge itself is `unsafe` because it takes
/// raw device pointers; see [`sys::innr_cuda_exchange_merge_dev`].
pub struct Exchange {
    h: *mut innr_cuda_exchange,
    n_ranks: usize,
}
unsafe impl Send for Exchange {}

impl Drop for Exchange {
    fn drop(&mut self) {
        if !self.h.is_null() {
            unsafe { innr_cuda_exchange_free(self.h) };
        }
    }
}

impl Exchange {
    /// On the calling thread's device; `slot_keys == 0` selects the default capacity (16384 keys per rank and call).
    pub fn create(n_ranks: usize, rank: usize, slot_keys: usize) -> Result<Self> {
        let mut h = core::ptr::null_mut();
        check(unsafe { innr_cuda_exchange_create(n_ranks as c_int, rank as c_int, slot_keys, &mut h) })?;
        Ok(Self { h, n_ranks })
    }

    /// The 64-byte IPC handle of this rank's mailbox, to be sent to the other processes.
    pub fn ipc_handle(&self) -> Result<[u8; 64]> {
        let mut out = [0u8; 64];
        check(unsafe { innr_cuda_exchange_ipc_handle(self.h, out.as_mut_ptr() as *mut c_void) })?;
        Ok(out)
    }

    /// `handles`: every rank's handle in rank order.
    pub fn connect_ipc(&mut self, handles: &[[u8; 64]]) -> Result<()> {
        assert_eq!(handles.len(), self.n_ranks);
        check(unsafe { innr_cuda_exchange_connect_ipc(self.h, handles.as_ptr() as *const c_void) })
    }

    /// All ranks of one exchange living in this process (possibly on different devices).
    pub fn connect_local(all: &mut [Exchange]) -> Result<()> {
        let ptrs: Vec<*mut innr_cuda_exchange> = all.iter().map(|x| x.h).collect();
        check(unsafe { innr_cuda_exchange_connect_local(ptrs.as_ptr(), ptrs.len() as c_int) })
    }

    /// 0, or 1 after a call whose peers did not publish within the timeout.
    pub fn status(&self) -> Result<i32> {
        let mut s: c_int = 0;
        check(unsafe { innr_cuda_exchange_status(self.h, &mut s) })?;
        Ok(s as i32)
    }

    /// Raw handle for [`sys::innr_cuda_exchange_merge_dev`].
    pub fn as_ptr(&self) -> *mut innr_cuda_exchange {
        self.h
    }
}
