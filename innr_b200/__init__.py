"""innr_b200 -- B200-native (sm_100a) device path for innr's batch similarity-search hot path.

The product is libinnr_cuda.so (hand-written CUDA behind the C-ABI in include/innr_cuda.h). This package is the
host-side mirror of the reference's API for that path (same names, arguments and error behaviour as
innr::batch / innr::binary / innr::scalar / innr::maxsim / innr::backend) so the parity tests read like the
reference's own tests. No CPU fallback: without the shared library or a CUDA device, calls raise.
"""
from ._lib import (InnrCudaError, backend_name, build, init, knn_tc_last_stats, last_kernel_ms,  # noqa: F401
                   launch_count, lib, set_option)
from .backend import Backend, dense_backend  # noqa: F401
from .batch import (BatchKnnResult, DeviceBatch, VerticalBatch, batch_cosine, batch_cosine_into,  # noqa: F401
                    batch_dimension_variance, batch_dot, batch_dot_into, batch_knn, batch_knn_adaptive, batch_knn_cosine,
                    batch_knn_dot,
                    batch_knn_filtered, batch_knn_many, batch_knn_reordered, batch_knn_subset, batch_l2_squared,
                    batch_l2_squared_into, batch_l2_squared_pruning, batch_norms, batch_norms_into, knn_tc_debug_bounds,
                    knn_screen_debug_bounds)
from .binary import (BinaryCorpus, PackedBinary, binary_dot, binary_dot_all, binary_hamming, binary_jaccard,  # noqa: F401
                     binary_jaccard_all, binary_topk, encode_binary, hamming_all,
                     hamming_topk, hamming_topk_many)
from .maxsim import TokenCorpus, maxsim, maxsim_corpus, maxsim_corpus_batch, maxsim_cosine  # noqa: F401
from .scalar import (QuantizationParams, QuantizedU8, QueryContext, U8Corpus, asymmetric_dot_u8,  # noqa: F401
                     asymmetric_dot_u8_all, asymmetric_dot_u8_precomputed, batch_knn_u8, batch_knn_u8_many,
                     mixed_dot_u8_all, mixed_dot_u8_f32, quantize_u8, query_context)
from .ternary import (PackedTernary, TernaryCorpus, encode_ternary, ternary_asymmetric_dot, ternary_dot,  # noqa: F401
                      ternary_hamming, ternary_scores_all, ternary_sparsity, ternary_topk)
from .topk import TopK, topk_from_distances  # noqa: F401
