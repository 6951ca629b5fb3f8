// layout.cu -- upload-time layout kernels and on-device synthetic generators.
//
//  * rows -> PDX transpose: VerticalBatch::from_flat / from_rows (src/batch.rs:103-183) done on the device;
//  * G-ref generator: generate_embedding (examples/batch_demo.rs:233-242), bit-identical to the Rust code
//    (u64 wrapping arithmetic, u64->f32 RNE conversion, exact power-of-two scaling, one rounded subtract);
//  * G-hash generator (SURVEY.md 8d): splitmix64(salt + row*d + j) -> 24-bit uniform in [-1, 1).
// Generators are stateless so any row can be re-derived on the CPU by the oracle without holding the corpus.
#include "common.cuh"
#include "kernels.cuh"
#include "pdx.cuh"

namespace innr {

namespace {

// rows: n x d row-major (a chunk of the corpus); pdx: first column of the chunk inside the PDX matrix (row pitch ld);
// columns [0, cols) are written (cols >= n: the tail of the last chunk zero-fills the pitch padding)
__global__ void transpose_rows_to_pdx_kernel(const float* __restrict__ rows, unsigned n, unsigned d, const PdxDst dst,
                                             unsigned cols) {
  __shared__ float tile[32][33];
  const unsigned i0 = blockIdx.x * 32, d0 = blockIdx.y * 32;
  // read rows[i][d0 + tx] coalesced along d
  for (unsigned r = threadIdx.y; r < 32; r += blockDim.y) {
    unsigned i = i0 + r, dd = d0 + threadIdx.x;
    tile[r][threadIdx.x] = (i < n && dd < d) ? rows[(size_t)i * d + dd] : 0.0f;
  }
  __syncthreads();
  // write pdx[dd][i0 + tx] coalesced along i
  for (unsigned r = threadIdx.y; r < 32; r += blockDim.y) {
    unsigned dd = d0 + r, i = i0 + threadIdx.x;
    if (dd < d && i < cols) pdx_store1(dst.data, dst.hi, dst.lo, (size_t)dd * dst.ld + i, tile[threadIdx.x][r]);
  }
}

__global__ void generate_f32_pdx_kernel(int generator, uint64_t salt, uint64_t first_row, unsigned n, unsigned d,
                                        const PdxDst dst) {
  const size_t ld = dst.ld, total = (size_t)d * ld;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t dd = t / ld, i = t % ld;
    float v = 0.0f;
    if (i < n) {
      const uint64_t row = first_row + i;
      v = generator == 0 ? ghash_value(salt, row * d + dd) : gref_value(salt + row, dd);
    }
    pdx_store1(dst.data, dst.hi, dst.lo, t, v);
  }
}

__global__ void pdx_rows_to_dst_kernel(const float* __restrict__ src, unsigned rows, unsigned n, const PdxDst dst) {
  const size_t total = (size_t)rows * dst.ld;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const size_t dd = t / dst.ld, i = t % dst.ld;
    pdx_store1(dst.data, dst.hi, dst.lo, t, i < n ? src[dd * n + i] : 0.0f);
  }
}

// The sketch, one thread per column of the pitch (padding columns are zero: code 128, scale 0, bound 0). Two passes over
// the row: absmax, then codes and the residual bound. Any code is valid because r is computed against the code stored:
// the exact residual x - s c lies between its RD and RU roundings, and the squares are summed rounding upward, so r
// bounds the true norm from above (also where the squares underflow). A row of zeros or of subnormals below 127 * 2^-150
// gets s = 0, codes 128 and r = its norm. NaN elements do not enter the absmax but make r NaN.
__global__ void pdx_sketch_kernel(const PdxView v, const float* __restrict__ norms, const PdxSketch sk,
                                  unsigned* __restrict__ nonfinite) {
  const size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= v.ld) return;
  float m = 0.0f;
  for (unsigned dd = 0; dd < v.d; ++dd) m = fmaxf(m, fabsf(pdx_load1(v, (size_t)dd * v.ld + i)));
  const float s = __fdiv_rn(m, 127.0f);
  float acc = 0.0f;
  for (unsigned dd = 0; dd < v.d; ++dd) {
    const float x = pdx_load1(v, (size_t)dd * v.ld + i);
    const float c = s > 0.0f ? fminf(fmaxf(rintf(__fdiv_rn(x, s)), -127.0f), 127.0f) : 0.0f;
    sk.codes[pdx_sketch_off(v.ld, dd, i)] = (uint8_t)((int)c + 128);
    const float e = fmaxf(fabsf(__fmaf_rd(-s, c, x)), fabsf(__fmaf_ru(-s, c, x)));
    acc = __fmaf_ru(e, e, acc);
  }
  const float r = __fsqrt_ru(acc);
  sk.scale[i] = s;
  sk.resid[i] = r;
  if (i < v.n && (!isfinite(s) || !isfinite(r) || !isfinite(norms[i]))) atomicOr(nonfinite, 1u);
}

__global__ void generate_tokens_kernel(uint64_t salt, uint64_t first_row, size_t n_rows, unsigned dim,
                                       float* __restrict__ out) {
  const size_t total = n_rows * dim;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x)
    out[t] = ghash_value(salt, first_row * dim + t);
}

}  // namespace

cudaError_t launch_transpose_rows_to_pdx(const float* dev_rows, size_t n, size_t d, const PdxDst& dst, size_t cols,
                                         cudaStream_t s, LaunchCounter* launches) {
  if (cols == 0 || d == 0) return cudaSuccess;
  dim3 grid((unsigned)((cols + 31) / 32), (unsigned)((d + 31) / 32));
  transpose_rows_to_pdx_kernel<<<grid, dim3(32, 8), 0, s>>>(dev_rows, (unsigned)n, (unsigned)d, dst, (unsigned)cols);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_generate_f32_pdx(int generator, uint64_t salt, uint64_t first_row, size_t n, size_t d,
                                    const PdxDst& dst, cudaStream_t s, LaunchCounter* launches) {
  if (n == 0 || d == 0) return cudaSuccess;
  generate_f32_pdx_kernel<<<148 * 16, 256, 0, s>>>(generator, salt, first_row, (unsigned)n, (unsigned)d, dst);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_pdx_rows_to_dst(const float* dev_src, size_t rows, size_t n, const PdxDst& dst, cudaStream_t s,
                                   LaunchCounter* launches) {
  if (rows == 0) return cudaSuccess;
  pdx_rows_to_dst_kernel<<<148 * 16, 256, 0, s>>>(dev_src, (unsigned)rows, (unsigned)n, dst);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_pdx_sketch(const PdxView& v, const float* dev_norms, const PdxSketch& sk, unsigned* dev_nonfinite,
                              cudaStream_t s, LaunchCounter* launches) {
  cudaError_t e = cudaMemsetAsync(dev_nonfinite, 0, sizeof(unsigned), s);
  if (e != cudaSuccess || v.ld == 0) return e;
  pdx_sketch_kernel<<<(unsigned)((v.ld + 255) / 256), 256, 0, s>>>(v, dev_norms, sk, dev_nonfinite);
  ++*launches;
  return cudaGetLastError();
}

cudaError_t launch_generate_tokens(uint64_t salt, uint64_t first_row, size_t n_rows, size_t dim, float* dev_tokens,
                                   cudaStream_t s, LaunchCounter* launches) {
  if (n_rows == 0 || dim == 0) return cudaSuccess;
  generate_tokens_kernel<<<148 * 16, 256, 0, s>>>(salt, first_row, n_rows, (unsigned)dim, dev_tokens);
  ++*launches;
  return cudaGetLastError();
}

}  // namespace innr
