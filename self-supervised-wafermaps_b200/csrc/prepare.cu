// prepare.cu — one-off relayout of caller tensors into the K-major row layout
// the tcgen05 kernels stream with TMA.
//
// The reference hands knn_predict a (D,N) contiguous fp32 bank
// (src/ssl_wafermap/models/knn.py:80 `.t().contiguous()`) and (B,D) fp32
// queries (:90).  The tensor cores want both operands K-major (vector
// dimension contiguous), so the bank is transposed once per validation epoch
// and cached by the host shim; queries only need the cast.
//
//   MODE_BF16  : dst_hi (n_vec, dim_pad) bf16, round-to-nearest-even
//   MODE_TF32X3: dst_hi (n_vec, dim_pad) f32 = rna_tf32(x); dst_lo = x - hi
//   MODE_BF16X3: dst_hi (n_vec, dim_pad) bf16 = rn(x); dst_lo = rn(x - hi)
//   MODE_F16   : dst_hi only, as MODE_F16X2's
//   MODE_F16X2 : dst_hi (n_vec, dim_pad) fp16 = rn(sat(x)); dst_lo (optional: bank only) = rn(sat(x - hi));
//                sat clamps to +-65504 so that no inf/NaN ever enters the contraction
//   MODE_F32ROWS: dst_hi (n_vec, dim_pad) f32 = x  (row-major shadow the exact re-scoring gathers)
// dim_pad = dim rounded up to 64; pad columns are written as zero.
//
// HBM-bound: reads n_vec*dim*sizeof(src), writes n_vec*dim_pad*(2 | 8) bytes.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "../../include/b200knn.h"
#include "common.cuh"
#include "kernels.h"

namespace b200knn {
namespace {

__device__ __forceinline__ float ld_f32(const void* p, int dtype, int64_t i) {
  if (dtype == B200KNN_F32) return static_cast<const float*>(p)[i];
  if (dtype == B200KNN_F16) return __half2float(static_cast<const __half*>(p)[i]);
  return __bfloat162float(static_cast<const __nv_bfloat16*>(p)[i]);
}

__device__ __forceinline__ void emit(int mode, float x, void* hi, void* lo, int64_t o) {
  if (mode == B200KNN_MODE_BF16) {
    static_cast<__nv_bfloat16*>(hi)[o] = __float2bfloat16_rn(x);
  } else if (mode == B200KNN_MODE_F32ROWS) {
    static_cast<float*>(hi)[o] = x;
  } else if (mode == B200KNN_MODE_BF16X3) {
    const __nv_bfloat16 h = __float2bfloat16_rn(x);
    static_cast<__nv_bfloat16*>(hi)[o] = h;
    static_cast<__nv_bfloat16*>(lo)[o] = __float2bfloat16_rn(x - __bfloat162float(h));
  } else if (mode == B200KNN_MODE_F16X2 || mode == B200KNN_MODE_F16) {
    const __half h = f16_operand(x);
    static_cast<__half*>(hi)[o] = h;
    if (lo != nullptr) static_cast<__half*>(lo)[o] = f16_operand(x - __half2float(h));
  } else {
    uint32_t u;
    asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(u) : "f"(x));
    const float h = __uint_as_float(u);
    static_cast<float*>(hi)[o] = h;
    static_cast<float*>(lo)[o] = x - h;
  }
}

// vectors are columns of src: element (n, d) at src[d*ld + n]
__global__ void __launch_bounds__(256)
    prepare_dn_kernel(const void* __restrict__ src, int dtype, int64_t n_vec, int dim, int dim_pad,
                      int64_t ld, int mode, void* __restrict__ hi, void* __restrict__ lo) {
  __shared__ float tile[64][65];
  const int64_t n0 = int64_t(blockIdx.x) * 64;
  const int d0 = blockIdx.y * 64;
  const int tx = threadIdx.x & 63, ty = threadIdx.x >> 6;
#pragma unroll
  for (int r = ty; r < 64; r += 4) {
    const int d = d0 + r;
    const int64_t n = n0 + tx;
    tile[r][tx] = (d < dim && n < n_vec) ? ld_f32(src, dtype, int64_t(d) * ld + n) : 0.0f;
  }
  __syncthreads();
#pragma unroll
  for (int r = ty; r < 64; r += 4) {
    const int64_t n = n0 + r;
    const int d = d0 + tx;
    if (n < n_vec && d < dim_pad) emit(mode, tile[tx][r], hi, lo, n * dim_pad + d);
  }
}

// vectors are rows of src: element (n, d) at src[n*ld + d]
__global__ void __launch_bounds__(256)
    prepare_nd_kernel(const void* __restrict__ src, int dtype, int64_t n_vec, int dim, int dim_pad,
                      int64_t ld, int mode, void* __restrict__ hi, void* __restrict__ lo) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n_vec * dim_pad) return;
  const int64_t n = i / dim_pad;
  const int d = int(i - n * dim_pad);
  const float x = d < dim ? ld_f32(src, dtype, n * ld + d) : 0.0f;
  emit(mode, x, hi, lo, i);
}

// F.normalize(x, dim=1) of row vectors (reference: src/ssl_wafermap/models/knn.py:77 for bank
// rows, :90 for queries) fused with the relayout into padded fp32 rows: one warp per row.
// Defined order, reproducible on the CPU (oracle.normalize_rows_ref): lane l adds the squares
// of columns l, l+32, ... in fp64 (each square is exact), the 32 partials are combined by an
// xor butterfly (16, 8, 4, 2, 1), norm = float(sqrt(total)), y = x / max(norm, eps) in fp32.
__global__ void __launch_bounds__(256)
    normalize_rows_kernel(const void* __restrict__ src, int dtype, int64_t n_vec, int dim, int dim_pad,
                          int64_t ld, float eps, float* __restrict__ dst) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (row >= n_vec) return;
  double acc = 0.0;
  for (int d = lane; d < dim; d += 32) {
    const double v = double(ld_f32(src, dtype, row * ld + d));
    acc += v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  const float denom = fmaxf(float(sqrt(acc)), eps);
  for (int d = lane; d < dim_pad; d += 32)
    dst[row * dim_pad + d] = d < dim ? __fdiv_rn(ld_f32(src, dtype, row * ld + d), denom) : 0.0f;
}

// ||row||^2 in the same defined order as normalize_rows_kernel, rounded once to fp32
__global__ void __launch_bounds__(256)
    row_sqnorm_kernel(const void* __restrict__ src, int dtype, int64_t n_vec, int dim, int64_t ld,
                      float* __restrict__ out) {
  const int lane = threadIdx.x & 31;
  const int64_t row = (int64_t(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  if (row >= n_vec) return;
  double acc = 0.0;
  for (int d = lane; d < dim; d += 32) {
    const double v = double(ld_f32(src, dtype, row * ld + d));
    acc += v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
  if (lane == 0) out[row] = float(acc);
}

}  // namespace

cudaError_t launch_row_sqnorm(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld, float* out,
                              cudaStream_t stream) {
  if (n_vec == 0) return cudaSuccess;
  const int64_t blocks = (n_vec * 32 + 255) / 256;
  row_sqnorm_kernel<<<unsigned(blocks), 256, 0, stream>>>(src, src_dtype, n_vec, dim, ld, out);
  return cudaGetLastError();
}

cudaError_t launch_normalize_rows(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld,
                                  float eps, float* dst, cudaStream_t stream) {
  if (n_vec == 0) return cudaSuccess;
  const int dim_pad = (dim + 63) / 64 * 64;
  const int64_t blocks = (n_vec * 32 + 255) / 256;
  normalize_rows_kernel<<<unsigned(blocks), 256, 0, stream>>>(src, src_dtype, n_vec, dim, dim_pad, ld, eps,
                                                              dst);
  return cudaGetLastError();
}

cudaError_t launch_prepare(const void* src, int src_dtype, int src_layout, int64_t n_vec, int dim,
                           int64_t ld, int mode, void* dst_hi, void* dst_lo, cudaStream_t stream) {
  if (n_vec == 0) return cudaSuccess;
  const int dim_pad = (dim + 63) / 64 * 64;
  if (src_layout == B200KNN_LAYOUT_DN) {
    dim3 grid(unsigned((n_vec + 63) / 64), unsigned(dim_pad / 64));
    prepare_dn_kernel<<<grid, 256, 0, stream>>>(src, src_dtype, n_vec, dim, dim_pad, ld, mode,
                                                dst_hi, dst_lo);
  } else {
    const int64_t total = n_vec * dim_pad;
    prepare_nd_kernel<<<unsigned((total + 255) / 256), 256, 0, stream>>>(
        src, src_dtype, n_vec, dim, dim_pad, ld, mode, dst_hi, dst_lo);
  }
  return cudaGetLastError();
}

}  // namespace b200knn
