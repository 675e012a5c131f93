// exact.cu — MODE_EXACT: fused fp32 similarity + streaming top-k on CUDA cores.
//
// sim(q, n) = fmaf chain over d = 0..D-1 in that order starting from +0.0f, so
// every similarity is bitwise independent of tiling, batch size, split and
// shard count, and bitwise reproducible on a CPU with fmaf (oracle/seqfma.c).
// This is the on-device golden the tensor-core modes are validated against at
// sizes the CPU oracle cannot cover, and the exact re-scoring reference.
//
// Replaces torch.mm + Tensor.topk of lightly's knn_predict (reference call
// site src/ssl_wafermap/models/knn.py:91-98); the (B,N) similarity matrix is
// never written to HBM.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"
#include "kernels.h"

namespace b200knn {

namespace {

constexpr int TM = 128, TN = 128, TD = 16;
constexpr int S_LD = TN + 1;

__device__ __forceinline__ float load_f32(const void* p, int dtype, int64_t i) {
  if (dtype == 0) return static_cast<const float*>(p)[i];
  if (dtype == 1) return __half2float(static_cast<const __half*>(p)[i]);
  return __bfloat162float(static_cast<const __nv_bfloat16*>(p)[i]);
}

// EXCL: bank columns of the query row's group (ExactParams::q_gid / bank_gid) are never admitted;
// the filter sits next to the peeling bound, so every pass of a peeled search applies it.
template <int ITEMS, bool EXCL>
__global__ void __launch_bounds__(256) exact_topk_kernel(ExactParams p) {
  extern __shared__ float smem[];
  float* As = smem;              // [TD][TM]  queries, d-major
  float* Bs = As + TD * TM;      // [TD][TN]  bank
  float* S = Bs + TD * TN;       // [TM][S_LD] similarity tile
  constexpr int CAP = ITEMS * 32;

  const int tid = threadIdx.x;
  const int lane = tid & 31, warp = tid >> 5;
  const int tx = tid & 15, ty = tid >> 4;
  const float neg_inf = __int_as_float(0xff800000);
  const float pos_inf = __int_as_float(0x7f800000);

  uint64_t* warp_lists = p.lists + (size_t(blockIdx.x) * TM + size_t(warp) * 32) * CAP;

  for (int64_t item = blockIdx.x; item < p.n_items; item += gridDim.x) {
    const int64_t qt = item % p.n_qtiles;
    const int64_t sp = item / p.n_qtiles;
    const int64_t m0 = qt * TM;
    const int64_t n_begin = sp * p.split_rows;
    const int64_t n_end = (n_begin + p.split_rows < p.N) ? n_begin + p.split_rows : p.N;

    RowState st;
    st.cnt = 0;
    st.tau = (m0 + tid < p.B) ? neg_inf : pos_inf;  // only meaningful for tid < TM
    // k > 992 is served in passes ("peeling", b200knn/knn.py): pass i admits only keys strictly
    // below the last key of pass i-1.  Filtering the stream keeps the threshold logic valid.
    const uint64_t upper = (p.upper != nullptr && tid < TM && m0 + tid < p.B) ? p.upper[m0 + tid] : ~0ull;
    int32_t my_gid = 0;
    if constexpr (EXCL) my_gid = (tid < TM && m0 + tid < p.B) ? p.q_gid[m0 + tid] : 0;

    for (int64_t n0 = n_begin; n0 < n_end; n0 += TN) {
      float acc[8][8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.0f;

      for (int d0 = 0; d0 < p.D; d0 += TD) {
        float ra[8], rb[8];
        {
          const int m = tid >> 1, dd0 = (tid & 1) * 8;
          const int64_t gm = m0 + m;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int d = d0 + dd0 + e;
            ra[e] = (gm < p.B && d < p.D) ? load_f32(p.q, p.q_dtype, gm * p.q_ld + d) : 0.0f;
          }
        }
        {
          const int dd = tid >> 4, nn0 = (tid & 15) * 8;
          const int d = d0 + dd;
#pragma unroll
          for (int e = 0; e < 8; ++e) {
            const int64_t gn = n0 + nn0 + e;
            rb[e] = (gn < n_end && d < p.D)
                        ? load_f32(p.bank, p.bank_dtype, int64_t(d) * p.bank_sd + gn * p.bank_sn)
                        : 0.0f;
          }
        }
        __syncthreads();
        {
          const int m = tid >> 1, dd0 = (tid & 1) * 8;
#pragma unroll
          for (int e = 0; e < 8; ++e) As[(dd0 + e) * TM + m] = ra[e];
          const int dd = tid >> 4, nn0 = (tid & 15) * 8;
#pragma unroll
          for (int e = 0; e < 8; ++e) Bs[dd * TN + nn0 + e] = rb[e];
        }
        __syncthreads();
#pragma unroll
        for (int dd = 0; dd < TD; ++dd) {
          float a[8], b[8];
          const float4 a0 = *reinterpret_cast<const float4*>(&As[dd * TM + ty * 4]);
          const float4 a1 = *reinterpret_cast<const float4*>(&As[dd * TM + 64 + ty * 4]);
          const float4 b0 = *reinterpret_cast<const float4*>(&Bs[dd * TN + tx * 4]);
          const float4 b1 = *reinterpret_cast<const float4*>(&Bs[dd * TN + 64 + tx * 4]);
          a[0] = a0.x; a[1] = a0.y; a[2] = a0.z; a[3] = a0.w;
          a[4] = a1.x; a[5] = a1.y; a[6] = a1.z; a[7] = a1.w;
          b[0] = b0.x; b[1] = b0.y; b[2] = b0.z; b[3] = b0.w;
          b[4] = b1.x; b[5] = b1.y; b[6] = b1.z; b[7] = b1.w;
#pragma unroll
          for (int i = 0; i < 8; ++i)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[i][j] = __fmaf_rn(a[i], b[j], acc[i][j]);
        }
      }

#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const int r = (i < 4) ? ty * 4 + i : 64 + ty * 4 + (i - 4);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          const int c = (j < 4) ? tx * 4 + j : 64 + tx * 4 + (j - 4);
          S[r * S_LD + c] = acc[i][j];
        }
      }
      __syncthreads();

      if (tid < TM) {
        uint64_t* my_list = warp_lists + size_t(lane) * CAP;
        for (int c0 = 0; c0 < TN; c0 += 32) {
          float s[32];
#pragma unroll
          for (int j = 0; j < 32; ++j) s[j] = S[tid * S_LD + c0 + j];
          uint32_t c = st.cnt;
#pragma unroll
          for (int j = 0; j < 32; ++j) {
            if (s[j] > st.tau) {
              const int64_t gn = n0 + c0 + j;
              const uint64_t key = make_key(s[j], uint32_t(gn + p.idx_offset));
              bool ok = gn < n_end && key < upper;
              if constexpr (EXCL) ok = ok && __ldg(p.bank_gid + gn) != my_gid;
              if (ok) my_list[c++] = key;
            }
          }
          st.cnt = c;
          warp_maintain<ITEMS>(warp_lists, st, p.k, lane, 32);
        }
      }
      __syncthreads();
    }

    if (tid < TM) {
      const int64_t row0 = m0 + int64_t(warp) * 32;
      unsigned valid = 0;
      if (row0 < p.B) {
        const int64_t nv = p.B - row0;
        valid = nv >= 32 ? kFull : ((1u << nv) - 1u);
      }
      uint64_t* out = p.out + (size_t(sp) * p.B + row0) * p.k;
      warp_flush<ITEMS>(warp_lists, st, p.k, lane, valid,
                        [&](int r) { return out + size_t(r) * size_t(p.k); });
    }
    __syncthreads();
  }
}

template <int ITEMS, bool EXCL>
cudaError_t launch_exact_t(const ExactParams& p, int grid, cudaStream_t stream) {
  const size_t smem = sizeof(float) * (TD * TM + TD * TN + TM * S_LD);
  cudaError_t e = cudaFuncSetAttribute(exact_topk_kernel<ITEMS, EXCL>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) return e;
  exact_topk_kernel<ITEMS, EXCL><<<grid, 256, smem, stream>>>(p);
  return cudaGetLastError();
}

template <bool EXCL>
cudaError_t launch_exact_cap(const ExactParams& p, int grid, int cap, cudaStream_t stream) {
  switch (cap) {
    case 64: return launch_exact_t<2, EXCL>(p, grid, stream);
    case 128: return launch_exact_t<4, EXCL>(p, grid, stream);
    case 256: return launch_exact_t<8, EXCL>(p, grid, stream);
    case 512: return launch_exact_t<16, EXCL>(p, grid, stream);
    case 1024: return launch_exact_t<32, EXCL>(p, grid, stream);
    default: return cudaErrorInvalidValue;
  }
}

}  // namespace

cudaError_t launch_exact(const ExactParams& p, int grid, int cap, cudaStream_t stream) {
  return p.bank_gid != nullptr ? launch_exact_cap<true>(p, grid, cap, stream)
                               : launch_exact_cap<false>(p, grid, cap, stream);
}

}  // namespace b200knn
