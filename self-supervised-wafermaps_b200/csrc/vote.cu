// vote.cu — exp(sim/t)-weighted class vote and class ranking.
//
// Replaces the tail of lightly's knn_predict (gather -> div/exp -> zeros +
// scatter one-hot -> mul/sum -> argsort(descending); reference call site
// src/ssl_wafermap/models/knn.py:91-98, consumer :99 `pred_labels[:, 0]`).
// No (B*K, C) one-hot is materialised.  Scores are accumulated in fp64 in rank
// order j = 0..k-1, so they do not depend on the launch geometry; classes are
// ranked by (score desc, class asc), which fixes the tie order torch's argsort
// leaves unspecified for C > 16 (SURVEY.md §7.3).
//
// HBM-bound: per row k*8 B of keys + k gathered labels in, C*8 B out.
#include "common.cuh"
#include "kernels.h"

namespace b200knn {
namespace {

constexpr int kVoteWarps = 4;

__global__ void __launch_bounds__(kVoteWarps * 32)
    vote_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ labels, int64_t B,
                int k, int64_t n_labels, int64_t label_offset, int C, double t,
                int64_t* __restrict__ pred, int64_t pred_ld, int status_col,
                double* __restrict__ scores, int32_t* __restrict__ err_flag) {
  extern __shared__ unsigned char vote_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // per warp: w[k] f64 | sc[C] f64 | lab[k] i32
  const size_t per_warp = size_t(k) * 8 + size_t(C) * 8 + size_t(k) * 4;
  unsigned char* base = vote_smem + size_t(warp) * ((per_warp + 7) / 8 * 8);
  double* w = reinterpret_cast<double*>(base);
  double* sc = w + k;
  int* lab = reinterpret_cast<int*>(sc + C);

  const int64_t row = int64_t(blockIdx.x) * kVoteWarps + warp;
  if (row >= B) return;

  int bad = 0;  // per-row status: 1 empty k-th slot (starved row), 2 label / 4 index out of range
  for (int j = lane; j < k; j += 32) {
    const uint64_t key = keys[row * k + j];
    int l = -1;
    double wj = 0.0;
    if (key != 0) {
      const int64_t li = key_idx(key) - label_offset;
      if (li >= 0 && li < n_labels) {
        const int64_t c = labels[li];
        if (c >= 0 && c < C) {
          l = int(c);
          wj = exp(double(key_sim(key)) / t);
        } else {
          atomicExch(err_flag, 1);
          bad |= 2;
        }
      } else {
        atomicExch(err_flag, 2);
        bad |= 4;
      }
    } else if (j == k - 1) {
      bad |= 1;
    }
    lab[j] = l;
    w[j] = wj;
  }
  if (status_col >= 0) {
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (lane == 0) pred[row * pred_ld + status_col] = bad;
  }
  __syncwarp();
  for (int c = lane; c < C; c += 32) {
    double acc = 0.0;
    for (int j = 0; j < k; ++j)
      if (lab[j] == c) acc += w[j];
    sc[c] = acc;
    if (scores) scores[row * C + c] = acc;
  }
  __syncwarp();
  for (int c = lane; c < C; c += 32) {
    const double s = sc[c];
    int rank = 0;
    for (int o = 0; o < C; ++o) {
      const double so = sc[o];
      rank += (so > s || (so == s && o < c)) ? 1 : 0;
    }
    pred[row * pred_ld + rank] = c;
  }
}

// vote_kernel for a grid of (k, t) settings from one top-k_max list per row: block (i, j) of a
// row's output is vote_kernel's ranking of its first ks[i] keys at temperature ts[j].  Per t the
// warp evaluates w[j] = exp(double(sim_j) / t) across its lanes (vote_kernel's expression), then a
// lane per class accumulates them in rank order j = 0, 1, ... (vote_kernel's order) and, whenever
// j + 1 reaches ks[i], the warp ranks the accumulators (vote_kernel's rank rule): every block is
// bitwise vote_kernel's result.  (Evaluating the exps in the lane that owns the class instead
// leaves most lanes idle at C = 9: the grid call cost 1.089x one k = 200 call at the north
// star that way, 1.003-1.050x this way; DESIGN §7.)
__global__ void __launch_bounds__(kVoteWarps * 32)
    vote_multi_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ labels, int64_t B,
                      int64_t n_labels, int64_t label_offset, int C, VoteGrid grid,
                      int64_t* __restrict__ pred, int64_t pred_ld, int status_col,
                      int32_t* __restrict__ err_flag) {
  extern __shared__ unsigned char vote_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = grid.ks[grid.n_k - 1], n_t = grid.n_t;
  // per warp: w[k] f64 | sc[C] f64 | sim[k] f32 | lab[k] i32
  const size_t per_warp = size_t(k) * 16 + size_t(C) * 8;
  unsigned char* base = vote_smem + size_t(warp) * per_warp;
  double* w = reinterpret_cast<double*>(base);
  double* sc = w + k;
  float* sim = reinterpret_cast<float*>(sc + C);
  int* lab = reinterpret_cast<int*>(sim + k);

  const int64_t row = int64_t(blockIdx.x) * kVoteWarps + warp;
  if (row >= B) return;

  int bad = 0;  // vote_kernel's status bits
  for (int j = lane; j < k; j += 32) {
    const uint64_t key = keys[row * k + j];
    int l = -1;
    if (key != 0) {
      const int64_t li = key_idx(key) - label_offset;
      if (li >= 0 && li < n_labels) {
        const int64_t c = labels[li];
        if (c >= 0 && c < C) {
          l = int(c);
        } else {
          atomicExch(err_flag, 1);
          bad |= 2;
        }
      } else {
        atomicExch(err_flag, 2);
        bad |= 4;
      }
    } else if (j == k - 1) {
      bad |= 1;
    }
    lab[j] = l;
    sim[j] = key_sim(key);
  }
  if (status_col >= 0) {
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (lane == 0) pred[row * pred_ld + status_col] = bad;
  }
  int64_t* out = pred + row * pred_ld;
  for (int ti = 0; ti < n_t; ++ti) {
    const double t = grid.ts[ti];
    __syncwarp();  // lab / sim written; the previous t's ranking is done with w
    for (int j = lane; j < k; j += 32) w[j] = lab[j] >= 0 ? exp(double(sim[j]) / t) : 0.0;
    for (int c = lane; c < C; c += 32) sc[c] = 0.0;
    __syncwarp();
    int j0 = 0;
    for (int s = 0; s < grid.n_k; ++s) {
      const int j1 = grid.ks[s];
      for (int c = lane; c < C; c += 32) {
        double acc = sc[c];
        for (int j = j0; j < j1; ++j)
          if (lab[j] == c) acc += w[j];
        sc[c] = acc;
      }
      j0 = j1;
      __syncwarp();
      int64_t* o = out + (int64_t(s) * n_t + ti) * C;
      for (int c = lane; c < C; c += 32) {
        const double v = sc[c];
        int rank = 0;
        for (int q = 0; q < C; ++q) {
          const double sq = sc[q];
          rank += (sq > v || (sq == v && q < c)) ? 1 : 0;
        }
        o[rank] = c;
      }
      __syncwarp();  // every lane has read sc before the next segment adds to it
    }
  }
}

// counts[t * C + p] += 1 for every (target t, prediction p): the confusion matrix the
// reference builds with torchmetrics after each validation epoch
// (src/ssl_wafermap/models/knn.py:104-129).  Block-private histograms in shared memory
// (C <= 64), one global atomic per non-zero cell per block.
__global__ void __launch_bounds__(256)
    confusion_kernel(const int64_t* __restrict__ pred, const int64_t* __restrict__ target, int64_t n, int C,
                     unsigned long long* __restrict__ counts, int32_t* __restrict__ err_flag) {
  extern __shared__ unsigned int cm_smem[];
  for (int i = threadIdx.x; i < C * C; i += blockDim.x) cm_smem[i] = 0u;
  __syncthreads();
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t p = pred[i], t = target[i];
    if (p >= 0 && p < C && t >= 0 && t < C) atomicAdd(&cm_smem[t * C + p], 1u);
    else atomicExch(err_flag, 1);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < C * C; i += blockDim.x)
    if (cm_smem[i]) atomicAdd(&counts[i], static_cast<unsigned long long>(cm_smem[i]));
}

}  // namespace

cudaError_t launch_confusion(const int64_t* pred, const int64_t* target, int64_t n, int C, int64_t* counts,
                             int32_t* err_flag, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  if (C > 64) return cudaErrorInvalidValue;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  confusion_kernel<<<unsigned(blocks), 256, size_t(C) * C * sizeof(unsigned int), stream>>>(
      pred, target, n, C, reinterpret_cast<unsigned long long*>(counts), err_flag);
  return cudaGetLastError();
}

cudaError_t launch_vote(const uint64_t* keys, const int64_t* labels, int64_t B, int k,
                        int64_t n_labels, int64_t label_offset, int C, double t, int64_t* pred,
                        int64_t pred_ld, int status_col, double* scores, int32_t* err_flag,
                        cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const size_t per_warp = (size_t(k) * 8 + size_t(C) * 8 + size_t(k) * 4 + 7) / 8 * 8;
  const size_t smem = per_warp * kVoteWarps;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(vote_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(smem));
    if (e != cudaSuccess) return e;
  }
  const int64_t blocks = (B + kVoteWarps - 1) / kVoteWarps;
  vote_kernel<<<unsigned(blocks), kVoteWarps * 32, smem, stream>>>(
      keys, labels, B, k, n_labels, label_offset, C, t, pred, pred_ld, status_col, scores, err_flag);
  return cudaGetLastError();
}

cudaError_t launch_vote_multi(const uint64_t* keys, const int64_t* labels, int64_t B, int64_t n_labels,
                              int64_t label_offset, int C, const VoteGrid& grid, int64_t* pred, int64_t pred_ld,
                              int status_col, int32_t* err_flag, cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const size_t per_warp = size_t(grid.ks[grid.n_k - 1]) * 16 + size_t(C) * 8;
  const size_t smem = per_warp * kVoteWarps;
  if (smem > 200 * 1024) return cudaErrorInvalidValue;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(vote_multi_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         int(smem));
    if (e != cudaSuccess) return e;
  }
  const int64_t blocks = (B + kVoteWarps - 1) / kVoteWarps;
  vote_multi_kernel<<<unsigned(blocks), kVoteWarps * 32, smem, stream>>>(
      keys, labels, B, n_labels, label_offset, C, grid, pred, pred_ld, status_col, err_flag);
  return cudaGetLastError();
}

}  // namespace b200knn
