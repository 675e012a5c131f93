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
constexpr int kConfusionSmemClasses = 64;  // larger C counts with global atomics

// Shared memory per warp for chunks of kc keys and C classes:
//   vote_kernel        w[kc] f64 | sc[C] f64 | lab[kc] i32            (8-byte aligned)
//   vote_multi_kernel  w[kc] f64 | sc[C] f64 | sim[kc] f32 | lab[kc] i32
__host__ __device__ inline size_t vote_warp_bytes(int kc, int C, bool multi) {
  return multi ? size_t(kc) * 16 + size_t(C) * 8 : (size_t(kc) * 12 + size_t(C) * 8 + 7) / 8 * 8;
}

__global__ void __launch_bounds__(kVoteWarps * 32)
    vote_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ labels, int64_t B,
                int k, int64_t n_labels, int64_t label_offset, int C, double t,
                int64_t* __restrict__ pred, int64_t pred_ld, int status_col,
                double* __restrict__ scores, int32_t* __restrict__ err_flag) {
  extern __shared__ unsigned char vote_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int kc = k < kVoteChunk ? k : kVoteChunk;  // k <= kVoteChunk: the whole row is one chunk
  unsigned char* base = vote_smem + size_t(warp) * vote_warp_bytes(kc, C, false);
  double* w = reinterpret_cast<double*>(base);
  double* sc = w + kc;
  int* lab = reinterpret_cast<int*>(sc + C);

  const int64_t row = int64_t(blockIdx.x) * kVoteWarps + warp;
  if (row >= B) return;

  int bad = 0;  // per-row status: 1 empty k-th slot (starved row), 2 label / 4 index out of range
  for (int j0 = 0; j0 < k; j0 += kc) {
    const int n = k - j0 < kc ? k - j0 : kc;
    __syncwarp();  // every lane is done with the previous chunk
    for (int i = lane; i < n; i += 32) {
      const int j = j0 + i;
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
      lab[i] = l;
      w[i] = wj;
    }
    __syncwarp();
    // sc[c] carries the class's score from chunk to chunk: the adds run in rank order j = 0..k-1,
    // so the score does not depend on the chunk length
    for (int c = lane; c < C; c += 32) {
      double acc = j0 ? sc[c] : 0.0;
      for (int i = 0; i < n; ++i)
        if (lab[i] == c) acc += w[i];
      sc[c] = acc;
      if (scores && j0 + n == k) scores[row * C + c] = acc;
    }
  }
  if (status_col >= 0) {
    bad = __reduce_or_sync(0xffffffffu, bad);
    if (lane == 0) pred[row * pred_ld + status_col] = bad;
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
// CHUNKED (k_max > kVoteChunk): the row is walked in chunks once per t.  t is the outer loop, so one
// score array serves every t and the class bound does not depend on n_t.  Otherwise the row is read
// once and kept for every t; a separate instantiation keeps that path's registers and occupancy.
template <bool CHUNKED>
__global__ void __launch_bounds__(kVoteWarps * 32)
    vote_multi_kernel(const uint64_t* __restrict__ keys, const int64_t* __restrict__ labels, int64_t B,
                      int64_t n_labels, int64_t label_offset, int C, VoteGrid grid,
                      int64_t* __restrict__ pred, int64_t pred_ld, int status_col,
                      int32_t* __restrict__ err_flag) {
  extern __shared__ unsigned char vote_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int k = grid.ks[grid.n_k - 1], n_t = grid.n_t;
  const int kc = k < kVoteChunk ? k : kVoteChunk;
  unsigned char* base = vote_smem + size_t(warp) * vote_warp_bytes(kc, C, true);
  double* w = reinterpret_cast<double*>(base);
  double* sc = w + kc;
  float* sim = reinterpret_cast<float*>(sc + C);
  int* lab = reinterpret_cast<int*>(sim + kc);

  const int64_t row = int64_t(blockIdx.x) * kVoteWarps + warp;
  if (row >= B) return;

  int bad = 0;  // vote_kernel's status bits
  auto load = [&](int j0, int n) {  // keys [j0, j0 + n) of the row -> lab / sim
    for (int i = lane; i < n; i += 32) {
      const int j = j0 + i;
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
      lab[i] = l;
      sim[i] = key_sim(key);
    }
  };
  auto add = [&](int a, int e) {  // keys [a, e) of the chunk onto the lane's classes
    for (int c = lane; c < C; c += 32) {
      double acc = sc[c];
      for (int i = a; i < e; ++i)
        if (lab[i] == c) acc += w[i];
      sc[c] = acc;
    }
  };
  int64_t* out = pred + row * pred_ld;
  auto rank_into = [&](int s, int ti) {  // vote_kernel's ranking of sc into block (s, ti)
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
  };
  auto store_status = [&]() {
    if (status_col >= 0) {
      bad = __reduce_or_sync(0xffffffffu, bad);
      if (lane == 0) out[status_col] = bad;
    }
  };
  if constexpr (!CHUNKED) {
    load(0, k);
    store_status();
    for (int ti = 0; ti < n_t; ++ti) {
      const double t = grid.ts[ti];
      __syncwarp();  // lab / sim written; the previous t's ranking is done with w
      for (int j = lane; j < k; j += 32) w[j] = lab[j] >= 0 ? exp(double(sim[j]) / t) : 0.0;
      for (int c = lane; c < C; c += 32) sc[c] = 0.0;
      __syncwarp();
      int j0 = 0;
      for (int s = 0; s < grid.n_k; ++s) {
        add(j0, grid.ks[s]);
        j0 = grid.ks[s];
        rank_into(s, ti);
      }
    }
  } else {
    for (int ti = 0; ti < n_t; ++ti) {
      const double t = grid.ts[ti];
      int s = 0;  // the next segment ends at ks[s]
      for (int j0 = 0; j0 < k; j0 += kc) {
        const int n = k - j0 < kc ? k - j0 : kc;
        __syncwarp();  // every lane is done with the previous chunk
        load(j0, n);
        __syncwarp();
        for (int i = lane; i < n; i += 32) w[i] = lab[i] >= 0 ? exp(double(sim[i]) / t) : 0.0;
        if (j0 == 0)
          for (int c = lane; c < C; c += 32) sc[c] = 0.0;
        __syncwarp();
        for (int a = 0; a < n;) {  // the segments of this chunk; a boundary may fall anywhere in it
          const int e = grid.ks[s] - j0 < n ? grid.ks[s] - j0 : n;
          add(a, e);
          a = e;
          if (j0 + e == grid.ks[s]) rank_into(s++, ti);
        }
      }
    }
    store_status();  // the bits of every pass: the same on each
  }
}

// counts[t * C + p] += 1 for every (target t, prediction p): the confusion matrix the
// reference builds with torchmetrics after each validation epoch
// (src/ssl_wafermap/models/knn.py:104-129).  Up to kConfusionSmemClasses classes: block-private
// histograms in shared memory, one global atomic per non-zero cell per block; above, one global
// atomic per prediction (the C*C matrix no longer fits, and its cells are rarely contended).
__global__ void __launch_bounds__(256)
    confusion_kernel(const int64_t* __restrict__ pred, const int64_t* __restrict__ target, int64_t n, int C,
                     unsigned long long* __restrict__ counts, int32_t* __restrict__ err_flag) {
  extern __shared__ unsigned int cm_smem[];
  const bool in_smem = C <= kConfusionSmemClasses;
  if (in_smem)
    for (int i = threadIdx.x; i < C * C; i += blockDim.x) cm_smem[i] = 0u;
  __syncthreads();
  for (int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x; i < n; i += int64_t(gridDim.x) * blockDim.x) {
    const int64_t p = pred[i], t = target[i];
    if (p >= 0 && p < C && t >= 0 && t < C) {
      if (in_smem) atomicAdd(&cm_smem[t * C + p], 1u);
      else atomicAdd(&counts[t * C + p], 1ull);
    } else {
      atomicExch(err_flag, 1);
    }
  }
  if (!in_smem) return;
  __syncthreads();
  for (int i = threadIdx.x; i < C * C; i += blockDim.x)
    if (cm_smem[i]) atomicAdd(&counts[i], static_cast<unsigned long long>(cm_smem[i]));
}

}  // namespace

cudaError_t launch_confusion(const int64_t* pred, const int64_t* target, int64_t n, int C, int64_t* counts,
                             int32_t* err_flag, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  int64_t blocks = (n + 255) / 256;
  if (blocks > 148 * 4) blocks = 148 * 4;
  const size_t smem = C <= kConfusionSmemClasses ? size_t(C) * C * sizeof(unsigned int) : 0;
  confusion_kernel<<<unsigned(blocks), 256, smem, stream>>>(
      pred, target, n, C, reinterpret_cast<unsigned long long*>(counts), err_flag);
  return cudaGetLastError();
}

cudaError_t launch_vote(const uint64_t* keys, const int64_t* labels, int64_t B, int k,
                        int64_t n_labels, int64_t label_offset, int C, double t, int64_t* pred,
                        int64_t pred_ld, int status_col, double* scores, int32_t* err_flag,
                        cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const size_t smem = vote_warp_bytes(k < kVoteChunk ? k : kVoteChunk, C, false) * kVoteWarps;
  if (smem > size_t(kVoteSmemBytes)) return cudaErrorInvalidValue;
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
  const int k = grid.ks[grid.n_k - 1];
  const size_t smem = vote_warp_bytes(k < kVoteChunk ? k : kVoteChunk, C, true) * kVoteWarps;
  if (smem > size_t(kVoteSmemBytes)) return cudaErrorInvalidValue;
  const auto kernel = k > kVoteChunk ? vote_multi_kernel<true> : vote_multi_kernel<false>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
  }
  const int64_t blocks = (B + kVoteWarps - 1) / kVoteWarps;
  kernel<<<unsigned(blocks), kVoteWarps * 32, smem, stream>>>(
      keys, labels, B, n_labels, label_offset, C, grid, pred, pred_ld, status_col, err_flag);
  return cudaGetLastError();
}

}  // namespace b200knn
