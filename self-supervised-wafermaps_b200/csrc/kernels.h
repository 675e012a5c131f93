// kernels.h — internal launch interfaces between api.cu and the kernel files.
#pragma once
#include <cstddef>
#include <cstdint>
#include <cuda_runtime.h>

namespace b200knn {

struct ExactParams {
  const void* q;
  int q_dtype;
  int64_t q_ld;
  const void* bank;
  int bank_dtype;
  int64_t bank_sd;  // element stride between consecutive d of one bank vector
  int64_t bank_sn;  // element stride between consecutive bank vectors
  int64_t B, N;
  int D, k;
  int64_t idx_offset;
  int64_t n_qtiles, n_items, split_rows;
  uint64_t* lists;
  uint64_t* out;  // (splits, B, k)
  const uint64_t* upper = nullptr;  // optional (B,): only keys strictly below upper[row] are admitted
  // optional group exclusion (both or neither): q_gid (B,), bank_gid (N,) indexed before idx_offset;
  // bank row n is never admitted to query row b's list when bank_gid[n] == q_gid[b]
  const int32_t* q_gid = nullptr;
  const int32_t* bank_gid = nullptr;
};

cudaError_t launch_exact(const ExactParams& p, int grid, int cap, cudaStream_t stream);

// merge G sorted lists per row: in (G,B,k_in) -> out (B,k_out)
cudaError_t launch_merge(const uint64_t* in, int G, int64_t B, int k_in, int k_out, uint64_t* out,
                         cudaStream_t stream);
cudaError_t launch_decode(const uint64_t* keys, int64_t n, float* sims, int64_t* idx,
                          cudaStream_t stream);
// (B, k_in) sorted keys -> (B, k_in - 1) without bank row b + self_offset's key (else the last)
cudaError_t launch_drop_self(const uint64_t* in, int64_t B, int k_in, int64_t self_offset, uint64_t* out,
                             cudaStream_t stream);
// (B, k_in) sorted keys -> (B, k_out): the first k_out keys outside row row_ids[b]'s group
// (group_ids (N,)), zero-filled; err_flag = 2 on a key index or row id outside [0, N)
cudaError_t launch_drop_group(const uint64_t* in, int64_t B, int k_in, const int64_t* row_ids,
                              const int32_t* group_ids, int64_t N, int k_out, uint64_t* out, int32_t* err_flag,
                              cudaStream_t stream);
// The vote kernels stream a row's keys through shared memory in chunks of at most kVoteChunk, so
// k is unbounded; the per-warp fp64 score array of C classes is not.  A launch whose shared
// memory, 4 warps x (chunk arrays + 8 C bytes), exceeds kVoteSmemBytes returns
// cudaErrorInvalidValue (b200knn/knn.py restates the bound as vote_max_classes).
constexpr int kVoteChunk = 1024;
constexpr int kVoteSmemBytes = 200 * 1024;
cudaError_t launch_vote(const uint64_t* keys, const int64_t* labels, int64_t B, int k,
                        int64_t n_labels, int64_t label_offset, int C, double t, int64_t* pred,
                        int64_t pred_ld, int status_col, double* scores, int32_t* err_flag,
                        cudaStream_t stream);
// launch_vote for every (ks[i], ts[j]) from one (B, ks[n_k-1]) key list; ks strictly increasing.
// Passed by value, so a captured launch needs no device-side copy of the grid.
constexpr int kVoteMaxKs = 16, kVoteMaxTs = 8;
struct VoteGrid {
  int n_k, n_t;
  int ks[kVoteMaxKs];
  double ts[kVoteMaxTs];
};
cudaError_t launch_vote_multi(const uint64_t* keys, const int64_t* labels, int64_t B, int64_t n_labels,
                              int64_t label_offset, int C, const VoteGrid& grid, int64_t* pred, int64_t pred_ld,
                              int status_col, int32_t* err_flag, cudaStream_t stream);
// out[b] = similarity of keys[b, j] (-inf for an empty slot)
cudaError_t launch_key_sim_column(const uint64_t* keys, int64_t B, int k, int j, float* out,
                                  cudaStream_t stream);
cudaError_t launch_prepare(const void* src, int src_dtype, int src_layout, int64_t n_vec, int dim,
                           int64_t ld, int mode, void* dst_hi, void* dst_lo, cudaStream_t stream);

// fused F.normalize(dim=1) + relayout into (n_vec, dim_pad) fp32 rows (prepare.cu)
cudaError_t launch_normalize_rows(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld,
                                  float eps, float* dst, cudaStream_t stream);
cudaError_t launch_row_sqnorm(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld, float* out,
                              cudaStream_t stream);
// confusion-matrix counts (vote.cu): counts (C,C) int64 += histogram of (target, pred); any C
cudaError_t launch_confusion(const int64_t* pred, const int64_t* target, int64_t n, int C, int64_t* counts,
                             int32_t* err_flag, cudaStream_t stream);

// exact re-scoring of tensor-core candidates (rescore.cu)
struct RescoreParams {
  const void* q;        // caller queries (B, dim), row-major, ld = q_ld
  int q_dtype;
  int64_t q_ld;
  const float* rows_a;  // (N, dim_pad) fp32 bank rows; value = rows_a + rows_b when rows_b != nullptr
  const float* rows_b;
  int dim, dim_pad;
  const uint64_t* cand;  // (B, k_in) candidate keys, sorted descending under the approximate sims
  int64_t B;
  int k_in, k_out;
  int all_rows;  // k_in >= N: every bank row is a candidate, empty slots are legitimate
  int64_t idx_offset;
  float err_coef;              // E = err_coef * ||q|| * M + err_abs * (||q|| + M),  M = *bank_max_norm
  float err_abs;
  float max_abs;               // > 0: rows with ||q|| or M >= max_abs are uncertified (operand range)
  const float* bank_max_norm;  // device scalar
  uint64_t* out;               // (B, k_out)
  int32_t* uncertified;        // (B,)
  int32_t* n_uncertified;      // device counter (caller zeroes)
  // sharded re-scoring: the sorted exact keys of query row b are stored into the exchange buffer
  // of the GPU that owns b, at [my_rank][b - owner*rows_per_owner][:k_out] (peer memory); no
  // certificate is evaluated (out / uncertified / n_uncertified unused)
  uint64_t* peer_out[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int n_peers = 0, my_rank = 0;
  int64_t rows_per_owner = 0;
};
// workspace (optional, rescore_workspace_bytes): selects the TMA-pipelined two-kernel variant
cudaError_t launch_rescore(const RescoreParams& p, void* workspace, size_t workspace_bytes,
                           cudaStream_t stream);
size_t rescore_workspace_bytes(int64_t B, int k_in);
// the certificate alone: p.out = merged exact keys (read), p.cand = merged approximate candidates
cudaError_t launch_certify(const RescoreParams& p, cudaStream_t stream);
// split (n, k) key lists by owning shard: out (G, n, k), each shard's keys compacted to the front
cudaError_t launch_route_keys(const uint64_t* keys, int64_t n, int k, int64_t rows_per_shard, int G,
                              uint64_t* out, cudaStream_t stream);
// sharded_ops.cu
cudaError_t launch_route_scatter(const uint64_t* keys, int64_t n, int k, int64_t rows_per_shard, int G,
                                 uint64_t* const* inbox, int64_t row_offset, cudaStream_t stream);
cudaError_t launch_broadcast_f32(const float* src, int64_t n, float* const* dst, int G, int64_t dst_offset,
                                 cudaStream_t stream);
cudaError_t launch_compact_rows(const int64_t* status, int64_t ld, int64_t n, int64_t mask, int64_t* rows_out,
                                int cap, int32_t* count_out, cudaStream_t stream);
cudaError_t launch_scatter_rows(int64_t* dst, int64_t dst_ld, const int64_t* src, int64_t src_ld,
                                const int64_t* rows, int n, const int32_t* count, int width,
                                cudaStream_t stream);
cudaError_t launch_row_norm_max(const float* a, const float* b, int64_t n, int dim_pad, float* out,
                                cudaStream_t stream);

// tensor-core path (tc_topk.cu)
struct TcParams {
  int mode;  // B200KNN_MODE_BF16 / TF32X3
  const void* q_hi;
  const void* q_lo;
  const void* bank_hi;
  const void* bank_lo;
  int64_t B, N;
  int D, k;
  int64_t idx_offset;
  int64_t n_qtiles, n_items, split_rows;
  int n_chunks = 1, slots = 1;  // chunk-major order (plan.h): bank chunks per tile, open tiles per worker
  int64_t chunk_rows = 0;
  float* st_tau = nullptr;      // (B,) parked thresholds / list fills between the chunks of a tile
  uint32_t* st_cnt = nullptr;
  uint64_t* lists;
  uint64_t* out;  // (splits, B, k)
  int64_t bank_row_stride = 1;  // visit every bank_row_stride-th prepared row (sampling pre-pass)
  const float* tau0 = nullptr;  // optional (B,) initial admission thresholds
  // fused exchange: scatter each query row's keys into its owner GPU's buffer (peer memory)
  uint64_t* peer_out[8] = {nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
  int n_peers = 0, my_rank = 0;
  int64_t rows_per_owner = 0;
  bool sample = false;  // sampling pre-pass: k == 16 best SIMILARITIES per row (keys carry index 0)
  // optional group exclusion, as ExactParams (no tau0, sample, debug output or peers with it)
  const int32_t* q_gid = nullptr;
  const int32_t* bank_gid = nullptr;
};
// returns cudaErrorNotSupported if (D, k) is outside what the kernel handles
// `dump` (optional, (B,N) fp32) receives the raw similarity tiles (unit tests only);
// `diag` (optional, int32[4]) records which pipeline wait timed out before a trap.
cudaError_t launch_tc(const TcParams& p, int grid, int cap, cudaStream_t stream, float* dump,
                      int32_t* diag, int flags, const char** why);
int tc_tile_n(int mode, int dim);
bool tc_use_pair(int mode, int64_t B);  // resident-query modes run as CTA pairs (256-row query tiles) when B > 128

}  // namespace b200knn
