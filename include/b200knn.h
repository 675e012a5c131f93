/*
 * b200knn.h — C ABI of libb200knn.so: the B200 (sm_100a) kNN hot path.
 *
 * This is the drop-in boundary for the one hot path of
 * faris-k/self-supervised-wafermaps:  lightly's
 *     knn_predict(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t)
 * bound at   src/ssl_wafermap/models/knn.py:16   and called at
 *            src/ssl_wafermap/models/knn.py:91-98 and :205-212,
 * plus the brute-force neighbour retrieval of
 *            notebooks/2.0-Figures-nearest-neighbors.ipynb:54.
 * The reference is pure Python over ATen ops (mm -> topk -> gather -> exp ->
 * scatter -> sum -> argsort); there is no FFI in the reference, so these entry
 * points are what a ctypes binding for that path binds (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name says `host_`;
 *   - the caller owns every buffer, including workspaces (the library never
 *     allocates or frees device memory);
 *   - all work is enqueued on `stream` (a cudaStream_t passed as void*), no
 *     implicit synchronisation, no default-stream use;
 *   - return code 0 = ok; otherwise a negative B200KNN_E_* code and
 *     b200knn_last_error() returns a thread-local message;
 *   - no C++ exception crosses this boundary; the library never calls
 *     exit/abort.
 */
#ifndef B200KNN_H_
#define B200KNN_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define B200KNN_VERSION 150 /* 0.1.5: the b200knn_topk_* variants become options of b200knn_topk_opt; plan_info folds into
                              b200knn_plan_info_ex; 0.1.4.2: + the peer-memory threshold exchange, b200knn_broadcast_f32;
                              0.1.4.1: + b200knn_plan_info_ex; 0.1.4: + peeling (k > 992), b200knn_route_scatter,
                              b200knn_rescore_scatter, b200knn_compact_rows, b200knn_scatter_rows (sync-free sharded fp32 mode);
                              0.1.3: + B200KNN_MODE_F16; 0.1.2: + b200knn_route_keys, b200knn_certify (sharded fp32 mode);
                              0.1.1: b200knn_rescore workspace */

/* error codes */
#define B200KNN_OK 0
#define B200KNN_E_ARG (-1)       /* bad argument (shape, k > N, alignment ...) */
#define B200KNN_E_CUDA (-2)      /* a CUDA runtime/driver call failed */
#define B200KNN_E_WORKSPACE (-3) /* workspace too small */
#define B200KNN_E_UNSUPPORTED (-4)

/* element types of caller tensors */
#define B200KNN_F32 0
#define B200KNN_F16 1
#define B200KNN_BF16 2

/* layouts of a 2-D (rows = vectors) operand as the caller holds it */
#define B200KNN_LAYOUT_DN 0 /* (D,N) contiguous, vectors are COLUMNS: knn.py:80 `.t().contiguous()` */
#define B200KNN_LAYOUT_ND 1 /* (N,D) contiguous, vectors are rows: queries, notebook banks */

/* similarity-contraction modes */
#define B200KNN_MODE_EXACT 0 /* CUDA-core fp32, sim = sequential fmaf over d (the on-device golden) */
#define B200KNN_MODE_BF16 1  /* tcgen05 kind::f16, bf16 operands, fp32 TMEM accumulate */
#define B200KNN_MODE_TF32X3 2 /* tcgen05 kind::tf32, hi/lo split operands, 3 MMAs per k-step */
#define B200KNN_MODE_F32ROWS 3 /* b200knn_prepare_rows only: plain fp32 (n_vec, dim_pad) row-major copy */
#define B200KNN_MODE_BF16X3 4 /* tcgen05 kind::f16, bf16 hi/lo split operands, 3 MMAs per k-step:
                                 ~2^-16 relative operand error at twice the TF32X3 MMA rate */
#define B200KNN_MODE_F16X2 5 /* tcgen05 kind::f16, fp16 queries (one array) x fp16 hi/lo split bank, 2 MMAs per
                               k-step: one-sided operand error 2^-11 ||q|| ||x|| (+ 2^-25 per element below the
                               fp16 normal range); values beyond +-65504 saturate.  Candidate generator of the
                               "fp32" cascade (b200knn_rescore certifies with err_abs / max_abs). */
#define B200KNN_MODE_F16 6 /* tcgen05 kind::f16, fp16 queries x fp16 bank (one array each, the BF16 kernel on fp16
                             data): two-sided operand error 2^-10 ||q|| ||x||, 8x tighter than BF16 at the same speed;
                             same range rules as F16X2.  First level of the "fp32" cascade. */

int b200knn_version(void);
const char* b200knn_last_error(void);

/*
 * Operand preparation (replaces nothing in the reference; it is the cached,
 * one-off relayout of the bank that knn.py:80 produces and of the queries of
 * knn.py:90).  Converts `src` (element type src_dtype, layout src_layout,
 * n_vec vectors of dimension dim, leading dimension ld in ELEMENTS) into the
 * K-major row layout the tensor-core kernels stream with TMA:
 *   mode BF16  : dst_hi = (n_vec, dim) bf16 (round-to-nearest-even); dst_lo unused
 *   mode TF32X3: dst_hi = (n_vec, dim) f32 holding x rounded to tf32 (10 mantissa bits), to nearest
 *                with ties away from zero (cvt.rna),
 *                dst_lo = (n_vec, dim) f32 holding  x - hi  (exact)
 *   mode BF16X3: dst_hi = (n_vec, dim) bf16 = rn(x), dst_lo = (n_vec, dim) bf16 = rn(x - hi)
 *   mode F16 / F16X2: dst_hi = (n_vec, dim) fp16 = rn(sat(x)), sat clamping to +-65504; dst_lo
 *                (optional) = rn(sat(x - hi))
 *   mode F32ROWS: dst_hi = (n_vec, dim) f32 = x
 * rn = round to nearest, ties to even; dim is padded to a multiple of 64 with +0 columns.
 */
int b200knn_prepare_rows(const void* src, int src_dtype, int src_layout,
                         int64_t n_vec, int dim, int64_t ld, int mode,
                         void* dst_hi, void* dst_lo, void* stream);

/*
 * Fused similarity + streaming top-k   (replaces torch.mm + Tensor.topk,
 * a1.1/a1.2 of SURVEY.md §8; lightly knn_predict lines 1-2).
 *
 *   mode EXACT : q = (B,dim) caller tensor (q_dtype, row-major, ld = q_ld);
 *                bank = caller tensor (bank_dtype, bank_layout, ld = bank_ld)
 *   mode BF16 / TF32X3 / BF16X3 : q_hi/q_lo and bank_hi/bank_lo are b200knn_prepare_rows
 *                outputs (K-major rows); q_dtype/bank_dtype/layout args ignored.
 *
 * Output: out_keys = (B, k) uint64 selection keys sorted
 * descending under the canonical total order (sim desc, index asc):
 *     key = orderable_u32(sim) << 32 | (0xFFFFFFFF - (idx + idx_offset))
 * Decode with b200knn_decode_keys.  `idx_offset` is added to every bank row
 * index (bank row-sharding across GPUs).
 * workspace: at least b200knn_topk_workspace_bytes(...) bytes, 256-byte aligned.
 */
size_t b200knn_topk_workspace_bytes(int64_t B, int64_t N, int dim, int k, int mode);

int b200knn_topk(int mode,
                 const void* q_hi, const void* q_lo, int q_dtype, int64_t q_ld,
                 const void* bank_hi, const void* bank_lo, int bank_dtype,
                 int bank_layout, int64_t bank_ld,
                 int64_t B, int64_t N, int dim, int k, int64_t idx_offset,
                 uint64_t* out_keys,
                 void* workspace, size_t workspace_bytes, void* stream);

/*
 * b200knn_topk with options (no counterpart in the reference).  opts == NULL, or an all-zero
 * struct, is exactly b200knn_topk.  The options:
 *   bank_row_stride : 0 or 1 visit every bank row; s > 1 visits prepared rows 0, s, 2s, ...
 *                     (N of them, the "n_visit" of a sample); indices are the VISIT index
 *                     (+ idx_offset).  Tensor-core modes.
 *   tau0            : (B,) initial admission thresholds: only rows with sim > tau0[b] are
 *                     considered, so fewer than k may be found (the remaining key slots are 0).
 *                     A threshold taken from the r-th best similarity of a strided sample is
 *                     below the true k-th similarity except with negligible probability; the
 *                     host shim detects the exception (empty k-th slot) and recomputes that row
 *                     without tau0.  Tensor-core modes.
 *   upper_keys      : (B,) peeling bound: only keys strictly below upper_keys[b] (the last key of
 *                     row b from the previous pass).  Tensor.topk accepts any k <= N and the
 *                     streaming lists hold at most 992 keys, so larger k is served in passes of
 *                     <= 992 ("peeling").  MODE_EXACT.
 *   q_groups,       : (B,) and (N,) int32 group ids (bank ids indexed before idx_offset), both or
 *   bank_groups       neither: bank row n is never admitted to query row b's list when
 *                     bank_groups[n] == q_groups[b] (k-fold cross-validation, held-out queries whose
 *                     group also has rows in the bank).  Order, key format and indices are
 *                     unchanged; a row with fewer than k eligible bank rows gets empty (0) trailing
 *                     slots.  Every mode: alone in the tensor-core modes, with or without
 *                     upper_keys in MODE_EXACT.
 *   sample          : non-zero = the sampling pre-pass: for every query, the B200KNN_SAMPLE_R = 16
 *                     best 32-column CHUNK MAXIMA of its similarities with the visited rows, as
 *                     (B,16) keys sorted descending whose index field is 0 (values only: each
 *                     row's running top-16 lives in registers, no candidate lists).  Every value
 *                     is a sampled similarity and the 16-th is <= the 16-th best sampled
 *                     similarity, so it is a valid seed for tau0.  Needs k == 16 and N >= 16.
 *                     Tensor-core modes.
 *   host_peer_out,  : fused exchange for the bank-row-sharded mode: result rows are not returned
 *   n_peers,          locally (out_keys must be NULL) but stored, as each query tile finishes,
 *   my_rank,          straight into the exchange buffer of the GPU that owns that query (peer
 *   rows_per_owner    memory over NVLink, so the all-to-all overlaps the remaining tiles' math).
 *                     host_peer_out is a HOST array of n_peers (1..8) DEVICE pointers, each mapped
 *                     in this process; peer g's buffer is (n_peers, rows_per_owner, k) uint64.
 *                     Query row b's owner is b / rows_per_owner (rows_per_owner * n_peers >= B),
 *                     and its keys go to peer_out[owner][my_rank][b - owner*rows_per_owner][0..k).
 *                     After a cross-GPU barrier every GPU holds, for its own query rows, all
 *                     shards' sorted lists in b200knn_merge's input layout.  Only problems planned
 *                     without bank splits (b200knn_plan_info_ex splits == 1) are supported; others
 *                     return B200KNN_E_UNSUPPORTED.  Tensor-core modes, with tau0 at stride 1 or
 *                     with sample at any stride.
 * Combinations (anything else returns B200KNN_E_ARG, checked before any work is planned):
 *   MODE_EXACT        : upper_keys, groups, or both;
 *   tensor-core modes : bank_row_stride with tau0; sample with bank_row_stride, optionally with
 *                       the peer exchange; tau0 with the peer exchange at stride 1; groups alone.
 * Workspace: b200knn_topk_workspace_bytes(B, N, dim, k, mode) bytes, N the rows visited.
 */
#define B200KNN_SAMPLE_R 16
typedef struct b200knn_topk_options {
  int64_t bank_row_stride;          /* 0 or 1: every row; s > 1: rows 0, s, 2s, ... (tensor-core modes) */
  const float* tau0;                /* (B,) admission thresholds (tensor-core modes) */
  const uint64_t* upper_keys;       /* (B,) peeling bound: only keys strictly below (MODE_EXACT) */
  const int32_t* q_groups;          /* (B,) and (N,) group ids: both or neither */
  const int32_t* bank_groups;
  int sample;                       /* values-only B200KNN_SAMPLE_R best (tensor-core modes) */
  const void* const* host_peer_out; /* fused exchange: n_peers device pointers (HOST array) */
  int n_peers, my_rank;
  int64_t rows_per_owner;
} b200knn_topk_options;

int b200knn_topk_opt(int mode,
                     const void* q_hi, const void* q_lo, int q_dtype, int64_t q_ld,
                     const void* bank_hi, const void* bank_lo, int bank_dtype,
                     int bank_layout, int64_t bank_ld,
                     int64_t B, int64_t N, int dim, int k, int64_t idx_offset,
                     uint64_t* out_keys, void* workspace, size_t workspace_bytes,
                     const b200knn_topk_options* opts, void* stream);

/*
 * Merge G sorted candidate lists per query into one (replaces nothing in the
 * reference; it is the exchange step of the bank-row-sharded mode, applied to
 * the buffer an all-gather of per-shard b200knn_topk outputs produces).
 *   keys_in : (G, B, k_in) uint64, each (g,b,:) a zero-terminated set: its non-empty keys first,
 *             in any order (sorted descending is one such order), then only empty (0) keys.  The
 *             first empty key ends a list; keys may repeat within and across lists.
 *   keys_out: (B, k_out) uint64 sorted descending, the best k_out keys of the union (repeats
 *             counted), zero-filled, k_out <= G*k_in
 */
int b200knn_merge(const uint64_t* keys_in, int G, int64_t B, int k_in, int k_out,
                  uint64_t* keys_out, void* stream);

/*
 * Leave-one-out lists (no counterpart in the reference): row b of a search of bank rows
 * [self_offset, self_offset + B) against the whole bank, without the row itself.
 *   keys_in : (B, k_in) uint64, each row sorted descending, k_in >= 2
 *   keys_out: (B, k_in - 1) uint64, must not overlap keys_in: row b without the key whose bank
 *             index (the key's index field, idx_offset included) is b + self_offset, or without
 *             its last key when no key has that index.  Empty (0) keys are copied and never match.
 */
int b200knn_drop_self(const uint64_t* keys_in, int64_t B, int k_in, int64_t self_offset,
                      uint64_t* keys_out, void* stream);

/*
 * Leave-one-group-out lists (no counterpart in the reference; replaces one bank preparation and
 * search per group): row b of a search of bank row row_ids[b] against the whole bank, without
 * every row of that row's group.
 *   keys_in  : (B, k_in) uint64, each row sorted descending, k_in >= k_out
 *   row_ids  : (B,) int64, the bank row each list belongs to
 *   group_ids: (N,) int32, the group of every bank row (the key's index field, idx_offset included)
 *   keys_out : (B, k_out) uint64, must not overlap keys_in: the first k_out keys of row b whose
 *              group_ids entry differs from group_ids[row_ids[b]], in order; zero-filled when fewer
 *              survive.  Empty (0) keys are never dropped.
 *   err_flag : int32[1], set to 2 when a key index or row id is outside [0, N); such a key is
 *              kept, and a row id outside [0, N) drops nothing.  Keys after the k_out-th survivor
 *              may be left unread (and unchecked).
 * k_out >= 1; B == 0 launches nothing.
 */
int b200knn_drop_group(const uint64_t* keys_in, int64_t B, int k_in, const int64_t* row_ids,
                       const int32_t* group_ids, int64_t N, int k_out, uint64_t* keys_out,
                       int32_t* err_flag, void* stream);

/* keys (B,k) -> sims (B,k) f32 and idx (B,k) int64  (Tensor.topk's two outputs).
 * Empty slots (fewer than k finite candidates) decode to sim=-inf, idx=-1. */
int b200knn_decode_keys(const uint64_t* keys, int64_t n_keys, float* sims,
                        int64_t* idx, void* stream);

/*
 * Weighted class vote + ranking  (replaces gather / div+exp / zeros+scatter /
 * mul+sum / argsort, a1.3-a1.7 of SURVEY.md §8; lightly knn_predict lines 3-7).
 *   keys   : (B,k) selection keys (sorted descending)
 *   labels : (N,) int64 class ids of the bank rows, indexed by (idx - label_offset)
 *   pred   : (B,C) int64 classes ordered by (score desc, class asc)
 *   scores : optional (B,C) f64 class scores (may be NULL)
 *   err_flag: device int32, set to 1 if any label is outside [0,C) — the
 *             reference raises from scatter in that case (the host shim checks)
 * Scores are sum_j exp(double(sim_j) / double(t)) accumulated in rank order.
 * Any k (keys are read in chunks of 1024); C <= (51200 - 8*ceil(12*min(k, 1024) / 8)) / 8, i.e.
 * 4864 for k >= 1024, 6100 at k = 200; a larger C returns B200KNN_E_UNSUPPORTED.
 */
int b200knn_vote(const uint64_t* keys, const int64_t* labels, int64_t B, int k,
                 int64_t n_labels, int64_t label_offset, int C, double t,
                 int64_t* pred, double* scores, int32_t* err_flag, void* stream);

/*
 * b200knn_vote writing into a wider row-major buffer: pred has row stride pred_ld >= C, and
 * when status_col >= C a per-row status word is stored in that column: bit 0 = the row's
 * k-th key slot is empty (a tau0 threshold of b200knn_topk_opt starved it), bit 1 = a label outside
 * [0,C), bit 2 = a neighbour index outside the labels.  The sharded driver all-gathers this
 * (B_owned, C+1) buffer as it is.
 */
int b200knn_vote_ex(const uint64_t* keys, const int64_t* labels, int64_t B, int k,
                    int64_t n_labels, int64_t label_offset, int C, double t,
                    int64_t* pred, int64_t pred_ld, int status_col, double* scores,
                    int32_t* err_flag, void* stream);

/*
 * b200knn_vote_ex for a grid of settings from one neighbour list per row: keys (B, k_max) and
 * ks[0] < ks[1] < ... < ks[n_k-1] == k_max (1 <= n_k <= 16), ts[0..n_t) non-zero (1 <= n_t <= 8).
 * pred has row stride pred_ld >= n_k*n_t*C; columns [(i*n_t + j)*C, (i*n_t + j + 1)*C) of a row
 * hold exactly what b200knn_vote writes for that row's first ks[i] keys at t = ts[j].
 * status_col: -1, or a column >= n_k*n_t*C for b200knn_vote_ex's status word (bit 0: the
 * k_max-th slot is empty).  Any k_max; C <= (51200 - 16*min(k_max, 1024)) / 8, i.e. 4352 for
 * k_max >= 1024, 6000 at k_max = 200; a larger C returns B200KNN_E_UNSUPPORTED.
 */
int b200knn_vote_multi(const uint64_t* keys, const int64_t* labels, int64_t B, int k_max,
                       int64_t n_labels, int64_t label_offset, int C, const int* ks, int n_k,
                       const double* ts, int n_t, int64_t* pred, int64_t pred_ld, int status_col,
                       int32_t* err_flag, void* stream);

/* out[b] = similarity of keys[b, j] (-inf for an empty slot): the threshold a (B,r) sample
 * hands to b200knn_topk_opt as tau0 (j = r-1). */
int b200knn_key_sim_column(const uint64_t* keys, int64_t B, int k, int j, float* out,
                           void* stream);

/*
 * Exact re-scoring of tensor-core candidates (the "fp32" mode; no counterpart in
 * the reference — it is what makes the tensor-core contraction reproduce the
 * fp32 torch.mm + topk of lightly's knn_predict bit for bit).
 *   q        : caller queries (B, dim), q_dtype, row-major, ld = q_ld
 *   rows_a/b : (N, dim_pad) fp32 bank rows from b200knn_prepare_rows (F32ROWS: rows_b
 *              NULL; TF32X3: value = hi + lo, exact)
 *   cand_keys: (B, k_in) keys from b200knn_topk (approximate sims), k_in <= 1024
 *   out_keys : (B, k_out) keys with EXACT sims = fmaf chain over d (MODE_EXACT's
 *              definition), canonical order
 *   uncertified[b] = 1 when  exact_sim(rank k_out) <= approx_sim(rank k_in) + E,
 *              E = err_coef * ||q_b|| * M + err_abs * (||q_b|| + M),  M = *bank_max_norm
 *              — the candidate set is then not proven to contain the true top-k and the
 *              caller must recompute row b in MODE_EXACT; *n_uncertified counts such rows
 *              (caller zeroes it).  max_abs > 0 additionally refuses rows with ||q_b|| or M
 *              >= max_abs (operand range of a half-precision candidate pass).  A row whose
 *              k_in-th candidate slot is empty although k_in < N (a b200knn_topk_opt tau0
 *              threshold starved it) is uncertified as well.
 *   workspace: optional, b200knn_rescore_workspace_bytes(B, k_in) bytes of device memory.
 *              With it (and fp32 queries, rows_b NULL) the rows are gathered by a persistent
 *              TMA-pipelined kernel (cp.async.bulk per candidate row) and ranked by a second
 *              one; without it a single block-per-query kernel does both.  Same results.
 * b200knn_row_norm_max writes max_n ||row_n|| (x1.001) to *out_dev.
 */
int b200knn_row_norm_max(const float* rows_a, const float* rows_b, int64_t n,
                         int dim_pad, float* out_dev, void* stream);
int b200knn_rescore(const void* q, int q_dtype, int64_t q_ld, const float* rows_a,
                    const float* rows_b, int64_t N, int dim,
                    const uint64_t* cand_keys, int64_t B, int k_in, int k_out,
                    int64_t idx_offset, float err_coef, float err_abs, float max_abs,
                    const float* bank_max_norm, uint64_t* out_keys, int32_t* uncertified,
                    int32_t* n_uncertified, void* workspace, size_t workspace_bytes,
                    void* stream);
size_t b200knn_rescore_workspace_bytes(int64_t B, int k_in);

/*
 * Sharded fp32 mode (no counterpart in the reference, which is single-device): the owner of a
 * query merges every shard's approximate candidates, has each candidate re-scored by the shard
 * that holds its bank row, merges the exact keys that come back and certifies the result.
 * b200knn_route_keys: out (n_shards, n, k): out[g][r][:] = the keys of row r whose bank row lies in
 *   [g*rows_per_shard, (g+1)*rows_per_shard), in their original order, compacted to the front and
 *   zero-padded — the send buffer of that exchange.  The shards re-score what they receive with
 *   b200knn_rescore (k_out = k_in).  Candidate lists are filled from the FRONT (empty slots only behind the last
 *   candidate): the first empty 32-slot unit of a query ends it.
 * b200knn_certify: the certificate of b200knn_rescore on its own: exact_keys (B,k) merged exact
 *   keys, approx_keys (B,k_in) merged approximate candidates (both sorted descending);
 *   all_rows != 0 when k_in covers the whole bank.
 */
int b200knn_route_keys(const uint64_t* keys, int64_t n, int k, int64_t rows_per_shard, int n_shards,
                       uint64_t* out, void* stream);
int b200knn_certify(const void* q, int q_dtype, int64_t q_ld, int dim, const uint64_t* exact_keys, int k,
                    const uint64_t* approx_keys, int k_in, int64_t B, int all_rows, float err_coef,
                    float err_abs, float max_abs, const float* bank_max_norm, int32_t* uncertified,
                    int32_t* n_uncertified, void* stream);

/*
 * The same exchange without NCCL round trips or host synchronisation (peer memory over NVLink):
 * b200knn_route_scatter: b200knn_route_keys fused with its all-to-all — the candidates of owned query
 *   row r that shard g can re-score are stored, compacted, into row (row_offset + r) of shard g's
 *   inbox host_inbox[g] (a (Q_pad, k) buffer of every rank, mapped here; the receivers zero their
 *   inboxes before the barrier that precedes the call).  n_shards <= 8.
 * b200knn_rescore_scatter: b200knn_rescore (fp32 queries, one fp32 row array, k_out = k_in, no
 *   certificate) whose sorted exact keys of query row b go straight into the exchange buffer of
 *   the GPU that owns b: host_peer_out[b / rows_per_owner] + ((my_rank * rows_per_owner +
 *   b % rows_per_owner) * k_in); only non-empty slots are written (receivers zero their buffers).
 * b200knn_compact_rows: rows_out[0..min(count,cap)) = ascending row numbers i with
 *   (status[i*ld] & mask) != 0, the rest of rows_out = 0, *count_out = their number (may exceed
 *   cap): the rows a cascade level could not certify, chosen on the device so that the next level
 *   runs on a fixed-capacity sub-batch without a host read.
 * b200knn_scatter_rows: dst[rows[i]*dst_ld + c] = src[i*src_ld + c], c < width, i < min(n, *count).
 */
/* The sharded threshold exchange over peer memory: a sample (b200knn_topk_opt) with the peer exchange stores the
 * 16 values of query row b into the buffer of the GPU that owns b, and b200knn_broadcast_f32:
 * dst[g][dst_offset + i] = src[i] for every peer g (the owner publishes its thresholds). */
int b200knn_broadcast_f32(const float* src, int64_t n, const void* const* host_peer_dst, int n_peers,
                          int64_t dst_offset, void* stream);
int b200knn_route_scatter(const uint64_t* keys, int64_t n, int k, int64_t rows_per_shard, int n_shards,
                          const void* const* host_inbox, int64_t row_offset, void* stream);
int b200knn_rescore_scatter(const float* q, int64_t q_ld, const float* rows, int64_t N, int dim,
                            const uint64_t* cand_keys, int64_t B, int k_in, int64_t idx_offset,
                            const void* const* host_peer_out, int n_peers, int my_rank,
                            int64_t rows_per_owner, void* workspace, size_t workspace_bytes, void* stream);
int b200knn_compact_rows(const int64_t* status, int64_t ld, int64_t n, int64_t mask, int64_t* rows_out,
                         int cap, int32_t* count_out, void* stream);
int b200knn_scatter_rows(int64_t* dst, int64_t dst_ld, const int64_t* src, int64_t src_ld,
                         const int64_t* rows, int n, const int32_t* count, int width, void* stream);

/*
 * SURVEY.md §8(f) rows — the steps either side of knn_predict in the reference.
 *
 * b200knn_normalize_rows: F.normalize(x, dim=1) of n_vec row vectors (reference
 * src/ssl_wafermap/models/knn.py:77 bank rows, :90 queries) fused with the relayout into the
 * padded (n_vec, dim_pad) fp32 rows the kernels read; y = x / max(||x||_2, eps).  The norm is
 * accumulated in fp64 in a fixed order (see csrc/prepare.cu), so the result is reproducible.
 *
 * b200knn_confusion: counts[t*C + p] += #(target == t, pred == p) — the confusion matrix of
 * src/ssl_wafermap/models/knn.py:121-127; macro accuracy / F1 follow from it.  err_flag is
 * set to 1 if a prediction or target lies outside [0, C).
 */
int b200knn_normalize_rows(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld,
                           float eps, float* dst_rows, void* stream);
/* out[n] = float(sum_d x[n,d]^2) with the accumulation order of b200knn_normalize_rows: the
 * ||x||^2 column that turns a dot-product top-k into the L2 ranking of
 * notebooks/2.0-Figures-nearest-neighbors.ipynb:54 (argmin ||x-q|| = argmax 2 q.x - ||x||^2). */
int b200knn_row_sqnorms(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld,
                        float* out, void* stream);
int b200knn_confusion(const int64_t* pred, const int64_t* target, int64_t n, int C,
                      int64_t* counts, int32_t* err_flag, void* stream);

/* Device capability probe for the host shim: 1 if the current device is sm_100. */
int b200knn_device_ok(void);

/* How b200knn_topk decomposes a call (for the bench and the docs), HOST pointer:
 * out9 = {n_qtiles, splits, split_rows, n_items, grid, list_capacity, chunks, chunk_rows, slots}
 * (a tensor-core worker keeps `slots` query tiles open and scans the bank in `chunks` L2-sized pieces). */
int b200knn_plan_info_ex(int mode, int64_t B, int64_t N, int dim, int k, int64_t* host_out9);
/* Tuning knob: bytes of bank one chunk of the chunk-major order may occupy (default 40 MiB, or
 * $B200KNN_L2_CHUNK_MB; 0 = never chunk).  Process-wide; affects planning only, never results. */
int b200knn_set_l2_chunk_bytes(int64_t bytes);

/* TEST HOOK, not a product entry point: b200knn_topk for the tensor-core modes
 * that also dumps the raw (B,N) fp32 similarity tiles it selected from, and a
 * pipeline diagnostic word diag[4] written if a barrier wait times out.
 * flags (experiments; results are then meaningless): 1 no selection, 2 no TMEM
 * loads, 4 no MMA issue, 8 no bank TMA loads. */
int b200knn_debug_topk_dump(int mode, const void* q_hi, const void* q_lo,
                            const void* bank_hi, const void* bank_lo, int64_t B,
                            int64_t N, int dim, int k, uint64_t* out_keys,
                            void* workspace, size_t workspace_bytes, float* dump,
                            int32_t* diag, int flags, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* B200KNN_H_ */
