// api.cu — the extern "C" boundary declared in include/b200knn.h.
// Argument validation, work planning, workspace carving, kernel dispatch.
// No device allocation, no implicit synchronisation, no exceptions.
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>

#include "../../include/b200knn.h"
#include "common.cuh"
#include "kernels.h"
#include "plan.h"

namespace {

thread_local char g_err[512] = "";

int fail(int code, const char* fmt, const char* a = "", const char* b = "") {
  std::snprintf(g_err, sizeof(g_err), fmt, a, b);
  return code;
}
int fail_cuda(const char* where, cudaError_t e) {
  std::snprintf(g_err, sizeof(g_err), "%s: %s", where, cudaGetErrorString(e));
  return B200KNN_E_CUDA;
}

int sm_count() {
  int dev = 0, n = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess) return 0;
  return n;
}

bool is_tc_mode(int mode) {
  return mode == B200KNN_MODE_BF16 || mode == B200KNN_MODE_TF32X3 || mode == B200KNN_MODE_BF16X3 ||
         mode == B200KNN_MODE_F16X2 || mode == B200KNN_MODE_F16;
}

// Bytes of bank the chunk-major order keeps L2-resident per chunk phase (plan.h).  B200: 126 MB of
// L2 in two halves; 40 MB leaves room for the query tiles and the list traffic.  B200KNN_L2_CHUNK_MB=0
// switches chunking off (A/B experiments).
int64_t g_l2_chunk_bytes = -1;
int64_t l2_chunk_bytes() {
  if (g_l2_chunk_bytes < 0) {
    const char* e = getenv("B200KNN_L2_CHUNK_MB");
    g_l2_chunk_bytes = (e != nullptr ? atoll(e) : 40) << 20;
  }
  return g_l2_chunk_bytes;
}

bool plan_for(int mode, int64_t B, int64_t N, int dim, int k, b200knn::TopkPlan* plan) {
  const int cap = b200knn::list_capacity(k);
  if (cap == 0) return false;
  int sms = sm_count();
  if (sms <= 0) sms = 148;
  if (mode == B200KNN_MODE_EXACT) {
    *plan = b200knn::make_plan(B, N, k, cap, 128, 128, sms * 2);
  } else {
    // a worker of the tensor-core kernel is one CTA, or a CTA pair owning 256 query rows
    const int pair = b200knn::tc_use_pair(mode, B) ? 2 : 1;
    const int64_t d_pad = (dim + 63) / 64 * 64;
    const int64_t row_bytes = d_pad * (mode == B200KNN_MODE_TF32X3 ? 8 : (mode == B200KNN_MODE_BF16 || mode == B200KNN_MODE_F16) ? 2 : 4);
    *plan = b200knn::make_plan(B, N, k, cap, 128 * pair, b200knn::tc_tile_n(mode, dim), sms / pair, row_bytes,
                               l2_chunk_bytes());
  }
  return true;
}

// The operands and shape of one search, named as b200knn_topk_opt names them.
struct TopkOperands {
  const void* q_hi;
  const void* q_lo;
  int q_dtype;
  int64_t q_ld;
  const void* bank_hi;
  const void* bank_lo;
  int bank_dtype, bank_layout;
  int64_t bank_ld;
  uint64_t* out_keys;
  void* workspace;
  size_t workspace_bytes;
  void* stream;
};
struct TopkShape {
  int64_t B, N;
  int dim, k;
  int64_t idx_offset;
};

// Which options of b200knn_topk_opt go together (the table in include/b200knn.h).  Runs before
// any planning or launch, so every refusal here needs no GPU.
int check_options(int mode, const TopkShape& s, const uint64_t* out_keys, const b200knn_topk_options& o) {
  const bool groups = o.q_groups != nullptr || o.bank_groups != nullptr;
  const bool peers = o.n_peers != 0 || o.host_peer_out != nullptr;
  const bool strided = o.bank_row_stride > 1;
  if (groups && (o.q_groups == nullptr || o.bank_groups == nullptr))
    return fail(B200KNN_E_ARG, "topk: null group ids (q_groups and bank_groups go together)");
  if (o.bank_row_stride < 0) return fail(B200KNN_E_ARG, "topk: bank_row_stride must be >= 0");
  if (o.sample && (s.k != B200KNN_SAMPLE_R || s.N < B200KNN_SAMPLE_R))
    return fail(B200KNN_E_ARG, "topk: sample needs k == 16 and at least 16 rows to visit");
  if (peers) {
    if (o.host_peer_out == nullptr || o.n_peers < 1 || o.n_peers > 8 || o.my_rank < 0 || o.my_rank >= o.n_peers)
      return fail(B200KNN_E_ARG, "topk: 1..8 peers and a rank among them");
    if (o.rows_per_owner <= 0 || o.rows_per_owner * o.n_peers < s.B)
      return fail(B200KNN_E_ARG, "topk: rows_per_owner * n_peers must cover B");
    for (int g = 0; g < o.n_peers; ++g)
      if (o.host_peer_out[g] == nullptr) return fail(B200KNN_E_ARG, "topk: null peer buffer");
    if (out_keys != nullptr) return fail(B200KNN_E_ARG, "topk: the peer exchange stores the keys; out_keys must be NULL");
  }
  if (mode == B200KNN_MODE_EXACT) {
    if (strided || o.tau0 || o.sample || peers)
      return fail(B200KNN_E_ARG, "topk: MODE_EXACT takes no bank_row_stride, tau0, sample or peers");
    return B200KNN_OK;
  }
  if (o.upper_keys) return fail(B200KNN_E_ARG, "topk: upper_keys needs MODE_EXACT");
  if (groups && (strided || o.tau0 || o.sample || peers))
    return fail(B200KNN_E_ARG, "topk: group ids take no bank_row_stride, tau0, sample or peers");
  if (o.sample && o.tau0) return fail(B200KNN_E_ARG, "topk: sample takes no tau0");
  if (peers && !o.sample && strided)
    return fail(B200KNN_E_ARG, "topk: the peer exchange of a search visits every row (bank_row_stride 1)");
  return B200KNN_OK;
}

}  // namespace

extern "C" {

int b200knn_version(void) { return B200KNN_VERSION; }
const char* b200knn_last_error(void) { return g_err; }

int b200knn_device_ok(void) {
  int dev = 0, major = 0;
  if (cudaGetDevice(&dev) != cudaSuccess) return 0;
  if (cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev) != cudaSuccess) return 0;
  return major == 10 ? 1 : 0;
}

int b200knn_prepare_rows(const void* src, int src_dtype, int src_layout, int64_t n_vec, int dim,
                         int64_t ld, int mode, void* dst_hi, void* dst_lo, void* stream) {
  if (!src || !dst_hi || n_vec < 0 || dim <= 0) return fail(B200KNN_E_ARG, "prepare_rows: bad argument");
  if (src_dtype < B200KNN_F32 || src_dtype > B200KNN_BF16)
    return fail(B200KNN_E_ARG, "prepare_rows: unknown dtype");
  if (src_layout != B200KNN_LAYOUT_DN && src_layout != B200KNN_LAYOUT_ND)
    return fail(B200KNN_E_ARG, "prepare_rows: unknown layout");
  if (mode != B200KNN_MODE_BF16 && mode != B200KNN_MODE_TF32X3 && mode != B200KNN_MODE_F32ROWS &&
      mode != B200KNN_MODE_BF16X3 && mode != B200KNN_MODE_F16X2 && mode != B200KNN_MODE_F16)
    return fail(B200KNN_E_ARG, "prepare_rows: mode must be BF16, F16, TF32X3, BF16X3, F16X2 or F32ROWS");
  if ((mode == B200KNN_MODE_TF32X3 || mode == B200KNN_MODE_BF16X3) && !dst_lo)
    return fail(B200KNN_E_ARG, "prepare_rows: split modes need dst_lo");
  cudaError_t e = b200knn::launch_prepare(src, src_dtype, src_layout, n_vec, dim, ld, mode, dst_hi,
                                          dst_lo, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("prepare_rows", e);
}

size_t b200knn_topk_workspace_bytes(int64_t B, int64_t N, int dim, int k, int mode) {
  b200knn::TopkPlan plan;
  if (B <= 0 || N <= 0 || k <= 0 || !plan_for(mode, B, N, dim, k, &plan)) return 0;
  return plan.total_bytes + 256;
}

static int topk_impl(int mode, const TopkOperands& x, const TopkShape& s, const b200knn_topk_options& o,
                     float* dump, int32_t* diag, int flags) {
  const int64_t B = s.B, N = s.N;
  const int dim = s.dim, k = s.k;
  uint64_t* out_keys = x.out_keys;
  int rc = check_options(mode, s, out_keys, o);
  if (rc != B200KNN_OK) return rc;
  if (B < 0 || N <= 0 || dim <= 0) return fail(B200KNN_E_ARG, "topk: bad shape");
  if (k <= 0 || k > N) return fail(B200KNN_E_ARG, "topk: selected index k out of range");
  if (N + s.idx_offset >= 0xFFFFFFFFll || s.idx_offset < 0)
    return fail(B200KNN_E_ARG, "topk: bank index does not fit 32 bits");
  if (B == 0) return B200KNN_OK;
  if (!x.q_hi || !x.bank_hi || (!out_keys && o.n_peers == 0) || !x.workspace)
    return fail(B200KNN_E_ARG, "topk: null pointer");
  b200knn::TopkPlan plan;
  if (!plan_for(mode, B, N, dim, k, &plan)) return fail(B200KNN_E_UNSUPPORTED, "topk: k too large (max 992)");
  if (o.n_peers > 0 && plan.splits > 1)
    return fail(B200KNN_E_UNSUPPORTED, "topk: the peer exchange needs a problem planned without bank splits");
  uintptr_t ws = (reinterpret_cast<uintptr_t>(x.workspace) + 255) & ~uintptr_t(255);
  const size_t slack = ws - reinterpret_cast<uintptr_t>(x.workspace);
  if (x.workspace_bytes < plan.total_bytes + slack) return fail(B200KNN_E_WORKSPACE, "topk: workspace too small");
  uint64_t* lists = reinterpret_cast<uint64_t*>(ws);
  float* st_tau = plan.chunks > 1 ? reinterpret_cast<float*>(ws + plan.lists_bytes) : nullptr;
  uint32_t* st_cnt = plan.chunks > 1 ? reinterpret_cast<uint32_t*>(st_tau + B) : nullptr;
  uint64_t* partial =
      plan.splits > 1 ? reinterpret_cast<uint64_t*>(ws + plan.lists_bytes + plan.state_bytes) : out_keys;
  cudaStream_t st = static_cast<cudaStream_t>(x.stream);
  cudaError_t e;
  if (mode == B200KNN_MODE_EXACT) {
    if (x.q_dtype < 0 || x.q_dtype > 2 || x.bank_dtype < 0 || x.bank_dtype > 2)
      return fail(B200KNN_E_ARG, "topk: unknown dtype");
    b200knn::ExactParams p;
    p.q = x.q_hi;
    p.q_dtype = x.q_dtype;
    p.q_ld = x.q_ld;
    p.bank = x.bank_hi;
    p.bank_dtype = x.bank_dtype;
    if (x.bank_layout == B200KNN_LAYOUT_DN) {
      p.bank_sd = x.bank_ld;
      p.bank_sn = 1;
    } else if (x.bank_layout == B200KNN_LAYOUT_ND) {
      p.bank_sd = 1;
      p.bank_sn = x.bank_ld;
    } else {
      return fail(B200KNN_E_ARG, "topk: unknown bank layout");
    }
    p.B = B;
    p.N = N;
    p.D = dim;
    p.k = k;
    p.idx_offset = s.idx_offset;
    p.n_qtiles = plan.n_qtiles;
    p.n_items = plan.n_items;
    p.split_rows = plan.split_rows;
    p.lists = lists;
    p.out = partial;
    p.upper = o.upper_keys;
    p.q_gid = o.q_groups;
    p.bank_gid = o.bank_groups;
    e = b200knn::launch_exact(p, plan.grid, plan.cap, st);
    if (e != cudaSuccess) return fail_cuda("topk(exact)", e);
  } else if (is_tc_mode(mode)) {
    if (mode == B200KNN_MODE_F16X2 ? !x.bank_lo
                                   : (mode != B200KNN_MODE_BF16 && mode != B200KNN_MODE_F16 && (!x.q_lo || !x.bank_lo)))
      return fail(B200KNN_E_ARG, "topk: split modes need the lo operands");
    b200knn::TcParams p;
    p.mode = mode;
    p.q_hi = x.q_hi;
    p.q_lo = x.q_lo;
    p.bank_hi = x.bank_hi;
    p.bank_lo = x.bank_lo;
    p.B = B;
    p.N = N;
    p.D = dim;
    p.k = k;
    p.idx_offset = s.idx_offset;
    p.n_qtiles = plan.n_qtiles;
    p.n_items = plan.n_items;
    p.split_rows = plan.split_rows;
    p.n_chunks = plan.chunks;
    p.slots = plan.slots;
    p.chunk_rows = plan.chunk_rows;
    p.st_tau = st_tau;
    p.st_cnt = st_cnt;
    p.lists = lists;
    p.out = partial;
    p.bank_row_stride = o.bank_row_stride > 1 ? o.bank_row_stride : 1;
    p.tau0 = o.tau0;
    p.sample = o.sample != 0;
    p.n_peers = o.n_peers;
    p.my_rank = o.my_rank;
    p.rows_per_owner = o.rows_per_owner;
    for (int g = 0; g < o.n_peers; ++g)
      p.peer_out[g] = static_cast<uint64_t*>(const_cast<void*>(o.host_peer_out[g]));
    p.q_gid = o.q_groups;
    p.bank_gid = o.bank_groups;
    const char* why = "";
    e = b200knn::launch_tc(p, plan.grid, plan.cap, st, dump, diag, flags, &why);
    if (e == cudaErrorNotSupported) return fail(B200KNN_E_UNSUPPORTED, "topk(tc): %s", why);
    if (e != cudaSuccess) {
      std::snprintf(g_err, sizeof(g_err), "topk(tc): %s %s", cudaGetErrorString(e), why);
      return B200KNN_E_CUDA;
    }
  } else {
    return fail(B200KNN_E_ARG, "topk: unknown mode");
  }
  if (plan.splits > 1) {
    e = b200knn::launch_merge(partial, plan.splits, B, k, k, out_keys, st);
    if (e != cudaSuccess) return fail_cuda("topk(merge)", e);
  }
  return B200KNN_OK;
}

int b200knn_topk_opt(int mode, const void* q_hi, const void* q_lo, int q_dtype, int64_t q_ld,
                     const void* bank_hi, const void* bank_lo, int bank_dtype, int bank_layout,
                     int64_t bank_ld, int64_t B, int64_t N, int dim, int k, int64_t idx_offset,
                     uint64_t* out_keys, void* workspace, size_t workspace_bytes,
                     const b200knn_topk_options* opts, void* stream) {
  const b200knn_topk_options none = {};
  return topk_impl(mode,
                   {q_hi, q_lo, q_dtype, q_ld, bank_hi, bank_lo, bank_dtype, bank_layout, bank_ld, out_keys,
                    workspace, workspace_bytes, stream},
                   {B, N, dim, k, idx_offset}, opts ? *opts : none, nullptr, nullptr, 0);
}

int b200knn_topk(int mode, const void* q_hi, const void* q_lo, int q_dtype, int64_t q_ld,
                 const void* bank_hi, const void* bank_lo, int bank_dtype, int bank_layout,
                 int64_t bank_ld, int64_t B, int64_t N, int dim, int k, int64_t idx_offset,
                 uint64_t* out_keys, void* workspace, size_t workspace_bytes, void* stream) {
  return b200knn_topk_opt(mode, q_hi, q_lo, q_dtype, q_ld, bank_hi, bank_lo, bank_dtype, bank_layout, bank_ld, B,
                          N, dim, k, idx_offset, out_keys, workspace, workspace_bytes, nullptr, stream);
}

int b200knn_broadcast_f32(const float* src, int64_t n, const void* const* host_peer_dst, int n_peers,
                          int64_t dst_offset, void* stream) {
  if (!src || !host_peer_dst || n < 0 || n_peers < 1 || n_peers > 8 || dst_offset < 0)
    return fail(B200KNN_E_ARG, "broadcast_f32: bad argument (1..8 peers)");
  float* dst[8];
  for (int g = 0; g < n_peers; ++g) {
    if (!host_peer_dst[g]) return fail(B200KNN_E_ARG, "broadcast_f32: null peer buffer");
    dst[g] = static_cast<float*>(const_cast<void*>(host_peer_dst[g]));
  }
  cudaError_t e = b200knn::launch_broadcast_f32(src, n, dst, n_peers, dst_offset, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("broadcast_f32", e);
}

// Test hook (not part of the product path): same as b200knn_topk for the tensor-core
// modes, additionally dumping the raw (B,N) fp32 similarity tiles and the pipeline
// diagnostic word.  Used by tests/ to validate the MMA path against a plain GEMM.
int b200knn_debug_topk_dump(int mode, const void* q_hi, const void* q_lo, const void* bank_hi,
                            const void* bank_lo, int64_t B, int64_t N, int dim, int k,
                            uint64_t* out_keys, void* workspace, size_t workspace_bytes,
                            float* dump, int32_t* diag, int flags, void* stream) {
  return topk_impl(mode, {q_hi, q_lo, 0, 0, bank_hi, bank_lo, 0, 0, 0, out_keys, workspace, workspace_bytes, stream},
                   {B, N, dim, k, 0}, b200knn_topk_options{}, dump, diag, flags);
}

int b200knn_set_l2_chunk_bytes(int64_t bytes) {
  if (bytes < 0) return fail(B200KNN_E_ARG, "set_l2_chunk_bytes: negative");
  g_l2_chunk_bytes = bytes;
  return B200KNN_OK;
}

// Plan introspection for the host shim / bench (how the work was split).
int b200knn_plan_info_ex(int mode, int64_t B, int64_t N, int dim, int k, int64_t* out9) {
  b200knn::TopkPlan plan;
  if (!out9 || !plan_for(mode, B, N, dim, k, &plan)) return fail(B200KNN_E_ARG, "plan_info_ex: bad argument");
  out9[0] = plan.n_qtiles;
  out9[1] = plan.splits;
  out9[2] = plan.split_rows;
  out9[3] = plan.n_items;
  out9[4] = plan.grid;
  out9[5] = plan.cap;
  out9[6] = plan.chunks;
  out9[7] = plan.chunk_rows;
  out9[8] = plan.slots;
  return B200KNN_OK;
}

int b200knn_merge(const uint64_t* keys_in, int G, int64_t B, int k_in, int k_out, uint64_t* keys_out,
                  void* stream) {
  if (!keys_in || !keys_out || G <= 0 || B < 0 || k_in <= 0 || k_out <= 0)
    return fail(B200KNN_E_ARG, "merge: bad argument");
  if (int64_t(k_out) > int64_t(G) * k_in) return fail(B200KNN_E_ARG, "merge: k_out > G*k_in");
  if (b200knn::list_capacity(k_out) == 0) return fail(B200KNN_E_UNSUPPORTED, "merge: k too large (max 992)");
  cudaError_t e = b200knn::launch_merge(keys_in, G, B, k_in, k_out, keys_out,
                                        static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("merge", e);
}

int b200knn_drop_self(const uint64_t* keys_in, int64_t B, int k_in, int64_t self_offset, uint64_t* keys_out,
                      void* stream) {
  if (!keys_in || !keys_out || B < 0) return fail(B200KNN_E_ARG, "drop_self: bad argument (null pointer or B < 0)");
  if (k_in < 2) return fail(B200KNN_E_ARG, "drop_self: need k_in >= 2");
  cudaError_t e = b200knn::launch_drop_self(keys_in, B, k_in, self_offset, keys_out,
                                            static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("drop_self", e);
}

int b200knn_drop_group(const uint64_t* keys_in, int64_t B, int k_in, const int64_t* row_ids,
                       const int32_t* group_ids, int64_t N, int k_out, uint64_t* keys_out, int32_t* err_flag,
                       void* stream) {
  if (!keys_in || !row_ids || !group_ids || !keys_out || !err_flag || B < 0 || N < 0)
    return fail(B200KNN_E_ARG, "drop_group: bad argument (null pointer, B < 0 or N < 0)");
  if (k_out < 1 || k_in < k_out) return fail(B200KNN_E_ARG, "drop_group: need 1 <= k_out <= k_in");
  cudaError_t e = b200knn::launch_drop_group(keys_in, B, k_in, row_ids, group_ids, N, k_out, keys_out, err_flag,
                                             static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("drop_group", e);
}

int b200knn_radius_compact(const uint64_t* keys, int64_t n, int m, const int64_t* row_ids, float tau,
                           int64_t self_offset, int64_t cap, int64_t* counts, int32_t* full, const int64_t* offsets,
                           int64_t* indices, float* sims, void* stream) {
  if (!keys || n < 0 || m < 1 || cap < 1) return fail(B200KNN_E_ARG, "radius_compact: bad argument (null keys, n < 0, m < 1 or cap < 1)");
  if (std::isnan(tau)) return fail(B200KNN_E_ARG, "radius_compact: tau is NaN");
  if (offsets == nullptr ? !counts : (!indices || !sims))
    return fail(B200KNN_E_ARG, "radius_compact: the count pass needs counts, the emit pass indices and sims");
  cudaError_t e = b200knn::launch_radius_compact(keys, n, m, row_ids, tau, self_offset, cap, counts, full, offsets,
                                                 indices, sims, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("radius_compact", e);
}

int b200knn_union_edges(int32_t* parent, int64_t n, const int64_t* offsets, const int64_t* indices, int64_t n_rows,
                        int64_t row_offset, int32_t* err_flag, void* stream) {
  if (!parent || !offsets || !err_flag || n < 0 || n_rows < 0 || (n_rows > 0 && !indices))
    return fail(B200KNN_E_ARG, "union_edges: bad argument (null pointer, n < 0 or n_rows < 0)");
  if (n > INT32_MAX) return fail(B200KNN_E_ARG, "union_edges: more than 2^31 - 1 nodes");
  cudaError_t e = b200knn::launch_union_edges(parent, n, offsets, indices, n_rows, row_offset, err_flag,
                                              static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("union_edges", e);
}

int b200knn_components(const int32_t* parent, int64_t n, int64_t* labels, void* stream) {
  if (!parent || !labels || n < 0) return fail(B200KNN_E_ARG, "components: bad argument");
  if (n > INT32_MAX) return fail(B200KNN_E_ARG, "components: more than 2^31 - 1 nodes");
  cudaError_t e = b200knn::launch_components(parent, n, labels, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("components", e);
}

int b200knn_row_norm_max(const float* rows_a, const float* rows_b, int64_t n, int dim_pad,
                         float* out_dev, void* stream) {
  if (!rows_a || !out_dev || n < 0 || dim_pad <= 0) return fail(B200KNN_E_ARG, "row_norm_max: bad argument");
  cudaError_t e = b200knn::launch_row_norm_max(rows_a, rows_b, n, dim_pad, out_dev,
                                               static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("row_norm_max", e);
}

int b200knn_row_f16_residual_max(const float* rows, int64_t n, int dim_pad, float* out_dev, void* stream) {
  if (!rows || !out_dev || n < 0 || dim_pad <= 0) return fail(B200KNN_E_ARG, "row_f16_residual_max: bad argument");
  cudaError_t e = b200knn::launch_row_f16_residual_max(rows, n, dim_pad, out_dev, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("row_f16_residual_max", e);
}

int b200knn_rescore(const void* q, int q_dtype, int64_t q_ld, const float* rows_a, const float* rows_b,
                    int64_t N, int dim, const uint64_t* cand_keys, int64_t B, int k_in, int k_out,
                    int64_t idx_offset, float err_coef, float err_abs, float max_abs,
                    const float* bank_max_norm, uint64_t* out_keys, int32_t* uncertified,
                    int32_t* n_uncertified, void* workspace, size_t workspace_bytes, void* stream) {
  if (!q || !rows_a || !cand_keys || !bank_max_norm || !out_keys || !uncertified || !n_uncertified)
    return fail(B200KNN_E_ARG, "rescore: null pointer");
  if (B < 0 || N <= 0 || dim <= 0 || k_out <= 0 || k_in < k_out || k_in > 1024)
    return fail(B200KNN_E_ARG, "rescore: bad shape (need 0 < k_out <= k_in <= 1024)");
  if (q_dtype < 0 || q_dtype > 2) return fail(B200KNN_E_ARG, "rescore: unknown dtype");
  b200knn::RescoreParams p;
  p.q = q;
  p.q_dtype = q_dtype;
  p.q_ld = q_ld;
  p.rows_a = rows_a;
  p.rows_b = rows_b;
  p.dim = dim;
  p.dim_pad = (dim + 63) / 64 * 64;
  p.cand = cand_keys;
  p.B = B;
  p.k_in = k_in;
  p.k_out = k_out;
  p.all_rows = (int64_t(k_in) >= N) ? 1 : 0;
  p.idx_offset = idx_offset;
  p.err_coef = err_coef;
  p.err_abs = err_abs;
  p.max_abs = max_abs;
  p.bank_max_norm = bank_max_norm;
  p.out = out_keys;
  p.uncertified = uncertified;
  p.n_uncertified = n_uncertified;
  cudaError_t e = b200knn::launch_rescore(p, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("rescore", e);
}

int b200knn_radius_tau0(const float* q, int64_t q_ld, int64_t B, int dim, float tau, float err_coef, float err_abs,
                        float max_abs, const float* bank_max_norm, const float* bank_resid, float acc_coef,
                        float* tau0, int32_t* refused, float* e_out, void* stream) {
  if (!q || !bank_max_norm || !tau0 || !refused) return fail(B200KNN_E_ARG, "radius_tau0: null pointer");
  if (B < 0 || dim <= 0 || q_ld < dim) return fail(B200KNN_E_ARG, "radius_tau0: bad shape (need B >= 0, 0 < dim <= q_ld)");
  if (!std::isfinite(tau)) return fail(B200KNN_E_ARG, "radius_tau0: tau must be finite");
  b200knn::RescoreParams p{};
  p.q = q;
  p.q_dtype = B200KNN_F32;
  p.q_ld = q_ld;
  p.dim = dim;
  p.dim_pad = (dim + 63) / 64 * 64;
  p.B = B;
  p.err_coef = err_coef;
  p.err_abs = err_abs;
  p.max_abs = max_abs;
  p.bank_max_norm = bank_max_norm;
  p.bank_resid = bank_resid;
  p.acc_coef = acc_coef;
  cudaError_t e = b200knn::launch_radius_tau0(p, tau, tau0, refused, e_out, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("radius_tau0", e);
}

int b200knn_rescore_vote(const float* q, int64_t q_ld, const float* rows, int64_t N, int dim,
                         const uint64_t* cand_keys, int64_t B, int k_in, int k, float err_coef, float err_abs,
                         float max_abs, const float* bank_max_norm, const float* bank_resid, float acc_coef,
                         const int64_t* labels, int64_t n_labels,
                         int C, double t, uint64_t* band_keys, int32_t* band_info, int64_t* pred,
                         int32_t* uncertified, int32_t* status, void* workspace, size_t workspace_bytes,
                         void* stream) {
  if (!q || !rows || !cand_keys || !bank_max_norm || !labels || !band_keys || !band_info || !pred ||
      !uncertified || !status || !workspace)
    return fail(B200KNN_E_ARG, "rescore_vote: null pointer");
  if (B < 0 || dim <= 0 || k <= 0 || k_in < k || k_in > 1024 || int64_t(k_in) >= N)
    return fail(B200KNN_E_ARG, "rescore_vote: bad shape (need 0 < k <= k_in <= 1024, k_in < N)");
  if (C < 1 || C > B200KNN_RESCORE_VOTE_MAX_CLASSES || !(t != 0.0))
    return fail(B200KNN_E_ARG, "rescore_vote: need 1 <= C <= 256 and t != 0");
  if (reinterpret_cast<uintptr_t>(rows) % 16 != 0) return fail(B200KNN_E_ARG, "rescore_vote: rows must be 16-byte aligned");
  if (workspace_bytes < b200knn::rescore_workspace_bytes(B, k_in))
    return fail(B200KNN_E_WORKSPACE, "rescore_vote: workspace too small");
  b200knn::RescoreParams p = {};
  p.q = q;
  p.q_dtype = B200KNN_F32;
  p.q_ld = q_ld;
  p.rows_a = rows;
  p.dim = dim;
  p.dim_pad = (dim + 63) / 64 * 64;
  p.cand = cand_keys;
  p.B = B;
  p.k_in = k_in;
  p.k_out = k;
  p.err_coef = err_coef;
  p.err_abs = err_abs;
  p.max_abs = max_abs;
  p.bank_max_norm = bank_max_norm;
  p.bank_resid = bank_resid;
  p.acc_coef = acc_coef;
  p.uncertified = uncertified;
  p.n_uncertified = status + 1;
  cudaError_t e = b200knn::launch_rescore_vote(p, band_keys, band_info, labels, n_labels, C, t, pred, status,
                                               workspace, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("rescore_vote", e);
}

int b200knn_certify(const void* q, int q_dtype, int64_t q_ld, int dim, const uint64_t* exact_keys, int k,
                    const uint64_t* approx_keys, int k_in, int64_t B, int all_rows, float err_coef,
                    float err_abs, float max_abs, const float* bank_max_norm, int32_t* uncertified,
                    int32_t* n_uncertified, void* stream) {
  if (!q || !exact_keys || !approx_keys || !bank_max_norm || !uncertified || !n_uncertified)
    return fail(B200KNN_E_ARG, "certify: null pointer");
  if (B < 0 || dim <= 0 || k <= 0 || k_in < k) return fail(B200KNN_E_ARG, "certify: bad shape (need 0 < k <= k_in)");
  if (q_dtype < 0 || q_dtype > 2) return fail(B200KNN_E_ARG, "certify: unknown dtype");
  b200knn::RescoreParams p = {};
  p.q = q;
  p.q_dtype = q_dtype;
  p.q_ld = q_ld;
  p.dim = dim;
  p.dim_pad = (dim + 63) / 64 * 64;
  p.cand = approx_keys;
  p.B = B;
  p.k_in = k_in;
  p.k_out = k;
  p.all_rows = all_rows ? 1 : 0;
  p.err_coef = err_coef;
  p.err_abs = err_abs;
  p.max_abs = max_abs;
  p.bank_max_norm = bank_max_norm;
  p.out = const_cast<uint64_t*>(exact_keys);  // read only by the certificate kernel
  p.uncertified = uncertified;
  p.n_uncertified = n_uncertified;
  cudaError_t e = b200knn::launch_certify(p, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("certify", e);
}

int b200knn_route_keys(const uint64_t* keys, int64_t n, int k, int64_t rows_per_shard, int n_shards,
                       uint64_t* out, void* stream) {
  if (!keys || !out || n < 0 || k <= 0 || rows_per_shard <= 0 || n_shards <= 0)
    return fail(B200KNN_E_ARG, "route_keys: bad argument");
  cudaError_t e = b200knn::launch_route_keys(keys, n, k, rows_per_shard, n_shards, out,
                                             static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("route_keys", e);
}

int b200knn_route_scatter(const uint64_t* keys, int64_t n, int k, int64_t rows_per_shard, int n_shards,
                          const void* const* host_inbox, int64_t row_offset, void* stream) {
  if (!keys || !host_inbox || n < 0 || k <= 0 || rows_per_shard <= 0 || n_shards <= 0 || n_shards > 8 ||
      row_offset < 0)
    return fail(B200KNN_E_ARG, "route_scatter: bad argument (1..8 shards)");
  uint64_t* inbox[8];
  for (int g = 0; g < n_shards; ++g) {
    if (!host_inbox[g]) return fail(B200KNN_E_ARG, "route_scatter: null inbox");
    inbox[g] = static_cast<uint64_t*>(const_cast<void*>(host_inbox[g]));
  }
  cudaError_t e = b200knn::launch_route_scatter(keys, n, k, rows_per_shard, n_shards, inbox, row_offset,
                                                static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("route_scatter", e);
}

int b200knn_rescore_scatter(const float* q, int64_t q_ld, const float* rows, int64_t N, int dim,
                            const uint64_t* cand_keys, int64_t B, int k_in, int64_t idx_offset,
                            const void* const* host_peer_out, int n_peers, int my_rank,
                            int64_t rows_per_owner, void* workspace, size_t workspace_bytes, void* stream) {
  if (!q || !rows || !cand_keys || !host_peer_out || !workspace)
    return fail(B200KNN_E_ARG, "rescore_scatter: null pointer");
  if (B < 0 || N <= 0 || dim <= 0 || k_in <= 0 || k_in > 1024)
    return fail(B200KNN_E_ARG, "rescore_scatter: bad shape (need 0 < k_in <= 1024)");
  if (n_peers < 1 || n_peers > 8 || my_rank < 0 || my_rank >= n_peers || rows_per_owner <= 0 ||
      rows_per_owner * n_peers < B)
    return fail(B200KNN_E_ARG, "rescore_scatter: 1..8 peers, a rank among them, rows_per_owner * n_peers >= B");
  if (reinterpret_cast<uintptr_t>(rows) % 16 != 0)
    return fail(B200KNN_E_ARG, "rescore_scatter: rows must be 16-byte aligned");
  if (workspace_bytes < b200knn::rescore_workspace_bytes(B, k_in))
    return fail(B200KNN_E_WORKSPACE, "rescore_scatter: workspace too small");
  b200knn::RescoreParams p = {};
  p.q = q;
  p.q_dtype = B200KNN_F32;
  p.q_ld = q_ld;
  p.rows_a = rows;
  p.rows_b = nullptr;
  p.dim = dim;
  p.dim_pad = (dim + 63) / 64 * 64;
  p.cand = cand_keys;
  p.B = B;
  p.k_in = k_in;
  p.k_out = k_in;
  p.idx_offset = idx_offset;
  p.n_peers = n_peers;
  p.my_rank = my_rank;
  p.rows_per_owner = rows_per_owner;
  for (int g = 0; g < n_peers; ++g) {
    if (!host_peer_out[g]) return fail(B200KNN_E_ARG, "rescore_scatter: null peer buffer");
    p.peer_out[g] = static_cast<uint64_t*>(const_cast<void*>(host_peer_out[g]));
  }
  cudaError_t e = b200knn::launch_rescore(p, workspace, workspace_bytes, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("rescore_scatter", e);
}

int b200knn_compact_rows(const int64_t* status, int64_t ld, int64_t n, int64_t mask, int64_t* rows_out,
                         int cap, int32_t* count_out, void* stream) {
  if (!status || !rows_out || !count_out || ld <= 0 || n < 0 || cap <= 0)
    return fail(B200KNN_E_ARG, "compact_rows: bad argument");
  cudaError_t e = b200knn::launch_compact_rows(status, ld, n, mask, rows_out, cap, count_out,
                                               static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("compact_rows", e);
}

int b200knn_scatter_rows(int64_t* dst, int64_t dst_ld, const int64_t* src, int64_t src_ld,
                         const int64_t* rows, int n, const int32_t* count, int width, void* stream) {
  if (!dst || !src || !rows || !count || n < 0 || width < 0 || dst_ld < width || src_ld < width)
    return fail(B200KNN_E_ARG, "scatter_rows: bad argument");
  cudaError_t e = b200knn::launch_scatter_rows(dst, dst_ld, src, src_ld, rows, n, count, width,
                                               static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("scatter_rows", e);
}

size_t b200knn_rescore_workspace_bytes(int64_t B, int k_in) {
  if (B <= 0 || k_in <= 0) return 0;
  return b200knn::rescore_workspace_bytes(B, k_in);
}

int b200knn_decode_keys(const uint64_t* keys, int64_t n_keys, float* sims, int64_t* idx, void* stream) {
  if (!keys || n_keys < 0) return fail(B200KNN_E_ARG, "decode_keys: bad argument");
  cudaError_t e = b200knn::launch_decode(keys, n_keys, sims, idx, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("decode_keys", e);
}

int b200knn_vote_ex(const uint64_t* keys, const int64_t* labels, int64_t B, int k, int64_t n_labels,
                    int64_t label_offset, int C, double t, int64_t* pred, int64_t pred_ld,
                    int status_col, double* scores, int32_t* err_flag, void* stream) {
  if (!keys || !labels || !pred || !err_flag || B < 0 || k <= 0 || C <= 0 || n_labels <= 0)
    return fail(B200KNN_E_ARG, "vote: bad argument");
  if (pred_ld < C || status_col >= pred_ld || (status_col >= 0 && status_col < C))
    return fail(B200KNN_E_ARG, "vote: pred_ld / status_col do not describe a (B, >=C) output");
  if (!(t > 0.0) && !(t < 0.0)) return fail(B200KNN_E_ARG, "vote: temperature must be non-zero");
  cudaError_t e = b200knn::launch_vote(keys, labels, B, k, n_labels, label_offset, C, t, pred, pred_ld,
                                       status_col, scores, err_flag, static_cast<cudaStream_t>(stream));
  if (e == cudaErrorInvalidValue) return fail(B200KNN_E_UNSUPPORTED, "vote: num_classes too large for shared memory");
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("vote", e);
}

int b200knn_vote_multi(const uint64_t* keys, const int64_t* labels, int64_t B, int k_max, int64_t n_labels,
                       int64_t label_offset, int C, const int* ks, int n_k, const double* ts, int n_t,
                       int64_t* pred, int64_t pred_ld, int status_col, int32_t* err_flag, void* stream) {
  if (!keys || !labels || !pred || !err_flag || !ks || !ts || B < 0 || k_max <= 0 || C <= 0 || n_labels <= 0)
    return fail(B200KNN_E_ARG, "vote_multi: bad argument");
  if (n_k < 1 || n_k > b200knn::kVoteMaxKs || n_t < 1 || n_t > b200knn::kVoteMaxTs)
    return fail(B200KNN_E_ARG, "vote_multi: need 1 <= n_k <= 16 and 1 <= n_t <= 8");
  b200knn::VoteGrid grid{};
  grid.n_k = n_k;
  grid.n_t = n_t;
  for (int i = 0; i < n_k; ++i) {
    if (ks[i] <= 0 || (i > 0 && ks[i] <= ks[i - 1]))
      return fail(B200KNN_E_ARG, "vote_multi: ks must be positive and strictly increasing");
    grid.ks[i] = ks[i];
  }
  if (ks[n_k - 1] != k_max) return fail(B200KNN_E_ARG, "vote_multi: ks[n_k-1] must equal k_max");
  for (int j = 0; j < n_t; ++j) {
    if (!(ts[j] > 0.0) && !(ts[j] < 0.0)) return fail(B200KNN_E_ARG, "vote_multi: temperature must be non-zero");
    grid.ts[j] = ts[j];
  }
  const int64_t width = int64_t(n_k) * n_t * C;
  if (pred_ld < width || status_col >= pred_ld || (status_col >= 0 && status_col < width))
    return fail(B200KNN_E_ARG, "vote_multi: pred_ld / status_col do not describe a (B, >=n_k*n_t*C) output");
  cudaError_t e = b200knn::launch_vote_multi(keys, labels, B, n_labels, label_offset, C, grid, pred, pred_ld,
                                             status_col, err_flag, static_cast<cudaStream_t>(stream));
  if (e == cudaErrorInvalidValue)
    return fail(B200KNN_E_UNSUPPORTED, "vote_multi: num_classes too large for shared memory");
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("vote_multi", e);
}

int b200knn_vote_multilabel(const uint64_t* keys, const uint64_t* label_bits, int64_t B, int k_max,
                            int64_t n_labels, int64_t label_offset, int L, const int* ks, int n_k,
                            const double* ts, int n_t, double* scores, int64_t scores_ld, int32_t* err_flag,
                            void* stream) {
  if (!keys || !label_bits || !scores || !err_flag || !ks || !ts || B < 0 || k_max <= 0 || n_labels <= 0)
    return fail(B200KNN_E_ARG, "vote_multilabel: bad argument");
  if (L < 1 || L > 64) return fail(B200KNN_E_ARG, "vote_multilabel: need 1 <= L <= 64 labels");
  if (n_k < 1 || n_k > b200knn::kVoteMaxKs || n_t < 1 || n_t > b200knn::kVoteMaxTs)
    return fail(B200KNN_E_ARG, "vote_multilabel: need 1 <= n_k <= 16 and 1 <= n_t <= 8");
  b200knn::VoteGrid grid{};
  grid.n_k = n_k;
  grid.n_t = n_t;
  for (int i = 0; i < n_k; ++i) {
    if (ks[i] <= 0 || (i > 0 && ks[i] <= ks[i - 1]))
      return fail(B200KNN_E_ARG, "vote_multilabel: ks must be positive and strictly increasing");
    grid.ks[i] = ks[i];
  }
  if (ks[n_k - 1] != k_max) return fail(B200KNN_E_ARG, "vote_multilabel: ks[n_k-1] must equal k_max");
  for (int j = 0; j < n_t; ++j) {
    if (!(ts[j] > 0.0) || !std::isfinite(ts[j]))
      return fail(B200KNN_E_ARG, "vote_multilabel: temperature must be finite and > 0");
    grid.ts[j] = ts[j];
  }
  if (scores_ld < int64_t(n_k) * n_t * L)
    return fail(B200KNN_E_ARG, "vote_multilabel: scores_ld does not describe a (B, >=n_k*n_t*L) output");
  cudaError_t e = b200knn::launch_vote_multilabel(keys, label_bits, B, n_labels, label_offset, L, grid, scores,
                                                  scores_ld, err_flag, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("vote_multilabel", e);
}

int b200knn_vote(const uint64_t* keys, const int64_t* labels, int64_t B, int k, int64_t n_labels,
                 int64_t label_offset, int C, double t, int64_t* pred, double* scores,
                 int32_t* err_flag, void* stream) {
  return b200knn_vote_ex(keys, labels, B, k, n_labels, label_offset, C, t, pred, C, -1, scores, err_flag,
                         stream);
}

int b200knn_normalize_rows(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld, float eps,
                           float* dst_rows, void* stream) {
  if (!src || !dst_rows || n_vec < 0 || dim <= 0 || ld < dim) return fail(B200KNN_E_ARG, "normalize_rows: bad argument");
  if (src_dtype < B200KNN_F32 || src_dtype > B200KNN_BF16) return fail(B200KNN_E_ARG, "normalize_rows: unknown dtype");
  cudaError_t e = b200knn::launch_normalize_rows(src, src_dtype, n_vec, dim, ld, eps, dst_rows,
                                                 static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("normalize_rows", e);
}

int b200knn_row_sqnorms(const void* src, int src_dtype, int64_t n_vec, int dim, int64_t ld, float* out,
                        void* stream) {
  if (!src || !out || n_vec < 0 || dim <= 0 || ld < dim) return fail(B200KNN_E_ARG, "row_sqnorms: bad argument");
  if (src_dtype < B200KNN_F32 || src_dtype > B200KNN_BF16) return fail(B200KNN_E_ARG, "row_sqnorms: unknown dtype");
  cudaError_t e = b200knn::launch_row_sqnorm(src, src_dtype, n_vec, dim, ld, out, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("row_sqnorms", e);
}

int b200knn_confusion(const int64_t* pred, const int64_t* target, int64_t n, int C, int64_t* counts,
                      int32_t* err_flag, void* stream) {
  if (!pred || !target || !counts || !err_flag || n < 0 || C <= 0) return fail(B200KNN_E_ARG, "confusion: bad argument");
  cudaError_t e = b200knn::launch_confusion(pred, target, n, C, counts, err_flag, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("confusion", e);
}

int b200knn_key_sim_column(const uint64_t* keys, int64_t B, int k, int j, float* out, void* stream) {
  if (!keys || !out || B < 0 || k <= 0 || j < 0 || j >= k) return fail(B200KNN_E_ARG, "key_sim_column: bad argument");
  cudaError_t e = b200knn::launch_key_sim_column(keys, B, k, j, out, static_cast<cudaStream_t>(stream));
  return e == cudaSuccess ? B200KNN_OK : fail_cuda("key_sim_column", e);
}

}  // extern "C"
