// select.cu — candidate-list merge (the exchange step of the sharded mode and
// of bank splits inside one GPU), the self- and group-exclusion of leave-one-out
// lists and key decoding.
//
// Inputs are lists of 64-bit selection keys sorted descending under the
// canonical (sim desc, idx asc) order, so merging G lists is itself a top-k of
// their union under one integer compare; the result is independent of G and
// of how the bank was partitioned (SURVEY.md §8e invariant).
#include "common.cuh"
#include "kernels.h"

namespace b200knn {
namespace {

// One warp per query row.  The warp streams the G lists into a CAP-slot buffer in shared
// memory, SKIPPING empty slots (lists are sorted descending, so the first empty key ends a
// list): shards and bank splits that ran under a shared admission threshold return mostly
// empty lists, and the union of their non-empty keys usually fits the buffer, i.e. one sort
// per row instead of one per list.  When the buffer fills it is pruned (sort, keep k_out).
// HBM-bound: reads <= G*k_in*8 B, writes k_out*8 B per row.
// wpr > 1 (few rows, many lists — the reference-shaped B = 64 call over a bank split 74 ways):
// wpr warps share a row, warp s ingests lists s, s+wpr, ... into its own buffer, and the row's
// first warp then folds the other buffers into its own; the list fetches of a row are then
// wpr-way parallel instead of one dependent chain (45 us -> ~10 us for 64 rows x 74 lists).
template <int ITEMS>
__device__ __forceinline__ void merge_rows_body(const uint64_t* __restrict__ in, int G, int64_t B, int k_in,
                                                int k_out, uint64_t* __restrict__ out, int wpr,
                                                uint64_t* merge_smem) {
  constexpr int CAP = ITEMS * 32;
  const int lane = threadIdx.x & 31;
  const int warp = threadIdx.x >> 5;
  const int n_warps = blockDim.x >> 5;
  const int sub = warp % wpr;
  const int64_t row = int64_t(blockIdx.x) * (n_warps / wpr) + warp / wpr;
  if (wpr == 1 && row >= B) return;
  const bool active = row < B;
  uint64_t* buf = merge_smem + size_t(warp) * CAP;
  int* cnts = reinterpret_cast<int*>(merge_smem + size_t(n_warps) * CAP);
  const unsigned lt_mask = (1u << lane) - 1u;
  int cnt = 0;

  auto prune = [&]() {  // cut the buffer to ~k_out: radix-select, or sort when ties defeat it
    __syncwarp();
    if (cnt > k_out) {
      int kept = -1;
      warp_prune_select<ITEMS>(buf, cnt, k_out, lane, &kept);
      __syncwarp();
      if (kept >= 0) {
        cnt = kept;
        return;
      }
    }
    uint64_t v[ITEMS];
#pragma unroll
    for (int r = 0; r < ITEMS; ++r) {
      const int i = r * 32 + lane;
      v[r] = i < cnt ? buf[i] : 0ull;
    }
    warp_sort_desc<ITEMS>(v, lane);
#pragma unroll
    for (int r = 0; r < ITEMS; ++r) {
      const int i = r * 32 + lane;
      if (i < k_out) buf[i] = v[r];
    }
    cnt = cnt < k_out ? cnt : k_out;
    __syncwarp();
  };
  // returns true when the chunk held an empty key (the rest of that list is empty too)
  auto push = [&](uint64_t key) -> bool {
    const bool nz = key != 0ull;
    const unsigned bm = __ballot_sync(kFull, nz);
    if (bm == 0u) return true;
    if (cnt + 32 > CAP) prune();
    if (nz) buf[cnt + __popc(bm & lt_mask)] = key;
    cnt += __popc(bm);
    return bm != kFull;
  };

  constexpr int kAhead = 4;  // first chunks of several lists are fetched together (latency)
  for (int g0 = sub; active && g0 < G; g0 += kAhead * wpr) {
    uint64_t first[kAhead];
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      const int g = g0 + u * wpr;
      first[u] = (g < G && lane < k_in) ? in[(int64_t(g) * B + row) * k_in + lane] : 0ull;
    }
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      const int g = g0 + u * wpr;
      if (g >= G) break;
      bool done = push(first[u]);
      const uint64_t* list = in + (int64_t(g) * B + row) * k_in;
      for (int j0 = 32; j0 < k_in && !done; j0 += 32)
        done = push(j0 + lane < k_in ? list[j0 + lane] : 0ull);
    }
  }
  if (wpr > 1) {
    __syncwarp();
    if (lane == 0) cnts[warp] = cnt;
    __syncthreads();
    if (sub != 0 || !active) return;
    for (int w = 1; w < wpr; ++w) {
      const uint64_t* src = buf + size_t(w) * CAP;
      const int n = cnts[warp + w];
      for (int j0 = 0; j0 < n; j0 += 32) push(j0 + lane < n ? src[j0 + lane] : 0ull);
    }
  }
  // final sort, with the network sized to what survived (long buffers are first cut to ~k_out
  // by radix-select, which is several times cheaper than the 512-key network)
  __syncwarp();
  uint64_t* o = out + row * k_out;
  if (ITEMS > 8 && cnt > 256 && cnt > k_out) {
    int kept = -1;
    warp_prune_select<ITEMS>(buf, cnt, k_out, lane, &kept);
    if (kept >= 0) cnt = kept;
    __syncwarp();
  }
  if (cnt <= 32) sort_store<1>(buf, cnt, k_out, lane, o);
  else if (cnt <= 64) sort_store<2>(buf, cnt, k_out, lane, o);
  else if (ITEMS >= 4 && cnt <= 128) sort_store<(ITEMS >= 4 ? 4 : ITEMS)>(buf, cnt, k_out, lane, o);
  else if (ITEMS >= 8 && cnt <= 256) sort_store<(ITEMS >= 8 ? 8 : ITEMS)>(buf, cnt, k_out, lane, o);
  else if (ITEMS >= 16 && cnt <= 512) sort_store<(ITEMS >= 16 ? 16 : ITEMS)>(buf, cnt, k_out, lane, o);
  else sort_store<ITEMS>(buf, cnt, k_out, lane, o);
}

template <int ITEMS>
__global__ void __launch_bounds__(256) merge_kernel(const uint64_t* __restrict__ in, int G,
                                                    int64_t B, int k_in, int k_out,
                                                    uint64_t* __restrict__ out, int wpr) {
  extern __shared__ __align__(16) uint64_t merge_smem[];
  merge_rows_body<ITEMS>(in, G, B, k_in, k_out, out, wpr, merge_smem);
}

// Few rows, many lists (the reference-shaped B = 64 call: one list per bank split and row, ~138 of
// them, mostly short because every split ran under the sampled threshold).  One 8-warp block per
// row: (1) all warps gather the non-empty keys of the row's lists into shared memory (slots from
// one atomic counter); (2) if more than the sorting network holds survive, a block-wide radix
// select on the 64-bit keys finds a threshold that keeps between k_out and CAP of them (early
// exit, a handful of counting rounds); (3) one warp sorts the survivors once.  The warp-serial
// variant above spends its time folding eight partial buffers through one warp (60 us for 64 rows
// x 138 lists at k = 240; this one: one gather, ~3 counting rounds, one sort).  Rows whose lists
// do not fit the staging buffer (no threshold: every split returns k_in keys) or whose keys tie
// beyond the network take the warp-serial path inside the same block.
constexpr int kStage = 4096;  // keys staged per row
template <int ITEMS>
__global__ void __launch_bounds__(256, 2) merge_small_kernel(const uint64_t* __restrict__ in, int G, int64_t B,
                                                          int k_in, int k_out, uint64_t* __restrict__ out) {
  constexpr int CAP = ITEMS * 32;
  constexpr int kPerThread = kStage / 256;
  extern __shared__ __align__(16) uint64_t merge_smem[];
  __shared__ int s_n, s_over, s_red[8];
  __shared__ unsigned long long s_and[8], s_or[8];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
  const int64_t row = blockIdx.x;
  const unsigned lt_mask = (1u << lane) - 1u;
  if (tid == 0) {
    s_n = 0;
    s_over = 0;
  }
  __syncthreads();
  // (1) gather: one THREAD per list (the lists are short and sit at unrelated addresses, so the
  // parallelism that hides the load latency is across lists, 256 at a time); a list longer than
  // kLong keys means it ran without a useful threshold, and the row takes the warp-serial path
  constexpr int kLong = 64;
  const bool pairs = (k_in % 2) == 0;  // 16-byte loads of two keys (list bases are then 16-byte aligned)
  for (int g = tid; g < G; g += 256) {
    const uint64_t* list = in + (int64_t(g) * B + row) * k_in;
    for (int j = 0; j < k_in;) {
      uint64_t k0, k1 = 0ull;
      if (pairs) {
        const ulonglong2 kk = *reinterpret_cast<const ulonglong2*>(list + j);
        k0 = kk.x;
        k1 = kk.y;
      } else {
        k0 = list[j];
      }
      const int c = (k0 != 0ull ? 1 : 0) + ((k0 != 0ull && k1 != 0ull) ? 1 : 0);
      if (c == 0) break;
      if (j + c > kLong) {
        s_over = 1;
        break;
      }
      const int base = atomicAdd(&s_n, c);
      if (base + c <= kStage) {
        merge_smem[base] = k0;
        if (c == 2) merge_smem[base + 1] = k1;
      } else {
        s_over = 1;
        break;
      }
      if (c < (pairs ? 2 : 1)) break;
      j += pairs ? 2 : 1;
    }
  }
  __syncthreads();
  int n = s_n;
  bool slow = s_over != 0;
  uint64_t* o = out + row * k_out;
  if (!slow && n > CAP) {
    // (2) block-wide radix select: threshold T with k_out <= #{key >= T} <= CAP
    uint64_t v[kPerThread];
    uint64_t a = ~0ull, r = 0ull;
#pragma unroll
    for (int i = 0; i < kPerThread; ++i) {
      const int idx = i * 256 + tid;
      v[i] = idx < n ? merge_smem[idx] : 0ull;
      if (idx < n) {
        a &= v[i];
        r |= v[i];
      }
    }
    a = (uint64_t(__reduce_and_sync(kFull, uint32_t(a >> 32))) << 32) | __reduce_and_sync(kFull, uint32_t(a));
    r = (uint64_t(__reduce_or_sync(kFull, uint32_t(r >> 32))) << 32) | __reduce_or_sync(kFull, uint32_t(r));
    if (lane == 0) {
      s_and[warp] = a;
      s_or[warp] = r;
    }
    __syncthreads();
#pragma unroll
    for (int w = 0; w < 8; ++w) {
      a &= s_and[w];
      r |= s_or[w];
    }
    uint64_t T = a, open_bits = a ^ r;
    int c = n;
    while (open_bits) {
      const uint64_t bit = 1ull << (63 - __clzll(open_bits));
      open_bits &= ~bit;
      const uint64_t cand = T | bit;
      int cc = 0;
#pragma unroll
      for (int i = 0; i < kPerThread; ++i) cc += (v[i] >= cand) ? 1 : 0;
      cc = __reduce_add_sync(kFull, cc);
      __syncthreads();  // previous round's s_red reads are done
      if (lane == 0) s_red[warp] = cc;
      __syncthreads();
      cc = 0;
#pragma unroll
      for (int w = 0; w < 8; ++w) cc += s_red[w];
      if (cc >= k_out) {
        T = cand;
        c = cc;
        if (c <= CAP) break;
      }
    }
    if (c > CAP) {
      slow = true;  // ties beyond the network (identical keys of the sampling variant): sort-based path
    } else {
      // compact the survivors to the front of the staging buffer (every key is in registers by now)
      __syncthreads();
      if (tid == 0) s_n = 0;
      __syncthreads();
#pragma unroll
      for (int i = 0; i < kPerThread; ++i) {
        const bool keep = v[i] >= T && v[i] != 0ull;
        const unsigned bm = __ballot_sync(kFull, keep);
        int base = 0;
        if (lane == 0 && bm != 0u) base = atomicAdd(&s_n, __popc(bm));
        base = __shfl_sync(kFull, base, 0);
        if (keep) merge_smem[base + __popc(bm & lt_mask)] = v[i];
      }
      __syncthreads();
      n = s_n;
    }
  }
  if (slow) {  // uniform over the block
    __syncthreads();
    merge_rows_body<ITEMS>(in, G, B, k_in, k_out, out, 8, merge_smem);
    return;
  }
  // (3) one sort of what is left (n <= CAP)
  if (warp != 0) return;
  if (n == 0) {
    for (int i = lane; i < k_out; i += 32) o[i] = 0ull;
  } else if (n <= 32) sort_store<1>(merge_smem, n, k_out, lane, o);
  else if (n <= 64) sort_store<2>(merge_smem, n, k_out, lane, o);
  else if (ITEMS >= 4 && n <= 128) sort_store<(ITEMS >= 4 ? 4 : ITEMS)>(merge_smem, n, k_out, lane, o);
  else if (ITEMS >= 8 && n <= 256) sort_store<(ITEMS >= 8 ? 8 : ITEMS)>(merge_smem, n, k_out, lane, o);
  else if (ITEMS >= 16 && n <= 512) sort_store<(ITEMS >= 16 ? 16 : ITEMS)>(merge_smem, n, k_out, lane, o);
  else sort_store<ITEMS>(merge_smem, n, k_out, lane, o);
}

__global__ void decode_kernel(const uint64_t* __restrict__ keys, int64_t n, float* __restrict__ sims,
                              int64_t* __restrict__ idx) {
  const int64_t i = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const uint64_t key = keys[i];
  if (sims) sims[i] = key_sim(key);
  if (idx) idx[i] = key_idx(key);
}

// One warp per row: (B, k_in) sorted keys -> (B, k_in - 1) without the key of bank row
// b + self_offset, or without the last key when that row is not in the list (a row need not be
// among its own nearest neighbours, and an exact duplicate of lower index ranks before it).
// A ballot finds the self key's position p; each lane stores its key j at j - (j > p).  Empty (0)
// keys never match.  HBM-bound: 8 B in and 8 B out per key; kAhead chunks are loaded before the
// first ballot so that several loads per warp are in flight.
__global__ void __launch_bounds__(256) drop_self_kernel(const uint64_t* __restrict__ in, int64_t B, int k_in,
                                                        int64_t self_offset, uint64_t* __restrict__ out) {
  constexpr int kAhead = 4;
  const int lane = threadIdx.x & 31;
  const int64_t row = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B) return;
  const int64_t self = row + self_offset;
  const uint64_t* src = in + row * k_in;
  uint64_t* dst = out + row * (k_in - 1);
  int p = k_in - 1;  // the position dropped: the self key's once found, the last one otherwise
  bool found = false;
  for (int j0 = 0; j0 < k_in; j0 += 32 * kAhead) {
    uint64_t v[kAhead];
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      const int j = j0 + u * 32 + lane;
      v[u] = j < k_in ? src[j] : 0ull;
    }
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      const int j = j0 + u * 32 + lane;
      const unsigned m = __ballot_sync(kFull, !found && v[u] != 0ull && key_idx(v[u]) == self);
      if (m) {
        p = j0 + u * 32 + __ffs(m) - 1;
        found = true;
      }
      if (j < k_in && j != p) dst[j - (j > p ? 1 : 0)] = v[u];
    }
  }
}

// One warp per row: (B, k_in) sorted keys -> (B, k_out), the first k_out keys whose bank row is
// not in the group of bank row row_ids[b], in order, zero-filled when fewer survive (leave-one-
// group-out lists).  Each lane gathers group_ids[key index] (4 B per bank row: 3.2 MB at
// N = 811k, so L2-resident) and compares it with the row's own id; a ballot plus a prefix
// popcount gives each survivor its output position.  Empty (0) keys are never dropped.  A key
// index or row id outside [0, N) sets *err_flag = 2 (the vote's "index outside the labels"); such
// a key is kept, such a row drops nothing.  kAhead chunks (and their group gathers) are issued
// before the first ballot, as in drop_self_kernel.  The warp stops after the chunk group in which
// the k_out-th survivor appears (a row of a large group searched at k + p keeps k keys): keys past
// it are neither read nor checked.
__global__ void __launch_bounds__(256) drop_group_kernel(const uint64_t* __restrict__ in, int64_t B, int k_in,
                                                         const int64_t* __restrict__ row_ids,
                                                         const int32_t* __restrict__ group_ids, int64_t N,
                                                         int k_out, uint64_t* __restrict__ out,
                                                         int32_t* __restrict__ err_flag) {
  constexpr int kAhead = 4;
  const int lane = threadIdx.x & 31;
  const int64_t row = int64_t(blockIdx.x) * (blockDim.x >> 5) + (threadIdx.x >> 5);
  if (row >= B) return;
  const uint64_t* src = in + row * k_in;
  uint64_t* dst = out + row * k_out;
  const int64_t self = row_ids[row];
  const bool self_ok = self >= 0 && self < N;
  const int32_t own = self_ok ? group_ids[self] : 0;
  bool bad = !self_ok;
  const unsigned lt_mask = (1u << lane) - 1u;
  int n = 0;  // survivors so far (warp-uniform)
  for (int j0 = 0; j0 < k_in && n < k_out; j0 += 32 * kAhead) {
    uint64_t v[kAhead];
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      const int j = j0 + u * 32 + lane;
      v[u] = j < k_in ? src[j] : 0ull;
    }
    bool keep[kAhead];
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      keep[u] = j0 + u * 32 + lane < k_in;
      if (v[u] != 0ull) {
        const int64_t i = key_idx(v[u]);
        if (i < N) keep[u] &= !(self_ok && group_ids[i] == own);  // key_idx of a non-empty key is >= 0
        else bad = true;
      }
    }
#pragma unroll
    for (int u = 0; u < kAhead; ++u) {
      const unsigned m = __ballot_sync(kFull, keep[u]);
      const int pos = n + __popc(m & lt_mask);
      if (keep[u] && pos < k_out) dst[pos] = v[u];
      n += __popc(m);
    }
  }
  for (int j = n + lane; j < k_out; j += 32) dst[j] = 0ull;
  if (bad) atomicExch(err_flag, 2);
}

__global__ void key_sim_column_kernel(const uint64_t* __restrict__ keys, int64_t B, int k, int j,
                                      float* __restrict__ out) {
  const int64_t b = int64_t(blockIdx.x) * blockDim.x + threadIdx.x;
  if (b < B) out[b] = key_sim(keys[b * k + j]);
}

template <int ITEMS>
cudaError_t launch_merge_t(const uint64_t* in, int G, int64_t B, int k_in, int k_out, uint64_t* out,
                           cudaStream_t stream) {
  // few rows: one row per CTA so that the rows spread over the SMs, and — when there are many
  // lists — several warps per row
  if (B < 148 * 8 && G >= 8) {  // few rows, many lists: one block per row, block-wide select
    const size_t stage = size_t(kStage) > size_t(8) * ITEMS * 32 ? size_t(kStage) : size_t(8) * ITEMS * 32;
    const size_t smem = stage * sizeof(uint64_t) + sizeof(int) * 8;
    auto kern = merge_small_kernel<ITEMS>;
    if (smem > 48 * 1024) {
      cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
      if (e != cudaSuccess) return e;
    }
    kern<<<unsigned(B), 256, smem, stream>>>(in, G, B, k_in, k_out, out);
    return cudaGetLastError();
  }
  int warps = 4, wpr = 1;
  const int64_t blocks = (B + warps / wpr - 1) / (warps / wpr);
  const size_t smem = size_t(warps) * ITEMS * 32 * sizeof(uint64_t) + sizeof(int) * warps;
  auto kern = merge_kernel<ITEMS>;
  if (smem > 48 * 1024) {
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
    if (e != cudaSuccess) return e;
  }
  kern<<<unsigned(blocks), warps * 32, smem, stream>>>(in, G, B, k_in, k_out, out, wpr);
  return cudaGetLastError();
}

}  // namespace

cudaError_t launch_merge(const uint64_t* in, int G, int64_t B, int k_in, int k_out, uint64_t* out,
                         cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  const int cap = list_capacity(k_out);
  switch (cap) {
    case 64: return launch_merge_t<2>(in, G, B, k_in, k_out, out, stream);
    case 128: return launch_merge_t<4>(in, G, B, k_in, k_out, out, stream);
    case 256: return launch_merge_t<8>(in, G, B, k_in, k_out, out, stream);
    case 512: return launch_merge_t<16>(in, G, B, k_in, k_out, out, stream);
    case 1024: return launch_merge_t<32>(in, G, B, k_in, k_out, out, stream);
    default: return cudaErrorInvalidValue;
  }
}

cudaError_t launch_key_sim_column(const uint64_t* keys, int64_t B, int k, int j, float* out,
                                  cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  key_sim_column_kernel<<<unsigned((B + 255) / 256), 256, 0, stream>>>(keys, B, k, j, out);
  return cudaGetLastError();
}

cudaError_t launch_drop_self(const uint64_t* in, int64_t B, int k_in, int64_t self_offset, uint64_t* out,
                             cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  constexpr int kWarps = 8;
  drop_self_kernel<<<unsigned((B + kWarps - 1) / kWarps), kWarps * 32, 0, stream>>>(in, B, k_in, self_offset, out);
  return cudaGetLastError();
}

cudaError_t launch_drop_group(const uint64_t* in, int64_t B, int k_in, const int64_t* row_ids,
                              const int32_t* group_ids, int64_t N, int k_out, uint64_t* out, int32_t* err_flag,
                              cudaStream_t stream) {
  if (B == 0) return cudaSuccess;
  constexpr int kWarps = 8;
  drop_group_kernel<<<unsigned((B + kWarps - 1) / kWarps), kWarps * 32, 0, stream>>>(
      in, B, k_in, row_ids, group_ids, N, k_out, out, err_flag);
  return cudaGetLastError();
}

cudaError_t launch_decode(const uint64_t* keys, int64_t n, float* sims, int64_t* idx,
                          cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  const int threads = 256;
  decode_kernel<<<unsigned((n + threads - 1) / threads), threads, 0, stream>>>(keys, n, sims, idx);
  return cudaGetLastError();
}

}  // namespace b200knn
