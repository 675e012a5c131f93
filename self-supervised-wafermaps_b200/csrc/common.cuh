// common.cuh — selection keys, warp bitonic sort and the streaming per-row top-k
// state shared by every similarity kernel (exact fp32 and tcgen05 paths).
//
// Canonical total order (SURVEY.md §7.3): neighbours are ranked by
// (sim desc, bank index asc).  A 64-bit key makes that one integer compare:
//     key = orderable_u32(sim) << 32 | (0xFFFFFFFF - idx)      larger = better
// This replaces the unspecified tie order of Tensor.topk in lightly's
// knn_predict (call site: src/ssl_wafermap/models/knn.py:91-98).
#pragma once
#include <cstdint>
#include <cuda_fp16.h>
#include <cuda_runtime.h>

namespace b200knn {

constexpr uint32_t kFull = 0xffffffffu;

__device__ __forceinline__ uint32_t f32_to_orderable(float s) {
  s = s + 0.0f;  // -0.0 -> +0.0 so that equal values compare equal
  uint32_t b = __float_as_uint(s);
  return (b & 0x80000000u) ? ~b : (b | 0x80000000u);
}
__device__ __forceinline__ float orderable_to_f32(uint32_t u) {
  uint32_t b = (u & 0x80000000u) ? (u & 0x7fffffffu) : ~u;
  return __uint_as_float(b);
}
__device__ __forceinline__ uint64_t make_key(float s, uint32_t idx) {
  return (uint64_t(f32_to_orderable(s)) << 32) | uint64_t(0xFFFFFFFFu - idx);
}
__device__ __forceinline__ float key_sim(uint64_t key) {
  return key == 0 ? __int_as_float(0xff800000)  // empty slot -> -inf
                  : orderable_to_f32(uint32_t(key >> 32));
}
__device__ __forceinline__ int64_t key_idx(uint64_t key) {
  return key == 0 ? int64_t(-1) : int64_t(0xFFFFFFFFu - uint32_t(key & 0xFFFFFFFFu));
}

// The fp16 operand of x in the F16 / F16X2 modes: rn(sat(x)), sat clamping to +-65504 so that no
// inf/NaN ever enters the contraction.  The bank and query preparation and the certificate's
// residual norms (rescore.cu) all round through this one function.
__device__ __forceinline__ __half f16_operand(float x) {
  return __float2half_rn(fminf(fmaxf(x, -65504.0f), 65504.0f));
}

// Bitonic sort, descending, of ITEMS*32 keys held as v[r] on lane l <-> element
// index r*32 + l.  Strides >= 32 are register-to-register, < 32 are shuffles.
// The (size, stride) loops are deliberately NOT unrolled: a fully unrolled
// 512-key network is ~120 KB of SASS that is executed once per prune and
// thrashes the instruction cache (measured: stall_no_instruction was the top
// stall reason of the fused kernel); rolled, the body is a few hundred
// instructions that stay resident.
template <int ITEMS, int D>
__device__ __forceinline__ void sort_stage_inreg(uint64_t (&v)[ITEMS], int size) {
#pragma unroll
  for (int r = 0; r < ITEMS; ++r) {
    const int pr = r ^ D;
    if (pr > r && pr < ITEMS) {
      const bool desc = (((r * 32) & size) == 0);
      const uint64_t a = v[r], b = v[pr];
      const bool sw = desc ? (a < b) : (a > b);
      v[r] = sw ? b : a;
      v[pr] = sw ? a : b;
    }
  }
}

template <int ITEMS>
__device__ __forceinline__ void warp_sort_desc(uint64_t (&v)[ITEMS], int lane) {
  constexpr int N = ITEMS * 32;
#pragma unroll 1
  for (int size = 2; size <= N; size <<= 1) {
#pragma unroll 1
    for (int stride = size >> 1; stride > 0; stride >>= 1) {
      if (stride >= 32) {
        switch (stride >> 5) {
          case 1: sort_stage_inreg<ITEMS, 1>(v, size); break;
          case 2: sort_stage_inreg<ITEMS, 2>(v, size); break;
          case 4: sort_stage_inreg<ITEMS, 4>(v, size); break;
          case 8: sort_stage_inreg<ITEMS, 8>(v, size); break;
          default: sort_stage_inreg<ITEMS, 16>(v, size); break;
        }
      } else {
        const bool lower = ((lane & stride) == 0);
#pragma unroll
        for (int r = 0; r < ITEMS; ++r) {
          const int i = r * 32 + lane;
          const uint64_t other = __shfl_xor_sync(kFull, v[r], stride);
          const bool desc = ((i & size) == 0);
          const bool keep_max = (desc == lower);
          const bool gt = v[r] > other;
          v[r] = (gt == keep_max) ? v[r] : other;
        }
      }
    }
  }
}

// Smallest supported list capacity (power of two, multiple of 32) for a given k.
// The capacity leaves slack above k so that a prune (sort + cut to k) happens
// once per (cap - k - 32) insertions rather than per insertion.
__host__ __device__ inline int list_capacity(int k) {
  int cap = 64;
  while (cap < 2 * k + 32 && cap < 1024) cap <<= 1;
  if (cap < k + 32) cap = 0;  // k too large for the in-register sort (k <= 992)
  return cap;
}

// Warp-cooperative prune of one row's candidate list (global scratch, `cap`
// = ITEMS*32 slots, `n_valid` filled): sort descending, keep the best k in
// place (sorted).  Returns the new admission threshold: the sim of the k-th
// best, or -inf while fewer than k candidates exist.
template <int ITEMS>
__device__ __forceinline__ float warp_prune(uint64_t* list, int n_valid, int k, int lane) {
  uint64_t v[ITEMS];
#pragma unroll
  for (int r = 0; r < ITEMS; ++r) {
    const int i = r * 32 + lane;
    v[r] = (i < n_valid) ? list[i] : 0ull;
  }
  warp_sort_desc<ITEMS>(v, lane);
  uint64_t kth = 0;
#pragma unroll
  for (int r = 0; r < ITEMS; ++r) {
    const int i = r * 32 + lane;
    if (i < k) list[i] = v[r];
    kth = (i == k - 1) ? v[r] : kth;  // lane-dependent select: stays in registers
  }
  kth = __shfl_sync(kFull, kth, (k - 1) & 31);
  return (n_valid >= k && kth != 0) ? orderable_to_f32(uint32_t(kth >> 32))
                                    : __int_as_float(0xff800000);
}

// Cheaper prune for the streaming phase: the new threshold only needs the k-th largest
// SIMILARITY, not a sorted list.  Radix-select over the 32 orderable bits of the sims (one
// warp-wide count per bit), then compact the keys with sim >= T in place (unsorted; the
// final flush sorts once).  All keys tied at T are kept, so the kept count can exceed k;
// returns it in *kept, or -1 if the ties would not leave room to keep appending (the caller
// then falls back to the exact sort-based prune, which breaks ties by index).
template <int ITEMS>
__device__ __forceinline__ float warp_prune_select(uint64_t* list, int n_valid, int k, int lane,
                                                   int* kept) {
  constexpr int CAP = ITEMS * 32;
  uint64_t v[ITEMS];
  uint32_t hi[ITEMS];
  uint32_t all_and = 0xffffffffu, all_or = 0u;
#pragma unroll
  for (int r = 0; r < ITEMS; ++r) {
    const int i = r * 32 + lane;
    v[r] = (i < n_valid) ? list[i] : 0ull;
    hi[r] = uint32_t(v[r] >> 32);
    if (i < n_valid) {
      all_and &= hi[r];
      all_or |= hi[r];
    }
  }
  all_and = __reduce_and_sync(kFull, all_and);
  all_or = __reduce_or_sync(kFull, all_or);
  // Every caller may append up to 32 more keys before it checks the list again, so the kept
  // count must also leave 32 free slots (k close to CAP: one tie at the cut would otherwise let
  // the next chunk of appends run past the list).
  const int room = (k + (CAP - k) / 4 < CAP - 32) ? k + (CAP - k) / 4 : CAP - 32;
  // bits on which all sims agree are fixed; search the others from the most significant down.
  // The search stops as soon as the count above the candidate threshold lies in [k, room]: the
  // threshold need not be the exact k-th similarity, any value that keeps between k and `room`
  // keys is as good (a few extra keys survive until the next prune / the final sort).  That
  // ends the search after the few bits that separate ~CAP values down to a window of room - k,
  // instead of walking all ~22 open mantissa bits — prunes sit on the accumulator hand-over's
  // critical path (one late warp of 16 stalls the MMA issuer), so their latency is what matters.
  uint32_t T = all_and;
  uint32_t open_bits = all_and ^ all_or;
  int c = n_valid;  // keys with hi >= T
  while (open_bits) {
    const uint32_t bit = 0x80000000u >> __clz(open_bits);
    open_bits &= ~bit;
    const uint32_t cand = T | bit;
    int cc = 0;
#pragma unroll
    for (int r = 0; r < ITEMS; ++r) cc += (hi[r] >= cand) ? 1 : 0;
    cc = __reduce_add_sync(kFull, cc);
    if (cc >= k) {
      T = cand;
      c = cc;
      if (c <= room) break;
    }
  }
  // now count(hi >= T) = c >= k (n_valid >= k is the caller's precondition); ties at T are all kept
  if (c > room) {
    *kept = -1;
    return 0.0f;
  }
  __syncwarp();
  const unsigned lt_mask = (1u << lane) - 1u;
  int base = 0;
#pragma unroll
  for (int r = 0; r < ITEMS; ++r) {
    const bool keep = hi[r] >= T;  // empty slots have hi == 0 < T
    const unsigned bm = __ballot_sync(kFull, keep);
    if (keep) list[base + __popc(bm & lt_mask)] = v[r];
    base += __popc(bm);
  }
  *kept = base;
  return orderable_to_f32(T);
}

// Per-row streaming state owned by the row's scanning thread.
struct RowState {
  float tau;     // admit sims strictly greater than tau (ties lose: bank is scanned in ascending idx)
  uint32_t cnt;  // filled slots of the row's list
};

// After a chunk of at most CHUNK appends per row: prune every row of the warp
// whose list could overflow during the next chunk.  `lists` points at the
// warp's first row; row r of the warp is lane r.
// slack = free slots every row must keep: the hard bound is the most a row can
// append before the next call (32 per chunk); callers that run off the critical
// path pass a larger value to prune early, where it stalls nobody.
// SELECT: prune by radix-select (threshold + unsorted compaction) instead of a full sort.
template <int ITEMS, bool SELECT = false>
__device__ __forceinline__ void warp_maintain(uint64_t* lists, RowState& st, int k, int lane,
                                              int slack) {
  constexpr int CAP = ITEMS * 32;
  const bool need = (int(st.cnt) + slack > CAP) && (int(st.cnt) > k);
  unsigned m = __ballot_sync(kFull, need);
  if (m == 0) return;
  __syncwarp();  // owner's appends visible to the whole warp
  while (m) {
    const int src = __ffs(m) - 1;
    m &= m - 1;
    const int n_valid = __shfl_sync(kFull, int(st.cnt), src);
    int kept = -1;
    float t = 0.0f;
    if (SELECT) t = warp_prune_select<ITEMS>(lists + size_t(src) * CAP, n_valid, k, lane, &kept);
    if (kept < 0) {
      t = warp_prune<ITEMS>(lists + size_t(src) * CAP, n_valid, k, lane);
      kept = n_valid < k ? n_valid : k;
    }
    if (lane == src) {
      st.tau = fmaxf(st.tau, t);  // never below a caller-supplied initial threshold
      st.cnt = uint32_t(kept);
    }
  }
  __syncwarp();
}

// Sort the first n (<= S*32) keys of `list` descending and write the best k to `o`
// (zero-padded).
template <int S>
__device__ __forceinline__ void sort_store(const uint64_t* list, int n, int k, int lane, uint64_t* o) {
  uint64_t v[S];
#pragma unroll
  for (int r = 0; r < S; ++r) {
    const int i = r * 32 + lane;
    v[r] = (i < n) ? list[i] : 0ull;
  }
  warp_sort_desc<S>(v, lane);
#pragma unroll
  for (int r = 0; r < S; ++r) {
    const int i = r * 32 + lane;
    if (i < k) o[i] = v[r];
  }
  for (int i = S * 32 + lane; i < k; i += 32) o[i] = 0ull;  // k beyond this network: empty slots
}

// End of a work item: every row of the warp is pruned one last time and its
// best k keys (sorted descending, zero-padded) are written out if row_valid.  The sorting network is sized to
// the row's candidate count (rows that ran under a good threshold hold few), and
// long lists are first cut to ~k by radix-select.
// `out_of(r)` returns where row r of the warp goes (a local buffer, or a peer GPU's exchange
// buffer when the kernel scatters its results over NVLink).
// unsorted_ok: the consumer is merge_kernel (bank splits, or the exchange buffer of a peer GPU),
// which treats a list as a zero-terminated SET: rows that hold at most k keys are then copied as
// they are — no sorting network on the item's tail, where the MMA pipe waits for the epilogue.
template <int ITEMS, typename OutFn>
__device__ __forceinline__ void warp_flush(uint64_t* lists, const RowState& st, int k, int lane,
                                           unsigned valid_mask, OutFn out_of, bool unsorted_ok = false) {
  constexpr int CAP = ITEMS * 32;
  __syncwarp();
  for (int src = 0; src < 32; ++src) {
    if (!((valid_mask >> src) & 1u)) continue;
    int n_valid = __shfl_sync(kFull, int(st.cnt), src);
    uint64_t* list = lists + size_t(src) * CAP;
    uint64_t* o = out_of(src);
    if (unsorted_ok && n_valid <= k) {
      for (int i = lane; i < k; i += 32) o[i] = i < n_valid ? list[i] : 0ull;
      continue;
    }
    if (ITEMS > 8 && n_valid > 256 && n_valid > k) {
      int kept = -1;
      warp_prune_select<ITEMS>(list, n_valid, k, lane, &kept);
      if (kept >= 0) n_valid = kept;
      __syncwarp();
    }
    // short lists (rows that ran under a good threshold in a small work item: the reference-shaped
    // B = 64 call flushes ~146 of them per row) must not pay for a 64-key network each
    if (n_valid == 0) {
      for (int i = lane; i < k; i += 32) o[i] = 0ull;
    } else if (n_valid <= 32) sort_store<1>(list, n_valid, k, lane, o);
    else if (n_valid <= 64) sort_store<2>(list, n_valid, k, lane, o);
    else if (ITEMS >= 4 && n_valid <= 128) sort_store<(ITEMS >= 4 ? 4 : ITEMS)>(list, n_valid, k, lane, o);
    else if (ITEMS >= 8 && n_valid <= 256) sort_store<(ITEMS >= 8 ? 8 : ITEMS)>(list, n_valid, k, lane, o);
    else if (ITEMS >= 16 && n_valid <= 512) sort_store<(ITEMS >= 16 ? 16 : ITEMS)>(list, n_valid, k, lane, o);
    else sort_store<ITEMS>(list, n_valid, k, lane, o);
  }
  __syncwarp();
}

}  // namespace b200knn
