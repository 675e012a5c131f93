// rescore.cu — exact re-scoring of tensor-core candidates ("fp32" mode).
//
// The tensor-core pass (tc_topk.cu) returns, per query, the k_in > k best bank
// rows under APPROXIMATE similarities (bf16 or 3xTF32 products, fp32 TMEM
// accumulation).  This kernel recomputes the similarity of every candidate
// exactly as MODE_EXACT defines it — an fmaf chain over d = 0..D-1 from +0.0f on
// the caller's fp32 values — re-ranks them under the canonical (sim desc, idx
// asc) order and keeps the best k.  The result is bitwise the MODE_EXACT result
// whenever the candidate set contains the true top-k, which is CERTIFIED per row:
//     exact_sim(rank k)  >  approx_sim(rank k_in) + E,
//     E = err_coef * ||q|| * max_n ||bank_n||      (Cauchy-Schwarz bound on the
//         approximation error of any non-candidate row)
// Rows that fail the certificate are flagged; the host shim re-runs those rows in
// MODE_EXACT, so the mode as a whole reproduces lightly's fp32 knn_predict
// neighbours (reference call site src/ssl_wafermap/models/knn.py:91-98) bit for
// bit against the oracle (oracle/seqfma.c).
//
// HBM/L2-bound gather: per query k_in rows of D fp32 (k_in*D*4 B, x2 in TF32X3
// where x = hi + lo is reassembled), 8*k B out.
//
// Two implementations of the same arithmetic:
//  * rescore_dot_kernel + rescore_select_kernel (fp32 queries, one fp32 row array, caller
//    workspace): persistent warps, each owning a ring of shared-memory stages that the
//    TMA engine fills with 32 candidate rows x CHUNK columns (one cp.async.bulk per row, the
//    query chunk by cp.async, all completing on the stage's mbarrier).  Lane c then walks
//    row c with conflict-free LDS.128 (row pitch CHUNK+4 floats) — the fma chain of one
//    candidate is sequential by definition, so the parallelism is 32 candidates per warp
//    and the copies of the next stage are in flight while the chain runs.  The exact keys go
//    to the workspace; a second kernel sorts them per query and evaluates the certificate.
//  * rescore_kernel (any query dtype, optional lo array, no workspace): one block per
//    query, rows staged by plain loads.  Kept for the TF32X3 operands and small calls.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <cstdlib>

#include "../../include/b200knn.h"
#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace b200knn {
namespace {

// The bound E >= |approx - exact| of one query against every bank row (DESIGN §4.1c, §5).
// qn = ||q||, qtn = ||f16(q)||, rho = ||q - f16(q)||, each rounded up / inflated by the caller.
//   E = err_coef ||q|| M + err_abs (||q|| + M)              the level's model (b200knn.knn LEVELS), M = *bank_max_norm
//     + qtn R + rho M~ + rho R + acc_coef qtn M~            with the bank's measured fp16 residuals [R, M~] (bank_resid)
//     + dim_pad 2^-149                                       underflow of the exact fma chain
// A level without residuals (bank_resid == nullptr) gets its worst-case model alone; with them the
// caller passes err_coef = gamma_D (the exact chain's own rounding) and err_abs = 0.  The last term
// changes no E above 2^-100 and covers the fp32 evaluation of a tiny E; the inflated norms cover
// it above.
__device__ __forceinline__ float cert_bound(const RescoreParams& p, float qn, float qtn, float rho) {
  const float m = *p.bank_max_norm;
  float e = p.err_coef * qn * m + p.err_abs * (qn + m);
  if (p.bank_resid != nullptr) {
    const float r = p.bank_resid[0], mt = p.bank_resid[1];
    e += qtn * r + rho * mt + rho * r + p.acc_coef * qtn * mt;
  }
  return e + float(p.dim_pad) * 0x1p-149f;
}

// Certificate of one row (see the header): kth = exact key at rank k_out, last = approximate key
// at rank k_in, qn = ||q|| (inflated by the caller for its rounding).
__device__ __forceinline__ int certified(const RescoreParams& p, uint64_t kth, uint64_t last, float qn) {
  if (last == 0) {
    // an empty slot certifies the row only when every bank row was a candidate (k_in >= N);
    // otherwise the candidate pass ran under an admission threshold that starved this row
    return p.all_rows ? 1 : 0;
  }
  const float m = *p.bank_max_norm;
  if (p.max_abs > 0.0f && !(qn < p.max_abs && m < p.max_abs)) return 0;  // operand range of the candidate pass
  const float e = cert_bound(p, qn, 0.0f, 0.0f);
  return (kth != 0) && (key_sim(kth) > key_sim(last) + e);
}

// slots per query in the workspace of the pipelined variant: k_in rounded up to 64 (work units of
// up to 64 candidate slots)
inline int ws_slots(int k_in) { return (k_in + 63) / 64 * 64; }

constexpr int kWarps = 4;
constexpr int kChunk = 64;            // d-columns staged per step
constexpr int kTileLd = kChunk + 1;   // padded: lane c walks row c conflict-free

__device__ __forceinline__ float ldq(const void* p, int dtype, int64_t i) {
  if (dtype == B200KNN_F32) return static_cast<const float*>(p)[i];
  if (dtype == B200KNN_F16) return __half2float(static_cast<const __half*>(p)[i]);
  return __bfloat162float(static_cast<const __nv_bfloat16*>(p)[i]);
}

template <int ITEMS>
__global__ void __launch_bounds__(kWarps * 32)
    rescore_kernel(RescoreParams p) {
  extern __shared__ __align__(16) unsigned char rs_smem[];
  float* qs = reinterpret_cast<float*>(rs_smem);                       // [dim_pad]
  float* tiles = qs + p.dim_pad;                                        // [kWarps][32][kTileLd]
  uint64_t* keys = reinterpret_cast<uint64_t*>(tiles + kWarps * 32 * kTileLd);  // [ITEMS*32]
  float* red = reinterpret_cast<float*>(keys + ITEMS * 32);             // [kWarps]

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = blockIdx.x;
  const uint64_t* cand = p.cand + b * p.k_in;

  float qq = 0.0f;
  for (int d = threadIdx.x; d < p.dim_pad; d += kWarps * 32) {
    const float v = d < p.dim ? ldq(p.q, p.q_dtype, b * p.q_ld + d) : 0.0f;
    qs[d] = v;
    qq = fmaf(v, v, qq);
  }
  for (int i = threadIdx.x; i < ITEMS * 32; i += kWarps * 32) keys[i] = 0ull;
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) qq += __shfl_xor_sync(kFull, qq, o);
  if (lane == 0) red[warp] = qq;
  __syncthreads();

  float* tile = tiles + warp * 32 * kTileLd;
  for (int c0 = warp * 32; c0 < p.k_in; c0 += kWarps * 32) {
    const int c = c0 + lane;
    const uint64_t key = c < p.k_in ? cand[c] : 0ull;
    const int64_t row = key != 0 ? key_idx(key) - p.idx_offset : -1;
    float acc = 0.0f;
    for (int d0 = 0; d0 < p.dim_pad; d0 += kChunk) {
      // cooperative, coalesced: lane l fetches columns d0+2l, d0+2l+1 of each of the 32 rows
      for (int cc = 0; cc < 32; ++cc) {
        const int64_t r = __shfl_sync(kFull, row, cc);
        float2 v = make_float2(0.0f, 0.0f);
        if (r >= 0) {
          v = *reinterpret_cast<const float2*>(p.rows_a + r * p.dim_pad + d0 + 2 * lane);
          if (p.rows_b != nullptr) {
            const float2 w = *reinterpret_cast<const float2*>(p.rows_b + r * p.dim_pad + d0 + 2 * lane);
            v.x += w.x;  // hi + lo is exact: lo = x - rna_tf32(x)
            v.y += w.y;
          }
        }
        tile[cc * kTileLd + 2 * lane] = v.x;
        tile[cc * kTileLd + 2 * lane + 1] = v.y;
      }
      __syncwarp();
#pragma unroll 8
      for (int dd = 0; dd < kChunk; ++dd) acc = __fmaf_rn(qs[d0 + dd], tile[lane * kTileLd + dd], acc);
      __syncwarp();
    }
    if (c < p.k_in) keys[c] = row >= 0 ? make_key(acc, uint32_t(row + p.idx_offset)) : 0ull;
  }
  __syncthreads();

  if (warp == 0) {
    uint64_t v[ITEMS];
#pragma unroll
    for (int r = 0; r < ITEMS; ++r) v[r] = keys[r * 32 + lane];
    warp_sort_desc<ITEMS>(v, lane);
    uint64_t kth = 0;
#pragma unroll
    for (int r = 0; r < ITEMS; ++r) {
      const int i = r * 32 + lane;
      if (i < p.k_out) p.out[b * p.k_out + i] = v[r];
      kth = (i == p.k_out - 1) ? v[r] : kth;
    }
    kth = __shfl_sync(kFull, kth, (p.k_out - 1) & 31);
    if (lane == 0) {
      const uint64_t last = cand[p.k_in - 1];  // worst candidate under the approximate order
      const float qn = sqrtf(red[0] + red[1] + red[2] + red[3]) * 1.001f;
      const int ok = certified(p, kth, last, qn);
      p.uncertified[b] = ok ? 0 : 1;
      if (!ok) atomicAdd(p.n_uncertified, 1);
    }
  }
}


// ------------------------------------------------------------------ pipelined variant
// One work unit = 32*R consecutive candidate slots of one query (lane l owns slots l, l+32, ...);
// a step = one unit x one CHUNK of columns.  Each warp owns STAGES stages and a contiguous range
// of units.  R = 2 (two independent fma chains per lane) is an experiment that did not pay, see
// launch_rescore.
template <int CHUNK, int R>
struct DotStage {
  static constexpr int kPitch = CHUNK + 4;  // floats; lane c reads float4 j of row c: bank group (c + j) mod 8
  float rows[32 * R * kPitch];
  float q[CHUNK];
  uint32_t klo[32 * R];  // low key word (0xFFFFFFFF - idx) of each candidate, 0 = empty slot
};

__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void* src, uint32_t bytes, uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
__device__ __forceinline__ void cp_async16_zfill(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async4_zfill(uint32_t dst, const void* src, uint32_t src_bytes) {
  asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;" ::"r"(dst), "l"(src), "r"(src_bytes) : "memory");
}
__device__ __forceinline__ void cp_async_arrive_noinc(uint32_t bar) {
  asm volatile("cp.async.mbarrier.arrive.noinc.shared::cta.b64 [%0];" ::"r"(bar) : "memory");
}

// tmp: (B, n_groups * 32 * R) exact keys, slot c of query b at tmp[b * n_groups*32*R + c]
template <int CHUNK, int STAGES, int R>
__global__ void __launch_bounds__(384)
    rescore_dot_kernel(RescoreParams p, uint64_t* __restrict__ tmp, int n_groups, int64_t n_units,
                       int q_vec16) {
  using Stage = DotStage<CHUNK, R>;
  constexpr int kSlots = 32 * R;
  extern __shared__ __align__(16) unsigned char rs_smem[];
  const int n_warps = blockDim.x >> 5;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  Stage* stages = reinterpret_cast<Stage*>(rs_smem) + size_t(warp) * STAGES;
  uint64_t* bars = reinterpret_cast<uint64_t*>(rs_smem + sizeof(Stage) * size_t(n_warps) * STAGES) +
                   warp * STAGES;
  if (lane == 0) {
    // per phase: lane 0's arrive.expect_tx + one cp.async "noinc" arrival per lane (query chunk)
    for (int s = 0; s < STAGES; ++s) ptx::mbar_init(ptx::smem_u32(&bars[s]), 33);
    ptx::fence_barrier_init();
  }
  __syncwarp();

  const int64_t wg = int64_t(blockIdx.x) * n_warps + warp, tw = int64_t(gridDim.x) * n_warps;
  const int64_t u_begin = n_units * wg / tw, u_end = n_units * (wg + 1) / tw;
  if (u_begin >= u_end) return;
  const int n_chunks = (p.dim_pad + CHUNK - 1) / CHUNK;
  const float* q32 = static_cast<const float*>(p.q);

  struct Keys {
    uint64_t k[R];
  };
  auto load_keys = [&](int64_t b, int g) -> Keys {
    Keys ks;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      const int c = g * kSlots + r * 32 + lane;
      ks.k[r] = (b < p.B && g < n_groups && c < p.k_in) ? p.cand[b * p.k_in + c] : 0ull;
    }
    return ks;
  };

  // producer cursor: unit (pb, pg), chunk pc; this lane's keys of that unit, of the next unit of the
  // same query and of the first unit of the next query (candidate lists are filled from the front:
  // the first empty unit of a query ends it, and the cursor jumps to the next query)
  int64_t pu = u_begin, pb = u_begin / n_groups;
  int pg = int(u_begin - pb * n_groups), pc = 0, ps = 0;
  Keys p_key = load_keys(pb, pg);
  Keys p_key_next = load_keys(pb, pg + 1);
  Keys p_key_nq = load_keys(pb + 1, 0);

  // One pipeline step = (unit, chunk).  The first unit of a query without candidates (routed lists
  // of the sharded mode use ~1/G of their slots) takes ONE step — no copies, just the barrier
  // handshake — and ends the query: producer and consumer, which sees the same all-empty key
  // words, both jump to the next query.
  auto produce = [&]() {
    Stage& st = stages[ps];
    const uint32_t bar = ptx::smem_u32(&bars[ps]);
    const int d0 = pc * CHUNK;
    const int len = min(CHUNK, p.dim_pad - d0);
    int64_t row[R];
    unsigned n_valid = 0;
#pragma unroll
    for (int r = 0; r < R; ++r) {
      row[r] = p_key.k[r] != 0 ? key_idx(p_key.k[r]) - p.idx_offset : -1;
      n_valid += __popc(__ballot_sync(kFull, row[r] >= 0));
    }
    if (lane == 0) ptx::mbar_expect_tx(bar, n_valid * uint32_t(len) * 4u);
#pragma unroll
    for (int r = 0; r < R; ++r)
      if (row[r] >= 0)
        bulk_g2s(ptx::smem_u32(st.rows + (r * 32 + lane) * Stage::kPitch), p.rows_a + row[r] * p.dim_pad + d0,
                 uint32_t(len) * 4u, bar);
    const float* qrow = q32 + pb * p.q_ld;
    if (n_valid == 0u) {
    } else if (q_vec16) {
      for (int i = lane; i < len / 4; i += 32) {
        const int d = d0 + 4 * i;
        const int nb = max(0, min(16, (p.dim - d) * 4));
        cp_async16_zfill(ptx::smem_u32(st.q + 4 * i), qrow + (nb > 0 ? d : 0), uint32_t(nb));
      }
    } else {
      for (int i = lane; i < len; i += 32) {
        const int d = d0 + i;
        cp_async4_zfill(ptx::smem_u32(st.q + i), qrow + (d < p.dim ? d : 0), d < p.dim ? 4u : 0u);
      }
    }
    cp_async_arrive_noinc(bar);
    if (pc == 0) {
#pragma unroll
      for (int r = 0; r < R; ++r) st.klo[r * 32 + lane] = row[r] >= 0 ? uint32_t(p_key.k[r]) : 0u;
    }
    if (++ps == STAGES) ps = 0;
    if (n_valid == 0u || ++pc == n_chunks) {
      pc = 0;
      if (n_valid == 0u || pg + 1 == n_groups) {  // on to the next query
        pu += n_groups - pg;
        ++pb;
        pg = 0;
        p_key = p_key_nq;
        p_key_nq = load_keys(pb + 1, 0);
      } else {
        ++pu;
        ++pg;
        p_key = p_key_next;
      }
      p_key_next = load_keys(pb, pg + 1);
    }
  };

  for (int t = 0; t < STAGES && pu < u_end; ++t) produce();

  int cs = 0, cc = 0;
  uint32_t phase = 0;
  uint32_t klo[R];
  float acc[R];
#pragma unroll
  for (int r = 0; r < R; ++r) {
    klo[r] = 0u;
    acc[r] = 0.0f;
  }
  int64_t cu = u_begin;
  int cg = int(u_begin % n_groups);
  bool live = true;  // the unit holds at least one candidate
  while (cu < u_end) {
    Stage& st = stages[cs];
    ptx::mbar_wait(ptx::smem_u32(&bars[cs]), phase, nullptr, 7);
    if (cc == 0) {
      bool any = false;
#pragma unroll
      for (int r = 0; r < R; ++r) {
        acc[r] = 0.0f;
        klo[r] = st.klo[r * 32 + lane];
        any = any || klo[r] != 0u;
      }
      live = __any_sync(kFull, any);
    }
    if (live) {
      const int len4 = min(CHUNK, p.dim_pad - cc * CHUNK) / 4;
      const float4* qr = reinterpret_cast<const float4*>(st.q);
      const float4* xr[R];
#pragma unroll
      for (int r = 0; r < R; ++r) xr[r] = reinterpret_cast<const float4*>(st.rows + (r * 32 + lane) * Stage::kPitch);
      // len4 is a multiple of 16 (dim_pad is a multiple of 64).  The loads of a block of 4 float4 per
      // row are issued before its fma chains start, and the next block's loads while they run; the
      // R chains of a lane are independent and interleave in the pipeline.
      constexpr int kBlk = 4;
      float4 x[R][kBlk], w[kBlk];
#pragma unroll
      for (int i = 0; i < kBlk; ++i) {
        w[i] = qr[i];
#pragma unroll
        for (int r = 0; r < R; ++r) x[r][i] = xr[r][i];
      }
#pragma unroll 1
      for (int j = 0; j < len4; j += kBlk) {
        float4 xn[R][kBlk], wn[kBlk];
        const int jn = (j + kBlk < len4) ? j + kBlk : j;
#pragma unroll
        for (int i = 0; i < kBlk; ++i) {
          wn[i] = qr[jn + i];
#pragma unroll
          for (int r = 0; r < R; ++r) xn[r][i] = xr[r][jn + i];
        }
#pragma unroll
        for (int i = 0; i < kBlk; ++i) {
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = __fmaf_rn(w[i].x, x[r][i].x, acc[r]);
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = __fmaf_rn(w[i].y, x[r][i].y, acc[r]);
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = __fmaf_rn(w[i].z, x[r][i].z, acc[r]);
#pragma unroll
          for (int r = 0; r < R; ++r) acc[r] = __fmaf_rn(w[i].w, x[r][i].w, acc[r]);
        }
#pragma unroll
        for (int i = 0; i < kBlk; ++i) {
          w[i] = wn[i];
#pragma unroll
          for (int r = 0; r < R; ++r) x[r][i] = xn[r][i];
        }
      }
    }
    if (!live) {  // the rest of this query is empty (the select kernel masks by the candidate keys)
      cc = 0;
      cu += n_groups - cg;
      cg = 0;
    } else if (++cc == n_chunks) {
      cc = 0;
#pragma unroll
      for (int r = 0; r < R; ++r)
        tmp[cu * kSlots + r * 32 + lane] =
            klo[r] != 0 ? ((uint64_t(f32_to_orderable(acc[r])) << 32) | uint64_t(klo[r])) : 0ull;
      ++cu;
      if (++cg == n_groups) cg = 0;
    }
    // the stage is free: order this warp's generic-proxy reads before the async-proxy refill
    __syncwarp();
    ptx::fence_proxy_async();
    if (pu < u_end) produce();
    if (++cs == STAGES) {
      cs = 0;
      phase ^= 1;
    }
  }
}

// Sort the first `groups` 32-key groups of v descending with the smallest network that covers
// them (the other groups are empty and stay where they are: zeros sort last anyway).
template <int ITEMS>
__device__ __forceinline__ void sort_groups(uint64_t (&v)[ITEMS], int groups, int lane) {
  if (ITEMS > 2 && groups <= 2) {
    uint64_t w[2] = {v[0], v[1]};
    warp_sort_desc<2>(w, lane);
    v[0] = w[0];
    v[1] = w[1];
  } else if (ITEMS > 4 && groups <= 4) {
    uint64_t w[4] = {v[0], v[1], v[2], v[3]};
    warp_sort_desc<4>(w, lane);
#pragma unroll
    for (int r = 0; r < 4; ++r) v[r] = w[r];
  } else {
    warp_sort_desc<ITEMS>(v, lane);
  }
}

// exact keys of one query (n_groups*32 slots in the workspace) -> best k_out, sorted; certificate.
// Sharded re-scoring (p.n_peers > 0): the sorted exact keys of query b go straight into the
// exchange buffer of the GPU that owns query b (peer memory over NVLink), non-empty prefix only
// (the owner zeroes its buffer before the exchange); no certificate here — the owner evaluates
// it on the merged lists.
template <int ITEMS>
__global__ void __launch_bounds__(128)
    rescore_select_kernel(RescoreParams p, const uint64_t* __restrict__ tmp, int n_groups) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = int64_t(blockIdx.x) * 4 + warp;
  if (b >= p.B) return;
  const uint64_t* mine = tmp + b * n_groups * 32;
  uint64_t v[ITEMS];
  int groups = 0;  // groups holding at least one key (candidate lists are filled from the front)
#pragma unroll
  for (int r = 0; r < ITEMS; ++r) {
    // a slot holds an exact key only where the candidate list holds a candidate (lists are filled
    // from the front; the dot kernel does not touch the slots of empty units)
    const int c = r * 32 + lane;
    const bool has = r < n_groups && c < p.k_in && p.cand[b * p.k_in + c] != 0ull;
    v[r] = has ? mine[c] : 0ull;
    if (__any_sync(kFull, has)) groups = r + 1;
  }
  sort_groups<ITEMS>(v, groups, lane);
  if (p.n_peers > 0) {
    const int64_t owner = b / p.rows_per_owner;
    uint64_t* o = p.peer_out[owner] +
                  (int64_t(p.my_rank) * p.rows_per_owner + (b - owner * p.rows_per_owner)) * p.k_out;
#pragma unroll
    for (int r = 0; r < ITEMS; ++r) {
      const int i = r * 32 + lane;
      if (i < p.k_out && v[r] != 0ull) o[i] = v[r];
    }
    return;
  }
  const float* qrow = static_cast<const float*>(p.q) + b * p.q_ld;
  float qq = 0.0f;
  for (int d = lane; d < p.dim; d += 32) qq = fmaf(qrow[d], qrow[d], qq);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) qq += __shfl_xor_sync(kFull, qq, o);
  uint64_t kth = 0;
#pragma unroll
  for (int r = 0; r < ITEMS; ++r) {
    const int i = r * 32 + lane;
    if (i < p.k_out) p.out[b * p.k_out + i] = v[r];
    kth = (i == p.k_out - 1) ? v[r] : kth;
  }
  kth = __shfl_sync(kFull, kth, (p.k_out - 1) & 31);
  if (lane == 0) {
    const uint64_t last = p.cand[b * p.k_in + p.k_in - 1];  // worst candidate under the approximate order
    const int ok = certified(p, kth, last, sqrtf(qq) * 1.001f);
    p.uncertified[b] = ok ? 0 : 1;
    if (!ok) atomicAdd(p.n_uncertified, 1);
  }
}

// The certificate alone (sharded fp32 mode: the exact keys of a query come back from the shards
// that own the candidate rows and are merged by the query's owner): p.out holds the merged exact
// keys (B, k_out), p.cand the merged approximate candidates (B, k_in).  One warp per query.
__global__ void __launch_bounds__(128) certify_kernel(RescoreParams p) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = int64_t(blockIdx.x) * 4 + warp;
  if (b >= p.B) return;
  float qq = 0.0f;
  for (int d = lane; d < p.dim; d += 32) {
    const float v = ldq(p.q, p.q_dtype, b * p.q_ld + d);
    qq = fmaf(v, v, qq);
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) qq += __shfl_xor_sync(kFull, qq, o);
  if (lane == 0) {
    const int ok = certified(p, p.out[b * p.k_out + p.k_out - 1], p.cand[b * p.k_in + p.k_in - 1],
                             sqrtf(qq) * 1.001f);
    p.uncertified[b] = ok ? 0 : 1;
    if (!ok) atomicAdd(p.n_uncertified, 1);
  }
}

// out[g][r][:] = the keys of row r whose bank row belongs to shard g (rows [g*rows_per_shard, ...)),
// in their original order, compacted to the front and zero-padded: the query owner's candidate list
// split by the shard that can re-score each candidate.  Compact lists let the re-scoring kernel
// skip the empty 32-slot units (with G shards only ~1/G of the slots are used).  One warp per row.
__global__ void __launch_bounds__(128)
    route_keys_kernel(const uint64_t* __restrict__ keys, int64_t n, int k, int64_t rows_per_shard, int G,
                      uint64_t* __restrict__ out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t r = int64_t(blockIdx.x) * 4 + warp;
  if (r >= n) return;
  const unsigned lt_mask = (1u << lane) - 1u;
  const uint64_t* row = keys + r * k;
  for (int g = 0; g < G; ++g) {
    uint64_t* o = out + (int64_t(g) * n + r) * k;
    int cnt = 0;
    for (int j0 = 0; j0 < k; j0 += 32) {
      const uint64_t key = j0 + lane < k ? row[j0 + lane] : 0ull;
      const bool mine = key != 0 && key_idx(key) / rows_per_shard == g;
      const unsigned bm = __ballot_sync(kFull, mine);
      if (mine) o[cnt + __popc(bm & lt_mask)] = key;
      cnt += __popc(bm);
    }
    for (int j = cnt + lane; j < k; j += 32) o[j] = 0ull;
  }
}

// max over rows of ||row||_2 (fp32), inflated by 0.1 % for the rounding of the reduction
__global__ void __launch_bounds__(256)
    row_norm_max_kernel(const float* __restrict__ a, const float* __restrict__ b, int64_t n,
                        int dim_pad, float* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  float best = 0.0f;
  for (int64_t r = warp; r < n; r += n_warps) {
    float s = 0.0f;
    for (int d = lane; d < dim_pad; d += 32) {
      float v = a[r * dim_pad + d];
      if (b != nullptr) v += b[r * dim_pad + d];
      s = fmaf(v, v, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(kFull, s, o);
    best = fmaxf(best, s);
  }
  if (lane == 0) atomicMax(reinterpret_cast<int*>(out), __float_as_int(sqrtf(best) * 1.001f));
}

// out[0] = max over rows of ||x - f16(x)||, out[1] = of ||f16(x)|| (f16_operand, the bank's fp16
// operand).  fp64 sums of exact squares, padded for their rounding and rounded up to fp32; a row
// holding a NaN makes both +inf, which refuses the bound.  Non-negative floats order as ints.
__global__ void __launch_bounds__(256)
    row_f16_residual_max_kernel(const float* __restrict__ a, int64_t n, int dim_pad, float* __restrict__ out) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, lane = threadIdx.x & 31;
  const int n_warps = (gridDim.x * blockDim.x) >> 5;
  double best_r = 0.0, best_t = 0.0;
  for (int64_t row = warp; row < n; row += n_warps) {
    double rr = 0.0, tt = 0.0;
    for (int d = lane; d < dim_pad; d += 32) {
      const float x = a[row * dim_pad + d];
      const double t = __half2float(f16_operand(x)), r = double(x) - t;
      rr = fma(r, r, rr);
      tt = fma(t, t, tt);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      rr += __shfl_xor_sync(kFull, rr, o);
      tt += __shfl_xor_sync(kFull, tt, o);
    }
    const bool bad = isnan(rr) || isnan(tt);
    best_r = bad ? INFINITY : fmax(best_r, rr);
    best_t = bad ? INFINITY : fmax(best_t, tt);
  }
  if (lane == 0) {
    const double pad = 1.0 + 0x1p-36;  // > 1 + dim_pad 2^-53 for dim_pad < 2^17
    atomicMax(reinterpret_cast<int*>(out), __float_as_int(__double2float_ru(__dsqrt_ru(__dmul_ru(best_r, pad)))));
    atomicMax(reinterpret_cast<int*>(out + 1),
              __float_as_int(__double2float_ru(__dsqrt_ru(__dmul_ru(best_t, pad)))));
  }
}

template <int ITEMS>
cudaError_t launch_rescore_t(const RescoreParams& p, cudaStream_t stream) {
  const size_t smem = sizeof(float) * (size_t(p.dim_pad) + kWarps * 32 * kTileLd) +
                      sizeof(uint64_t) * ITEMS * 32 + sizeof(float) * kWarps;
  cudaError_t e = cudaFuncSetAttribute(rescore_kernel<ITEMS>,
                                       cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) return e;
  rescore_kernel<ITEMS><<<unsigned(p.B), kWarps * 32, smem, stream>>>(p);
  return cudaGetLastError();
}


template <int ITEMS>
cudaError_t launch_select_t(const RescoreParams& p, const uint64_t* tmp, int n_groups, cudaStream_t stream) {
  rescore_select_kernel<ITEMS><<<unsigned((p.B + 3) / 4), 128, 0, stream>>>(p, tmp, n_groups);
  return cudaGetLastError();
}

// experiment switches B200KNN_RESCORE_CHUNK=64|128 (columns per stage; 64 = two chains per lane) and B200KNN_RESCORE_STAGES=2|3
int dot_chunk() {
  static int v = 0;
  if (v == 0) {
    const char* e = getenv("B200KNN_RESCORE_CHUNK");
    v = (e != nullptr && atoi(e) == 128) ? 128 : 64;
  }
  return v;
}
int dot_rows() {
  static int v = 0;
  if (v == 0) {
    const char* e = getenv("B200KNN_RESCORE_ROWS");
    v = (e != nullptr && atoi(e) == 2) ? 2 : 1;
  }
  return v;
}
int dot_stages() {
  static int v = 0;
  if (v == 0) {
    const char* e = getenv("B200KNN_RESCORE_STAGES");
    const int x = e != nullptr ? atoi(e) : 0;
    v = (x == 3) ? 3 : 2;
  }
  return v;
}

// The norms cert_bound takes for one fp32 query row, computed by a whole warp: qn = ||q|| (the select
// kernel's fp32 sum of squares, so that E is the certificate's E) and, when the bank's fp16 residuals
// are given, qtn = ||f16(q)|| and rho = ||q - f16(q)|| (0 otherwise); each inflated for its rounding.
__device__ __forceinline__ void query_norms(const RescoreParams& p, const float* qrow, int lane, float* qn,
                                            float* qtn, float* rho) {
  const bool resid = p.bank_resid != nullptr;
  float qq = 0.0f;
  // ||f16(q)||^2 and ||q - f16(q)||^2 in fp64: the squares are exact and cannot underflow
  double tt = 0.0, rr = 0.0;
  for (int d = lane; d < p.dim; d += 32) {
    const float v = qrow[d];
    qq = fmaf(v, v, qq);
    if (resid) {
      const double t = __half2float(f16_operand(v)), r = double(v) - t;  // exact below the max_abs range
      tt = fma(t, t, tt);
      rr = fma(r, r, rr);
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) qq += __shfl_xor_sync(kFull, qq, o);
  *qtn = 0.0f;
  *rho = 0.0f;
  if (resid) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      tt += __shfl_xor_sync(kFull, tt, o);
      rr += __shfl_xor_sync(kFull, rr, o);
    }
    *qtn = __double2float_ru(sqrt(tt)) * 1.001f;
    *rho = __double2float_ru(sqrt(rr)) * 1.001f;
  }
  *qn = sqrtf(qq) * 1.001f;
}

// The largest fp32 value strictly below the exact real t - e (fp32 t, e >= 0): the rounded-down
// difference when the subtraction is inexact (it is then below the exact value), else the next
// value below the exact difference.
__device__ __forceinline__ float below_difference(float t, float e) {
  const float lo = __fsub_rd(t, e), hi = __fsub_ru(t, e);
  return lo == hi ? nextafterf(lo, -INFINITY) : lo;
}

// Admission thresholds of a radius search (b200knn_radius_tau0), one warp per fp32 query row:
// tau0[b] = the largest fp32 strictly below tau - E_b, E_b = cert_bound of the row.  Every column
// whose exact similarity is >= tau then has an approximate one > tau0[b], since |a - s| <= E_b.
// Rows the bound does not cover (operand range max_abs, non-finite E) get refused[b] = 1 and
// tau0[b] = +inf, which admits no column.  e_out (optional): E_b itself.
__global__ void __launch_bounds__(128)
    radius_tau0_kernel(RescoreParams p, float tau, float* __restrict__ tau0, int32_t* __restrict__ refused,
                       float* __restrict__ e_out) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = int64_t(blockIdx.x) * 4 + warp;
  if (b >= p.B) return;
  float qn, qtn, rho;
  query_norms(p, static_cast<const float*>(p.q) + b * p.q_ld, lane, &qn, &qtn, &rho);
  const float m = *p.bank_max_norm;
  const float e = cert_bound(p, qn, qtn, rho);
  const bool ok = isfinite(e) && !(p.max_abs > 0.0f && !(qn < p.max_abs && m < p.max_abs));
  if (lane == 0) {
    tau0[b] = ok ? below_difference(tau, e) : INFINITY;
    refused[b] = ok ? 0 : 1;
    if (e_out != nullptr) e_out[b] = e;
  }
}

// ------------------------------------------------------------------ certified class vote (DESIGN §4.1c)
// knn_predict needs the class ranking, not the neighbour keys.  Per query (warp), with the
// approximate candidates a_1 >= ... >= a_m (m = k_in) and the row's certificate bound E:
//   S    = {i <= k : a_i > a_{k+1} + 2E}  (p = |S|): certainly in the exact top k (a_{k+1} := a_m
//          when k = m; every row outside the list has s <= a_m + E);
//   band = c_{p+1} .. c_r,  r = #{i : a_i + E >= a_k - E}: the only candidates re-scored.
// band_kernel writes the band front-filled (zero tail) into `band` (B, k_in), the list format the
// dot kernel reads, and info[b] = (p, r, E bits, 0); p = -1 marks a row it cannot serve (starved
// list, operand range, non-finite E), whose band is empty.
__global__ void __launch_bounds__(128)
    band_kernel(RescoreParams p, uint64_t* __restrict__ band, int4* __restrict__ info) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int64_t b = int64_t(blockIdx.x) * 4 + warp;
  if (b >= p.B) return;
  const uint64_t* cand = p.cand + b * p.k_in;
  float qn, qtn, rho;
  query_norms(p, static_cast<const float*>(p.q) + b * p.q_ld, lane, &qn, &qtn, &rho);
  const float m = *p.bank_max_norm;
  const float e = cert_bound(p, qn, qtn, rho);
  const bool ok = cand[p.k_in - 1] != 0ull && isfinite(e) &&
                  !(p.max_abs > 0.0f && !(qn < p.max_abs && m < p.max_abs));
  int n_s = -1, r = 0;
  if (ok) {
    const double E = e;
    const double ak = key_sim(cand[p.k_out - 1]);
    const double ak1 = key_sim(cand[p.k_out < p.k_in ? p.k_out : p.k_in - 1]);
    n_s = 0;
    for (int j0 = 0; j0 < p.k_in; j0 += 32) {
      const int j = j0 + lane;
      const double a = j < p.k_in ? double(key_sim(cand[j])) : -INFINITY;
      n_s += __popc(__ballot_sync(kFull, j < p.k_out && a > ak1 + 2.0 * E));
      r += __popc(__ballot_sync(kFull, a + E >= ak - E));
    }
  }
  uint64_t* o = band + b * p.k_in;
  for (int j = lane; j < p.k_in; j += 32) o[j] = (ok && j < r - n_s) ? cand[n_s + j] : 0ull;
  if (lane == 0) info[b] = make_int4(n_s, r, __float_as_int(e), 0);
}

// The exact keys of the band (tmp, from the dot kernel over `band`) -> the class ranking, when it
// is certified; otherwise uncertified[b] = 1 and *n_uncertified counts the row (pred row unset).
//  set:     the (k-p)-th exact band key must beat a_{r+1} + E (a_m + E when r = m): then S and the
//           best k - p of the band are the exact top k (today's certificate, applied to the band);
//  ranking: S members vote with the interval [exp((a-E)/t), exp((a+E)/t)] (ends swapped for
//           t < 0), the chosen band members with vote_kernel's exact exp(double(s)/t); intervals
//           are padded for the fp64 rounding of division, exp and summation (any order), and the
//           ranking is certified when the intervals of the present classes are pairwise disjoint
//           and each has a positive, finite lower / upper end.  Absent classes score exactly 0
//           and follow in class order, as in vote_kernel.  A certified ranking is vote_kernel's
//           ranking of the exact top k, element for element.
// Label / index errors of a row whose set is certified go to status[0] as in vote_kernel.
template <int ITEMS>
__global__ void __launch_bounds__(128)
    rescore_vote_kernel(RescoreParams p, const uint64_t* __restrict__ tmp, int n_groups,
                        const int4* __restrict__ info, const int64_t* __restrict__ labels, int64_t n_labels,
                        int C, double t, int64_t* __restrict__ pred, int32_t* __restrict__ status) {
  extern __shared__ __align__(16) unsigned char cv_smem[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  double* lo = reinterpret_cast<double*>(cv_smem) + size_t(warp) * 2 * C;
  double* hi = lo + C;
  int* cnt = reinterpret_cast<int*>(reinterpret_cast<double*>(cv_smem) + size_t(4) * 2 * C) + warp * C;
  const int64_t b = int64_t(blockIdx.x) * 4 + warp;
  if (b >= p.B) return;
  const int4 in = info[b];
  const int n_s = in.x, r = in.y;
  const float e = __int_as_float(in.z);
  const int k = p.k_out;
  const uint64_t* cand = p.cand + b * p.k_in;
  auto fail = [&]() {
    if (lane == 0) {
      p.uncertified[b] = 1;
      atomicAdd(p.n_uncertified, 1);
    }
  };
  if (n_s < 0) return fail();
  const int nb = r - n_s, need = k - n_s;
  uint64_t v[ITEMS];
  int groups = 0;
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) {
    const int c = i * 32 + lane;
    const bool has = c < nb;
    v[i] = has ? tmp[b * n_groups * 32 + c] : 0ull;
    if (__any_sync(kFull, has)) groups = i + 1;
  }
  sort_groups<ITEMS>(v, groups, lane);
  if (need > 0) {
    uint64_t kth = 0;
#pragma unroll
    for (int i = 0; i < ITEMS; ++i) kth = (i * 32 + lane == need - 1) ? v[i] : kth;
    kth = __shfl_sync(kFull, kth, (need - 1) & 31);
    const double bound = double(key_sim(cand[r < p.k_in ? r : p.k_in - 1])) + double(e);
    if (kth == 0ull || !(double(key_sim(kth)) > bound)) return fail();
  }

  for (int c = lane; c < C; c += 32) {
    lo[c] = 0.0;
    hi[c] = 0.0;
    cnt[c] = 0;
  }
  __syncwarp();
  auto add = [&](uint64_t key, double wl, double wh) {
    const int64_t li = key_idx(key) - p.idx_offset;
    if (li >= 0 && li < n_labels) {
      const int64_t c = labels[li];
      if (c >= 0 && c < C) {
        atomicAdd(&lo[c], wl);
        atomicAdd(&hi[c], wh);
        atomicAdd(&cnt[c], 1);
      } else {
        atomicExch(status, 1);
      }
    } else {
      atomicExch(status, 2);
    }
  };
  for (int i = lane; i < n_s; i += 32) {
    const uint64_t key = cand[i];
    const double a = key_sim(key);
    const double x1 = (a - double(e)) / t, x2 = (a + double(e)) / t;
    const double pad = (fabs(x1) + fabs(x2)) * 0x1p-48;  // rounding of a -+ E, of the division
    add(key, exp(fmin(x1, x2) - pad) * (1.0 - 0x1p-48), exp(fmax(x1, x2) + pad) * (1.0 + 0x1p-48));
  }
#pragma unroll
  for (int i = 0; i < ITEMS; ++i) {
    if (i * 32 + lane < need) {
      const double w = exp(double(key_sim(v[i])) / t);  // vote_kernel's weight
      add(v[i], w, w);
    }
  }
  __syncwarp();
  const double widen = double(k + 8) * 0x1p-48;  // fp64 sums of <= k positive terms, any order
  bool good = true;
  int n_present = 0;
  for (int c = 0; c < C; ++c) n_present += cnt[c] != 0;
  for (int c = lane; c < C; c += 32) {
    if (cnt[c] == 0) continue;
    const double l = lo[c] * (1.0 - widen), h = hi[c] * (1.0 + widen);
    if (!(l >= 2.2250738585072014e-308) || !(h < INFINITY)) good = false;
    for (int o = 0; o < C; ++o) {
      if (o == c || cnt[o] == 0) continue;
      if (!(l > hi[o] * (1.0 + widen) || lo[o] * (1.0 - widen) > h)) good = false;
    }
  }
  if (!__all_sync(kFull, good)) return fail();
  int64_t* out = pred + b * C;
  for (int c = lane; c < C; c += 32) {
    int rank = 0;
    if (cnt[c] != 0) {
      const double h = hi[c] * (1.0 + widen);
      for (int o = 0; o < C; ++o) rank += (cnt[o] != 0 && lo[o] * (1.0 - widen) > h) ? 1 : 0;
    } else {
      rank = n_present;
      for (int o = 0; o < c; ++o) rank += cnt[o] == 0 ? 1 : 0;
    }
    out[rank] = c;
  }
  if (lane == 0) p.uncertified[b] = 0;
}

template <int ITEMS>
cudaError_t launch_rescore_vote_t(const RescoreParams& p, const uint64_t* tmp, int n_groups, const int4* info,
                                  const int64_t* labels, int64_t n_labels, int C, double t, int64_t* pred,
                                  int32_t* status, cudaStream_t stream) {
  const size_t smem = size_t(4) * C * (2 * sizeof(double) + sizeof(int));
  rescore_vote_kernel<ITEMS><<<unsigned((p.B + 3) / 4), 128, smem, stream>>>(p, tmp, n_groups, info, labels,
                                                                             n_labels, C, t, pred, status);
  return cudaGetLastError();
}

template <int CHUNK, int STAGES, int R>
cudaError_t launch_dot_t(const RescoreParams& p, uint64_t* tmp, cudaStream_t stream) {
  constexpr int kSmem = 232448 - 1024;
  const size_t per_warp = STAGES * (sizeof(DotStage<CHUNK, R>) + sizeof(uint64_t));
  int warps = int(kSmem / per_warp);
  if (warps > 12) warps = 12;
  if (warps < 1) return cudaErrorNotSupported;
  const int n_groups = ws_slots(p.k_in) / (32 * R);
  const int64_t n_units = p.B * n_groups;
  int64_t blocks = (n_units + warps - 1) / warps;
  if (blocks > 148) blocks = 148;
  const size_t smem = per_warp * warps;
  auto kern = rescore_dot_kernel<CHUNK, STAGES, R>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) return e;
  const uintptr_t qa = reinterpret_cast<uintptr_t>(p.q);
  const int q_vec16 = (qa % 16 == 0 && p.q_ld % 4 == 0) ? 1 : 0;
  kern<<<unsigned(blocks), warps * 32, smem, stream>>>(p, tmp, n_groups, n_units, q_vec16);
  return cudaGetLastError();
}

// the exact keys of p.cand's candidates into tmp (B, ws_slots(k_in)); the first empty 32-slot unit of
// a list ends its query
cudaError_t launch_dot(const RescoreParams& p, uint64_t* tmp, cudaStream_t stream) {
  const int ch = dot_chunk(), stg = dot_stages();
  // default: 64 columns x 32 candidates per stage, 11 warps per SM.  Measured at the north-star step
  // (74.5 GB of candidate rows, power-capped clocks): 128 columns / 6 warps 14.95 ms, 64 columns / 11 warps
  // 13.96 ms, 3-4 stages with fewer warps 19.6-26.2 ms, two fma chains per lane over 64 candidates x 64
  // columns (B200KNN_RESCORE_ROWS=2) 23.1 ms: the kernel is bound by the rate of its per-row bulk copies and
  // by how many warps keep them in flight, not by the dependent-fma latency.
  // small calls (the reference-shaped B = 64) are latency-bound chains of steps: fewer, larger steps
  const bool small_call = p.B * int64_t(ws_slots(p.k_in) / 32) < 148 * 12 * 8;
  if (dot_rows() == 2) return launch_dot_t<64, 2, 2>(p, tmp, stream);
  if ((ch == 128 || small_call) && stg == 2) return launch_dot_t<128, 2, 1>(p, tmp, stream);
  if (ch == 128) return launch_dot_t<128, 3, 1>(p, tmp, stream);
  if (stg == 3) return launch_dot_t<64, 3, 1>(p, tmp, stream);
  return launch_dot_t<64, 2, 1>(p, tmp, stream);
}
}  // namespace

size_t rescore_workspace_bytes(int64_t B, int k_in) { return size_t(B) * size_t(ws_slots(k_in)) * sizeof(uint64_t); }

cudaError_t launch_rescore(const RescoreParams& p, void* workspace, size_t workspace_bytes,
                           cudaStream_t stream) {
  if (p.B == 0) return cudaSuccess;
  const int items = (p.k_in + 31) / 32;
  const bool pipelined = workspace != nullptr && workspace_bytes >= rescore_workspace_bytes(p.B, p.k_in) &&
                         p.rows_b == nullptr && p.q_dtype == B200KNN_F32 &&
                         reinterpret_cast<uintptr_t>(p.rows_a) % 16 == 0;
  if (p.n_peers > 0 && !pipelined) return cudaErrorInvalidValue;  // the scatter lives in the pipelined variant
  if (pipelined) {
    uint64_t* tmp = static_cast<uint64_t*>(workspace);
    const cudaError_t e = launch_dot(p, tmp, stream);
    if (e != cudaSuccess) return e;
    const int g32 = ws_slots(p.k_in) / 32;  // 32-slot groups per query in the workspace (always even)
    if (g32 <= 2) return launch_select_t<2>(p, tmp, g32, stream);
    if (g32 <= 4) return launch_select_t<4>(p, tmp, g32, stream);
    if (g32 <= 8) return launch_select_t<8>(p, tmp, g32, stream);
    if (g32 <= 16) return launch_select_t<16>(p, tmp, g32, stream);
    if (g32 <= 32) return launch_select_t<32>(p, tmp, g32, stream);
    return cudaErrorInvalidValue;
  }
  if (items <= 2) return launch_rescore_t<2>(p, stream);
  if (items <= 4) return launch_rescore_t<4>(p, stream);
  if (items <= 8) return launch_rescore_t<8>(p, stream);
  if (items <= 16) return launch_rescore_t<16>(p, stream);
  if (items <= 32) return launch_rescore_t<32>(p, stream);
  return cudaErrorInvalidValue;
}

cudaError_t launch_rescore_vote(const RescoreParams& p, uint64_t* band, int32_t* info, const int64_t* labels,
                                int64_t n_labels, int C, double t, int64_t* pred, int32_t* status,
                                void* workspace, cudaStream_t stream) {
  if (p.B == 0) return cudaSuccess;
  int4* inf = reinterpret_cast<int4*>(info);
  band_kernel<<<unsigned((p.B + 3) / 4), 128, 0, stream>>>(p, band, inf);
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) return e;
  RescoreParams pb = p;
  pb.cand = band;
  uint64_t* tmp = static_cast<uint64_t*>(workspace);
  e = launch_dot(pb, tmp, stream);
  if (e != cudaSuccess) return e;
  const int g32 = ws_slots(p.k_in) / 32;
  if (g32 <= 2) return launch_rescore_vote_t<2>(p, tmp, g32, inf, labels, n_labels, C, t, pred, status, stream);
  if (g32 <= 4) return launch_rescore_vote_t<4>(p, tmp, g32, inf, labels, n_labels, C, t, pred, status, stream);
  if (g32 <= 8) return launch_rescore_vote_t<8>(p, tmp, g32, inf, labels, n_labels, C, t, pred, status, stream);
  if (g32 <= 16) return launch_rescore_vote_t<16>(p, tmp, g32, inf, labels, n_labels, C, t, pred, status, stream);
  if (g32 <= 32) return launch_rescore_vote_t<32>(p, tmp, g32, inf, labels, n_labels, C, t, pred, status, stream);
  return cudaErrorInvalidValue;
}

cudaError_t launch_radius_tau0(const RescoreParams& p, float tau, float* tau0, int32_t* refused, float* e_out,
                               cudaStream_t stream) {
  if (p.B == 0) return cudaSuccess;
  radius_tau0_kernel<<<unsigned((p.B + 3) / 4), 128, 0, stream>>>(p, tau, tau0, refused, e_out);
  return cudaGetLastError();
}

cudaError_t launch_certify(const RescoreParams& p, cudaStream_t stream) {
  if (p.B == 0) return cudaSuccess;
  certify_kernel<<<unsigned((p.B + 3) / 4), 128, 0, stream>>>(p);
  return cudaGetLastError();
}

cudaError_t launch_route_keys(const uint64_t* keys, int64_t n, int k, int64_t rows_per_shard, int G,
                              uint64_t* out, cudaStream_t stream) {
  if (n == 0) return cudaSuccess;
  route_keys_kernel<<<unsigned((n + 3) / 4), 128, 0, stream>>>(keys, n, k, rows_per_shard, G, out);
  return cudaGetLastError();
}

cudaError_t launch_row_norm_max(const float* a, const float* b, int64_t n, int dim_pad, float* out,
                                cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(out, 0, sizeof(float), stream);
  if (e != cudaSuccess) return e;
  if (n == 0) return cudaSuccess;
  const int blocks = int(n < 148 * 8 * 8 ? (n + 7) / 8 : 148 * 8);
  row_norm_max_kernel<<<blocks, 256, 0, stream>>>(a, b, n, dim_pad, out);
  return cudaGetLastError();
}

cudaError_t launch_row_f16_residual_max(const float* a, int64_t n, int dim_pad, float* out, cudaStream_t stream) {
  cudaError_t e = cudaMemsetAsync(out, 0, 2 * sizeof(float), stream);
  if (e != cudaSuccess) return e;
  if (n == 0) return cudaSuccess;
  const int blocks = int(n < 148 * 8 * 8 ? (n + 7) / 8 : 148 * 8);
  row_f16_residual_max_kernel<<<blocks, 256, 0, stream>>>(a, n, dim_pad, out);
  return cudaGetLastError();
}

}  // namespace b200knn
