// tc_topk_impl.cuh — MODE_BF16 / MODE_TF32X3: the fused similarity contraction +
// streaming per-row top-k on the sm_100a tensor cores.
//
// Replaces torch.mm(feature, feature_bank) + sim_matrix.topk(k) of lightly's
// knn_predict (reference call site src/ssl_wafermap/models/knn.py:91-98).  The
// (B,N) similarity matrix lives only in TMEM: one 128 x BLOCK_N fp32 tile at a
// time, double buffered, drained by the epilogue warps straight into the
// per-row candidate lists of common.cuh.
//
// CTA = 10 warps, one CTA per SM, persistent over work items
// (query tile of 128 rows) x (bank split):
//   warp 0  : TMA producer  (one elected lane)   global -> smem, SWIZZLE_128B
//   warp 1  : tcgen05.mma issuer (one lane); owns the TMEM allocation
//   warp 2-9: epilogue; warp w may only touch TMEM lanes 32*(w%4)..+31, so two
//             warps share each lane quarter and each owns 16 of its 32 query
//             rows (two warps per scheduler hide each other's latencies; the
//             selection code is latency-bound, measured CPI 8 with one warp).
// Candidate extraction is warp-cooperative: a row whose 32-column chunk holds a
// similarity above its threshold is staged through 128 B of shared memory so
// that lane j tests column j (one ballot, coalesced appends), instead of one
// thread walking its 32 registers through 32 divergent branches.
// Pipelines (mbarrier): smem stage full/empty (TMA <-> MMA), TMEM accumulator
// full/empty (MMA <-> epilogue), query tile full/empty (BF16 mode keeps the
// 128 x D query tile resident in smem for the whole work item).
//
// MODE_BF16  : operands bf16 K-major, kind::f16, UMMA 128 x BLOCK_N x 16.
// MODE_BF16X3: operands bf16 hi/lo split (prepare.cu), kind::f16; same three products per
//              k-step as TF32X3 at twice its MMA rate (~2^-16 relative operand error).
// MODE_F16X2 : queries fp16 (one array, resident like BF16), bank fp16 hi/lo split; per k-block
//              q*lo + q*hi, the two bank arrays streamed as alternating pipeline stages.  Runs
//              as CTA pairs like BF16: two MMAs per k-step instead of BF16X3's three, one-sided
//              operand error 2^-11 (the query rounding) — candidate generator of the default
//              "fp32" cascade.
// MODE_F16   : the BF16 kernel on fp16 operands (one array each): two-sided operand error 2^-10,
//              8x smaller than bf16's 2^-7 at the same speed — first level of the "fp32" cascade.
// MODE_TF32X3: operands fp32 hi/lo split (prepare.cu), kind::tf32, UMMA
//              128 x BLOCK_N x 8; per k-step  hi*lo + lo*hi + hi*hi  accumulate
//              into the same TMEM tile; A and B are both streamed per k-block.
// The full D is accumulated in one fixed order in one MMA chain (no split-K),
// so sim(q, n) does not depend on tiling, batch size, split or shard count.
// This header holds the kernel template and its launcher; every (mode, CTA-pair) combination is
// instantiated in its own translation unit (tc_inst_*.cu) so that the library builds in parallel.
#pragma once
#include <cuda.h>

#include <cstdlib>

#include "../../include/b200knn.h"
#include "common.cuh"
#include "kernels.h"
#include "ptx.cuh"

namespace b200knn {
namespace {

constexpr int kTileM = 128;
constexpr int kMaxStages = 12;
constexpr int kMaxAccBufs = 4;  // TMEM accumulator buffers: 512 columns / BLOCK_N
constexpr int kRowBytes = 128;                   // one swizzle row = one k-block of a vector
constexpr int kABlockBytes = kTileM * kRowBytes;  // 16 KB: 128 query rows x one k-block
#ifndef B200KNN_EPI_PER_QUARTER
#define B200KNN_EPI_PER_QUARTER 2
#endif
constexpr int kEpiPerQuarter = B200KNN_EPI_PER_QUARTER;  // epilogue warps per TMEM lane quarter
constexpr int kEpiWarps = 4 * kEpiPerQuarter;
constexpr int kRowsPerWarp = 32 / kEpiPerQuarter;
constexpr int kThreads = 64 + 32 * kEpiWarps;
constexpr int kSmemLimit = 232448;  // 227 KB
constexpr int kMaxPeers = 8;        // GPUs of one NVSwitch domain the fused exchange addresses
constexpr int kSampleR = 16;        // values kept per row by the SAMPLE variant (= its k)

struct alignas(16) Barriers {
  uint64_t full[kMaxStages];
  uint64_t empty[kMaxStages];
  uint64_t tmem_full[kMaxAccBufs];
  uint64_t tmem_empty[kMaxAccBufs];
  uint64_t q_full;
  uint64_t q_empty;
  uint32_t tmem_base;
  uint32_t pad;
};

struct TcKernelArgs {
  int64_t B, N;
  int k;
  int n_kblocks;  // D_pad / elements-per-128B-row
  int n_stages;
  int64_t idx_offset;
  int64_t n_qtiles, n_items, split_rows;  // n_qtiles counts 128-row tiles (256-row tile pairs when PAIR)
  // Chunk-major order (n_chunks > 1; only with one bank split): a worker keeps up to `slots` query
  // tiles "open" at once and scans the bank chunk by chunk — every open tile over chunk 0, then
  // every open tile over chunk 1, ... — so the chunk being scanned (sized to stay in L2) is read
  // from HBM once per group of tiles instead of once per tile per drifting worker.  The per-row
  // selection state (threshold, list fill) of a tile survives between its chunks in st_tau /
  // st_cnt, its list in the worker's slot of `lists`.
  int n_chunks, slots;
  int64_t chunk_rows;
  float* st_tau;     // (B,)
  uint32_t* st_cnt;  // (B,)
  uint64_t* lists;
  uint64_t* out;
  const float* tau0;  // optional (B,) initial admission thresholds (nullptr: -inf)
  // Fused exchange (sharded mode): when n_peers > 0 the finished keys of query row g are stored
  // straight into the exchange buffer of the GPU that owns that query (peer memory over
  // NVLink), at [my_rank][g - owner*rows_per_owner][:], instead of into `out`.
  uint64_t* peer_out[kMaxPeers];
  int n_peers, my_rank;
  int64_t rows_per_owner;
  float* dump;  // optional (B, N) fp32 similarity dump for unit tests (nullptr in production)
  int32_t* diag;
  int flags;    // experiment switches of the debug entry point (0 in production):
                // 1 no selection, 2 no TMEM loads, 4 no MMA issue, 8 no bank TMA loads
  // EXCL: group ids of the query rows, (B,), and of the bank rows of this launch, (N,) indexed
  // before idx_offset; a column whose id equals its query row's id is never admitted to its list
  const int32_t* q_gid;
  const int32_t* bank_gid;
};

// PAIR: two CTAs of a cluster (one TPC) run one tcgen05.mma.cta_group::2 per k-step:
// M = 256 (each CTA's own resident 128-row query tile), N = BLOCK_N with each CTA
// loading HALF of the bank tile.  Per SM that halves the bank bytes pulled from L2
// per MMA cycle and doubles the number of pipeline stages the same smem buys — the
// 1-CTA kernel was bound by exactly that (3 stages of 32 KB, ~15 TB/s of L2->SM
// reads chip-wide; profiles/r01_call10_*).  The leader CTA (cluster rank 0) owns the
// barriers the MMA thread waits on (smem full, query full, TMEM empty); both CTAs'
// TMA transactions and epilogue arrivals are routed there, and the leader's commits
// are multicast to both CTAs' smem-empty / TMEM-full / query-empty barriers.
//
// SAMPLE: the sampling pre-pass.  Only a threshold is wanted: each row's thread keeps the 16
// best CHUNK MAXIMA (one value per 32 sampled columns) in registers, branch-free sorted
// insert — no candidate lists, no prunes, no indices.  Its 16-th value is <= the 16-th best
// sampled similarity, which is all the main pass's admission threshold needs.  The general
// list machinery spent 2/3 of the pre-pass warming up its lists.
//
// EXCL: group exclusion (product builds only, never with DEBUG or SAMPLE).  Only the hit path of
// the epilogue changes: an excluded column can turn a miss into a false hit, never the reverse, so
// the no-hit test stays as it is and the qualifying columns of a hit are filtered by their group
// ids (gathered from the L2-resident id array) before they are appended.
// One unit of work of a worker: query tile `qt` against bank rows [n_begin, n_end).
struct WorkItem {
  int64_t qt, sp, n_begin, n_end;
  int slot;          // which of the worker's list slots the tile's lists live in
  bool first, last;  // first / last visit of this tile (start from tau0 / flush the result)
};

// The sequence of work items of `worker` — identical for the producer, the MMA issuer and the
// epilogue warps, which is what keeps their barrier phases aligned.
template <typename F>
__device__ __forceinline__ void for_each_item(const TcKernelArgs& a, int64_t worker, int64_t n_workers, F&& body) {
  // Items are numbered split-major (item = sp * n_qtiles + qt) and dealt round-robin to the
  // workers, so concurrently running workers stream the same bank split.  Without chunks
  // (n_chunks == 1, slots == 1, chunk_rows == split_rows) this is one pass over the worker's items;
  // with chunks (one split only) the worker's tiles are taken in groups of `slots`, each group
  // scanned chunk by chunk.  ONE call site of `body` (it is large and must not be duplicated).
  const int64_t n_units = worker < a.n_items ? (a.n_items - worker + n_workers - 1) / n_workers : 0;
  WorkItem it;
  for (int64_t g0 = 0; g0 < n_units; g0 += a.slots) {
    const int glen = int(n_units - g0 < a.slots ? n_units - g0 : a.slots);
    for (int c = 0; c < a.n_chunks; ++c) {
      it.first = (c == 0);
      it.last = (c == a.n_chunks - 1);
      for (int j = 0; j < glen; ++j) {
        const int64_t item = worker + (g0 + j) * n_workers;
        it.qt = item % a.n_qtiles;
        it.sp = item / a.n_qtiles;
        const int64_t base = it.sp * a.split_rows;
        const int64_t span_end = (base + a.split_rows < a.N) ? base + a.split_rows : a.N;
        it.n_begin = base + int64_t(c) * a.chunk_rows;
        it.n_end = (it.n_begin + a.chunk_rows < span_end) ? it.n_begin + a.chunk_rows : span_end;
        it.slot = j;
        body(it);
      }
    }
  }
}

template <int MODE, int BLOCK_N, int ITEMS, bool DEBUG, bool PAIR, bool SAMPLE, bool EXCL>
__global__ void __launch_bounds__(kThreads, 1)
    tc_topk_kernel(const __grid_constant__ CUtensorMap map_q_hi,
                   const __grid_constant__ CUtensorMap map_q_lo,
                   const __grid_constant__ CUtensorMap map_b_hi,
                   const __grid_constant__ CUtensorMap map_b_lo, const TcKernelArgs a) {
  // query tile resident in smem, only bank tiles are streamed (BF16, F16X2)
  constexpr bool kBf16 = (MODE == B200KNN_MODE_BF16 || MODE == B200KNN_MODE_F16X2 || MODE == B200KNN_MODE_F16);
  constexpr int kBArrays = (MODE == B200KNN_MODE_F16X2) ? 2 : 1;  // bank arrays streamed per k-block (lo, hi)
  constexpr bool kHalf = (MODE != B200KNN_MODE_TF32X3);   // 2-byte elements (kind::f16)
  static_assert(!PAIR || kBf16, "CTA pairs are implemented for the resident-query modes");
  static_assert(!EXCL || (!DEBUG && !SAMPLE), "group exclusion is a product-build variant");
  constexpr int CAP = ITEMS * 32;
  constexpr int kCtas = PAIR ? 2 : 1;
  constexpr int kBRows = BLOCK_N / kCtas;  // bank rows of one tile this CTA loads
  constexpr int kBBlockBytes = kBRows * kRowBytes;
  constexpr int kStageBytes = kBf16 ? kBBlockBytes : 2 * (kABlockBytes + kBBlockBytes);
  constexpr int kElemsPerRow = kHalf ? 64 : 32;  // elements of one 128-byte k-block row
  constexpr int kUmmaKBytes = 32;                // one MMA consumes 32 bytes of k per row
  constexpr uint32_t kIdesc =
      ptx::make_idesc((MODE == B200KNN_MODE_F16X2 || MODE == B200KNN_MODE_F16) ? 0u : (kHalf ? 1u : 2u),
                      kTileM * kCtas, BLOCK_N);
  // all 512 TMEM columns: 2 accumulator buffers of 256 columns, or 4 of 128.  More buffers let the
  // MMA issuer run further ahead of the slowest of the 16 epilogue warps it hands tiles to (a warp
  // that prunes a list is late for a whole tile time).
  constexpr int kAccBufs = 512 / BLOCK_N;
  static_assert(kAccBufs >= 2 && kAccBufs <= kMaxAccBufs, "BLOCK_N must be 128 or 256");
  constexpr uint32_t kTmemCols = 512;

  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                             ~uintptr_t(1023));
  const int q_bytes = kBf16 ? a.n_kblocks * kABlockBytes : 0;
  uint8_t* q_smem = smem;
  uint8_t* stage_smem = smem + q_bytes;
  Barriers* bars = reinterpret_cast<Barriers*>(stage_smem + size_t(a.n_stages) * kStageBytes);

  // warp index through a shuffle so the compiler knows it is warp-uniform (role code then
  // lives in uniform registers instead of being re-broadcast around every TMA/MMA instruction)
  const int warp = __shfl_sync(kFull, int(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const uint32_t cta_rank = PAIR ? ptx::cluster_ctarank() : 0u;
  const bool leader = (cta_rank == 0);
  const int64_t worker = PAIR ? int64_t(blockIdx.x >> 1) : int64_t(blockIdx.x);
  const int64_t n_workers = PAIR ? int64_t(gridDim.x >> 1) : int64_t(gridDim.x);

  if (warp == 0 && lane == 0) {
    ptx::prefetch_tensormap(&map_q_hi);
    ptx::prefetch_tensormap(&map_b_hi);
    if (!kBf16) ptx::prefetch_tensormap(&map_q_lo);
    if (!kBf16 || kBArrays == 2) ptx::prefetch_tensormap(&map_b_lo);
    for (int s = 0; s < a.n_stages; ++s) {
      ptx::mbar_init(ptx::smem_u32(&bars->full[s]), 1);
      ptx::mbar_init(ptx::smem_u32(&bars->empty[s]), 1);
    }
    for (int b = 0; b < kAccBufs; ++b) {
      ptx::mbar_init(ptx::smem_u32(&bars->tmem_full[b]), 1);
      // one arrive per epilogue warp (of both CTAs of a pair: the leader's barrier collects them)
      ptx::mbar_init(ptx::smem_u32(&bars->tmem_empty[b]), kEpiWarps * kCtas);
    }
    ptx::mbar_init(ptx::smem_u32(&bars->q_full), 1);
    ptx::mbar_init(ptx::smem_u32(&bars->q_empty), 1);
    ptx::fence_barrier_init();
  }
  if (warp == 1) {
    if (PAIR) {
      ptx::tmem_alloc_pair(ptx::smem_u32(&bars->tmem_base), kTmemCols);
      ptx::tmem_relinquish_pair();
    } else {
      ptx::tmem_alloc(ptx::smem_u32(&bars->tmem_base), kTmemCols);
      ptx::tmem_relinquish();
    }
  }
  ptx::tc_fence_before();
  if (PAIR) ptx::cluster_sync(); else __syncthreads();
  ptx::tc_fence_after();
  const uint32_t tmem_base = bars->tmem_base;

  if (warp == 0) {
    // ------------------------------------------------------------ TMA producer
    // The whole warp runs the (uniform) loop and waits; one elected lane issues.
    {
      int stage = 0;
      uint32_t phase = 0, q_phase = 0;
      const uint32_t qbar = PAIR ? ptx::mapa(ptx::smem_u32(&bars->q_full), 0) : ptx::smem_u32(&bars->q_full);
      for_each_item(a, worker, n_workers, [&](const WorkItem& it) {
        const int m0 = int((it.qt * kCtas + cta_rank) * kTileM);
        const int64_t n_begin = it.n_begin, n_end = it.n_end;
        if (kBf16) {
          ptx::mbar_wait(ptx::smem_u32(&bars->q_empty), q_phase ^ 1, a.diag, 1);
          if (ptx::elect_one()) {
            if (leader) ptx::mbar_expect_tx(ptx::smem_u32(&bars->q_full), uint32_t(q_bytes) * kCtas);
            for (int kb = 0; kb < a.n_kblocks; ++kb) {
              if (PAIR)
                ptx::tma_load_2d_pair(ptx::smem_u32(q_smem + kb * kABlockBytes), &map_q_hi,
                                      kb * kElemsPerRow, m0, qbar);
              else
                ptx::tma_load_2d(ptx::smem_u32(q_smem + kb * kABlockBytes), &map_q_hi,
                                 kb * kElemsPerRow, m0, qbar);
            }
          }
          __syncwarp();
          q_phase ^= 1;
        }
        for (int64_t n0 = n_begin; n0 < n_end; n0 += BLOCK_N) {
          const int nrow = int(n0) + int(cta_rank) * kBRows;  // this CTA's half of the bank tile
          // resident-query modes: one pipeline stage per (k-block, bank array); F16X2 visits lo, hi
          for (int v = 0; v < a.n_kblocks * kBArrays; ++v) {
            const int kb = v / kBArrays;
            ptx::mbar_wait(ptx::smem_u32(&bars->empty[stage]), phase ^ 1, a.diag, 2);
            if (ptx::elect_one()) {
              const uint32_t full = ptx::smem_u32(&bars->full[stage]);
              const uint32_t st = ptx::smem_u32(stage_smem + size_t(stage) * kStageBytes);
              if (DEBUG && (a.flags & 8)) {
                if (leader) ptx::mbar_arrive(full);
              } else if (kBf16) {
                const CUtensorMap* mb = (kBArrays == 2 && (v & 1) == 0) ? &map_b_lo : &map_b_hi;
                if (leader) ptx::mbar_expect_tx(full, uint32_t(kStageBytes) * kCtas);
                if (PAIR)
                  ptx::tma_load_2d_pair(st, mb, kb * kElemsPerRow, nrow, ptx::mapa(full, 0));
                else
                  ptx::tma_load_2d(st, mb, kb * kElemsPerRow, nrow, full);
              } else {
                ptx::mbar_expect_tx(full, uint32_t(kStageBytes));
                ptx::tma_load_2d(st, &map_q_hi, kb * kElemsPerRow, m0, full);
                ptx::tma_load_2d(st + kABlockBytes, &map_q_lo, kb * kElemsPerRow, m0, full);
                ptx::tma_load_2d(st + 2 * kABlockBytes, &map_b_hi, kb * kElemsPerRow, nrow, full);
                ptx::tma_load_2d(st + 2 * kABlockBytes + kBBlockBytes, &map_b_lo, kb * kElemsPerRow,
                                 nrow, full);
              }
            }
            __syncwarp();
            if (++stage == a.n_stages) {
              stage = 0;
              phase ^= 1;
            }
          }
        }
      });
    }
  } else if (warp == 1) {
    // -------------------------------------------------------------- MMA issuer
    // Warp-uniform loop (all lanes wait on the barriers); one elected lane issues the MMAs
    // and commits.  Descriptors differ only in their 14-bit address field.
    if (leader) {
      int stage = 0;
      uint32_t phase = 0, q_phase = 0;
      uint32_t tcount = 0;
      const uint64_t desc0 = ptx::smem_desc_sw128(0);
      const uint32_t q_base = ptx::smem_u32(q_smem), st_base = ptx::smem_u32(stage_smem);
      for_each_item(a, worker, n_workers, [&](const WorkItem& it) {
        const int64_t n_begin = it.n_begin, n_end = it.n_end;
        if (kBf16) {
          ptx::mbar_wait(ptx::smem_u32(&bars->q_full), q_phase, a.diag, 3);
          q_phase ^= 1;
        }
        for (int64_t n0 = n_begin; n0 < n_end; n0 += BLOCK_N) {
          const uint32_t buf = tcount % kAccBufs, aphase = (tcount / kAccBufs) & 1u;
          ptx::mbar_wait(ptx::smem_u32(&bars->tmem_empty[buf]), aphase ^ 1, a.diag, 4);
          ptx::tc_fence_after();
          const uint32_t tmem_d = tmem_base + buf * BLOCK_N;
          for (int v = 0; v < a.n_kblocks * kBArrays; ++v) {
            const int kb = v / kBArrays;
            ptx::mbar_wait(ptx::smem_u32(&bars->full[stage]), phase, a.diag, 5);
            ptx::tc_fence_after();
            if (ptx::elect_one()) {
              const uint32_t st = st_base + uint32_t(stage) * uint32_t(kStageBytes);
              if (DEBUG && (a.flags & 4)) {
              } else if (kBf16) {
                const uint64_t da = desc0 + uint64_t(((q_base + uint32_t(kb) * kABlockBytes) & 0x3FFFFu) >> 4);
                const uint64_t db = desc0 + uint64_t((st & 0x3FFFFu) >> 4);
#pragma unroll
                for (int ks = 0; ks < kRowBytes / kUmmaKBytes; ++ks) {
                  const uint64_t o = uint64_t((ks * kUmmaKBytes) >> 4);
                  if (PAIR)
                    ptx::umma_f16_pair(tmem_d, da + o, db + o, kIdesc, uint32_t((v | ks) != 0));
                  else
                    ptx::umma_f16(tmem_d, da + o, db + o, kIdesc, uint32_t((v | ks) != 0));
                }
              } else {
                const uint64_t a_hi = desc0 + uint64_t((st & 0x3FFFFu) >> 4);
                const uint64_t a_lo = a_hi + uint64_t(kABlockBytes >> 4);
                const uint64_t b_hi = a_hi + uint64_t((2 * kABlockBytes) >> 4);
                const uint64_t b_lo = b_hi + uint64_t(kBBlockBytes >> 4);
#pragma unroll
                for (int ks = 0; ks < kRowBytes / kUmmaKBytes; ++ks) {
                  const uint64_t o = uint64_t((ks * kUmmaKBytes) >> 4);
                  if (kHalf) {  // BF16X3: bf16 hi/lo split, same three products at the bf16 rate
                    ptx::umma_f16(tmem_d, a_hi + o, b_lo + o, kIdesc, uint32_t((kb | ks) != 0));
                    ptx::umma_f16(tmem_d, a_lo + o, b_hi + o, kIdesc, 1u);
                    ptx::umma_f16(tmem_d, a_hi + o, b_hi + o, kIdesc, 1u);
                  } else {
                    ptx::umma_tf32(tmem_d, a_hi + o, b_lo + o, kIdesc, uint32_t((kb | ks) != 0));
                    ptx::umma_tf32(tmem_d, a_lo + o, b_hi + o, kIdesc, 1u);
                    ptx::umma_tf32(tmem_d, a_hi + o, b_hi + o, kIdesc, 1u);
                  }
                }
              }
              // frees the smem stage (in both CTAs of a pair)
              if (PAIR) ptx::umma_commit_pair(ptx::smem_u32(&bars->empty[stage]), 3);
              else ptx::umma_commit(ptx::smem_u32(&bars->empty[stage]));
              if (v + 1 == a.n_kblocks * kBArrays) {  // accumulator ready
                if (PAIR) ptx::umma_commit_pair(ptx::smem_u32(&bars->tmem_full[buf]), 3);
                else ptx::umma_commit(ptx::smem_u32(&bars->tmem_full[buf]));
              }
            }
            __syncwarp();
            if (++stage == a.n_stages) {
              stage = 0;
              phase ^= 1;
            }
          }
          ++tcount;
        }
        if (kBf16) {  // query tile reusable
          if (ptx::elect_one()) {
            if (PAIR) ptx::umma_commit_pair(ptx::smem_u32(&bars->q_empty), 3);
            else ptx::umma_commit(ptx::smem_u32(&bars->q_empty));
          }
          __syncwarp();
        }
      });
    }
  } else {
    // ---------------------------------------------------------------- epilogue
    const int quarter = warp & 3;             // TMEM lane quarter this warp may access
    const int sub = (warp - 2) / 4;           // which of the quarter's warps
    const bool owner = (lane / kRowsPerWarp) == sub;  // this lane's row is selected by this warp
    const int row_in_tile = quarter * 32 + lane;
    const float neg_inf = __int_as_float(0xff800000);
    const float pos_inf = __int_as_float(0x7f800000);
    // the barrier the MMA thread waits on before overwriting an accumulator buffer
    const uint32_t tmem_empty_bar0 = PAIR ? ptx::mapa(ptx::smem_u32(&bars->tmem_empty[0]), 0)
                                          : ptx::smem_u32(&bars->tmem_empty[0]);
    // free slots below which a row is pruned between tiles (off the critical path)
    const int soft_slack = min(40, (CAP - a.k) / 2);
    uint32_t tcount = 0;
    for_each_item(a, worker, n_workers, [&](const WorkItem& it) {
      const int64_t sp = it.sp;
      const int64_t m0 = (it.qt * kCtas + cta_rank) * kTileM;
      const int64_t n_begin = it.n_begin, n_end = it.n_end;
      const int64_t grow = m0 + row_in_tile;
      uint64_t* warp_lists =
          a.lists + ((size_t(blockIdx.x) * size_t(a.slots) + size_t(it.slot)) * kTileM + size_t(quarter) * 32) * CAP;
      uint64_t* my_list = warp_lists + size_t(lane) * CAP;
      const bool mine = owner && grow < a.B;  // this lane selects for a real query row
      int32_t my_gid = 0;
      if constexpr (EXCL) my_gid = mine ? a.q_gid[grow] : 0;
      RowState st;
      if (it.first || SAMPLE) {
        st.cnt = 0;
        st.tau = mine ? (a.tau0 != nullptr ? a.tau0[grow] : neg_inf) : pos_inf;
      } else {  // resume this tile where its previous chunk left it
        st.cnt = mine ? a.st_cnt[grow] : 0u;
        st.tau = mine ? a.st_tau[grow] : pos_inf;
      }
      float top[SAMPLE ? kSampleR : 1];  // SAMPLE: this row's best similarities, descending
#pragma unroll
      for (int i = 0; i < (SAMPLE ? kSampleR : 1); ++i) top[i] = neg_inf;
      for (int64_t n0 = n_begin; n0 < n_end; n0 += BLOCK_N) {
        const uint32_t buf = tcount % kAccBufs, aphase = (tcount / kAccBufs) & 1u;
        ptx::mbar_wait(ptx::smem_u32(&bars->tmem_full[buf]), aphase, a.diag, 6);
        ptx::tc_fence_after();
        const uint32_t taddr = tmem_base + (uint32_t(quarter * 32) << 16) + buf * BLOCK_N;
#pragma unroll 1
        for (int c0 = 0; c0 < BLOCK_N; c0 += 32) {
          float s[32];
          if (DEBUG && (a.flags & 2)) {
#pragma unroll
            for (int j = 0; j < 32; ++j) s[j] = neg_inf;
          } else {
            ptx::tmem_ld32(taddr + c0, s);
          }
          if (c0 + 32 == BLOCK_N) {
            // all of this warp's TMEM reads of the buffer are done: hand it back
            ptx::tc_fence_before();
            __syncwarp();
            if (lane == 0) {
              const uint32_t bar = tmem_empty_bar0 + buf * uint32_t(sizeof(uint64_t));  // same offset in the leader's smem
              if (PAIR) ptx::mbar_arrive_cluster(bar);
              else ptx::mbar_arrive(bar);
            }
          }
          if (DEBUG && a.dump != nullptr && owner && grow < a.B) {
#pragma unroll
            for (int j = 0; j < 32; ++j) {
              const int64_t gn = n0 + c0 + j;
              if (gn < n_end) a.dump[grow * a.N + gn] = s[j];
            }
          }
          if (n0 + c0 + 32 > n_end) {
            // ragged end of the split: columns past it (zero-filled by TMA) never qualify
            const int nv = int(n_end - (n0 + c0));
#pragma unroll
            for (int j = 0; j < 32; ++j)
              if (j >= nv) s[j] = neg_inf;
          }
          float m4[4] = {s[0], s[1], s[2], s[3]};
#pragma unroll
          for (int j = 4; j < 32; ++j) m4[j & 3] = fmaxf(m4[j & 3], s[j]);
          const float mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
          const bool hit = mx > st.tau;
          if (!__any_sync(kFull, hit) || (DEBUG && (a.flags & 1))) continue;
          // ---- some rows of this warp have candidates in this chunk.  Every such row's
          // thread appends its own candidates straight from its registers; rows proceed in
          // parallel, so the cost does not grow with the number of rows that hit.
          if (SAMPLE) {
            // Only the chunk maximum of a row is inserted.  The top-16 of a SUBSET of the
            // sample is still a valid (slightly lower) threshold, a second qualifying value in
            // the same 32 columns is rare after the first tiles, and the epilogue stays free
            // of per-column work: 32 min/max per hit, all hit rows in parallel.
            if (hit) {
              float x = mx;
#pragma unroll
              for (int i = 0; i < kSampleR; ++i) {
                const float hi = fmaxf(top[i], x);
                x = fminf(top[i], x);
                top[i] = hi;
              }
              st.tau = top[kSampleR - 1];  // only rows that can hit get here (others hold +inf)
            }
            continue;
          }
          if (hit) {
            // bit j of m: column j qualifies.  Only the column classes (j mod 4) whose partial
            // maximum qualifies are tested; no per-column branches.
            unsigned m = 0;
#pragma unroll
            for (int c = 0; c < 4; ++c) {
              if (m4[c] > st.tau) {
#pragma unroll
                for (int j = c; j < 32; j += 4) m |= (s[j] > st.tau) ? (1u << j) : 0u;
              }
            }
            const uint32_t gidx0 = uint32_t(n0 + c0 + a.idx_offset);
            bool one = (m & (m - 1u)) == 0u;
            if constexpr (EXCL) {
              // drop the qualifying columns of the row's own group; the row maximum may be one of
              // them, so a single survivor of a filtered mask takes the general path below
              const int32_t* g = a.bank_gid + (n0 + c0);
              unsigned keep = m;
              for (unsigned r = m; r != 0u; r &= r - 1u) {
                const int j = __ffs(r) - 1;
                if (__ldg(g + j) == my_gid) keep &= ~(1u << j);
              }
              one = one && keep == m;
              m = keep;
            }
            if (one) {
              // the common case, exactly one candidate: it is the row maximum
              my_list[st.cnt] = make_key(mx, gidx0 + uint32_t(__ffs(m) - 1));
              st.cnt += 1;
            } else {
              // several candidates: walk only the column classes that hold one (the list is
              // unordered until its prune / flush, so the class-major append order is immaterial)
              uint64_t* lp = my_list + st.cnt;
              uint32_t c = 0;
#pragma unroll
              for (int cl = 0; cl < 4; ++cl) {
                const unsigned mc = m & (0x11111111u << cl);
                if (mc != 0u) {
#pragma unroll
                  for (int j = cl; j < 32; j += 4) {
                    if ((mc >> j) & 1u) {
                      lp[c] = make_key(s[j], gidx0 + uint32_t(j));
                      ++c;
                    }
                  }
                }
              }
              st.cnt += c;
            }
          }
          __syncwarp();
          warp_maintain<ITEMS, true>(warp_lists, st, a.k, lane, 32);  // emergency only (list would overflow)
        }
        // The TMEM buffer went back to the MMA warp before the last chunk was processed:
        // prune here, off the accumulator's critical path, a little before it becomes mandatory.
        if (!SAMPLE) warp_maintain<ITEMS, true>(warp_lists, st, a.k, lane, soft_slack);
        ++tcount;
      }
      if (SAMPLE) {
        if (owner && grow < a.B) {
          uint64_t* o;
          if (a.n_peers > 0) {  // sharded threshold exchange: straight into the query owner's buffer
            const int64_t own = grow / a.rows_per_owner;
            o = a.peer_out[own] + (int64_t(a.my_rank) * a.rows_per_owner + (grow - own * a.rows_per_owner)) * kSampleR;
          } else {
            o = a.out + (size_t(sp) * a.B + grow) * kSampleR;
          }
#pragma unroll
          for (int i = 0; i < kSampleR; ++i) o[i] = top[i] > neg_inf ? make_key(top[i], 0u) : 0ull;
        }
        return;
      }
      if (!it.last) {  // more chunks of this tile to come: park the selection state
        if (mine) {
          a.st_cnt[grow] = st.cnt;
          a.st_tau[grow] = st.tau;
        }
        __syncwarp();  // this lane's list appends are read by the whole warp's prunes later
        return;
      }
      const int64_t row0 = m0 + quarter * 32;
      unsigned valid = 0;
      if (row0 < a.B) {
        const int64_t nv = a.B - row0;
        valid = nv >= 32 ? kFull : ((1u << nv) - 1u);
      }
      valid &= (kRowsPerWarp == 32 ? kFull : ((1u << kRowsPerWarp) - 1u)) << (sub * kRowsPerWarp);
      warp_flush<ITEMS>(warp_lists, st, a.k, lane, valid, [&](int r) -> uint64_t* {
        const int64_t g = row0 + r;
        if (a.n_peers > 0) {
          const int64_t owner = g / a.rows_per_owner;
          return a.peer_out[owner] +
                 (int64_t(a.my_rank) * a.rows_per_owner + (g - owner * a.rows_per_owner)) * a.k;
        }
        return a.out + (size_t(sp) * a.B + size_t(g)) * a.k;
      }, a.n_peers > 0 || a.n_items > a.n_qtiles);  // exchange buffers and bank splits are merged afterwards
    });
  }

  ptx::tc_fence_before();
  if (PAIR) ptx::cluster_sync(); else __syncthreads();
  if (warp == 1) {
    ptx::tc_fence_after();
    if (PAIR) ptx::tmem_dealloc_pair(tmem_base, kTmemCols);
    else ptx::tmem_dealloc(tmem_base, kTmemCols);
  }
}

// ------------------------------------------------------------------- host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode() {
  static EncodeTiledFn fn = nullptr;
  if (fn) return fn;
  void* p = nullptr;
  cudaDriverEntryPointQueryResult qres;
  if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) !=
          cudaSuccess ||
      qres != cudaDriverEntryPointSuccess)
    return nullptr;
  fn = reinterpret_cast<EncodeTiledFn>(p);
  return fn;
}

// rows x cols matrix of `esize`-byte elements, row pitch = cols*esize; box = box_rows x 128 bytes
bool make_map(CUtensorMap* m, const void* base, bool bf16, uint64_t rows, uint64_t cols,
              uint32_t box_rows, uint64_t row_stride = 1, bool fp16 = false) {
  EncodeTiledFn enc = get_encode();
  if (!enc) return false;
  const uint64_t esize = bf16 ? 2 : 4;
  cuuint64_t gdim[2] = {cols, rows};
  cuuint64_t gstride[1] = {cols * esize * row_stride};  // row_stride > 1: every row_stride-th row
  cuuint32_t box[2] = {cuuint32_t(kRowBytes / esize), box_rows};
  cuuint32_t estr[2] = {1, 1};
  CUresult r = enc(m, fp16 ? CU_TENSOR_MAP_DATA_TYPE_FLOAT16
                        : (bf16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT32), 2,
                   const_cast<void*>(base), gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                   CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  return r == CUDA_SUCCESS;
}

template <int MODE, int BLOCK_N, int ITEMS, bool DEBUG, bool PAIR, bool SAMPLE = false, bool EXCL = false>
cudaError_t launch_t(const TcParams& p, int grid, cudaStream_t stream, float* dump, int32_t* diag,
                     int flags, const char** why) {
  constexpr bool kBf16 = (MODE == B200KNN_MODE_BF16 || MODE == B200KNN_MODE_F16X2 ||
                          MODE == B200KNN_MODE_F16);  // resident query tile
  constexpr bool kF16 = (MODE == B200KNN_MODE_F16X2 || MODE == B200KNN_MODE_F16);  // fp16 tensor maps
  constexpr bool kTwoB = (MODE == B200KNN_MODE_F16X2);
  constexpr bool kHalf = (MODE != B200KNN_MODE_TF32X3);
  constexpr int kCtas = PAIR ? 2 : 1;
  constexpr int kBRows = BLOCK_N / kCtas;
  const int d_pad = (p.D + 63) / 64 * 64;
  const int elems_per_row = kHalf ? 64 : 32;
  TcKernelArgs a;
  a.B = p.B;
  a.N = p.N;
  a.k = p.k;
  a.n_kblocks = d_pad / elems_per_row;
  a.idx_offset = p.idx_offset;
  a.n_qtiles = p.n_qtiles;
  a.n_items = p.n_items;
  a.split_rows = p.split_rows;
  // the sampling variant keeps its row state in registers: always one chunk
  a.n_chunks = (SAMPLE || p.n_chunks < 1) ? 1 : p.n_chunks;
  a.slots = (SAMPLE || p.slots < 1) ? 1 : p.slots;
  a.chunk_rows = a.n_chunks > 1 ? p.chunk_rows : p.split_rows;
  a.st_tau = p.st_tau;
  a.st_cnt = p.st_cnt;
  a.lists = p.lists;
  a.out = p.out;
  a.tau0 = p.tau0;
  a.n_peers = p.n_peers;
  a.my_rank = p.my_rank;
  a.rows_per_owner = p.rows_per_owner;
  for (int g = 0; g < kMaxPeers; ++g) a.peer_out[g] = g < p.n_peers ? p.peer_out[g] : nullptr;
  a.dump = dump;
  a.diag = diag;
  a.flags = flags;
  a.q_gid = p.q_gid;
  a.bank_gid = p.bank_gid;
  const int b_block = kBRows * kRowBytes;
  const int stage_bytes = kBf16 ? b_block : 2 * (kABlockBytes + b_block);
  const int q_bytes = kBf16 ? a.n_kblocks * kABlockBytes : 0;
  const int fixed = q_bytes + int(sizeof(Barriers)) + 1024;  // 1024: manual alignment slack
  int stages = (kSmemLimit - fixed) / stage_bytes;
  if (stages > kMaxStages) stages = kMaxStages;
  if (stages < 2) {
    *why = "vector dimension too large for the resident query tile";
    return cudaErrorNotSupported;
  }
  a.n_stages = stages;
  const size_t smem = size_t(fixed) + size_t(stages) * stage_bytes;

  CUtensorMap mq_hi, mq_lo, mb_hi, mb_lo;
  bool ok = make_map(&mq_hi, p.q_hi, kHalf, uint64_t(p.B), uint64_t(d_pad), kTileM, 1, kF16) &&
            make_map(&mb_hi, p.bank_hi, kHalf, uint64_t(p.N), uint64_t(d_pad), kBRows, uint64_t(p.bank_row_stride), kF16);
  if (ok && !kBf16) ok = make_map(&mq_lo, p.q_lo, kHalf, uint64_t(p.B), uint64_t(d_pad), kTileM);
  if (ok && (!kBf16 || kTwoB))
    ok = make_map(&mb_lo, p.bank_lo, kHalf, uint64_t(p.N), uint64_t(d_pad), kBRows, uint64_t(p.bank_row_stride), kF16);
  if (!ok) {
    *why = "cuTensorMapEncodeTiled failed";
    return cudaErrorInvalidValue;
  }
  if (kBf16) mq_lo = mq_hi;
  if (kBf16 && !kTwoB) mb_lo = mb_hi;
  auto kern = tc_topk_kernel<MODE, BLOCK_N, ITEMS, DEBUG, PAIR, SAMPLE, EXCL>;
  cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, int(smem));
  if (e != cudaSuccess) return e;
  // `grid` counts workers: CTAs, or CTA pairs (clusters of 2 on one TPC) when PAIR
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = dim3(unsigned(grid * kCtas));
  cfg.blockDim = dim3(kThreads);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeClusterDimension;
  attr[0].val.clusterDim.x = kCtas;
  attr[0].val.clusterDim.y = 1;
  attr[0].val.clusterDim.z = 1;
  cfg.attrs = attr;
  cfg.numAttrs = 1;
  return cudaLaunchKernelEx(&cfg, kern, mq_hi, mq_lo, mb_hi, mb_lo, a);
}

template <int MODE, int BLOCK_N, bool DEBUG, bool PAIR>
cudaError_t launch_cap(const TcParams& p, int grid, int cap, cudaStream_t stream, float* dump,
                       int32_t* diag, int flags, const char** why) {
  // which options combine is checked before planning (api.cu); the debug hook passes none
  if (p.sample) return launch_t<MODE, BLOCK_N, 2, false, PAIR, true>(p, grid, stream, nullptr, diag, 0, why);
  if (p.bank_gid != nullptr) {
    switch (cap) {
      case 64: return launch_t<MODE, BLOCK_N, 2, false, PAIR, false, true>(p, grid, stream, nullptr, diag, 0, why);
      case 128: return launch_t<MODE, BLOCK_N, 4, false, PAIR, false, true>(p, grid, stream, nullptr, diag, 0, why);
      case 256: return launch_t<MODE, BLOCK_N, 8, false, PAIR, false, true>(p, grid, stream, nullptr, diag, 0, why);
      case 512: return launch_t<MODE, BLOCK_N, 16, false, PAIR, false, true>(p, grid, stream, nullptr, diag, 0, why);
      case 1024: return launch_t<MODE, BLOCK_N, 32, false, PAIR, false, true>(p, grid, stream, nullptr, diag, 0, why);
      default: *why = "unsupported k"; return cudaErrorNotSupported;
    }
  }
  switch (cap) {
    case 64: return launch_t<MODE, BLOCK_N, 2, DEBUG, PAIR>(p, grid, stream, dump, diag, flags, why);
    case 128: return launch_t<MODE, BLOCK_N, 4, DEBUG, PAIR>(p, grid, stream, dump, diag, flags, why);
    case 256: return launch_t<MODE, BLOCK_N, 8, DEBUG, PAIR>(p, grid, stream, dump, diag, flags, why);
    case 512: return launch_t<MODE, BLOCK_N, 16, DEBUG, PAIR>(p, grid, stream, dump, diag, flags, why);
    case 1024: return launch_t<MODE, BLOCK_N, 32, DEBUG, PAIR>(p, grid, stream, dump, diag, flags, why);
    default: *why = "unsupported k"; return cudaErrorNotSupported;
  }
}


// one (mode, pair) combination: both bank-tile widths, every list capacity, product + debug builds
template <int MODE, bool PAIR>
cudaError_t launch_variant(const TcParams& p, int grid, int cap, cudaStream_t stream, float* dump,
                           int32_t* diag, int flags, const char** why) {
  constexpr bool kResident = (MODE == B200KNN_MODE_BF16 || MODE == B200KNN_MODE_F16X2 || MODE == B200KNN_MODE_F16);
  const bool debug = dump != nullptr || flags != 0;  // only reachable from the test hook
  if constexpr (kResident) {  // 256-wide bank tiles exist for the resident-query modes only
    if (tc_tile_n(p.mode, p.D) == 256) {
      if (debug) return launch_cap<MODE, 256, true, PAIR>(p, grid, cap, stream, dump, diag, flags, why);
      return launch_cap<MODE, 256, false, PAIR>(p, grid, cap, stream, dump, diag, flags, why);
    }
  }
  if (debug) return launch_cap<MODE, 128, true, PAIR>(p, grid, cap, stream, dump, diag, flags, why);
  return launch_cap<MODE, 128, false, PAIR>(p, grid, cap, stream, dump, diag, flags, why);
}

}  // namespace
}  // namespace b200knn
