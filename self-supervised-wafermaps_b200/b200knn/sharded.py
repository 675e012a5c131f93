"""Bank row-sharded kNN over the GPUs of one node (SURVEY.md §8e).

Rank g owns bank rows [g*ceil(N/G), min(N,(g+1)*ceil(N/G))) and the matching
label slice is not needed locally: labels are replicated (N int64) so the vote
can look classes up by global index.  Every rank holds all queries.  One
exchange step of the per-shard (B,k) selection keys (8 B each), then the merge
kernel picks the global top-k under the same total order, so the G-GPU result
is bitwise the 1-GPU result.  Two exchanges are implemented:
  "allgather"  every rank receives every shard's (B,k) keys and merges all B rows
               (what ``topk_keys`` / ``knn_topk`` need: the full key matrix everywhere);
  "alltoall"   (default of ``knn_predict``) rank g receives only query rows
               [g*ceil(B/G), ...) from every shard, merges and votes that slice, and the
               (B,C) class rankings — 25x fewer bytes than the keys at k=200 — are
               all-gathered.  Moves G x fewer key bytes and does 1/G of the merge/vote
               work per rank.  The reference has no
distributed kNN (its DDP flag is off, ``scripts/WM811k_benchmark.py:54``); this
is the scale-out of its single-device bank (``src/ssl_wafermap/models/knn.py:80``).

The compute steps are injected (``ops``) so that the partition/exchange logic is
testable on CPU with gloo; the default ``ops`` is the CUDA library and there is
no CPU implementation in the product.
"""
from __future__ import annotations

import os
from typing import Optional, Tuple

import torch
import torch.distributed as dist

_TC_MODES = ("bf16", "tf32x3", "bf16x3", "f16x2", "f16")  # = knn.TC_MODES (raw tensor-core similarity modes)
_MAX_K = 992  # = knn.MAX_K (largest k of the streaming candidate lists)


def shard_bounds(n_rows: int, world_size: int, rank: int) -> Tuple[int, int]:
    """Rows [lo, hi) of the bank owned by `rank` (contiguous, ceil-divided)."""
    per = (n_rows + world_size - 1) // world_size
    lo = min(n_rows, rank * per)
    hi = min(n_rows, lo + per)
    return lo, hi


class _CudaOps:
    """Default compute backend: the C-ABI CUDA library."""

    @staticmethod
    def topk_keys(feature, bank_shard, k, mode, idx_offset, tau0=None):
        from .knn import topk_keys
        return topk_keys(feature, bank_shard, k, mode, idx_offset, tau0)

    @staticmethod
    def topk_into(feature, bank_shard, k, mode, idx_offset, tau0, out):
        """topk_keys writing into `out` when the mode allows it (tensor-core mode with a threshold)."""
        from .knn import topk_keys
        if tau0 is not None and mode in _TC_MODES:
            topk_keys(feature, bank_shard, k, mode, idx_offset, tau0, out=out)
        else:
            out.copy_(topk_keys(feature, bank_shard, k, mode, idx_offset, tau0))

    @staticmethod
    def scatter_supported(B, n_rows, D, k, mode):
        from .knn import plan_info
        try:
            return plan_info(B, n_rows, D, k, mode)["splits"] == 1
        except RuntimeError:
            return False

    @staticmethod
    def topk_scatter(feature, bank_shard, k, mode, idx_offset, tau0, peer_ptrs, rank, rows_per_owner):
        from .knn import topk_scatter
        return topk_scatter(feature, bank_shard, k, mode, idx_offset, tau0, peer_ptrs, rank, rows_per_owner)

    @staticmethod
    def sample_keys(feature, bank_shard, k, mode, n_rows_global):
        from .knn import sample_keys
        return sample_keys(feature, bank_shard, k, mode, n_rows_global)

    @staticmethod
    def sample_scatter_supported(B, n_rows, D, k, mode, n_rows_global):
        from .knn import sample_scatter_supported
        return sample_scatter_supported(B, n_rows, D, k, mode, n_rows_global)

    @staticmethod
    def sample_scatter(feature, bank_shard, k, mode, n_rows_global, peer_ptrs, rank, rows_per_owner):
        from .knn import sample_scatter
        return sample_scatter(feature, bank_shard, k, mode, n_rows_global, peer_ptrs, rank, rows_per_owner)

    @staticmethod
    def broadcast_f32(src, peer_ptrs, dst_offset):
        from .knn import broadcast_f32
        return broadcast_f32(src, peer_ptrs, dst_offset)

    @staticmethod
    def kth_sim(keys):
        from .knn import kth_sim
        return kth_sim(keys)

    @staticmethod
    def merge_keys(keys_in, k_out):
        from .knn import merge_keys
        return merge_keys(keys_in, k_out)

    @staticmethod
    def vote(keys, labels, num_classes, knn_t):
        from .knn import vote
        return vote(keys, labels, num_classes, knn_t)

    @staticmethod
    def vote_packed(keys, labels, num_classes, knn_t, n_rows_out):
        """(n_rows_out, C+1): class rankings + per-row status word (bit 0 starved row, bit 1 label
        out of range, bit 2 index out of range); no host synchronisation."""
        from .knn import vote_packed
        return vote_packed(keys, labels, num_classes, knn_t, n_rows_out)

    @staticmethod
    def vote_multi_packed(keys, labels, num_classes, knn_ks, knn_ts, n_rows_out):
        """vote_packed for a (knn_ks ascending, knn_ts) grid: (n_rows_out, n_k*n_t*C + 1)."""
        from .knn import vote_multi_packed
        return vote_multi_packed(keys, labels, num_classes, knn_ks, knn_ts, n_rows_out)

    @staticmethod
    def decode_keys(keys):
        from .knn import decode_keys
        return decode_keys(keys)

    # ---- sharded fp32 mode: candidate level, routing, re-scoring of routed candidates, certificate
    @staticmethod
    def cascade_levels(bank_shard, mode, boost=1):
        from .knn import RESCORED_MODES, cascade_levels
        return cascade_levels(bank_shard, mode, boost) if mode in RESCORED_MODES else None

    @staticmethod
    def route_keys(keys, rows_per_shard, n_shards):
        from .knn import route_keys
        return route_keys(keys, rows_per_shard, n_shards)

    @staticmethod
    def rescore_sparse(feature, bank_shard, cand, cand_mode, idx_offset):
        from .knn import rescore_sparse
        return rescore_sparse(feature, bank_shard, cand, cand_mode, idx_offset)

    @staticmethod
    def certify(exact, approx, feature, level, max_norm, all_rows):
        from .knn import certify
        return certify(exact, approx, feature, level, max_norm, all_rows)

    @staticmethod
    def bank_max_norm(bank_shard, cand_mode):
        from .knn import bank_max_norm
        return bank_max_norm(bank_shard, cand_mode)

    # ---- the same exchange over NVLink peer memory, and the device-side hand-over between levels
    @staticmethod
    def route_scatter(keys, rows_per_shard, n_shards, inbox_ptrs, row_offset):
        from .knn import route_scatter
        return route_scatter(keys, rows_per_shard, n_shards, inbox_ptrs, row_offset)

    @staticmethod
    def rescore_scatter(feature, bank_shard, cand, cand_mode, idx_offset, peer_ptrs, rank, rows_per_owner):
        from .knn import rescore_scatter
        return rescore_scatter(feature, bank_shard, cand, cand_mode, idx_offset, peer_ptrs, rank, rows_per_owner)

    @staticmethod
    def compact_rows(packed, col, mask, cap):
        from .knn import compact_rows
        return compact_rows(packed, col, mask, cap)

    @staticmethod
    def scatter_rows(dst, src, rows, count):
        from .knn import scatter_rows
        return scatter_rows(dst, src, rows, count)

    @staticmethod
    def local_exact_keys(feature, bank_shard, k, mode, idx_offset, n_shards=1):
        from .knn import local_exact_keys
        return local_exact_keys(feature, bank_shard, k, mode, idx_offset, n_shards)


class ShardedBank:
    """A (D, N) bank whose columns (bank rows) are partitioned over a process group.

    bank_shard: this rank's (D, hi-lo) slice; labels: all N labels (replicated).
    """

    def __init__(self, bank_shard: torch.Tensor, labels: torch.Tensor, n_rows: int,
                 group: Optional[dist.ProcessGroup] = None, mode: Optional[str] = None, ops=None):
        self.group = group
        self.world_size = dist.get_world_size(group) if dist.is_initialized() else 1
        self.rank = dist.get_rank(group) if dist.is_initialized() else 0
        self.n_rows = int(n_rows)
        self.lo, self.hi = shard_bounds(self.n_rows, self.world_size, self.rank)
        if bank_shard.shape[1] != self.hi - self.lo:
            raise ValueError(f"rank {self.rank}: shard has {bank_shard.shape[1]} rows, "
                             f"expected {self.hi - self.lo} for rows [{self.lo},{self.hi})")
        if labels.numel() != self.n_rows:
            raise ValueError("labels must hold all N bank labels (replicated)")
        self.bank_shard = bank_shard
        self.labels = labels
        self.mode = mode
        self.ops = ops or _CudaOps
        self._symm = {}

    @classmethod
    def from_full(cls, feature_bank: torch.Tensor, labels: torch.Tensor, **kw) -> "ShardedBank":
        """Slice a replicated (D, N) bank (testing / small banks)."""
        n = feature_bank.shape[1]
        ws = dist.get_world_size(kw.get("group")) if dist.is_initialized() else 1
        rk = dist.get_rank(kw.get("group")) if dist.is_initialized() else 0
        lo, hi = shard_bounds(n, ws, rk)
        return cls(feature_bank[:, lo:hi].contiguous(), labels, n, **kw)

    def local_keys(self, feature: torch.Tensor, k: int, tau0: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Per-shard top-min(k, shard rows) keys with GLOBAL indices, padded to k with empty keys."""
        rows = self.hi - self.lo
        k_loc = min(k, rows)
        B = feature.shape[0]
        keys = torch.zeros((B, k), dtype=torch.int64, device=feature.device)
        if k_loc > 0:
            keys[:, :k_loc] = self.ops.topk_keys(feature, self.bank_shard, k_loc, self.mode, self.lo, tau0)
        return keys

    def _gather(self, local: torch.Tensor) -> torch.Tensor:
        """all-gather of (B, c) keys -> (G, B, c), rank-major."""
        B, c = local.shape
        gathered = torch.empty((self.world_size * B, c), dtype=local.dtype, device=local.device)
        dist.all_gather_into_tensor(gathered, local.contiguous(), group=self.group)
        return gathered.view(self.world_size, B, c)

    def global_threshold(self, feature: torch.Tensor, k: int) -> Optional[torch.Tensor]:
        """Sampling pre-pass across shards: every rank samples its own rows, the per-rank sample
        lists are all-gathered (B*r keys per rank) and the r-th best of their union — a strided
        sample of the WHOLE bank — becomes the same admission threshold on every rank.  Shards
        then only collect rows that can still reach the global top-k, so the per-shard work no
        longer carries a fixed list warm-up (this is what lets the sharded mode scale)."""
        if self.mode not in _TC_MODES or self.world_size == 1:
            return None
        fused = self._global_threshold_fused(feature, k)
        if fused is not None:
            return fused
        sk = self.ops.sample_keys(feature, self.bank_shard, k, self.mode, self.n_rows)
        if sk is None:
            return None
        self._mark("  sample")
        B, r = sk.shape
        per, _, _ = self._owned(B)
        if B < 8 * self.world_size:  # tiny batches: one all-gather, every rank merges every row
            merged = self.ops.merge_keys(self._gather(sk), r)
            return self.ops.kth_sim(merged)
        # by query slice: rank g merges the G sample lists of its own rows only, then the (B,)
        # thresholds (4 B per query) are all-gathered
        padded = sk
        if per * self.world_size != B:
            padded = torch.zeros((per * self.world_size, r), dtype=sk.dtype, device=sk.device)
            padded[:B] = sk
        recv = self._exchange_owned(padded, per)
        self._mark("  all-to-all(B,16)")
        tau_own = self.ops.kth_sim(self.ops.merge_keys(recv, r))
        tau = torch.empty((per * self.world_size,), dtype=tau_own.dtype, device=tau_own.device)
        dist.all_gather_into_tensor(tau, tau_own.contiguous(), group=self.group)
        return tau[:B].contiguous()

    # OFF by default (B200KNN_FUSED_THRESHOLD=1 switches it on).  Measured at 8 GPUs
    # (profiles/r02_call25_* vs r02_call23_*): the resident step is unchanged (16.99 vs 16.78 ms fp32 — what
    # the phase log shows at a step's first synchronisation point is the ranks' arrival skew, whichever
    # primitive implements it), but the end-to-end step with the concurrent NCCL all-gather of the next
    # batch on the copy stream got 24-30 % slower, so the NCCL exchange stays the default.
    fused_threshold = os.environ.get("B200KNN_FUSED_THRESHOLD", "0") == "1"

    def _global_threshold_fused(self, feature: torch.Tensor, k: int) -> Optional[torch.Tensor]:
        """global_threshold over NVLink peer memory: the sampling kernel stores every query's 16
        values into the query owner's buffer, the owner merges the G samples of its rows and stores
        their thresholds into every rank's threshold buffer; three symmetric-memory barriers, no
        NCCL call."""
        if not (self.fused_threshold and self.fused_exchange and feature.is_cuda
                and hasattr(self.ops, "sample_scatter")):
            return None
        G = self.world_size
        B, D = feature.shape
        if G > 8 or B < 8 * G:
            return None
        for r in range(G):  # the same decision on every rank
            lo, hi = shard_bounds(self.n_rows, G, r)
            if not self.ops.sample_scatter_supported(B, hi - lo, D, k, self.mode, self.n_rows):
                return None
        per, _, _ = self._owned(B)
        r16 = 16
        try:
            (smp, tau64), hdl, (p_smp, p_tau), fresh = self._symmetric_regions(2, per, r16, feature.device, tag="thr")
        except Exception:
            type(self).fused_exchange = False
            return None
        if fresh:
            smp.zero_()  # rows past B are never written
        tau_all = tau64.view(-1).view(torch.float32)[:G * per]
        hdl.barrier(channel=0)  # every rank is done with the thresholds / samples of the previous call
        self.ops.sample_scatter(feature, self.bank_shard, k, self.mode, self.n_rows, p_smp, self.rank, per)
        self._mark("  sample + scatter")
        hdl.barrier(channel=1)
        tau_own = self.ops.kth_sim(self.ops.merge_keys(smp, r16))
        self.ops.broadcast_f32(tau_own, p_tau, self.rank * per)
        hdl.barrier(channel=2)
        self._mark("  merge + broadcast")
        return tau_all[:B]

    def topk_keys(self, feature: torch.Tensor, k: int) -> torch.Tensor:
        if k > self.n_rows:
            raise RuntimeError("selected index k out of range")
        if self.world_size == 1:
            return self.local_keys(feature, k)
        tau0 = self.global_threshold(feature, k)
        merged = self.ops.merge_keys(self._gather(self.local_keys(feature, k, tau0)), k)
        if tau0 is not None:
            # identical on every rank, so every rank takes the same branch (collectives stay matched)
            bad = merged[:, -1] == 0
            if bool(bad.any()):
                rows = bad.nonzero(as_tuple=False).view(-1)
                sub = feature[rows].contiguous()
                merged[rows] = self.ops.merge_keys(self._gather(self.local_keys(sub, k, None)), k)
        return merged

    last_uncertified = 0

    def knn_topk(self, feature: torch.Tensor, k: int):
        return self.ops.decode_keys(self.topk_keys(feature, k))

    # measurement hook (bench.py --phases): CUDA events between the phases of knn_predict
    phase_log = None

    def _mark(self, name: str) -> None:
        if self.phase_log is not None and torch.cuda.is_available():
            ev = torch.cuda.Event(enable_timing=True)
            ev.record()
            self.phase_log.append((name, ev))

    # ------------------------------------------------------------------ all-to-all exchange
    def _owned(self, B: int) -> Tuple[int, int, int]:
        """(rows per rank, first owned query row, one past the last owned row) for B queries."""
        per = (B + self.world_size - 1) // self.world_size
        lo = min(B, self.rank * per)
        return per, lo, min(B, lo + per)

    def _exchange_owned(self, local_padded: torch.Tensor, per: int) -> torch.Tensor:
        """local_padded: (G*per, k) this shard's keys for ALL (padded) queries.  Returns
        (G, per, k): every shard's keys for the query rows this rank owns."""
        recv = torch.empty_like(local_padded)
        dist.all_to_all_single(recv, local_padded, group=self.group)
        return recv.view(self.world_size, per, local_padded.shape[1])

    # ------------------------------------------------------------------ fused exchange (NVLink P2P)
    fused_exchange = os.environ.get("B200KNN_FUSED_EXCHANGE", "1") == "1"

    def _symmetric_regions(self, n_regions: int, per: int, k: int, device, tag: str = "buf"):
        """n_regions exchange buffers of shape (G, per, k) int64 carved out of ONE symmetric-memory
        allocation (every rank's copy is mapped into every process), plus the rendezvous handle and
        per region the list of all ranks' device pointers to it.  Allocations are bucketed by size
        (powers of two) and shared by every call shape that fits, so a new batch size or a new
        count of uncertified rows does not trigger a new allocation + rendezvous collective.
        Returns (regions, handle, ptrs, fresh): fresh is True when the layout differs from the
        previous call's, i.e. rows a kernel never writes may hold another layout's keys."""
        import torch.distributed._symmetric_memory as symm_mem

        G = self.world_size
        need = n_regions * G * per * k
        bucket = 1 << max(20, (need - 1).bit_length())
        hit = self._symm.get((tag, bucket))
        if hit is None:
            for key in [key for key in self._symm if key[0] == tag and key[1] < bucket]:
                self._symm.pop(key)  # superseded by the larger allocation
            flat = symm_mem.empty((bucket,), dtype=torch.int64, device=device)
            flat.zero_()
            hdl = symm_mem.rendezvous(flat, self.group if self.group is not None else dist.group.WORLD)
            hit = self._symm[(tag, bucket)] = [flat, hdl, None]
        flat, hdl, layout = hit
        fresh = layout != (n_regions, per, k)
        hit[2] = (n_regions, per, k)
        size = G * per * k
        regions = [flat[r * size:(r + 1) * size].view(G, per, k) for r in range(n_regions)]
        ptrs = [[int(base) + r * size * 8 for base in hdl.buffer_ptrs] for r in range(n_regions)]
        return regions, hdl, ptrs, fresh

    def _fused_ok(self, feature: torch.Tensor, k: int, mode: str) -> bool:
        """Whether the fused (peer-memory) exchange applies — decided from quantities every rank
        knows, so the decision is the same everywhere."""
        if not (self.fused_exchange and feature.is_cuda and hasattr(self.ops, "topk_scatter")):
            return False
        if self.world_size > 8 or mode not in _TC_MODES:
            return False
        B, D = feature.shape
        for r in range(self.world_size):
            lo, hi = shard_bounds(self.n_rows, self.world_size, r)
            if hi - lo < k or not self.ops.scatter_supported(B, hi - lo, D, k, mode):
                return False
        return True

    def _owned_keys_fused(self, feature: torch.Tensor, k: int, tau0, per: int) -> Optional[torch.Tensor]:
        """The compute step and its collective as ONE kernel: every shard's tc_topk kernel stores the
        keys of each query tile it finishes into the owner GPU's exchange buffer over NVLink, so the
        all-to-all overlaps the remaining tiles' math.  Returns None when not applicable."""
        if not self._fused_ok(feature, k, self.mode):
            return None
        try:
            (buf,), hdl, (ptrs,), fresh = self._symmetric_regions(1, per, k, feature.device)
        except Exception:  # symmetric memory unavailable on this system: NCCL exchange instead
            type(self).fused_exchange = False
            return None
        if fresh:
            buf.zero_()  # rows past B are never written: they must read as empty lists
        hdl.barrier(channel=0)  # every rank is done reading its buffer of the previous call
        ok = self.ops.topk_scatter(feature, self.bank_shard, k, self.mode, self.lo, tau0, ptrs, self.rank, per)
        self._mark("  local topk + scatter")
        hdl.barrier(channel=1)  # every rank's stores have landed
        if not ok:
            raise RuntimeError("b200knn: fused exchange refused after the collective decision to use it")
        self._mark("  barrier")
        return self.ops.merge_keys(buf, k)

    def owned_keys(self, feature: torch.Tensor, k: int, tau0: Optional[torch.Tensor]) -> torch.Tensor:
        """Merged global top-k keys of the query rows this rank owns: (per, k); rows past B and
        slots a too-high threshold starved are empty (0)."""
        B = feature.shape[0]
        per, _, _ = self._owned(B)
        rows = self.hi - self.lo
        k_loc = min(k, rows)
        if B > 0:
            fused = self._owned_keys_fused(feature, k, tau0, per)
            if fused is not None:
                return fused
        if k_loc == k and B > 0 and hasattr(self.ops, "topk_into"):
            # the kernel writes its keys straight into the exchange buffer; only the pad rows are zeroed
            local = torch.empty((per * self.world_size, k), dtype=torch.int64, device=feature.device)
            local[B:].zero_()
            self.ops.topk_into(feature, self.bank_shard, k, self.mode, self.lo, tau0, local[:B])
            self._mark("  local topk")
        else:
            local = torch.zeros((per * self.world_size, k), dtype=torch.int64, device=feature.device)
            if k_loc > 0 and B > 0:
                local[:B, :k_loc] = self.ops.topk_keys(feature, self.bank_shard, k_loc, self.mode, self.lo, tau0)
        recv = self._exchange_owned(local, per)
        self._mark("  all-to-all")
        return self.ops.merge_keys(recv, k)

    # ------------------------------------------------------------------ sharded fp32 (bit-exact) mode
    rescore_at_row_owner = os.environ.get("B200KNN_SHARDED_RESCORE", "1") == "1"

    def _global_max_norm(self, cand_mode: str) -> torch.Tensor:
        """max row norm over the WHOLE bank (all-reduce MAX of the shards' values), cached."""
        key = ("max_norm", cand_mode, getattr(self.bank_shard, "_version", 0))  # in-place bank updates
        hit = self._symm.get(key)
        if hit is None:
            hit = self.ops.bank_max_norm(self.bank_shard, cand_mode).clone()
            dist.all_reduce(hit, op=dist.ReduceOp.MAX, group=self.group)
            self._symm[key] = hit
        return hit

    def _owned_keys_rescored(self, feature: torch.Tensor, k: int, level: dict):
        """fp32-matching mode with the bank sharded, re-scoring work divided by the shard count:
        1. every shard's tensor-core candidates (k + margin, under one global sampled threshold) go
           to the owner of the query (fused scatter / all-to-all) and are merged there: the global
           approximate top-(k + margin), exactly what one GPU would have produced;
        2. the owner routes each candidate to the shard that holds its bank row, that shard
           re-scores it exactly (sequential fma) and returns the exact key;
        3. the owner merges the exact keys and evaluates the single-GPU certificate.
        Steps 2-3 run over NVLink peer memory when the fused exchange applies (route_scatter ->
        rescore_scatter, four symmetric-memory barriers, no NCCL call), else as two all-to-alls.
        Returns (exact keys (per, k), uncertified flags (n_owned,) int32) for the owned query rows."""
        import copy
        B = feature.shape[0]
        per, lo, hi = self._owned(B)
        G = self.world_size
        # the streaming lists hold MAX_K keys: near that limit the margin shrinks (as on one GPU)
        k_in = min(k + level["margin"], self.n_rows, max(k, _MAX_K))
        cand = copy.copy(self)  # same shard, buffers and phase log; candidate mode instead of "fp32"
        cand.mode = level["cand"]
        tau0 = cand.global_threshold(feature, k_in)
        self._mark("threshold")
        rows_per_shard = (self.n_rows + G - 1) // G
        max_norm = self._global_max_norm(level["cand"])
        fused = B > 0 and hasattr(self.ops, "rescore_scatter") and self._fused_ok(feature, k_in, level["cand"])
        if fused:
            try:
                (exch1, inbox, exch2), hdl, (p1, p_in, p2), fresh = \
                    self._symmetric_regions(3, per, k_in, feature.device)
            except Exception:
                type(self).fused_exchange = False
                fused = False
        if fused:
            if fresh:
                exch1.zero_()
            inbox.zero_()   # written sparsely by the peers (non-empty prefixes only)
            exch2.zero_()
            hdl.barrier(channel=0)  # every rank has zeroed its buffers and is done with the previous call
            if not self.ops.topk_scatter(feature, self.bank_shard, k_in, level["cand"], self.lo, tau0, p1,
                                         self.rank, per):
                raise RuntimeError("b200knn: fused exchange refused after the collective decision to use it")
            self._mark("  candidates + scatter")
            hdl.barrier(channel=1)
            approx = self.ops.merge_keys(exch1, k_in)                     # (per, k_in) global approximate top
            self.ops.route_scatter(approx[:hi - lo], rows_per_shard, G, p_in, self.rank * per)
            self._mark("  merge + route")
            hdl.barrier(channel=2)
            # my bank rows among the candidates of ALL queries -> exact keys -> each query's owner
            self.ops.rescore_scatter(feature, self.bank_shard, inbox.view(G * per, k_in)[:B], level["cand"],
                                     self.lo, p2, self.rank, per)
            self._mark("  re-score + scatter")
            hdl.barrier(channel=3)
            merged = self.ops.merge_keys(exch2, k)                        # (per, k) exact
        else:
            approx = cand.owned_keys(feature, k_in, tau0)                  # (per, k_in)
            self._mark("candidates+exchange+merge")
            routed = self.ops.route_keys(approx, rows_per_shard, G)       # (G, per, k_in)
            mine = self._exchange_owned(routed.view(G * per, k_in), per)   # (G, per, k_in): all queries, my rows
            self._mark("  route + all-to-all")
            exact_local = torch.zeros((G * per, k_in), dtype=torch.int64, device=feature.device)
            if B:
                exact_local[:B] = self.ops.rescore_sparse(feature, self.bank_shard, mine.view(G * per, k_in)[:B],
                                                          level["cand"], self.lo)
            self._mark("  re-score")
            back = self._exchange_owned(exact_local, per)                  # (G, per, k_in): my queries, every shard
            merged = self.ops.merge_keys(back, k)                          # (per, k) exact
        flags = self.ops.certify(merged[:hi - lo], approx[:hi - lo], feature[lo:hi], level, max_norm,
                                 k_in >= self.n_rows)
        self._mark("  merge + certify")
        return merged, flags

    def _predict_level_packed(self, feature, knn_k, W, vote_packed, level):
        """One cascade level for all (replicated) query rows: (G*per, W+1) int64, identical on every
        rank — class rankings (W = C columns, or n_k*n_t*C for a grid) in columns [0, W), status word
        in column W (bit 0 starved row, bits 1 / 2 label / index out of range, bit 3 uncertified).
        vote_packed(keys, n_rows_out): the call's vote step (``_CudaOps.vote_packed`` or
        ``vote_multi_packed`` with the call's settings bound)."""
        n = feature.shape[0]
        per, lo, hi = self._owned(n)
        merged, flags = self._owned_keys_rescored(feature, knn_k, level)
        packed = vote_packed(merged[:hi - lo], per)
        packed[:hi - lo, W] |= flags.to(torch.int64) << 3
        gathered = torch.empty((per * self.world_size, W + 1), dtype=torch.int64, device=feature.device)
        dist.all_gather_into_tensor(gathered, packed, group=self.group)
        self._mark("vote+gather")
        return gathered

    # capacity of the device-side second level, per batch size (doubles after an overflow), and the
    # first level's margin boost (knn.next_boost).  Both follow the all-gathered count of open rows
    # only, so every rank keeps the same values and takes the same decisions.
    _l2_cap = None
    _boost = 1
    _calm = 0

    def _knn_predict_rescored(self, feature, C, knn_k, W, vote_packed, levels) -> torch.Tensor:
        """Sharded fp32 mode, ONE host synchronisation per call.
        Level 1 (all rows): `_owned_keys_rescored` at the cascade's first level.  Rows it leaves
        uncertified or starved (status bits 3 / 0 — identical on every rank after the all-gather)
        are compacted ON THE DEVICE into a fixed-capacity sub-batch; level 2 recomputes that
        sub-batch exactly on every shard's own rows (one cascade level at base margin — fp16 again
        with 4 or more shards, fp16 x split-fp16 below that — + exact re-scoring + the shard-local
        certificate: a shard holds 1/G of the bank, so its rank gaps are G times wider), the per-shard
        exact top-k are all-gathered and merged and the rankings scattered back.  Only then is one status word read; rows still open (level 2
        uncertified on some shard, or more open rows than the capacity) take the host-driven path."""
        B = feature.shape[0]
        self._mark("start")
        packed = self._predict_level_packed(feature, knn_k, W, vote_packed, levels[0])
        out = packed[:B]
        n_open = None
        if hasattr(self.ops, "compact_rows"):
            if self._l2_cap is None:
                self._l2_cap = {}
            cap = self._l2_cap.get(B) or min(B, max(256, -(-B // 64)))  # first call: 1/64 of the batch
            rows, count = self.ops.compact_rows(out, W, 9, cap)
            sub = feature.index_select(0, rows)
            loc = self.ops.local_exact_keys(sub, self.bank_shard, knn_k, self.mode, self.lo,
                                            self.world_size)                                # (cap, k+1)
            allk = self._gather(loc)                                                        # (G, cap, k+1)
            keys2 = self.ops.merge_keys(allk[:, :, :knn_k].contiguous(), knn_k)
            pk2 = vote_packed(keys2, cap)
            pk2[:, W] |= (allk[:, :, knn_k].amax(0) != 0).to(torch.int64) << 3
            self.ops.scatter_rows(out, pk2, rows, count)
            n_open = count
            self._mark("level 2 (open rows, per shard)")
        # one host read: OR of the status bits over all rows + the number of rows level 1 left open
        shifts = torch.arange(4, device=out.device)
        bits = ((out[:, W:W + 1] >> shifts) & 1).amax(0)
        if n_open is None:
            host = bits.tolist() + [0]
        else:
            host = torch.cat([bits, n_open.view(1).to(bits.dtype)]).tolist()
        status = out[:, W]
        pred = out[:, :W].contiguous()
        self.last_uncertified = int(host[4]) if n_open is not None else int(((status & 9) != 0).sum().item())
        if n_open is not None:
            # the second level costs every shard the same whatever G is: size it to ~1.5x the rows
            # the first level really leaves open (rounded up to 256), at least 256
            self._l2_cap[B] = min(B, max(256, -(-int(1.5 * host[4]) // 256) * 256))
        if len(levels) > 1:
            from .knn import next_boost
            self._boost, self._calm = next_boost(self._boost, self._calm, B, self.last_uncertified)
        if host[0] or host[3]:
            # host-driven path (identical status on every rank -> matched collectives): per-shard
            # exact top-k through the single-GPU cascade, all-gathered and merged
            rows = ((status & 9) != 0).nonzero(as_tuple=False).view(-1)
            sub = feature[rows].contiguous()
            keys = self.ops.merge_keys(self._gather(self.local_keys(sub, knn_k, None)), knn_k)
            pk = vote_packed(keys, rows.numel())
            pred[rows] = pk[:, :W]
            worst = int(pk[:, W].max().item()) if rows.numel() else 0
            host[1] = host[1] or (worst & 2)
            host[2] = host[2] or (worst & 4)
        _raise_label_bits((2 if host[1] else 0) | (4 if host[2] else 0), C)
        return pred

    def knn_predict(self, feature: torch.Tensor, num_classes: int, knn_k: int = 200,
                    knn_t: float = 0.1, exchange: str = "alltoall") -> torch.Tensor:
        """Same contract as ``knn_predict`` with the bank sharded; identical on every rank."""
        if exchange == "allgather" or self.world_size == 1 or not hasattr(self.ops, "vote_packed"):
            return self.ops.vote(self.topk_keys(feature, knn_k), self.labels, num_classes, knn_t)
        C = int(num_classes)
        return self._predict(feature, C, knn_k, C,
                             lambda keys, n: self.ops.vote_packed(keys, self.labels, C, knn_t, n), exchange)

    def knn_predict_multi(self, feature: torch.Tensor, num_classes: int, knn_ks=(200,), knn_ts=(0.1,),
                          exchange: str = "alltoall") -> torch.Tensor:
        """Same contract as ``knn_predict_multi`` with the bank sharded: (n_k, n_t, B, C), identical on
        every rank and bitwise the 1-GPU result.  One sharded search at k_max (two when k_max is
        beyond a raw tensor-core mode's lists and some k is not, as on one GPU)."""
        from .knn import check_grid, get_default_mode, grid_parts, grid_view
        ks, ts, order = check_grid(knn_ks, knn_ts)
        C = int(num_classes)
        preds = []
        for part in grid_parts(tuple(ks[i] for i in order), self.mode or get_default_mode()):
            W = len(part) * len(ts) * C

            def vote_packed(keys, n, part=part):
                return self.ops.vote_multi_packed(keys, self.labels, C, part, tuple(ts), n)

            if exchange == "allgather" or self.world_size == 1:
                packed = vote_packed(self.topk_keys(feature, part[-1]), feature.shape[0])
                _raise_label_bits(int(packed[:, W].max().item()) if feature.shape[0] else 0, C)
                preds.append(packed[:, :W])
            else:
                preds.append(self._predict(feature, C, part[-1], W, vote_packed, exchange))
        return grid_view(torch.cat(preds, dim=1), order, len(ts), C)

    def _predict(self, feature, C, knn_k, W, vote_packed, exchange) -> torch.Tensor:
        """The all-to-all path of knn_predict / knn_predict_multi: (B, W) rankings; vote_packed(keys,
        n_rows_out) -> (n_rows_out, W+1) is the call's vote step (see ``_predict_level_packed``)."""
        if exchange != "alltoall":
            raise ValueError(f"unknown exchange {exchange!r}")
        if knn_k > self.n_rows:
            raise RuntimeError("selected index k out of range")
        levels = self.ops.cascade_levels(self.bank_shard, self.mode, self._boost) \
            if hasattr(self.ops, "cascade_levels") else None
        if levels and self.rescore_at_row_owner and feature.shape[0] > 0:
            return self._knn_predict_rescored(feature, C, knn_k, W, vote_packed, levels)
        B = feature.shape[0]
        per, lo, hi = self._owned(B)
        mark = self._mark
        mark("start")
        tau0 = self.global_threshold(feature, knn_k)
        mark("threshold")  # sample + all-gather of (B,16) + merge
        merged = self.owned_keys(feature, knn_k, tau0)
        mark("topk+exchange+merge")
        # (per, W+1): class rankings + a status column, for the owned rows only (pad rows stay 0)
        packed = vote_packed(merged[:hi - lo], per)
        gathered = torch.empty((per * self.world_size, W + 1), dtype=torch.int64, device=feature.device)
        dist.all_gather_into_tensor(gathered, packed, group=self.group)
        mark("vote+gather")
        status = gathered[:B, W]
        out = gathered[:B, :W].contiguous()
        worst = int(status.max().item()) if B else 0  # the one host synchronisation of the call
        _raise_label_bits(worst, C)
        if worst == 1:
            # identical on every rank -> every rank takes this branch: recompute the starved rows
            # (the ~1e-7 tail of the sampled threshold) without a threshold
            rows = (status == 1).nonzero(as_tuple=False).view(-1)
            sub = feature[rows].contiguous()
            keys = self.ops.merge_keys(self._gather(self.local_keys(sub, knn_k, None)), knn_k)
            pk = vote_packed(keys, rows.numel())
            out[rows] = pk[:, :W]
            _raise_label_bits(int(pk[:, W].max().item()), C)
        return out


def _raise_label_bits(status: int, C: int) -> None:
    """The errors of a status word (b200knn_vote_ex): bit 1 label / bit 2 neighbour index out of range."""
    if status & 2:
        raise RuntimeError("index out of bounds: a feature_labels entry is outside "
                           f"[0, num_classes={C})")
    if status & 4:
        raise RuntimeError("index out of bounds: neighbour index outside feature_labels")
