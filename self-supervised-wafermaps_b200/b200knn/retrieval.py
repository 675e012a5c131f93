"""Batch nearest-neighbour retrieval over the reference's embedding tables (SURVEY.md §8 a5, f2, f4).

The reference's notebooks search one query at a time in NumPy
(``notebooks/2.0-Figures-nearest-neighbors.ipynb:54``,
``notebooks/3.1-Embeddings-clustering.ipynb:1930``):

    np.argsort(np.linalg.norm(data - q, axis=1))[:6]          # rank 0 is the query itself

over tables written by ``notebooks/3.0-Embeddings-inference.ipynb:493-507``
(``data/interim/model_preds/{model}_preds_*.pkl.xz``: integer columns 0..D-1 hold the fp16
embedding, the others are wafer metadata).  Here the same search runs for any number of queries
at once through the fused similarity/top-k kernels: argmin ||x - q||  =  argmax 2 q.x - ||x||^2,
so the L2 ranking is a dot-product top-k over vectors extended by one column
(x' = [x, ||x||^2], q' = [2q, -1]).
"""
from __future__ import annotations

import math
from fractions import Fraction
from typing import NamedTuple, Optional, Tuple

import numpy as np
import torch

from . import knn as K
from .bank import FeatureBank


def load_embedding_table(path: str):
    """Read a reference embedding table (``*_preds_*.pkl.xz``).  Returns (embeddings, meta):
    an (N, D) NumPy array in the stored dtype (fp16) and a DataFrame of the remaining columns
    (``waferMap``, ``failureType``, ``failureCode`` ...).  Host-side; needs pandas."""
    import numpy as np
    import pandas as pd

    df = pd.read_pickle(path)
    emb_cols = [c for c in df.columns if isinstance(c, (int, np.integer))]
    if not emb_cols:
        raise ValueError(f"{path}: no integer-named embedding columns")
    emb = np.ascontiguousarray(df[sorted(emb_cols)].to_numpy())
    return emb, df.drop(columns=emb_cols)


def _augment_rows(x: torch.Tensor) -> torch.Tensor:
    """(N, D) -> (N, D+1) fp32 rows [x, ||x||^2]."""
    xf = x if x.dtype == torch.float32 else x.float()
    out = torch.empty((x.shape[0], x.shape[1] + 1), dtype=torch.float32, device=x.device)
    out[:, :-1] = xf
    out[:, -1] = K.row_sqnorms(x)
    return out


def _augment_queries(q: torch.Tensor) -> torch.Tensor:
    qf = q if q.dtype == torch.float32 else q.float()
    out = torch.empty((q.shape[0], q.shape[1] + 1), dtype=torch.float32, device=q.device)
    out[:, :-1] = qf * 2.0  # exact (power of two)
    out[:, -1] = -1.0
    return out


class L2Index:
    """Rows of an embedding table, extended once so that L2 search is a dot-product top-k."""

    def __init__(self, data_rows: torch.Tensor):
        K._require_cuda("data_rows", data_rows)
        if data_rows.dim() != 2:
            raise RuntimeError("data_rows must be (N, D)")
        self.n_rows, self.dim = data_rows.shape
        self._fb = FeatureBank.from_rows(_augment_rows(data_rows), normalize=False)

    def search(self, queries: torch.Tensor, k: int, mode: Optional[str] = None) -> Tuple[torch.Tensor, torch.Tensor]:
        """(dist (B,k) fp32 ascending, idx (B,k) int64): the k rows nearest to every query in L2;
        ties by lowest row index.  Same result as the notebooks' per-query argsort for the rows it
        can tell apart in fp32.  dist^2 = ||q||^2 - (2 q.x - ||x||^2) carries the fp32 rounding of
        ||x||^2, i.e. an absolute (not relative) error of about ulp(||x||^2)."""
        K._require_cuda("queries", queries)
        if queries.dim() != 2 or queries.shape[1] != self.dim:
            raise RuntimeError(f"queries must be (B, {self.dim})")
        s, idx = self._fb.knn_topk(_augment_queries(queries), k, mode=mode)  # s = 2 q.x - ||x||^2
        qq = K.row_sqnorms(queries).view(-1, 1)
        return torch.sqrt(torch.clamp(qq - s, min=0.0)), idx


def l2_topk(data_rows: torch.Tensor, queries: torch.Tensor, k: int, mode: Optional[str] = None):
    """One-shot ``L2Index(data_rows).search(queries, k)``."""
    return L2Index(data_rows).search(queries, k, mode)


def knn_graph(rows: torch.Tensor, k: int, normalize: bool = True, mode: Optional[str] = None,
              batch: int = 75776, include_self: bool = False,
              groups: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """k nearest neighbours (cosine when normalize=True) of EVERY row among all rows — the graph
    UMAP / HDBSCAN build from the embeddings (``notebooks/3.0-Embeddings-inference.ipynb:208-216``,
    ``3.2-Embeddings-SSL-categories.ipynb:51-53``; BASELINE.json config "811k x 512, top-10 for all
    811k queries").  Returns (sims (N,k) fp32, idx (N,k) int64); a row's own entry (rank 0 when
    rows are distinct) is dropped unless include_self.  groups: optional (N,) integer ids (lots,
    duplicate hashes); a row's k neighbours then exclude every row of its group, through the
    leave-one-group-out search of ``knn_predict_loo``; k <= N - (largest group size)."""
    if groups is not None:
        if include_self:
            raise ValueError("knn_graph: groups leaves a row's whole group out, so include_self must be False")
        plan = K._group_plan(groups, rows.shape[0], rows.device)
        if k > rows.shape[0] - plan[1]:
            raise RuntimeError("knn_graph: k must be smaller than the number of rows outside a row's group")
    fb = FeatureBank.from_rows(rows, normalize=normalize)
    n = fb.n_rows
    if groups is not None:
        sims = torch.empty((n, k), dtype=torch.float32, device=rows.device)
        idx = torch.empty((n, k), dtype=torch.int64, device=rows.device)
        flag = torch.zeros((1,), dtype=torch.int32, device=rows.device)
        for _, lo, hi, keys in K._group_searches(fb.bank, plan, (int(k),), mode or K.get_default_mode(), batch,
                                                 flag):
            sims[lo:hi], idx[lo:hi] = K.decode_keys(keys)
        if len(plan[3]) > 1:  # bucket order -> row order
            sims = torch.empty_like(sims).index_copy_(0, plan[2], sims)
            idx = torch.empty_like(idx).index_copy_(0, plan[2], idx)
        if int(flag.item()):
            raise RuntimeError("knn_graph: a neighbour index is outside the group ids")
        return sims, idx
    if not include_self and k >= n:
        raise RuntimeError("knn_graph: k must be smaller than the number of rows")
    kk = min(n, k if include_self else k + 1)
    sims = torch.empty((n, k), dtype=torch.float32, device=rows.device)
    idx = torch.empty((n, k), dtype=torch.int64, device=rows.device)
    for lo in range(0, n, batch):
        hi = min(n, lo + batch)
        if include_self:
            s, i = fb.knn_topk(fb.rows[lo:hi, :fb.dim], kk, mode=mode)
            sims[lo:hi], idx[lo:hi] = s[:, :k], i[:, :k]
            continue
        # drop the row itself by index (wherever it ranks among exact duplicates), else the last key
        keys = K.topk_keys(fb.rows[lo:hi, :fb.dim], fb.bank, kk, mode)
        sims[lo:hi], idx[lo:hi] = K.decode_keys(K.drop_self(keys, lo))
    return sims, idx


# ---- similarity-threshold (radius) search -------------------------------------------------------
# A radius row has no fixed length, so it is searched on a ladder of list depths: every row first at
# RADIUS_FIRST_DEPTH keys, a row whose list filled there again at RADIUS_SECOND_DEPTH (the longest
# streaming list), and a row that fills that too (only when max_per_row > RADIUS_SECOND_DEPTH) by
# the exact kernel's peeling in passes of <= MAX_K keys.  The tensor-core searches run under a
# per-row admission threshold tau0 (b200knn_topk_opt), so a list fills only when the row really has
# that many columns above it; with a high threshold almost every tile takes the epilogue's no-hit
# path.  Most rows have few near-duplicates and end at the first depth.
RADIUS_FIRST_DEPTH = 32
RADIUS_SECOND_DEPTH = K.MAX_K


class RadiusNeighbors(NamedTuple):
    """CSR rows of a radius search: row b is indices / sims [offsets[b], offsets[b + 1])."""
    offsets: torch.Tensor    # (B + 1,) int64
    indices: torch.Tensor    # (nnz,) int64
    sims: torch.Tensor       # (nnz,) fp32
    saturated: torch.Tensor  # (B,) bool: the row stopped at max_per_row and may miss neighbours


# rows per ladder level of the last radius search (bench): first / second depth, the certified
# top-max_per_row of fp32 modes, the self-join's own-row-excluded search at max_per_row = MAX_K,
# exact peeling
last_radius_stats = {"first": 0, "second": 0, "certify": 0, "self_excluded": 0, "peel": 0}


def admission_threshold(tau32: float, e: float = 0.0) -> np.float32:
    """The largest fp32 value strictly below the exact real tau32 - e (fp32 tau32, e >= 0): what
    b200knn_radius_tau0 computes per row, restated on the host (raw modes use e = 0)."""
    t, e = np.float32(tau32), np.float32(e)
    exact = Fraction(float(t)) - Fraction(float(e))
    r = np.float32(float(exact)) if math.isfinite(float(exact)) else np.float32(-np.inf)
    while r > -np.inf and Fraction(float(r)) >= exact:
        r = np.nextafter(r, np.float32(-np.inf))
    while True:
        up = np.nextafter(r, np.float32(np.inf))
        if not math.isfinite(float(up)) or Fraction(float(up)) >= exact:
            return r
        r = up


def radius_ladder(n_bank: int, cap_search: int) -> tuple:
    """The list depths of the ladder for a bank of n_bank rows and rows of at most cap_search keys
    (max_per_row, + 1 when the row's own key is dropped afterwards): (first,) or (first, second)."""
    m0 = min(n_bank, RADIUS_FIRST_DEPTH, cap_search)
    m1 = min(n_bank, RADIUS_SECOND_DEPTH, cap_search)
    return (m0,) if m1 == m0 else (m0, m1)


def radius_plan(depth: int, cap_search: int, n_bank: int, full: torch.Tensor, exact_order: bool):
    """(escalate, saturated) bool masks of the rows of a list searched at `depth`, from the count
    pass's `full` bits.  A list in the exact order (exact kernel, re-scored certified lists, raw
    modes' own order) may continue when its last key is a neighbour; a re-scored candidate list
    (fp32 modes) when its last slot is filled at all, since the columns past it were ranked by the
    approximate similarities.  A row that may continue is searched deeper while depth < cap_search;
    at cap_search it is saturated.  depth == n_bank holds every column: nothing continues."""
    go = (full & (2 if exact_order else 1)) != 0
    none = torch.zeros_like(go)
    if depth >= n_bank:
        return none, none
    return (go, none) if depth < cap_search else (none, go)


def _radius_peel(q: torch.Tensor, bank: torch.Tensor, tau32: float, cap_search: int,
                 first: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Exact keys of rows q by peeling: pass i takes the best min(MAX_K, left) keys strictly below
    the row's last key of pass i - 1 (b200knn_topk_opt's upper_keys); a row stops when its last key
    is below tau32 or it holds cap_search keys.  first: the rows' first exact list (all of them
    continue).  Returns (n, depth) keys, zero-filled behind the rows that stopped early."""
    n, D = q.shape
    N = bank.shape[1]
    limit = min(N, cap_search)
    qx, bx = K._exact_operands(q, bank)
    blocks, done, upper = [], 0, None
    active = torch.arange(n, device=q.device)
    if first is not None:
        blocks, done, upper = [first], first.shape[1], first[:, -1].contiguous()
    while done < limit and active.numel():
        kp = min(K.MAX_K, limit - done)
        qa = qx if active.numel() == n else qx.index_select(0, active)
        part = K._search("exact", qa, bx, active.numel(), N, D, kp, upper=upper)
        blocks.append(part if active.numel() == n else
                      torch.zeros((n, kp), dtype=torch.int64, device=q.device).index_copy_(0, active, part))
        done += kp
        cont = K.kth_sim(part) >= tau32
        active, upper = active[cont], part[cont, -1].contiguous()
    return torch.cat(blocks, 1) if len(blocks) > 1 else blocks[0]


def _radius_rows(q: torch.Tensor, bank: torch.Tensor, tau32: float, mode: str, cap: int,
                 self_offset: int) -> RadiusNeighbors:
    """Radius rows of queries q (B, D) in the (D, N) bank (see ``knn_radius``); self_offset >= 0
    drops bank row self_offset + b from row b."""
    B, D = q.shape
    N = bank.shape[1]
    dev = q.device
    cap_search = min(N, cap + (1 if self_offset >= 0 else 0))
    counts = torch.zeros((B,), dtype=torch.int64, device=dev)
    saturated = torch.zeros((B,), dtype=torch.bool, device=dev)
    pieces = []  # (keys, list row -> result row or None): every result row in exactly one piece
    stats = last_radius_stats

    def settle(keys, rows, depth, exact_order, n_bank=N, depth_cap=cap_search):
        """Count a list: (escalate, saturated) masks of its rows (radius_plan)."""
        with K._Timed("radius_compact"):
            full = K.radius_count(keys, rows, tau32, self_offset, cap, counts)
        return radius_plan(depth, depth_cap, n_bank, full, exact_order)

    def to_rows(mask, rows):
        return mask.nonzero().view(-1) if rows is None else rows[mask]

    def finish(keys, rows, leave):
        """Keep the list rows of the result rows that do not leave it."""
        if not bool(leave.any()):
            pieces.append((keys, rows))
        else:
            keep = (~leave).nonzero().view(-1)
            pieces.append((keys.index_select(0, keep), keep if rows is None else rows[keep]))

    peel = []     # (rows, first exact keys or None)
    certify = []  # rows whose re-scored candidate list filled at cap_search (fp32 modes)
    # A self-join row holds up to cap entries besides its own, so it is searched at cap + 1 keys; at
    # cap = MAX_K that is one more than the streaming lists hold.  Such rows are searched again at
    # depth cap with their own row left out inside the search (topk_keys' exclusion, every mode and
    # path), not peeled: peeling stays for max_per_row > MAX_K.
    self_excl = self_offset >= 0 and cap <= K.MAX_K < cap_search
    deeper = peel if not self_excl else []  # where rows past the last ladder depth go
    # An fp32 mode's exact top list at k >= MAX_K has no candidate margin beyond k, so no cascade level
    # can certify it and the cascade would end in the exact kernel after its tensor-core passes:
    # such lists come from the exact kernel directly (the same keys).
    top_mode = "exact" if mode in K.RESCORED_MODES and cap_search >= K.MAX_K else mode
    if mode == "exact":
        keys = K.topk_keys(q, bank, min(N, RADIUS_FIRST_DEPTH, cap_search), "exact")
        stats["first"] += B
        esc, sat = settle(keys, None, keys.shape[1], True)
        saturated |= sat
        finish(keys, None, esc)
        go = esc.nonzero().view(-1)
        if go.numel():
            deeper.append((go, keys.index_select(0, go)))
    else:
        fp32 = mode in K.RESCORED_MODES
        if fp32:
            cfg = K.level_config(K._cascade_levels(bank, mode, track=False)[0], D)
            cand = K.effective_mode(cfg["cand"], D)
            with K._Timed("radius_admission"):
                tau0, refused = K.radius_tau0(q, bank, tau32, cfg, cand)
            refused = refused != 0
        else:
            cand = mode
            tau0 = torch.full((B,), float(admission_threshold(tau32)), dtype=torch.float32, device=dev)
            refused = None
        rows = None
        depths = radius_ladder(N, cap_search)
        for level, depth in enumerate(depths):
            ql = q if rows is None else q.index_select(0, rows)
            stats["first" if level == 0 else "second"] += ql.shape[0]
            with K._Timed("radius_candidates" if level == 0 else "radius_second"):
                keys = K.topk_keys(ql, bank, depth, cand, tau0=tau0 if rows is None else tau0[rows])
                if fp32:
                    with K._Timed("radius_rescore"):
                        keys = K.rescore_sparse(ql, bank, keys, cand, 0)
            esc, sat = settle(keys, rows, depth, not fp32)
            leave = esc | sat if fp32 else esc.clone()
            if not fp32:
                saturated[slice(None) if rows is None else rows] |= sat
            if refused is not None and rows is None:
                leave |= refused
                if bool(refused.any()):
                    deeper.append((refused.nonzero().view(-1), None))
            finish(keys, rows, leave)
            if fp32 and bool(sat.any()):
                certify.append(to_rows(sat, rows))
            rows = to_rows(esc, rows)
            if rows.numel() == 0:
                break
            if level == len(depths) - 1:
                deeper.append((rows, None))
    for rows in certify:
        # the approximate top-cap_search is not the exact one: the cascade's certified exact top list
        stats["certify"] += rows.numel()
        with K._Timed("radius_certify"):
            keys = K.topk_keys(q.index_select(0, rows), bank, cap_search, top_mode) if top_mode == "exact" else \
                K._topk_keys_rescored(q.index_select(0, rows), bank, cap_search, mode, track=False)
        _, sat = settle(keys, rows, cap_search, True)
        saturated[rows] |= sat
        pieces.append((keys, rows))
    if self_excl:
        bank_ids = torch.arange(N, dtype=torch.int32, device=dev) if deeper else None
        for rows, _ in deeper:
            stats["self_excluded"] += rows.numel()
            with K._Timed("radius_self_excluded"):
                keys = K.topk_keys(q.index_select(0, rows), bank, cap, top_mode,
                                   exclude=((rows + self_offset).to(torch.int32), bank_ids, 1))
            # a list of the bank without the row: it continues when its last key is a neighbour
            _, sat = settle(keys, rows, cap, True, n_bank=N - 1, depth_cap=cap)
            saturated[rows] |= sat
            pieces.append((keys, rows))
    for rows, first in peel:
        stats["peel"] += rows.numel()
        with K._Timed("radius_peel"):
            keys = _radius_peel(q.index_select(0, rows), bank, tau32, cap_search, first)
        _, sat = settle(keys, rows, keys.shape[1], True)
        saturated[rows] |= sat
        pieces.append((keys, rows))
    offsets = torch.zeros((B + 1,), dtype=torch.int64, device=dev)
    torch.cumsum(counts, 0, out=offsets[1:])
    nnz = int(offsets[-1])
    indices = torch.empty((nnz,), dtype=torch.int64, device=dev)
    sims = torch.empty((nnz,), dtype=torch.float32, device=dev)
    with K._Timed("radius_compact"):
        for keys, rows in pieces:
            K.radius_emit(keys, rows, tau32, self_offset, offsets, indices, sims)
    return RadiusNeighbors(offsets, indices, sims, saturated)


def _radius_args(threshold, max_per_row, mode):
    """(tau32, max_per_row or None, mode) after the checks every radius entry point makes first;
    resets last_radius_stats."""
    t = float(threshold)
    with np.errstate(over="ignore"):
        tau32 = np.float32(t) if math.isfinite(t) else np.float32(np.nan)
    if not math.isfinite(t) or not np.isfinite(tau32):
        raise ValueError(f"threshold must be finite in fp32, got {threshold!r}")
    if max_per_row is not None and int(max_per_row) < 1:
        raise ValueError(f"max_per_row must be >= 1 or None, got {max_per_row!r}")
    mode = mode or K.get_default_mode()
    if mode not in K.ALL_MODES:
        raise ValueError(f"unknown mode {mode!r}; expected one of {sorted(K.ALL_MODES)}")
    for level in last_radius_stats:  # a new public call: its own ladder statistics
        last_radius_stats[level] = 0
    return float(tau32), (None if max_per_row is None else int(max_per_row)), mode


def _empty_radius(B: int, device) -> RadiusNeighbors:
    return RadiusNeighbors(torch.zeros((B + 1,), dtype=torch.int64, device=device),
                           torch.empty((0,), dtype=torch.int64, device=device),
                           torch.empty((0,), dtype=torch.float32, device=device),
                           torch.zeros((B,), dtype=torch.bool, device=device))


def knn_radius(feature: torch.Tensor, feature_bank: torch.Tensor, threshold: float, mode: Optional[str] = None,
               max_per_row: Optional[int] = 992) -> RadiusNeighbors:
    """Every bank column n with sim(b, n) >= tau32 for every query row b, tau32 = fp32(threshold)
    rounded to nearest: the question ``knn_topk`` cannot ask ("everything closer than tau", e.g.
    which validation wafers have a near-copy in the bank).  feature (B, D) and feature_bank (D, N)
    as ``knn_topk`` takes them.  Returns ``RadiusNeighbors(offsets, indices, sims, saturated)``: CSR
    rows in the canonical (sim desc, index asc) order.  A row stops at max_per_row entries and
    saturated[b] says it did and may miss neighbours; max_per_row=None: no limit.

    Per mode: "exact" and every "fp32*" mode give bitwise the same rows, with the sequential-fma
    similarities of the "exact" mode (the fp32 modes search tensor-core candidates under a per-row
    threshold tau32 - E lowered by the bound E their certificate uses, then re-score them exactly).
    A raw tensor-core mode gives the columns whose similarity IN THAT MODE is >= tau32, bitwise the
    keys of ``topk_keys(..., mode)`` above tau32.  Rows deeper than MAX_K = 992 (max_per_row > 992
    only) come from the exact kernel's peeling in every mode, as ``topk_keys`` serves k > 992."""
    tau32, cap, mode = _radius_args(threshold, max_per_row, mode)
    K._check_feature_bank(feature, feature_bank)
    B, N = feature.shape[0], feature_bank.shape[1]
    if B == 0 or N == 0:
        return _empty_radius(B, feature.device)
    with torch.cuda.device(feature.device):
        return _radius_rows(feature, feature_bank, tau32, mode, N if cap is None else cap, -1)


def _radius_graph_batches(rows, threshold, normalize, mode, max_per_row, batch, include_self):
    """Yields (lo, RadiusNeighbors of rows lo..hi-1) of the self-join, after every argument check."""
    tau32, cap, mode = _radius_args(threshold, max_per_row, mode)
    K._require_cuda("rows", rows)
    if rows.dim() != 2:
        raise RuntimeError("rows must be (N, D)")
    if int(batch) <= 0:
        raise ValueError(f"batch must be positive, got {batch}")
    n = rows.shape[0]
    if n == 0:
        return
    fb = FeatureBank.from_rows(rows, normalize=normalize)
    with torch.cuda.device(rows.device):
        for lo in range(0, n, int(batch)):
            hi = min(n, lo + int(batch))
            yield lo, _radius_rows(fb.rows[lo:hi, :fb.dim], fb.bank, tau32, mode, n if cap is None else cap,
                                   -1 if include_self else lo)


def radius_graph(rows: torch.Tensor, threshold: float, normalize: bool = True, mode: Optional[str] = None,
                 max_per_row: Optional[int] = 992, batch: int = 75776,
                 include_self: bool = False) -> RadiusNeighbors:
    """The radius self-join of (N, D) rows (cosine when normalize=True), shaped like ``knn_graph``:
    ``knn_radius`` of every row against all rows, N CSR rows.  A row's own entry is dropped by
    index, unless include_self (an exact duplicate of lower index is another row and stays), and
    max_per_row counts the entries left.  The result does not depend on `batch`, the number of
    rows searched at once.  A row's own entry takes one slot of its search, so a row with
    max_per_row or more neighbours is searched again with itself left out inside the search
    (``topk_keys``' exclusion: the mode's own similarities, no peeling) when max_per_row <= 992;
    rows deeper than 992 are peeled by the exact kernel, as in ``knn_radius``."""
    parts = list(_radius_graph_batches(rows, threshold, normalize, mode, max_per_row, batch, include_self))
    if not parts:
        return _empty_radius(rows.shape[0], rows.device)
    if len(parts) == 1:
        return parts[0][1]
    base = [0]
    for _, r in parts[:-1]:
        base.append(base[-1] + r.indices.numel())
    offsets = torch.cat([parts[0][1].offsets[:1]] + [r.offsets[1:] + b for b, (_, r) in zip(base, parts)])
    return RadiusNeighbors(offsets, torch.cat([r.indices for _, r in parts]), torch.cat([r.sims for _, r in parts]),
                           torch.cat([r.saturated for _, r in parts]))


def near_duplicate_groups(rows: torch.Tensor, threshold: float, normalize: bool = True,
                          mode: Optional[str] = None, max_per_row: Optional[int] = 992,
                          batch: int = 75776) -> Tuple[torch.Tensor, int]:
    """(group_ids (N,) int64, n_saturated): the connected components of ``radius_graph(rows,
    threshold, ...)`` with its edges taken as undirected, each labelled by its smallest row index;
    n_saturated counts the rows whose radius row stopped at max_per_row (their missing edges can
    only split a group, never merge two).  Deterministic and independent of `batch`; the edges of
    each batch are unioned on the device as they come (b200knn_union_edges), so the edge list is
    never held whole.  The ids plug into the leave-one-group-out evaluation:

        groups, _ = near_duplicate_groups(rows, 0.999)
        knn_predict_loo(bank, labels, C, ks, groups=groups)

    Components chain (single linkage): rows a and c share a group when a ~ b ~ c even if a and c are
    far apart, so a low threshold merges whole clusters."""
    parent = None
    n_sat = None
    for lo, r in _radius_graph_batches(rows, threshold, normalize, mode, max_per_row, batch, False):
        if parent is None:
            parent = torch.arange(rows.shape[0], dtype=torch.int32, device=rows.device)
            flag = torch.zeros((1,), dtype=torch.int32, device=rows.device)
            n_sat = torch.zeros((), dtype=torch.int64, device=rows.device)
        with K._Timed("radius_union"):
            K.union_edges(parent, r.offsets, r.indices, lo, flag)
        n_sat += r.saturated.sum()
    if parent is None:
        return torch.empty((0,), dtype=torch.int64, device=rows.device), 0
    with K._Timed("radius_flatten"):
        labels = K.components(parent)
    if int(flag.item()):
        raise RuntimeError("near_duplicate_groups: a neighbour index is outside the rows")
    return labels, int(n_sat)
