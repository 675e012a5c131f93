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

from typing import Optional, Tuple

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
