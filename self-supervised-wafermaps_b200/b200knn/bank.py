"""FeatureBank — the bank build of the reference's validation epoch, laid out for the kernels.

The reference builds its bank in ``KNNBenchmarkModule.on_validation_epoch_start``
(``src/ssl_wafermap/models/knn.py:67-81``): per dataloader batch ``F.normalize(feature, dim=1)``
(``:77``), then ``torch.cat(...).t().contiguous()`` (``:80``) — an (N,D) fp32 concatenation, an
(N,D) normalised copy and a (D,N) transposed copy, which ``knn_predict`` then has to re-lay-out
again for the tensor cores.  ``FeatureBank`` does the normalisation and the relayout in ONE
kernel (``b200knn_normalize_rows``: rows -> zero-padded (N, D_pad) fp32 rows) and hands the
result to the kernels as it is; the (D,N) tensor the reference interface expects is exposed as
a zero-copy view (``.bank``), so every ``b200knn`` entry point — and the reference's own
``knn_predict(feature, bank.bank, bank.labels, ...)`` call — works on it unchanged.

SURVEY.md §8(f1).  CUDA only, like the rest of the path.
"""
from __future__ import annotations

from typing import Iterable, List, Optional, Tuple

import torch

from . import knn as K


class FeatureBank:
    def __init__(self, rows_padded: torch.Tensor, dim: int, labels: Optional[torch.Tensor] = None):
        if rows_padded.dim() != 2 or rows_padded.dtype != torch.float32 or not rows_padded.is_contiguous() \
                or rows_padded.shape[1] != K.padded_dim(dim):
            raise ValueError("rows_padded must be contiguous (N, padded_dim(dim)) fp32 with zero pad columns")
        self.rows = rows_padded                     # (N, D_pad) fp32: exact-mode operand and re-scoring rows
        self.dim = int(dim)
        self.bank = rows_padded[:, :dim].t()        # (D, N) view: the reference's feature_bank interface
        self.labels = labels
        K.register_padded_rows(self.bank, rows_padded)

    # ------------------------------------------------------------------ construction
    @classmethod
    def from_rows(cls, rows: torch.Tensor, labels: Optional[torch.Tensor] = None,
                  normalize: bool = True) -> "FeatureBank":
        """rows: (N, D) embeddings (fp32/fp16/bf16, CUDA).  normalize=True applies the reference's
        ``F.normalize(dim=1)`` (``knn.py:77``) in the same kernel that lays the rows out."""
        K._require_cuda("rows", rows)
        if rows.dim() != 2:
            raise RuntimeError("rows must be (N, D)")
        dim = rows.shape[1]
        if normalize:
            padded = K.normalize_rows(rows)._base
        else:
            padded = K.prepare_rows(rows, "f32rows", vectors_are_columns=False).hi
        if labels is not None:
            labels = labels.to(rows.device).long().contiguous().view(-1)
            if labels.numel() != rows.shape[0]:
                raise RuntimeError(f"labels has {labels.numel()} entries for {rows.shape[0]} rows")
        return cls(padded, dim, labels)

    @classmethod
    def from_batches(cls, batches: Iterable[Tuple[torch.Tensor, torch.Tensor]], normalize: bool = True,
                     total_rows: Optional[int] = None) -> "FeatureBank":
        """The loop of ``on_validation_epoch_start`` (``knn.py:70-81``): (features, targets) per
        dataloader batch.  Each batch is normalised and laid out by one kernel straight into its
        slice of ONE (N, D_pad) buffer — the reference's list of per-batch tensors, its ``torch.cat``
        copy and its ``.t().contiguous()`` copy never exist.  total_rows (``len(dataloader.dataset)``)
        sizes the buffer up front; without it (or if more rows arrive) the buffer grows geometrically."""
        buf: Optional[torch.Tensor] = None
        labs: Optional[torch.Tensor] = None
        n = 0
        dim = None
        for feat, target in batches:
            K._require_cuda("feature batch", feat)
            if feat.dim() != 2:
                raise RuntimeError("feature batches must be (b, D)")
            b = feat.shape[0]
            if dim is None:
                dim = feat.shape[1]
                cap = max(int(total_rows or 0), b)
                buf = torch.empty((cap, K.padded_dim(dim)), dtype=torch.float32, device=feat.device)
                labs = torch.empty((cap,), dtype=torch.int64, device=feat.device)
            elif feat.shape[1] != dim:
                raise RuntimeError(f"feature batch has dimension {feat.shape[1]}, expected {dim}")
            if n + b > buf.shape[0]:
                cap = max(n + b, 2 * buf.shape[0])
                buf = torch.cat([buf[:n], torch.empty((cap - n, buf.shape[1]), dtype=buf.dtype, device=buf.device)])
                labs = torch.cat([labs[:n], torch.empty((cap - n,), dtype=labs.dtype, device=labs.device)])
            if normalize:
                K.normalize_rows(feat, out=buf[n:n + b])
            else:
                buf[n:n + b] = K.prepare_rows(feat, "f32rows", vectors_are_columns=False).hi
            labs[n:n + b] = target.to(feat.device).view(-1)
            n += b
        if dim is None:
            raise RuntimeError("no batches")
        return cls(buf[:n], dim, labs[:n])

    # ------------------------------------------------------------------ the reference's calls
    @property
    def n_rows(self) -> int:
        return self.rows.shape[0]

    def _queries(self, feature: torch.Tensor, normalize: bool) -> torch.Tensor:
        return K.normalize_rows(feature) if normalize else feature  # knn.py:90

    def knn_predict(self, feature: torch.Tensor, num_classes: int, knn_k: int = 200, knn_t: float = 0.1,
                    normalize: bool = False) -> torch.Tensor:
        """``validation_step``'s kNN call (``knn.py:90-98``); normalize=True also fuses its
        ``F.normalize(feature, dim=1)``."""
        if self.labels is None:
            raise RuntimeError("this FeatureBank was built without labels")
        return K.knn_predict(self._queries(feature, normalize), self.bank, self.labels, num_classes, knn_k, knn_t)

    def knn_predict_multi(self, feature: torch.Tensor, num_classes: int, knn_ks=(200,), knn_ts=(0.1,),
                          normalize: bool = False, query_groups: Optional[torch.Tensor] = None,
                          bank_groups: Optional[torch.Tensor] = None) -> torch.Tensor:
        """``knn_predict`` over a (knn_ks, knn_ts) grid from one neighbour search (``K.knn_predict_multi``):
        (len(knn_ks), len(knn_ts), B, C); normalize=True fuses the query ``F.normalize``.
        query_groups (B,) / bank_groups (N,): each query's group left out of its search."""
        if self.labels is None:
            raise RuntimeError("this FeatureBank was built without labels")
        return K.knn_predict_multi(self._queries(feature, normalize), self.bank, self.labels, num_classes,
                                   knn_ks, knn_ts, query_groups, bank_groups)

    def knn_predict_loo(self, num_classes: int, knn_ks=(200,), knn_ts=(0.1,), batch: int = 75776,
                        groups: Optional[torch.Tensor] = None) -> torch.Tensor:
        """Leave-one-out class rankings of the bank's own rows and labels (``K.knn_predict_loo``):
        (len(knn_ks), len(knn_ts), N, C).  The queries are views of the padded rows, no copy.
        groups: (N,) integer ids, each row's whole group left out of its vote."""
        if self.labels is None:
            raise RuntimeError("this FeatureBank was built without labels")
        return K.knn_predict_loo(self.bank, self.labels, num_classes, knn_ks, knn_ts, batch, groups)

    def knn_topk(self, feature: torch.Tensor, k: int, normalize: bool = False, mode: Optional[str] = None,
                 query_groups: Optional[torch.Tensor] = None, bank_groups: Optional[torch.Tensor] = None):
        return K.knn_topk(self._queries(feature, normalize), self.bank, k, mode, query_groups, bank_groups)
