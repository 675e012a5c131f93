"""On-device kNN validation metrics (SURVEY.md §8 f3).

The reference scores its kNN predictions after every validation epoch with torchmetrics
(``src/ssl_wafermap/models/knn.py:52-53, 104-129``): ``MulticlassAccuracy(average="macro")``,
``MulticlassF1Score(average="macro")`` and ``MulticlassConfusionMatrix(normalize="true")``,
followed by a ``.cpu().numpy()`` of the matrix.  Everything follows from the (C,C) count matrix,
which one small kernel (``b200knn_confusion``) builds from ``pred_labels[:, 0]`` and the
targets; the derived numbers stay on the device until the caller reads them.

torchmetrics semantics restated [recalled — torchmetrics is not installed here]:
  macro accuracy = mean over classes of recall_c = tp_c / (tp_c + fn_c),
  macro F1       = mean over classes of 2 tp_c / (2 tp_c + fp_c + fn_c),
  both with 0/0 := 0 and classes that occur neither in the predictions nor in the targets left
  out of the mean; normalize="true" divides every row (true class) by its sum, 0/0 := 0.
The tests check them against scikit-learn's recall_score / f1_score / confusion_matrix.
"""
from __future__ import annotations

from typing import Dict

import torch

from . import _lib
from . import knn as K


def confusion_counts(pred: torch.Tensor, target: torch.Tensor, num_classes: int) -> torch.Tensor:
    """(C, C) int64 counts[t, p] = #(target == t and pred == p)."""
    K._require_cuda("pred", pred)
    K._require_cuda("target", target)
    pred = pred.long().contiguous().view(-1)
    target = target.to(pred.device).long().contiguous().view(-1)
    if pred.numel() != target.numel():
        raise RuntimeError(f"pred has {pred.numel()} entries, target {target.numel()}")
    C = int(num_classes)
    counts = torch.zeros((C, C), dtype=torch.int64, device=pred.device)
    if pred.numel():
        with torch.cuda.device(pred.device):
            flag = torch.zeros((1,), dtype=torch.int32, device=pred.device)
            _lib.check(_lib.load().b200knn_confusion(pred.data_ptr(), target.data_ptr(), pred.numel(), C,
                                                     counts.data_ptr(), flag.data_ptr(), K._stream()), "confusion")
            if int(flag.item()):
                raise RuntimeError(f"a prediction or target is outside [0, num_classes={C})")
    return counts


def metrics_from_counts(counts: torch.Tensor) -> Dict[str, torch.Tensor]:
    """macro accuracy, macro F1 (0-dim fp64 tensors) and the row-normalised confusion matrix."""
    c = counts.double()
    tp = c.diagonal()
    support = c.sum(1)            # tp + fn
    predicted = c.sum(0)          # tp + fp
    present = (support + predicted) > 0
    n_present = present.sum().clamp(min=1)
    recall = torch.where(support > 0, tp / support.clamp(min=1), torch.zeros_like(tp))
    denom = support + predicted   # 2 tp + fp + fn
    f1 = torch.where(denom > 0, 2 * tp / denom.clamp(min=1), torch.zeros_like(tp))
    return {
        "accuracy": (recall * present).sum() / n_present,
        "f1": (f1 * present).sum() / n_present,
        "confusion": torch.where(support.view(-1, 1) > 0, c / support.clamp(min=1).view(-1, 1), torch.zeros_like(c)),
        "counts": counts,
    }


def knn_metrics(pred: torch.Tensor, target: torch.Tensor, num_classes: int) -> Dict[str, torch.Tensor]:
    """``on_validation_epoch_end`` of the reference (``knn.py:104-129``) for predictions
    ``pred_labels[:, 0]`` and their targets."""
    return metrics_from_counts(confusion_counts(pred, target, num_classes))


def multilabel_metrics_from_scores(scores: torch.Tensor, target: torch.Tensor,
                                   threshold: float = 0.5) -> Dict[str, torch.Tensor]:
    """Multi-label metrics of per-label scores (Q, L) against 0/1 targets (Q, L), on any device, with
    no host synchronisation.  A label is predicted when its score is > threshold.

      counts          (L, 4) int64: per label tp, fp, fn, tn
      f1_macro        mean over labels of 2 tp / (2 tp + fp + fn), 0/0 := 0, labels absent from both
                      the predictions and the targets left out (metrics_from_counts' convention)
      f1_micro        2 TP / (2 TP + FP + FN) over all labels, 0/0 := 0
      subset_accuracy share of rows whose predicted label set equals the target set
      hamming_loss    share of (row, label) cells predicted wrongly
      auc             (L,) fp64 ROC AUC per label: the Mann-Whitney statistic with average ranks for
                      ties; NaN for a label whose targets do not contain both values
      auc_macro       mean of auc over the labels where it is defined (NaN if there are none)
    The scalars are 0-dim fp64 tensors."""
    if scores.dim() != 2 or scores.shape != target.shape:
        raise RuntimeError(f"scores {tuple(scores.shape)} and target {tuple(target.shape)} must be the same (Q, L)")
    s = scores.double()
    pos = target != 0
    pred = s > threshold
    tp = (pred & pos).sum(0)
    fp = (pred & ~pos).sum(0)
    fn = (~pred & pos).sum(0)
    tn = (~pred & ~pos).sum(0)
    counts = torch.stack([tp, fp, fn, tn], dim=1)
    tp_d, fp_d, fn_d = tp.double(), fp.double(), fn.double()
    denom = 2 * tp_d + fp_d + fn_d
    present = denom > 0
    f1 = torch.where(present, 2 * tp_d / denom.clamp(min=1), torch.zeros_like(tp_d))
    micro_denom = denom.sum()
    cells = max(s.numel(), 1)
    # average ranks (1-based) within each label's column: (#below + #below-or-equal + 1) / 2
    cols = s.t().contiguous()
    srt = cols.sort(dim=1).values
    rank = (torch.searchsorted(srt, cols, right=False) + torch.searchsorted(srt, cols, right=True) + 1).double() / 2
    n_pos = pos.sum(0).double()
    n_neg = s.shape[0] - n_pos
    rank_sum = (rank * pos.t()).sum(1)
    defined = (n_pos > 0) & (n_neg > 0)
    auc = torch.where(defined, (rank_sum - n_pos * (n_pos + 1) / 2) / (n_pos * n_neg).clamp(min=1),
                      torch.full_like(rank_sum, float("nan")))
    return {
        "counts": counts,
        "f1_macro": (f1 * present).sum() / present.sum().clamp(min=1),
        "f1_micro": torch.where(micro_denom > 0, 2 * tp_d.sum() / micro_denom.clamp(min=1), micro_denom * 0),
        "subset_accuracy": (pred == pos).all(1).double().sum() / max(s.shape[0], 1),
        "hamming_loss": (pred != pos).double().sum() / cells,
        "auc": auc,
        "auc_macro": auc.nanmean() if auc.numel() else torch.tensor(float("nan"), dtype=torch.float64,
                                                                      device=s.device),
    }


def knn_multilabel_metrics(scores: torch.Tensor, target: torch.Tensor, threshold: float = 0.5) -> Dict[str, torch.Tensor]:
    """``multilabel_metrics_from_scores`` on the device for ``knn_predict_multilabel``'s scores [i, j]
    (Q, L) and the queries' 0/1 label matrix (Q, L), bool or integer (a non-zero entry is a positive):
    per-label counts, macro / micro F1, subset accuracy, Hamming loss and per-label / macro ROC AUC."""
    K._require_cuda("scores", scores)
    K._require_cuda("target", target)
    if target.dtype.is_floating_point or target.dtype.is_complex:
        raise RuntimeError(f"target must be bool or integer 0/1 entries, got {target.dtype}")
    return multilabel_metrics_from_scores(scores, target.to(scores.device), threshold)
