"""Replacement validation hooks for the reference's ``KNNBenchmarkModule`` (SURVEY.md §8 f1/f3).

``b200knn.install(hooks=True)`` patches, on ``ssl_wafermap.models.knn.KNNBenchmarkModule`` (and the
copy of that class ``scripts/WM811k_benchmark.py`` defines for itself),

    on_validation_epoch_start   knn.py:67-81    bank build: per-batch ``F.normalize`` + ``torch.cat`` +
                                                ``.t().contiguous()``  ->  ``FeatureBank.from_batches``
                                                (one kernel per batch, straight into ONE (N, D_pad) buffer)
    validation_step             knn.py:87-101   ``F.normalize`` + ``knn_predict`` + ``pred[:, 0]``
                                                ->  ``FeatureBank.knn_predict(normalize=True)``
    on_validation_epoch_end     knn.py:104-133  torchmetrics accuracy / F1 / confusion matrix
                                                ->  ``knn_metrics`` (one confusion-count kernel)

and on ``WandBKNNBenchmarkModule`` (``knn.py:181-215``) the first two — its epoch-end hook also draws
and uploads a W&B figure (``knn.py:241-272``), which is not this path and stays as it is.

The hooks keep the module's observable state: ``feature_bank`` ((D,N), a zero-copy view),
``targets_bank``, ``all_preds`` / ``all_targets``, ``max_accuracy`` / ``max_f1``, the
``knn_accuracy`` / ``knn_f1`` log keys and the ``confusion_matrix`` list of numpy arrays.

Opt-in kNN grid: a module with ``b200knn_knn_grid = (ks, ts)`` is scored in ``validation_step`` by one
``FeatureBank.knn_predict_multi`` over ks x ts extended by its own (knn_k, knn_t); its state above
stays that of its own setting, and ``on_validation_epoch_end`` also logs ``knn_accuracy_k{k}_t{t}`` and
``knn_f1_k{k}_t{t}`` for every setting of the extended grid.
"""
from __future__ import annotations

import sys
from typing import Dict, List, Tuple

import torch

from . import bank as _bank
from . import metrics as _metrics

_EPOCH_HOOKS = ("on_validation_epoch_start", "validation_step", "on_validation_epoch_end")
_TARGETS = {
    "KNNBenchmarkModule": _EPOCH_HOOKS,
    "WandBKNNBenchmarkModule": _EPOCH_HOOKS[:2],
}
_MODULES = ("ssl_wafermap.models.knn", "__main__")

_saved: List[Tuple[type, str, object]] = []


def _total_rows(loader):
    try:
        return len(loader.dataset)
    except Exception:
        return None


def on_validation_epoch_start(self):
    def batches():
        for img, target in self.dataloader_kNN:
            img = img.to(self.device)
            yield self.backbone(img).squeeze(), target.to(self.device)

    fb = _bank.FeatureBank.from_batches(batches(), normalize=True, total_rows=_total_rows(self.dataloader_kNN))
    self._b200knn_bank = fb
    self.__dict__.pop("_b200knn_grid_preds", None)  # an epoch whose end hook is not ours (W&B twin)
    self.feature_bank = fb.bank        # (D, N): what the reference's own knn_predict call would read
    self.targets_bank = fb.labels


def _grid(self):
    """The module's opt-in ``b200knn_knn_grid = (ks, ts)`` extended by its own (knn_k, knn_t), or None."""
    grid = getattr(self, "b200knn_knn_grid", None)
    if grid is None:
        return None
    ks, ts = [int(k) for k in grid[0]], [float(t) for t in grid[1]]
    if int(self.knn_k) not in ks:
        ks.append(int(self.knn_k))
    if float(self.knn_t) not in ts:
        ts.append(float(self.knn_t))
    return ks, ts


def validation_step(self, batch, batch_idx):
    images, targets = batch
    feature = self.backbone(images).squeeze()
    grid = _grid(self)
    if grid is None:
        pred_labels = self._b200knn_bank.knn_predict(feature, self.num_classes, self.knn_k, self.knn_t,
                                                     normalize=True)
    else:
        # every setting of the grid from one neighbour search; the module's own setting is one of them
        ks, ts = grid
        pred = self._b200knn_bank.knn_predict_multi(feature, self.num_classes, ks, ts, normalize=True)
        pred_labels = pred[ks.index(int(self.knn_k)), ts.index(float(self.knn_t))]
        preds = self.__dict__.setdefault("_b200knn_grid_preds", {})
        for i, k in enumerate(ks):
            for j, t in enumerate(ts):
                preds.setdefault((k, t), []).append(pred[i, j, :, 0])
    self.all_preds.append(pred_labels[:, 0])
    self.all_targets.append(targets)


def on_validation_epoch_end(self):
    all_preds = torch.cat(self.all_preds, dim=0)
    all_targets = torch.cat(self.all_targets, dim=0)
    m = _metrics.knn_metrics(all_preds, all_targets, self.num_classes)
    acc, f1 = float(m["accuracy"]), float(m["f1"])
    if acc > self.max_accuracy:
        self.max_accuracy = acc
    if f1 > self.max_f1:
        self.max_f1 = f1
    self.log("knn_accuracy", acc, on_epoch=True, prog_bar=True)
    self.log("knn_f1", f1, on_epoch=True, prog_bar=True)
    self.confusion_matrix.append(m["confusion"].detach().cpu().numpy())
    for (k, t), preds in self.__dict__.pop("_b200knn_grid_preds", {}).items():
        g = _metrics.knn_metrics(torch.cat(preds, dim=0), all_targets, self.num_classes)
        self.log(f"knn_accuracy_k{k}_t{t:g}", float(g["accuracy"]), on_epoch=True)
        self.log(f"knn_f1_k{k}_t{t:g}", float(g["f1"]), on_epoch=True)
    self.all_preds.clear()
    self.all_targets.clear()


_IMPL = {"on_validation_epoch_start": on_validation_epoch_start, "validation_step": validation_step,
         "on_validation_epoch_end": on_validation_epoch_end}


def patch_class(cls: type, hook_names=_EPOCH_HOOKS) -> None:
    """Replace the named hooks of one module class (idempotent)."""
    for name in hook_names:
        cur = cls.__dict__.get(name)
        if cur is _IMPL[name]:
            continue
        _saved.append((cls, name, cur))
        setattr(cls, name, _IMPL[name])


def install_hooks(extra_classes: Tuple[type, ...] = ()) -> Dict[str, bool]:
    """Patch every reference kNN module class that is importable / already imported."""
    done: Dict[str, bool] = {}
    for mod_name in _MODULES:
        mod = sys.modules.get(mod_name)
        if mod is None and mod_name != "__main__":
            try:
                mod = __import__(mod_name, fromlist=["KNNBenchmarkModule"])
            except Exception:
                mod = None
        for cls_name, hook_names in _TARGETS.items():
            cls = getattr(mod, cls_name, None) if mod is not None else None
            ok = isinstance(cls, type) and all(hasattr(cls, h) for h in hook_names)
            if ok:
                patch_class(cls, hook_names)
            done[f"{mod_name}.{cls_name}"] = bool(ok)
    for cls in extra_classes:
        patch_class(cls)
        done[f"{cls.__module__}.{cls.__name__}"] = True
    return done


def uninstall_hooks() -> None:
    while _saved:
        cls, name, orig = _saved.pop()
        if orig is None:
            delattr(cls, name)
        else:
            setattr(cls, name, orig)
