"""The slice of the reference project's ``src/ssl_wafermap/models/knn.py`` (faris-k/self-supervised-wafermaps)
that ``b200knn.install(hooks=True)`` acts on, restated so that tests/test_hooks_cpu.py runs from this
repository alone.  That test imports this file as ``ssl_wafermap.models.knn`` with the third-party
modules below stubbed out, as it would import the reference's own file.

TEST INFRASTRUCTURE, like the oracle.  It keeps what the hooks and ``install()`` depend on:
  * the module-level ``from lightly.utils.benchmarking import knn_predict`` (``knn.py:16``), looked up
    at call time by ``validation_step``;
  * ``KNNBenchmarkModule`` (``knn.py:28-138``): constructor arguments and state, the bank build
    (``:67-81``: per-batch ``F.normalize``, ``cat``, ``.t().contiguous()``), the query step
    (``:87-101``: ``F.normalize``, ``knn_predict``, ``pred_labels[:, 0]``) and the torchmetrics
    epoch end (``:104-133``);
  * ``WandBKNNBenchmarkModule`` (``knn.py:142-281``): the same two first hooks, and an epoch end that
    also draws and uploads the confusion matrix to W&B;
  * one of the model classes that subclass ``KNNBenchmarkModule`` (``knn.py:284-1116``).
"""
import matplotlib.pyplot as plt
import pytorch_lightning as pl
import seaborn as sns
import torch
import torch.nn as nn
import torch.nn.functional as F
import wandb
from lightly.models.modules import heads
from lightly.utils.benchmarking import knn_predict
from torchmetrics.classification import MulticlassAccuracy, MulticlassConfusionMatrix, MulticlassF1Score


class KNNBenchmarkModule(pl.LightningModule):
    def __init__(self, dataloader_kNN, num_classes, knn_k=5, knn_t=0.1):
        super().__init__()
        self.backbone = nn.Module()
        self.max_accuracy = 0.0
        self.max_f1 = 0.0
        self.dataloader_kNN = dataloader_kNN
        self.num_classes = num_classes
        self.knn_k = knn_k
        self.knn_t = knn_t
        self.confusion_matrix = []
        self.all_preds = []
        self.all_targets = []

    def on_validation_epoch_start(self):
        train_feature_bank = []
        train_targets_bank = []
        with torch.no_grad():
            for img, target in self.dataloader_kNN:
                img = img.to(self.device)
                target = target.to(self.device)
                feature = self.backbone(img).squeeze()
                feature = F.normalize(feature, dim=1)
                train_feature_bank.append(feature)
                train_targets_bank.append(target)
        self.feature_bank = torch.cat(train_feature_bank, dim=0).t().contiguous()
        self.targets_bank = torch.cat(train_targets_bank, dim=0).t().contiguous()

    def validation_step(self, batch, batch_idx):
        if hasattr(self, "feature_bank") and hasattr(self, "targets_bank"):
            images, targets = batch
            feature = self.backbone(images).squeeze()
            feature = F.normalize(feature, dim=1)
            pred_labels = knn_predict(
                feature, self.feature_bank, self.targets_bank, self.num_classes, self.knn_k, self.knn_t
            )
            self.all_preds.append(pred_labels[:, 0])
            self.all_targets.append(targets)

    def _epoch_metrics(self):
        all_preds = torch.cat(self.all_preds, dim=0)
        all_targets = torch.cat(self.all_targets, dim=0)
        accuracy = MulticlassAccuracy(num_classes=self.num_classes, average="macro").to(self.device)
        f1 = MulticlassF1Score(num_classes=self.num_classes, average="macro").to(self.device)
        confmat = MulticlassConfusionMatrix(num_classes=self.num_classes, normalize="true").to(self.device)
        acc = accuracy(all_preds, all_targets).item()
        f1_score = f1(all_preds, all_targets).item()
        if acc > self.max_accuracy:
            self.max_accuracy = acc
        if f1_score > self.max_f1:
            self.max_f1 = f1_score
        self.log("knn_accuracy", acc, on_epoch=True, prog_bar=True)
        self.log("knn_f1", f1_score, on_epoch=True, prog_bar=True)
        cm = confmat(all_preds, all_targets).cpu().numpy()
        self.confusion_matrix.append(cm)
        self.all_preds.clear()
        self.all_targets.clear()
        return cm

    def on_validation_epoch_end(self):
        self._epoch_metrics()


class WandBKNNBenchmarkModule(pl.LightningModule):
    def __init__(self, dataloader_kNN, num_classes, knn_k=5, knn_t=0.1):
        super().__init__()
        self.backbone = nn.Module()
        self.max_accuracy = 0.0
        self.max_f1 = 0.0
        self.dataloader_kNN = dataloader_kNN
        self.num_classes = num_classes
        self.knn_k = knn_k
        self.knn_t = knn_t
        self.confusion_matrix = []
        self.all_preds = []
        self.all_targets = []

    on_validation_epoch_start = KNNBenchmarkModule.on_validation_epoch_start
    validation_step = KNNBenchmarkModule.validation_step
    _epoch_metrics = KNNBenchmarkModule._epoch_metrics

    def on_validation_epoch_end(self):
        cm = self._epoch_metrics()
        fig, ax = plt.subplots(figsize=(8, 8))
        sns.heatmap(cm, annot=True, fmt=".2f", ax=ax)
        wandb.log({"confusion_matrix": wandb.Image(fig)})
        plt.close(fig)


class SimCLR(KNNBenchmarkModule):
    def __init__(self, dataloader_kNN, num_classes, knn_k=5, knn_t=0.1):
        super().__init__(dataloader_kNN, num_classes, knn_k, knn_t)
        self.backbone = nn.Identity()
        self.projection_head = heads.SimCLRProjectionHead(512, 512, 128)
