"""A stand-in for the reference's ``KNNBenchmarkModule`` (``src/ssl_wafermap/models/knn.py:28-138``)
for driving the hooks on the GPU without pytorch_lightning and torchmetrics.

TEST INFRASTRUCTURE, like the oracle: it restates the three validation hooks' data flow (what the
hooks read and write on the module: ``backbone``, ``dataloader_kNN``, ``num_classes``, ``knn_k``,
``knn_t``, ``feature_bank`` (D,N), ``targets_bank``, ``all_preds`` / ``all_targets``,
``max_accuracy`` / ``max_f1``, ``confusion_matrix``, ``log``) so that ``b200knn.install(hooks=True,
hook_classes=(StandInKNNModule,))`` can be driven end to end and compared with the un-hooked flow.
The un-hooked hooks look the module-global ``knn_predict`` up at call time, exactly like the
reference does after ``from lightly.utils.benchmarking import knn_predict`` (``knn.py:16``).
tests/test_hooks_cpu.py runs the same comparison on CPU against the reference's module file as
restated in tests/reference_knn.py, imported with its third-party dependencies stubbed.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F

from oracle import knn_oracle as O

knn_predict = None  # bound by the test (b200knn.knn_predict, or the oracle's R32 on CPU)
normalize = F.normalize  # the test may inject the oracle's bit-defined normalisation


class StandInKNNModule(nn.Module):
    def __init__(self, dataloader_kNN, num_classes, knn_k=5, knn_t=0.1):
        super().__init__()
        self.backbone = nn.Identity()
        self.max_accuracy = 0.0
        self.max_f1 = 0.0
        self.dataloader_kNN = dataloader_kNN
        self.num_classes = num_classes
        self.knn_k = knn_k
        self.knn_t = knn_t
        self.confusion_matrix = []
        self.all_preds = []
        self.all_targets = []
        self.logged = {}
        self._device = torch.device("cpu")

    @property
    def device(self):
        return self._device

    def log(self, name, value, **kw):
        self.logged[name] = float(value)

    def on_validation_epoch_start(self):           # data flow of knn.py:67-81
        feats, targets = [], []
        for img, target in self.dataloader_kNN:
            feats.append(normalize(self.backbone(img.to(self.device)).squeeze(), dim=1))
            targets.append(target.to(self.device))
        self.feature_bank = torch.cat(feats, dim=0).t().contiguous()
        self.targets_bank = torch.cat(targets, dim=0).t().contiguous()

    def validation_step(self, batch, batch_idx):   # data flow of knn.py:87-101
        images, targets = batch
        feature = normalize(self.backbone(images).squeeze(), dim=1)
        pred_labels = knn_predict(feature, self.feature_bank, self.targets_bank, self.num_classes, self.knn_k,
                                  self.knn_t)
        self.all_preds.append(pred_labels[:, 0])
        self.all_targets.append(targets)

    def on_validation_epoch_end(self):             # data flow of knn.py:104-133 (torchmetrics -> oracle restatement)
        p = torch.cat(self.all_preds).cpu().numpy()
        t = torch.cat(self.all_targets).cpu().numpy()
        m = O.metrics_ref(p, t, self.num_classes)
        self.max_accuracy = max(self.max_accuracy, float(m["accuracy"]))
        self.max_f1 = max(self.max_f1, float(m["f1"]))
        self.log("knn_accuracy", m["accuracy"])
        self.log("knn_f1", m["f1"])
        self.confusion_matrix.append(np.asarray(m["confusion"]))
        self.all_preds.clear()
        self.all_targets.clear()


def run_validation_epoch(module, val_batches):
    module.on_validation_epoch_start()
    for i, batch in enumerate(val_batches):
        module.validation_step(batch, i)
    preds = torch.cat(module.all_preds).clone()
    module.on_validation_epoch_end()
    return preds
