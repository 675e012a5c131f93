"""CPU: b200knn.install(hooks=True) against the reference's kNN module file
(src/ssl_wafermap/models/knn.py, restated in tests/reference_knn.py and imported under the
reference's module name with its absent third-party dependencies — lightly, pytorch_lightning,
timm, torchmetrics, wandb, matplotlib, seaborn — stubbed out).  Checks that the reference's classes
get their three validation hooks replaced (KNNBenchmarkModule) / two (WandBKNNBenchmarkModule,
whose epoch-end also draws a W&B figure), that the module global `knn_predict` is rebound, and —
with the CUDA-only compute steps served by the oracle — that one validation epoch through the hooks
gives the un-hooked flow's predictions and metrics
(tests/test_gpu_round2.py::test_hooks_equal_unhooked_flow drives the hooks on the device)."""
import importlib.util
import os
import sys
import types

import numpy as np
import pytest
import torch
import torch.nn as nn

import datagen
from oracle import knn_oracle as O

REF_FILE = os.path.join(os.path.dirname(os.path.abspath(__file__)), "reference_knn.py")


class _Anything:
    """Stands for any class / function / constant of a stubbed third-party module."""

    def __init__(self, *a, **k):
        pass

    def __call__(self, *a, **k):
        return _Anything()

    def __getattr__(self, name):
        return _Anything()

    def __mro_entries__(self, bases):
        return (nn.Module,)


class _StubModule(types.ModuleType):
    def __getattr__(self, name):
        if name.startswith("__"):
            raise AttributeError(name)
        return _Anything()


class _LightningModule(nn.Module):
    """The slice of pl.LightningModule the kNN hooks use."""

    def __init__(self):
        super().__init__()
        self.logged = {}

    @property
    def device(self):
        return torch.device("cpu")

    def log(self, name, value, **kw):
        self.logged[name] = value


class _Metric:
    def __init__(self, *a, **k):
        pass

    def to(self, *a):
        return self


STUBS = ["lightly", "lightly.models", "lightly.models.modules", "lightly.utils", "lightly.utils.benchmarking",
         "matplotlib", "matplotlib.pyplot", "pytorch_lightning", "seaborn", "timm", "timm.optim", "timm.optim.lars",
         "wandb", "torchmetrics", "torchmetrics.classification", "ssl_wafermap", "ssl_wafermap.models"]


@pytest.fixture()
def reference_module():
    saved = {n: sys.modules.get(n) for n in STUBS + ["ssl_wafermap.models.knn"]}
    for n in STUBS:
        sys.modules[n] = _StubModule(n)
    sys.modules["pytorch_lightning"].LightningModule = _LightningModule
    sys.modules["lightly.utils.benchmarking"].knn_predict = O.knn_predict_r32  # what lightly would provide
    for cls in ("MulticlassAccuracy", "MulticlassConfusionMatrix", "MulticlassF1Score"):
        setattr(sys.modules["torchmetrics.classification"], cls, _Metric)
    spec = importlib.util.spec_from_file_location("ssl_wafermap.models.knn", REF_FILE)
    mod = importlib.util.module_from_spec(spec)
    sys.modules["ssl_wafermap.models.knn"] = mod
    spec.loader.exec_module(mod)
    try:
        yield mod
    finally:
        import b200knn

        b200knn.uninstall()
        for n, m in saved.items():
            if m is None:
                sys.modules.pop(n, None)
            else:
                sys.modules[n] = m


class _OracleBank:
    """FeatureBank's interface (from_batches / knn_predict / bank / labels) served by the oracle."""

    def __init__(self, rows, labels):
        self.rows, self.labels = rows, labels
        self.bank = rows.t()

    @classmethod
    def from_batches(cls, batches, normalize=True, total_rows=None):
        feats, labs = zip(*[(f, t) for f, t in batches])
        rows = torch.from_numpy(O.normalize_rows_ref(torch.cat(feats).numpy()))
        cls.last_total_rows = total_rows
        return cls(rows, torch.cat(labs).long())

    def knn_predict(self, feature, num_classes, knn_k=200, knn_t=0.1, normalize=False):
        q = O.normalize_rows_ref(feature.numpy()) if normalize else feature.numpy()
        s, i = O.topk_seqfma(q, np.ascontiguousarray(self.rows.numpy().T), knn_k)
        return torch.from_numpy(O.vote_o64(s, i, self.labels.numpy(), num_classes, knn_t)[0])


def _oracle_metrics(pred, target, num_classes):
    m = O.metrics_ref(pred.numpy(), target.numpy(), num_classes)
    return {"accuracy": torch.tensor(m["accuracy"], dtype=torch.float64), "f1": torch.tensor(m["f1"], dtype=torch.float64),
            "confusion": torch.from_numpy(m["confusion"]), "counts": torch.from_numpy(m["counts"])}


class _Loader(list):
    """A list of batches with the `.dataset` attribute the hooks size the bank from."""

    def __init__(self, batches, n):
        super().__init__(batches)
        self.dataset = range(n)


def test_install_hooks_patches_the_reference_classes(reference_module, monkeypatch):
    import b200knn

    ref = reference_module
    orig = {(c, h): getattr(getattr(ref, c), h) for c in ("KNNBenchmarkModule", "WandBKNNBenchmarkModule")
            for h in ("on_validation_epoch_start", "validation_step", "on_validation_epoch_end")}
    done = b200knn.install(hooks=True)
    assert done["ssl_wafermap.models.knn"] and ref.knn_predict is b200knn.knn_predict
    assert done["ssl_wafermap.models.knn.KNNBenchmarkModule"] and done["ssl_wafermap.models.knn.WandBKNNBenchmarkModule"]
    H = b200knn.hooks
    assert ref.KNNBenchmarkModule.on_validation_epoch_start is H.on_validation_epoch_start
    assert ref.KNNBenchmarkModule.validation_step is H.validation_step
    assert ref.KNNBenchmarkModule.on_validation_epoch_end is H.on_validation_epoch_end
    assert ref.WandBKNNBenchmarkModule.on_validation_epoch_start is H.on_validation_epoch_start
    assert ref.WandBKNNBenchmarkModule.validation_step is H.validation_step
    # the W&B twin keeps its own epoch-end hook (it also draws and uploads the confusion-matrix figure)
    assert ref.WandBKNNBenchmarkModule.on_validation_epoch_end is orig[("WandBKNNBenchmarkModule", "on_validation_epoch_end")]
    # subclasses (the 16 model classes of knn.py:284-1116) inherit the patched hooks
    assert ref.SimCLR.validation_step is H.validation_step
    b200knn.install(hooks=True)  # idempotent
    b200knn.uninstall()
    for (c, h), fn in orig.items():
        assert getattr(getattr(ref, c), h) is fn
    assert ref.knn_predict is O.knn_predict_r32


def test_hooked_epoch_equals_reference_epoch(reference_module, monkeypatch):
    """One validation epoch of the reference's KNNBenchmarkModule, un-hooked (its own code with
    lightly's knn_predict = the oracle's R32) and hooked (compute served by the oracle through
    FeatureBank's interface): same predictions, metrics, confusion matrix, module state."""
    import b200knn

    ref = reference_module
    C, D, n_bank, n_val, bs = 9, 64, 700, 200, 64
    rng = np.random.default_rng(5)
    lab = datagen.labels(n_bank, C, 1)
    emb = (datagen.clustered(n_bank, D, C, 2, lab) * rng.uniform(0.5, 9, (n_bank, 1))).astype(np.float32)
    vlab = datagen.labels(n_val, C, 3)
    vemb = (datagen.clustered(n_val, D, C, 4, vlab) * rng.uniform(0.5, 9, (n_val, 1))).astype(np.float32)
    loader = _Loader([(torch.from_numpy(emb[i:i + bs]), torch.from_numpy(lab[i:i + bs])) for i in range(0, n_bank, bs)], n_bank)
    val = [(torch.from_numpy(vemb[i:i + bs]), torch.from_numpy(vlab[i:i + bs])) for i in range(0, n_val, bs)]

    def epoch(module, with_end):
        module.backbone = nn.Identity()
        module.on_validation_epoch_start()
        for i, b in enumerate(val):
            module.validation_step(b, i)
        preds, targets = torch.cat(module.all_preds).clone(), torch.cat(module.all_targets).clone()
        if with_end:
            module.on_validation_epoch_end()
        return preds, targets

    plain = ref.KNNBenchmarkModule(loader, C, knn_k=5, knn_t=0.1)
    p0, t0 = epoch(plain, with_end=False)  # the reference's epoch-end needs torchmetrics: compared via the oracle
    assert plain.feature_bank.shape == (D, n_bank) and plain.targets_bank.shape == (n_bank,)

    b200knn.install(hooks=True)
    monkeypatch.setattr(b200knn.hooks._bank, "FeatureBank", _OracleBank)
    monkeypatch.setattr(b200knn.hooks._metrics, "knn_metrics", _oracle_metrics)
    hooked = ref.KNNBenchmarkModule(loader, C, knn_k=5, knn_t=0.1)
    p1, t1 = epoch(hooked, with_end=True)
    assert _OracleBank.last_total_rows == n_bank
    assert torch.equal(t0, t1)
    # R32 (torch CPU mm + topk) and the sequential-fma oracle agree except on fp32 near-ties
    assert float((p0 == p1).float().mean()) >= 0.99
    assert hooked.feature_bank.shape == (D, n_bank) and torch.equal(hooked.targets_bank, plain.targets_bank)
    assert float((hooked.feature_bank - plain.feature_bank).abs().max()) <= 2.5e-7
    want = O.metrics_ref(p1.numpy(), t1.numpy(), C)
    assert abs(hooked.max_accuracy - want["accuracy"]) < 1e-12 and abs(hooked.max_f1 - want["f1"]) < 1e-12
    assert abs(hooked.logged["knn_accuracy"] - want["accuracy"]) < 1e-12
    assert abs(hooked.logged["knn_f1"] - want["f1"]) < 1e-12
    assert len(hooked.confusion_matrix) == 1 and np.allclose(hooked.confusion_matrix[0], want["confusion"])
    assert hooked.all_preds == [] and hooked.all_targets == []
