"""CPU: multi-label kNN — the C ABI's argument checks of b200knn_vote_multilabel, the Python argument
errors of knn_predict_multilabel (all raised before any search), the label bitmask packing, and the
multi-label metric arithmetic against scikit-learn."""
import ctypes
import math

import numpy as np
import pytest
import torch

import b200knn
from b200knn import _lib
from b200knn import knn as K
from b200knn import metrics as M


def _grid_args(ks, ts):
    return (ctypes.c_int * max(1, len(ks)))(*ks), len(ks), (ctypes.c_double * max(1, len(ts)))(*ts), len(ts)


def test_vote_multilabel_abi_refuses_bad_arguments_without_gpu():
    lib = _lib.load()

    def call(ks, ts, k_max=None, L=8, scores_ld=None, n_labels=10, keys=1):
        k_max = ks[-1] if k_max is None and ks else (k_max or 1)
        ka, nk, ta, nt = _grid_args(ks, ts)
        ld = scores_ld if scores_ld is not None else max(1, nk * nt * L)
        return lib.b200knn_vote_multilabel(keys, 1, 4, k_max, n_labels, 0, L, ka, nk, ta, nt, 1, ld, 1, None)

    for kw, what in [(dict(ks=(5,), ts=(0.1,), L=0), b"L <= 64"),
                     (dict(ks=(5,), ts=(0.1,), L=65), b"L <= 64"),
                     (dict(ks=(5, 3, 8), ts=(0.1,)), b"strictly increasing"),
                     (dict(ks=(3, 3), ts=(0.1,)), b"strictly increasing"),
                     (dict(ks=(0, 3), ts=(0.1,)), b"strictly increasing"),
                     (dict(ks=(3, 5), ts=(0.1,), k_max=6), b"k_max"),
                     (dict(ks=(), ts=(0.1,), k_max=5), b"n_k"),
                     (dict(ks=tuple(range(1, 18)), ts=(0.1,)), b"n_k"),
                     (dict(ks=(5,), ts=()), b"n_t"),
                     (dict(ks=(5,), ts=tuple(0.1 * i for i in range(1, 10))), b"n_t"),
                     (dict(ks=(5,), ts=(0.1, 0.0)), b"finite and > 0"),
                     (dict(ks=(5,), ts=(-0.1,)), b"finite and > 0"),
                     (dict(ks=(5,), ts=(math.inf,)), b"finite and > 0"),
                     (dict(ks=(5,), ts=(math.nan,)), b"finite and > 0"),
                     (dict(ks=(3, 5), ts=(0.1, 0.2), scores_ld=31), b"scores_ld"),
                     (dict(ks=(5,), ts=(0.1,), keys=None), b"bad argument"),
                     (dict(ks=(5,), ts=(0.1,), n_labels=0), b"bad argument")]:
        assert call(**kw) == -1, kw
        assert what in lib.b200knn_last_error(), (kw, lib.b200knn_last_error())


def _case(N=300, D=16, B=7, L=8, seed=0):
    g = torch.Generator().manual_seed(seed)
    bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g), dim=1).t().contiguous()
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g), dim=1)
    return q, bank, torch.rand((N, L), generator=g) < 0.3


@pytest.mark.parametrize("ks,ts,match", [
    ((), (0.1,), "empty"), ((5, 5), (0.1,), "duplicate"), ((0, 5), (0.1,), "positive"), ((5,), (0.0,), "non-zero"),
    (tuple(range(1, 18)), (0.1,), "at most"), ((2.5,), (0.1,), "integers"),
    ((5,), (0.1, -0.1), "finite and > 0"), ((5,), (math.inf,), "finite and > 0"),
])
def test_python_grid_errors(ks, ts, match):
    q, bank, m = _case()
    with pytest.raises(ValueError, match=match):
        b200knn.knn_predict_multilabel(q, bank, m, ks, ts)


def test_python_label_matrix_errors():
    q, bank, m = _case()
    N = bank.shape[1]
    for bad, match in [(m[:, 0], "must be \\(N, L\\)"), (m[None], "must be \\(N, L\\)"), (m[:-1], "rows for a bank"),
                       (m[:, :0], "1 to 64 labels"), (torch.zeros((N, 65), dtype=torch.bool), "1 to 64 labels"),
                       (m.float(), "bool or integer"), (m.to(torch.int32) * 2, "0 or 1"),
                       (m.to(torch.int8) - 1, "0 or 1")]:
        with pytest.raises(ValueError, match=match):
            b200knn.knn_predict_multilabel(q, bank, bad, (5,), (0.1,))
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        b200knn.knn_predict_multilabel(q, bank, m, (5, N + 1), (0.1,))
    for dtype in (torch.bool, torch.uint8, torch.int64):  # valid: only the CPU tensors are refused
        with pytest.raises(RuntimeError, match="no CPU fallback"):
            b200knn.knn_predict_multilabel(q, bank, m.to(dtype), (5, N), (0.1,))


@pytest.mark.parametrize("L", [1, 8, 64])
def test_label_bits_round_trip(L):
    g = torch.Generator().manual_seed(L)
    m = torch.rand((500, L), generator=g) < 0.5
    m[0] = True   # every bit, bit 63 included at L = 64
    m[1] = False  # the empty set
    bits = b200knn.pack_label_bits(m.to(torch.uint8))
    assert bits.dtype == torch.int64 and bits.shape == (500,)
    back = (bits.view(-1, 1) >> torch.arange(L)) & 1
    assert torch.equal(back.bool(), m)
    assert int(bits[1]) == 0 and int(bits[0]) == (-1 if L == 64 else (1 << L) - 1)
    want = [sum(1 << b for b in range(L) if m[n, b]) for n in range(500)]
    assert [int(x) & ((1 << 64) - 1) for x in bits] == want
    assert bool((bits < 0).any()) == (L == 64)


def _metric_inputs(Q=400, L=7, seed=3, threshold=0.5):
    rng = np.random.default_rng(seed)
    scores = rng.integers(0, 11, (Q, L)) / 10.0  # a grid of 11 values: many ties, some exactly at 0.5
    target = rng.random((Q, L)) < np.linspace(0.1, 0.6, L)
    target[:, 2] = False                          # a label that is never positive
    target[:, 4] = scores[:, 4] > 0.3             # a well-separated label
    scores[:5, 0] = threshold                     # exactly at the threshold: not predicted
    return scores, target.astype(np.int64)


@pytest.mark.parametrize("threshold", [0.5, 0.3])
def test_metrics_arithmetic_equals_sklearn(threshold):
    from sklearn.metrics import accuracy_score, f1_score, hamming_loss, roc_auc_score

    scores, target = _metric_inputs(threshold=threshold)
    got = M.multilabel_metrics_from_scores(torch.from_numpy(scores), torch.from_numpy(target), threshold)
    pred = (scores > threshold).astype(np.int64)
    assert pred[:5, 0].sum() == 0 and (scores == threshold).any()
    present = [l for l in range(target.shape[1]) if pred[:, l].any() or target[:, l].any()]
    tol = 1e-12
    assert abs(float(got["f1_macro"]) - f1_score(target, pred, average="macro", labels=present,
                                                 zero_division=0)) < tol
    assert abs(float(got["f1_micro"]) - f1_score(target, pred, average="micro", zero_division=0)) < tol
    assert abs(float(got["subset_accuracy"]) - accuracy_score(target, pred)) < tol
    assert abs(float(got["hamming_loss"]) - hamming_loss(target, pred)) < tol
    defined = [l for l in range(target.shape[1]) if 0 < target[:, l].sum() < target.shape[0]]
    want_auc = roc_auc_score(target[:, defined], scores[:, defined], average=None)
    auc = got["auc"].numpy()
    assert np.abs(auc[defined] - want_auc).max() < tol
    assert np.isnan(np.delete(auc, defined)).all() and 2 not in defined
    assert abs(float(got["auc_macro"]) - want_auc.mean()) < tol
    tp = (pred & target).sum(0)
    fp = (pred & (1 - target)).sum(0)
    fn = ((1 - pred) & target).sum(0)
    tn = ((1 - pred) & (1 - target)).sum(0)
    assert np.array_equal(got["counts"].numpy(), np.stack([tp, fp, fn, tn], axis=1))
    for key in ("f1_macro", "f1_micro", "subset_accuracy", "hamming_loss", "auc_macro"):
        assert got[key].dtype == torch.float64 and got[key].dim() == 0, key


def test_metrics_edge_cases():
    s = torch.zeros((4, 3), dtype=torch.float64)
    t = torch.zeros((4, 3), dtype=torch.bool)
    got = M.multilabel_metrics_from_scores(s, t)
    assert float(got["f1_macro"]) == 0.0 and float(got["f1_micro"]) == 0.0
    assert float(got["subset_accuracy"]) == 1.0 and float(got["hamming_loss"]) == 0.0
    assert torch.isnan(got["auc"]).all() and math.isnan(float(got["auc_macro"]))
    with pytest.raises(RuntimeError, match="same"):
        M.multilabel_metrics_from_scores(s, t[:, :2])


def test_public_metrics_refuse_cpu_tensors():
    scores, target = _metric_inputs()
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        b200knn.knn_multilabel_metrics(torch.from_numpy(scores), torch.from_numpy(target))


def test_multilabel_spec_stays_off_tuple_paths():
    """The spec is not a tuple, so the class-ranking grid, the certified vote and the CUDA-graph key
    never take it for theirs."""
    spec = K._MultiLabelVote((5, 20), (0.1,))
    assert not isinstance(spec, tuple)
    bank = torch.zeros((4, 2000))
    assert not K._certified_vote_applies(None, bank, 8, 20, spec, "fp32", None)
