"""GPU: knn_predict_multilabel and b200knn_vote_multilabel — per-label kNN scores of multi-hot banks over
a (k, t) grid from one neighbour search: bitwise the separate single-(k, t) calls in every mode, the
fp32 cascade bitwise the exact mode, each raw mode bitwise the vote of its own neighbour lists, the fp64
oracle within the bound of a not correctly rounded exp, batch invariance, deep (chunked, peeled) lists,
L = 1 and 64, index errors, agreement with knn_predict on one-hot banks, and the metrics against
scikit-learn."""
import functools

import numpy as np
import pytest
import torch

import b200knn
from b200knn import knn as K

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KS, TS = (20, 1, 200, 5), (0.1, 0.5, 0.07)  # not ascending: the output follows the caller's order
L8 = 8
# label sets of an 8-pattern bank shaped like MixedWM38: none, each single pattern, and 29 fixed
# mixtures of 2-4 patterns (pattern ids 0..7)
MIXTURES = [(0, 2), (0, 3), (0, 4), (0, 6), (1, 2), (1, 3), (1, 4), (1, 6), (2, 4), (2, 6), (3, 4), (3, 6), (4, 6),
            (0, 2, 4), (0, 2, 6), (0, 3, 4), (0, 3, 6), (0, 4, 6), (1, 2, 4), (1, 2, 6), (1, 3, 4), (1, 3, 6),
            (1, 4, 6), (2, 4, 6), (3, 4, 6), (0, 2, 4, 6), (0, 3, 4, 6), (1, 2, 4, 6), (1, 3, 4, 6)]
LABEL_SETS = [()] + [(l,) for l in range(L8)] + MIXTURES
assert len(MIXTURES) == 29 and len(set(LABEL_SETS)) == 38


def _rows(m: np.ndarray, centroids: np.ndarray, rng, noise: float = 0.1) -> np.ndarray:
    """Rows of label matrix m: the normalised sum of their labels' centroids plus Gaussian noise."""
    x = m.astype(np.float32) @ centroids + noise * rng.standard_normal((m.shape[0], centroids.shape[1]))
    return (x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-12)).astype(np.float32)


def _label_matrix(n: int, L: int, rng) -> np.ndarray:
    if L == L8:
        m = np.zeros((n, L), dtype=bool)
        for r, s in enumerate(rng.integers(0, len(LABEL_SETS), n)):
            m[r, list(LABEL_SETS[s])] = True
        return m
    return rng.random((n, L)) < 0.25


@functools.lru_cache(maxsize=8)
def _data(N: int, D: int, B: int, L: int = L8, seed: int = 0):
    """(queries (B, D), bank (D, N), bank label matrix (N, L) bool, query label matrix (B, L) bool)"""
    rng = np.random.default_rng(seed)
    centroids = rng.standard_normal((L, D)).astype(np.float32)
    centroids /= np.linalg.norm(centroids, axis=1, keepdims=True)
    m, mq = _label_matrix(N, L, rng), _label_matrix(B, L, rng)
    bank = _rows(m, centroids, rng)
    q = _rows(mq, centroids, rng)
    t = lambda x: torch.from_numpy(np.ascontiguousarray(x)).to(DEV)  # noqa: E731
    return t(q), t(bank.T), t(m), t(mq)


@pytest.fixture()
def mode_guard():
    old = b200knn.get_default_mode()
    yield
    b200knn.set_default_mode(old)


def _separate(q, bank, m, ks, ts):
    return torch.stack([torch.stack([b200knn.knn_predict_multilabel(q, bank, m, (k,), (t,))[0, 0] for t in ts])
                        for k in ks])


def _own_vote(keys, m, ks, ts):
    """b200knn_vote_multilabel of each (k, t) alone on the first k of the given keys."""
    bits = b200knn.pack_label_bits(m)
    return torch.stack([torch.stack([K.vote_multilabel(keys[:, :k], bits, m.shape[1], (k,), (t,)) for t in ts])
                        for k in ks])


def vote_multilabel_o64(sims: np.ndarray, idx: np.ndarray, bits: np.ndarray, ks, ts) -> np.ndarray:
    """The fp64 oracle: per-label kNN scores of multi-hot bank rows, restated from include/b200knn.h
    (b200knn_vote_multilabel) with numpy: bits (N, L) 0/1, bit l of bank row n; sims / idx (B, >= max(ks))
    the neighbour lists in rank order.  Returns (len(ks), len(ts), B, L) f64 with [i, j, b, l] = S_l / W,
    w_r = exp((f64(s_r) - f64(s_0)) / t), W = sum_{r<k} w_r and S_l the sum over the ranks whose row
    carries l, both added in rank order."""
    bits = np.asarray(bits)
    B, L = sims.shape[0], bits.shape[1]
    s = sims.astype(np.float64)
    out = np.zeros((len(ks), len(ts), B, L), dtype=np.float64)
    for j, t in enumerate(ts):
        W = np.zeros(B)
        S = np.zeros((B, L))
        for r in range(max(ks)):  # rank order
            w = np.exp((s[:, r] - s[:, 0]) / np.float64(t))
            W += w
            S += np.where(bits[idx[:, r]] != 0, w[:, None], 0.0)  # adding +0.0 leaves S unchanged
            for i, k in enumerate(ks):
                if k == r + 1:
                    out[i, j] = S / W[:, None]
    return out


def _bound(k: int) -> float:
    return (2 * k + 6) * 2.0 ** -52


def _check_oracle(got: np.ndarray, want: np.ndarray, ks, threshold: float = 0.5) -> None:
    for i, k in enumerate(ks):
        g, w = got[i], want[i]
        bound = _bound(k)
        assert np.all(np.abs(g - w) <= bound * w), (k, np.max(np.abs(g - w) / np.maximum(w, 1e-300)))
        exact = (w == 0.0) | (w == 1.0)
        assert np.array_equal(g[exact], w[exact]), k
        far = np.abs(w - threshold) > bound
        assert np.array_equal((g > threshold)[far], (w > threshold)[far]), k
        assert g.min() >= 0.0 and g.max() <= 1.0


@pytest.mark.parametrize("mode", ["fp32", "exact", "fp32_f16x2", "f16", "bf16", "bf16x3"])
@pytest.mark.parametrize("B", [64, 1000, 5000])
def test_grid_bitwise_equals_separate_calls(mode, B, mode_guard):
    q, bank, m, _ = _data(20000, 512, B)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_multilabel(q, bank, m, KS, TS)
    assert got.shape == (4, 3, B, L8) and got.dtype == torch.float64
    assert torch.equal(got, _separate(q, bank, m, KS, TS))


@pytest.mark.parametrize("mode", ["fp32", "fp32_f16x2", "f16", "bf16", "bf16x3"])
def test_mode_equality(mode, mode_guard):
    """fp32 modes: bitwise the exact mode.  Raw modes: bitwise the vote of the mode's own neighbour lists."""
    q, bank, m, _ = _data(20000, 512, 1000)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_multilabel(q, bank, m, KS, TS)
    if mode in K.TC_MODES:
        want = _own_vote(K.topk_keys(q, bank, max(KS), mode), m, KS, TS)
    else:
        b200knn.set_default_mode("exact")
        want = b200knn.knn_predict_multilabel(q, bank, m, KS, TS)
    assert torch.equal(got, want)


@pytest.mark.parametrize("mode", ["exact", "fp32"])
def test_equals_fp64_oracle(mode, mode_guard):
    q, bank, m, _ = _data(20000, 512, 1000)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_multilabel(q, bank, m, KS, TS).cpu().numpy()
    sims, idx = b200knn.knn_topk(q, bank, max(KS), mode="exact")
    want = vote_multilabel_o64(sims.cpu().numpy(), idx.cpu().numpy(), m.cpu().numpy(), KS, TS)
    _check_oracle(got, want, KS)
    assert (want == 0.0).any() and (want == 1.0).any()  # both exact cases occur


def test_batch_invariance(mode_guard):
    q, bank, m, _ = _data(20000, 512, 1000)
    b200knn.set_default_mode("fp32")
    full = b200knn.knn_predict_multilabel(q, bank, m, KS, TS)
    for a, b in ((0, 64), (64, 581), (581, 1000), (997, 1000)):
        assert torch.equal(b200knn.knn_predict_multilabel(q[a:b], bank, m, KS, TS), full[:, :, a:b]), (a, b)
    empty = b200knn.knn_predict_multilabel(q[:0], bank, m, KS, TS)
    assert empty.shape == (4, 3, 0, L8)
    # the kernel alone, on one raw mode's keys: a row's scores do not depend on the rows beside it
    keys = K.topk_keys(q, bank, 200, "bf16")
    bits = b200knn.pack_label_bits(m)
    whole = K.vote_multilabel(keys, bits, L8, (5, 200), (0.1, 0.07))
    for a, b in ((0, 1), (3, 8), (5, 1000)):
        assert torch.equal(K.vote_multilabel(keys[a:b], bits, L8, (5, 200), (0.1, 0.07)), whole[a:b])


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_deep_lists_chunked_and_peeled(mode, mode_guard):
    q, bank, m, _ = _data(6000, 256, 70, seed=7)
    b200knn.set_default_mode(mode)
    ks, ts = (1500, 5, 1000), (0.1, 0.07)
    got = b200knn.knn_predict_multilabel(q, bank, m, ks, ts)
    assert torch.equal(got, _separate(q, bank, m, ks, ts))
    if mode != "bf16":
        keys = K.topk_keys(q, bank, 1500, "exact")
        # the chunked kernel's k = 1000 block is the single-chunk kernel's k = 1000 call
        assert torch.equal(got, _own_vote(keys, m, ks, ts))
        sims, idx = b200knn.knn_topk(q, bank, 1500, mode="exact")
        _check_oracle(got.cpu().numpy(), vote_multilabel_o64(sims.cpu().numpy(), idx.cpu().numpy(),
                                                             m.cpu().numpy(), ks, ts), ks)
    with pytest.raises(RuntimeError, match="k out of range"):
        b200knn.knn_predict_multilabel(q, bank, m, (5, 6001), ts)


@pytest.mark.parametrize("L", [1, 64])
def test_label_counts(L, mode_guard):
    q, bank, m, _ = _data(8000, 128, 300, L=L, seed=L)
    if L == 64:
        assert bool(m[:, 63].any())  # bit 63: negative int64 masks
    b200knn.set_default_mode("fp32")
    ks, ts = (10, 100), (0.1, 0.05)
    got = b200knn.knn_predict_multilabel(q, bank, m.to(torch.uint8), ks, ts)
    assert got.shape == (2, 2, 300, L)
    sims, idx = b200knn.knn_topk(q, bank, 100, mode="exact")
    _check_oracle(got.cpu().numpy(), vote_multilabel_o64(sims.cpu().numpy(), idx.cpu().numpy(),
                                                         m.cpu().numpy(), ks, ts), ks)


def test_index_outside_labels(mode_guard):
    q, bank, m, _ = _data(3000, 128, 64, seed=5)
    keys = K.topk_keys(q, bank, 20, "exact")
    bits = b200knn.pack_label_bits(m)
    short = bits[:1000]  # neighbours with index >= 1000 fall outside
    assert bool((b200knn.decode_keys(keys)[1] >= 1000).any())
    flag = torch.zeros((1,), dtype=torch.int32, device=DEV)
    K.vote_multilabel(keys, short, L8, (5, 20), (0.1,), check_labels=False, flag=flag)
    assert int(flag.item()) == 2
    with pytest.raises(RuntimeError, match="neighbour index outside feature_labels"):
        K.vote_multilabel(keys, short, L8, (5, 20), (0.1,))
    flag.zero_()
    K.vote_multilabel(keys, bits, L8, (5, 20), (0.1,), check_labels=False, flag=flag)
    assert int(flag.item()) == 0


@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_one_hot_bank_agrees_with_knn_predict(mode, mode_guard):
    import datagen

    C, k, t = 9, 200, 0.1
    lab = datagen.labels(20000, C, 3)
    bank = torch.from_numpy(np.ascontiguousarray(datagen.clustered(20000, 512, C, 4, lab).T)).to(DEV)
    q = torch.from_numpy(datagen.clustered(2000, 512, C, 5)).to(DEV)
    lab = torch.from_numpy(lab).to(DEV)
    b200knn.set_default_mode(mode)
    scores = b200knn.knn_predict_multilabel(q, bank, torch.nn.functional.one_hot(lab, C), (k,), (t,))[0, 0]
    assert torch.allclose(scores.sum(1), torch.ones(2000, dtype=torch.float64, device=DEV), rtol=0, atol=1e-12)
    pred = b200knn.knn_predict(q, bank, lab, C, k, t)[:, 0]
    top2 = scores.topk(2, dim=1).values
    clear = (top2[:, 0] - top2[:, 1]) > 1e-12 * top2[:, 0]
    assert clear.float().mean() > 0.9
    assert torch.equal(scores.argmax(1)[clear], pred[clear])


def test_metrics_on_device_equal_sklearn(mode_guard):
    from sklearn.metrics import accuracy_score, f1_score, hamming_loss, roc_auc_score

    q, bank, m, mq = _data(20000, 512, 1000)
    b200knn.set_default_mode("fp32")
    scores = b200knn.knn_predict_multilabel(q, bank, m, (20, 200), (0.07,))[0, 0]
    got = b200knn.knn_multilabel_metrics(scores, mq)
    assert all(v.device.type == "cuda" for v in got.values())
    s, t = scores.cpu().numpy(), mq.cpu().numpy().astype(np.int64)
    p = (s > 0.5).astype(np.int64)
    present = [l for l in range(L8) if p[:, l].any() or t[:, l].any()]
    assert abs(float(got["f1_macro"]) - f1_score(t, p, average="macro", labels=present, zero_division=0)) < 1e-12
    assert abs(float(got["f1_micro"]) - f1_score(t, p, average="micro", zero_division=0)) < 1e-12
    assert abs(float(got["subset_accuracy"]) - accuracy_score(t, p)) < 1e-12
    assert abs(float(got["hamming_loss"]) - hamming_loss(t, p)) < 1e-12
    auc = roc_auc_score(t, s, average=None)
    assert np.abs(got["auc"].cpu().numpy() - auc).max() < 1e-12
    assert abs(float(got["auc_macro"]) - auc.mean()) < 1e-12
    assert float(got["f1_micro"]) > 0.5  # the scores carry the labels' signal
