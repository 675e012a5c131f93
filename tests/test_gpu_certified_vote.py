"""knn_predict's certified class vote (b200knn_rescore_vote, DESIGN §4.1c) against the exact mode
and against the full re-scoring path (switch off): bitwise equal rankings, the same label errors."""
import numpy as np
import pytest
import torch

import datagen
from b200knn import knn as K

pytestmark = pytest.mark.gpu

DEV = "cuda:0"
N, D = 6000, 128


def _bank(kind: str, C: int, seed: int = 5):
    lab = datagen.labels(N, C, seed)
    if kind == "clustered":
        x = datagen.clustered(N, D, C, seed, lab)
    elif kind == "relu":
        x = datagen.relu(N, D, C, seed, lab)
    elif kind == "gauss":
        x = datagen.gauss(N, D, seed)
    else:
        x = datagen.absgauss(N, D, seed)
    return x, lab


def _queries(kind: str, B: int, C: int, seed: int = 9):
    return _bank(kind, C, seed)[0][:B] if B <= N else np.concatenate(
        [_bank(kind, C, seed + i)[0] for i in range((B + N - 1) // N)])[:B]


def _three_ways(q, bank, lab, C, k, t):
    """(certified vote, full re-scoring, exact mode) rankings of one call."""
    old = K.CERTIFIED_VOTE["enabled"]
    try:
        K.CERTIFIED_VOTE["enabled"] = True
        on = K._predict(q, bank, lab, C, k, t, "fp32")
        K.CERTIFIED_VOTE["enabled"] = False
        off = K._predict(q, bank, lab, C, k, t, "fp32")
    finally:
        K.CERTIFIED_VOTE["enabled"] = old
    ex = K._predict(q, bank, lab, C, k, t, "exact")
    return on, off, ex


def _check(q, bank, lab, C, k, t):
    on, off, ex = _three_ways(q, bank, lab, C, k, t)
    assert torch.equal(on, ex), (C, k, t)
    assert torch.equal(off, ex), (C, k, t)


@pytest.mark.parametrize("kind", ["clustered", "gauss", "relu", "absgauss"])
@pytest.mark.parametrize("C", [2, 9, 38])
def test_equals_exact_mode(kind, C):
    x, lab = _bank(kind, C)
    bank = torch.from_numpy(x).to(DEV).t().contiguous()
    lab = torch.from_numpy(lab).to(DEV)
    qs = torch.from_numpy(_queries(kind, 513, C)).to(DEV)
    for B in (1, 64, 513):
        q = qs[:B].contiguous()
        for k in (1, 5, 200, 992):
            for t in (0.1, 0.01, -0.1):
                _check(q, bank, lab, C, k, t)


@pytest.mark.parametrize("kind", ["clustered", "gauss", "relu", "absgauss"])
def test_large_batch(kind):
    x, lab = _bank(kind, 9)
    bank = torch.from_numpy(x).to(DEV).t().contiguous()
    lab = torch.from_numpy(lab).to(DEV)
    q = torch.from_numpy(_queries(kind, 37888, 9)).to(DEV)
    _check(q, bank, lab, 9, 200, 0.1)
    info = K.last_rescore_stats["band_info"]
    assert info.shape == (37888, 4)
    served = info[:, 0] >= 0
    assert bool(served.all())
    assert bool(((info[:, 1] >= 200) & (info[:, 0] <= 200)).all())


def _fallbacks_after(q, bank, lab, C, k, t):
    old = K.CERTIFIED_VOTE["enabled"]
    K.CERTIFIED_VOTE["enabled"] = True
    try:
        K.last_rescore_stats.pop("vote_fallback", None)
        pred = K._predict(q, bank, lab, C, k, t, "fp32")
        n = K.last_rescore_stats.get("vote_fallback")
    finally:
        K.CERTIFIED_VOTE["enabled"] = old
    assert torch.equal(pred, K._predict(q, bank, lab, C, k, t, "exact"))
    return n


def test_tie_beyond_the_list_falls_back():
    # rule 2: more copies of one row than the list holds, so the k-th exact key cannot beat a_m + E
    x, lab = _bank("gauss", 9)
    x[100:1200] = x[0]
    q = torch.from_numpy(x[:1].copy()).to(DEV)
    bank = torch.from_numpy(x).to(DEV).t().contiguous()
    assert _fallbacks_after(q, bank, torch.from_numpy(lab).to(DEV), 9, 992, 0.1) == 1


def test_close_class_scores_fall_back():
    # rule 3: two neighbours of different classes within the error bound, k = 2, C = 2
    rng = np.random.default_rng(3)
    x, _ = _bank("gauss", 2)
    lab = np.zeros(N, dtype=np.int64)
    lab[N // 2:] = 1
    q = datagen.gauss(1, D, 77)
    for row in (10, N - 10):
        v = q[0] + 1e-4 * rng.standard_normal(D).astype(np.float32)
        x[row] = v / np.linalg.norm(v)
    bank = torch.from_numpy(x).to(DEV).t().contiguous()
    n = _fallbacks_after(torch.from_numpy(q).to(DEV), bank, torch.from_numpy(lab).to(DEV), 2, 2, 0.1)
    assert n == 1


def test_underflow_and_overflow_fall_back():
    x, lab = _bank("clustered", 9)
    bank = torch.from_numpy(x).to(DEV).t().contiguous()
    lab = torch.from_numpy(lab).to(DEV)
    q = torch.from_numpy(x[:64].copy()).to(DEV)
    assert _fallbacks_after(q, bank, lab, 9, 200, -1e-3) is not None  # exp(-s/1e-3) underflows
    assert _fallbacks_after(q, bank, lab, 9, 200, 1e-3) == 64  # exp(1/1e-3) of the row itself overflows
    assert _fallbacks_after(q * 1000.0, bank, lab, 9, 200, 0.1) == 64  # unnormalised: exp overflows


@pytest.mark.parametrize("bad", [9, -1])
def test_label_errors_raise_the_same(bad):
    x, lab = _bank("clustered", 9)
    q = torch.from_numpy(x[:8].copy()).to(DEV)
    bank = torch.from_numpy(x).to(DEV).t().contiguous()
    lab[3] = bad  # row 3 is query 3's own nearest neighbour
    lab = torch.from_numpy(lab).to(DEV)
    msgs = []
    for mode, on in (("fp32", True), ("fp32", False), ("exact", True)):
        old = K.CERTIFIED_VOTE["enabled"]
        K.CERTIFIED_VOTE["enabled"] = on
        try:
            with pytest.raises(RuntimeError) as e:
                K._predict(q, bank, lab, 9, 200, 0.1, mode)
            msgs.append(str(e.value))
        finally:
            K.CERTIFIED_VOTE["enabled"] = old
    assert msgs[0] == msgs[1] == msgs[2]
    assert "num_classes=9" in msgs[0]
