"""GPU: knn_predict_loo — the leave-one-out ranking of bank row r is bitwise knn_predict_multi of that
row against the bank with row r deleted: across modes, C = 9 and 38, the caller's order of ks,
exact duplicates, rows that are not among their own nearest neighbours, the k boundaries (peeling,
the raw modes' k = 992, k = N - 1), batching, the cascade's repair levels, FeatureBank and fp16
banks.  Also the SEQ oracle on the real golden table, drop_self against a NumPy restatement and
knn_graph's self-exclusion on duplicate and small-norm rows."""
import os

import numpy as np
import pytest
import torch

import b200knn
import datagen
from b200knn import knn as K
from oracle import knn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KS, TS = (1, 5, 20, 200), (0.07, 0.1, 0.5)


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _bank(N, D, C, seed):
    lab = datagen.labels(N, C, seed)
    return _t(datagen.clustered(N, D, C, seed + 1, lab).T), _t(lab)


def _deleted(bank, lab, C, ks, ts, r):
    """knn_predict_multi of row r against the bank without column r: (n_k, n_t, C)."""
    keep = torch.ones(bank.shape[1], dtype=torch.bool, device=bank.device)
    keep[r] = False
    q = bank[:, r:r + 1].t()
    return b200knn.knn_predict_multi(q, bank[:, keep].contiguous(), lab[keep].contiguous(), C, ks, ts)[:, :, 0]


def _assert_equals_deletion(got, bank, lab, C, ks, ts, rows):
    for r in rows:
        want = _deleted(bank, lab, C, ks, ts, int(r))
        assert torch.equal(got[:, :, int(r)], want), int(r)


def _rows(N, n, seed):
    return np.sort(np.random.default_rng(seed).choice(N, n, replace=False))


@pytest.fixture()
def mode_guard():
    yield
    b200knn.set_default_mode("exact")
    K.GRAPHS["enabled"] = True


@pytest.mark.parametrize("mode", ["fp32", "exact", "fp32_f16x2", "f16", "bf16", "bf16x3"])
@pytest.mark.parametrize("C", [9, 38])
def test_loo_bitwise_equals_row_deletion(mode, C, mode_guard):
    N = 20000
    bank, lab = _bank(N, 512, C, 300 + C)
    b200knn.set_default_mode(mode)
    ks, ts = (20, 1, 200, 5), (0.1, 0.5, 0.07)  # not ascending: output follows the caller's order
    before = dict(K.graph_stats)
    got = b200knn.knn_predict_loo(bank, lab, C, ks, ts, batch=400)  # batches small enough for a graph
    assert K.graph_stats == before  # ... but they never use the graph cache
    assert got.shape == (4, 3, N, C) and got.dtype == torch.int64
    rows = np.concatenate([[0, N - 1], _rows(N, 46, C)])
    _assert_equals_deletion(got, bank, lab, C, ks, ts, rows)


@pytest.mark.parametrize("mode", ["exact", "fp32"])
def test_loo_equals_seq_oracle_on_golden(mode, golden_dir, mode_guard):
    g = np.load(os.path.join(golden_dir, "real_FastSiam.npz"))
    b = g["bank_rows_f16"].astype(np.float32)
    b = b / np.maximum(np.linalg.norm(b, axis=1, keepdims=True), 1e-12)
    bank, labels, C = np.ascontiguousarray(b.T), g["bank_labels"].astype(np.int64), 9
    sims = O.sims_seqfma(b, bank)
    np.fill_diagonal(sims, -np.inf)  # each row's own column
    ss, si = O.canonical_topk_c(sims, max(KS))
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_loo(_t(bank), _t(labels), C, KS, TS).cpu().numpy()
    assert got.shape == (len(KS), len(TS), 3000, C)
    for i, k in enumerate(KS):
        for j, t in enumerate(TS):
            assert np.array_equal(got[i, j], O.vote_o64(ss[:, :k], si[:, :k], labels, C, t)[0]), (k, t)


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_loo_exact_duplicates_keep_the_twin(mode, mode_guard):
    N, D, C = 6000, 256, 9
    bank, lab = _bank(N, D, C, 41)
    bank[:, 3000:3100] = bank[:, 100:200]  # rows 3000.. are exact twins of rows 100..
    b200knn.set_default_mode(mode)
    ks, ts = (1, 5, 50), (0.1,)
    got = b200knn.knn_predict_loo(bank, lab, C, ks, ts)
    # the twin is the deleted row's nearest neighbour on both sides of the pair
    keys = K.topk_keys(bank[:, [100, 3000]].t().contiguous(), bank, 2, "exact")
    _, idx = K.decode_keys(K.drop_self(keys[0:1], 100))
    assert int(idx[0, 0]) == 3000
    _, idx = K.decode_keys(K.drop_self(keys[1:2], 3000))
    assert int(idx[0, 0]) == 100
    _assert_equals_deletion(got, bank, lab, C, ks, ts, [100, 150, 199, 3000, 3050, 3099, 7, 5999])


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_loo_rows_outside_their_own_top_list(mode, mode_guard):
    """Un-normalised bank, a few rows at 1e-2 of the others' norm: their self-similarity ranks far
    down, so the drop-last branch runs."""
    N, D, C = 6000, 256, 9
    bank, lab = _bank(N, D, C, 52)
    small = [3, 777, 4242, 5998]
    bank[:, small] *= 1e-2
    b200knn.set_default_mode(mode)
    ks, ts = (3, 30), (0.1, 0.07)
    keys = K.topk_keys(bank[:, small].t().contiguous(), bank, 31, "exact")
    _, idx = K.decode_keys(keys)
    assert not bool((idx == torch.tensor(small, device=DEV).view(-1, 1)).any())
    got = b200knn.knn_predict_loo(bank, lab, C, ks, ts)
    _assert_equals_deletion(got, bank, lab, C, ks, ts, small + [0, 1000])


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_loo_beyond_max_k_takes_peeling_path(mode, mode_guard):
    bank, lab = _bank(6000, 256, 9, 7)
    b200knn.set_default_mode(mode)
    ks, ts = (5, 1000), (0.1, 0.07)
    got = b200knn.knn_predict_loo(bank, lab, 9, ks, ts)
    _assert_equals_deletion(got, bank, lab, 9, ks, ts, _rows(6000, 6, 1))


def test_loo_k992_in_raw_mode_is_exact_modes_result(mode_guard):
    bank, lab = _bank(6000, 256, 9, 8)
    ks, ts = (991, 992), (0.1,)
    b200knn.set_default_mode("exact")
    exact = b200knn.knn_predict_loo(bank, lab, 9, ks, ts)
    b200knn.set_default_mode("bf16")
    got = b200knn.knn_predict_loo(bank, lab, 9, ks, ts)
    assert torch.equal(got[1], exact[1])  # k + 1 = 993 > MAX_K: the exact kernel's list
    rows = _rows(6000, 6, 2)
    _assert_equals_deletion(got[:1], bank, lab, 9, ks[:1], ts, rows)  # k = 991 keeps the contract


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_loo_k_up_to_n_minus_1(mode, mode_guard):
    N = 300
    bank, lab = _bank(N, 128, 9, 9)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_loo(bank, lab, 9, (N - 1, 4), (0.1,))
    _assert_equals_deletion(got, bank, lab, 9, (N - 1, 4), (0.1,), [0, 17, N - 1])
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        b200knn.knn_predict_loo(bank, lab, 9, (4, N), (0.1,))


@pytest.mark.parametrize("mode", ["fp32", "bf16", "exact"])
def test_loo_independent_of_batch(mode, mode_guard):
    N = 9000
    bank, lab = _bank(N, 512, 9, 10)
    b200knn.set_default_mode(mode)
    ks, ts = (5, 20, 200), (0.1, 0.07)
    ref = b200knn.knn_predict_loo(bank, lab, 9, ks, ts, batch=N)
    for batch in (1000, 4099, N + 5):
        assert torch.equal(b200knn.knn_predict_loo(bank, lab, 9, ks, ts, batch=batch), ref), batch


def test_loo_repair_levels(mode_guard):
    """Rows the cascade's first level leaves uncertified are repaired at k_max + 1 by the later levels."""
    c = datagen.make_case("absgauss_small")
    bank, lab, C = _t(c["bank"]), _t(c["labels"]), c["C"]
    reached = []
    for mode in ("fp32", "fp32_bf16"):
        b200knn.set_default_mode(mode)
        got = b200knn.knn_predict_loo(bank, lab, C, KS, TS)
        reached.append(len(K.last_rescore_stats["levels"]) > 1)
        _assert_equals_deletion(got, bank, lab, C, KS, TS, _rows(bank.shape[1], 12, 3))
    assert any(reached), K.last_rescore_stats


def test_feature_bank_and_fp16_bank(mode_guard):
    rng = np.random.default_rng(4)
    C = 9
    rows = _t(rng.standard_normal((8000, 512)).astype(np.float32) * 3)
    lab = _t(datagen.labels(8000, C, 4))
    fb = b200knn.FeatureBank.from_rows(rows, lab)
    b200knn.set_default_mode("fp32")
    got = fb.knn_predict_loo(C, KS, TS)
    assert torch.equal(got, b200knn.knn_predict_loo(fb.bank, fb.labels, C, KS, TS))
    _assert_equals_deletion(got, fb.bank, fb.labels, C, KS, TS, [0, 4321, 7999])
    # an fp16 (D, N) bank: the queries keep the bank's dtype
    bank16 = fb.bank.half().contiguous()
    for mode in ("fp32", "bf16"):
        b200knn.set_default_mode(mode)
        got16 = b200knn.knn_predict_loo(bank16, lab, C, (5, 20), (0.1,))
        _assert_equals_deletion(got16, bank16, lab, C, (5, 20), (0.1,), [1, 2500, 7998])


def test_loo_label_errors(mode_guard):
    bank, lab = _bank(3000, 128, 9, 5)
    bad = lab.clone()
    bad[:] = 9
    for mode in ("fp32", "exact"):
        b200knn.set_default_mode(mode)
        with pytest.raises(RuntimeError, match="num_classes=9"):
            b200knn.knn_predict_loo(bank, bad, 9, (5, 20), (0.1,))
        with pytest.raises(RuntimeError, match="feature_labels has 2999 entries for a bank of 3000"):
            b200knn.knn_predict_loo(bank, lab[1:], 9, (5,), (0.1,))


def _drop_self_np(keys, self_offset):
    B, k_in = keys.shape
    out = np.empty((B, k_in - 1), dtype=np.uint64)
    _, idx = O.decode_keys(keys)
    for b in range(B):
        hit = np.flatnonzero((keys[b] != 0) & (idx[b] == b + self_offset))
        p = hit[0] if hit.size else k_in - 1
        out[b] = np.delete(keys[b], p)
    return out


@pytest.mark.parametrize("k_in", [2, 31, 32, 33, 201, 1001])
def test_drop_self_against_numpy(k_in):
    rng = np.random.default_rng(k_in)
    B, off = 777, 12345
    sims = -np.sort(-rng.standard_normal((B, k_in)).astype(np.float32), axis=1)
    idx = rng.integers(0, 50000, (B, k_in))
    own = rng.random(B) < 0.6  # the row's own index at a random position of 60 % of the rows
    pos = rng.integers(0, k_in, B)
    idx[own, pos[own]] = np.arange(B)[own] + off
    idx[~own] = np.where(idx[~own] == (np.arange(B)[~own] + off)[:, None], 0, idx[~own])
    keys = O.make_keys(sims, idx)
    empty = rng.random(B) < 0.2  # trailing empty slots
    cut = rng.integers(0, k_in, B)
    for b in np.flatnonzero(empty):
        keys[b, cut[b]:] = 0
    got = K.drop_self(_t(keys.view(np.int64)), off).cpu().numpy().view(np.uint64)
    assert np.array_equal(got, _drop_self_np(keys, off))


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_knn_graph_drops_self_by_index(mode):
    g = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn(4000, 256, generator=g, device=DEV)
    x[2000:2050] = x[10:60]                    # exact duplicates
    x[[7, 999, 3333]] *= 1e-2                  # rows far down their own lists
    k = 12
    sims, idx = b200knn.knn_graph(x, k, normalize=False, mode=mode, batch=1500)
    own = torch.arange(4000, device=DEV).view(-1, 1)
    assert not bool((idx == own).any())
    assert bool((idx[2000:2050, 0] == own[10:60, 0]).all())  # the lower-index twin ranks first and stays
    keys = K.topk_keys(x, x.t().contiguous(), k + 1, mode)
    s_all, i_all = K.decode_keys(keys)
    keep = i_all != own
    keep &= keep.cumsum(1) <= k
    assert torch.equal(idx, i_all[keep].view(4000, k)) and torch.equal(sims, s_all[keep].view(4000, k))
    with pytest.raises(RuntimeError, match="smaller than the number of rows"):
        b200knn.knn_graph(x[:10], 10, normalize=False, mode=mode)
