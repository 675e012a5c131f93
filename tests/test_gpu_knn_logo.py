"""GPU: knn_predict_loo(groups=...) — the leave-one-group-out ranking of bank row r is bitwise
knn_predict_multi of that row against the bank without every row of r's group: across modes, C = 9
and 38, lot-like groups (contiguous runs, random sizes with negative non-contiguous int32 ids), a
group beyond MAX_K (the peeling path), the k boundary N - max group size, batching, the cascade's
repair levels, FeatureBank and fp16 banks.  groups = arange(N) is bitwise plain leave-one-out.  Also
the SEQ oracle on the real golden table, drop_group against a NumPy restatement and knn_graph's group
exclusion."""
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
MODES = ["fp32", "exact", "fp32_f16x2", "f16", "bf16", "bf16x3"]


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _bank(N, D, C, seed):
    lab = datagen.labels(N, C, seed)
    return _t(datagen.clustered(N, D, C, seed + 1, lab).T), _t(lab)


def _random_size_groups(N, seed):
    """Groups of 1 to 40 rows, scattered over the bank, with negative non-contiguous int32 ids."""
    rng = np.random.default_rng(seed)
    sizes = rng.integers(1, 41, N)
    sizes = sizes[:np.searchsorted(np.cumsum(sizes), N) + 1]
    ids = -1 - rng.choice(10 ** 6, sizes.size, replace=False) * 7
    g = np.repeat(ids, sizes)[:N].astype(np.int32)
    rng.shuffle(g)
    return g


def _lot_bank(N, D, C, seed, groups):
    """Lot-mates are small perturbations of their lot's centre, so they fill the top of each other's
    lists; a lot's rows share its label, 20 % of the rows carry another one."""
    rng = np.random.default_rng(seed)
    _, lot = np.unique(groups, return_inverse=True)
    n_lots = lot.max() + 1
    lot_lab = datagen.labels(n_lots, C, seed + 1)
    centre = datagen.clustered(n_lots, D, C, seed + 2, lot_lab)
    x = centre[lot] + 0.1 * rng.standard_normal((N, D)).astype(np.float32) / np.sqrt(D)
    lab = lot_lab[lot].copy()
    flip = rng.random(N) < 0.2
    lab[flip] = rng.integers(0, C, int(flip.sum()))
    return _t(x.astype(np.float32).T), _t(lab.astype(np.int64))


def _deleted(bank, lab, C, ks, ts, groups, r):
    """knn_predict_multi of row r against the bank without r's group: (n_k, n_t, C)."""
    keep = groups != groups[r]
    q = bank[:, r:r + 1].t()
    return b200knn.knn_predict_multi(q, bank[:, keep].contiguous(), lab[keep].contiguous(), C, ks, ts)[:, :, 0]


def _assert_equals_deletion(got, bank, lab, C, ks, ts, groups, rows):
    for r in rows:
        want = _deleted(bank, lab, C, ks, ts, groups, int(r))
        assert torch.equal(got[:, :, int(r)], want), int(r)


def _rows(N, n, seed):
    return np.sort(np.random.default_rng(seed).choice(N, n, replace=False))


@pytest.fixture()
def mode_guard():
    yield
    b200knn.set_default_mode("exact")
    K.GRAPHS["enabled"] = True


@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("C", [9, 38])
def test_singleton_groups_are_plain_loo(mode, C, mode_guard):
    N = 6000
    bank, lab = _bank(N, 256, C, 500 + C)
    b200knn.set_default_mode(mode)
    ks, ts = (20, 1, 200, 5), (0.1, 0.5, 0.07)
    plain = b200knn.knn_predict_loo(bank, lab, C, ks, ts, batch=1500)
    assert torch.equal(b200knn.knn_predict_loo(bank, lab, C, ks, ts, batch=1500,
                                               groups=torch.arange(N, device=DEV)), plain)
    perm = torch.from_numpy(np.random.default_rng(C).permutation(N)).to(DEV)
    assert torch.equal(b200knn.knn_predict_loo(bank, lab, C, ks, ts, batch=1500, groups=perm), plain)


@pytest.mark.parametrize("kind", ["runs_of_25", "random_sizes"])
@pytest.mark.parametrize("mode", MODES)
@pytest.mark.parametrize("C", [9, 38])
def test_logo_bitwise_equals_group_deletion(kind, mode, C, mode_guard):
    N = 10000
    g_np = np.arange(N) // 25 if kind == "runs_of_25" else _random_size_groups(N, C)
    bank, lab = _lot_bank(N, 256, C, 600 + C, g_np)
    groups = _t(g_np)
    b200knn.set_default_mode(mode)
    ks, ts = (20, 1, 200, 5), (0.1, 0.5, 0.07)  # not ascending: output follows the caller's order
    before = dict(K.graph_stats)
    got = b200knn.knn_predict_loo(bank, lab, C, ks, ts, batch=700, groups=groups)
    assert K.graph_stats == before
    assert got.shape == (4, 3, N, C) and got.dtype == torch.int64
    rows = np.concatenate([[0, N - 1], _rows(N, 38, C)])
    _assert_equals_deletion(got, bank, lab, C, ks, ts, groups, rows)
    # the leakage this removes: with its lot-mates in the vote, a row's ranking is another one
    plain = b200knn.knn_predict_loo(bank, lab, C, ks, ts, batch=700)
    sizes = np.bincount(np.unique(g_np, return_inverse=True)[1])[np.unique(g_np, return_inverse=True)[1]]
    lot_rows = [int(r) for r in rows if sizes[r] >= 5]
    assert len(lot_rows) >= 20
    differ = sum(not torch.equal(plain[:, :, r], got[:, :, r]) for r in lot_rows)
    assert differ >= 0.9 * len(lot_rows), (differ, len(lot_rows))


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_group_beyond_max_k_takes_peeling_path(mode, mode_guard):
    N, C = 6000, 9
    bank, lab = _bank(N, 256, C, 17)
    rng = np.random.default_rng(17)
    g_np = np.arange(N, dtype=np.int64)
    big = np.sort(rng.choice(N, 1500, replace=False))
    g_np[big] = -3  # one group of 1,500 rows: it searches at k + 2048 > MAX_K
    groups = _t(g_np)
    ks, ts = (5, 50), (0.1, 0.07)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_loo(bank, lab, C, ks, ts, groups=groups)
    in_big = big[rng.choice(big.size, 5, replace=False)]
    others = np.setdiff1d(_rows(N, 12, 18), big)[:5]
    if mode == "bf16":
        b200knn.set_default_mode("exact")
        exact = b200knn.knn_predict_loo(bank, lab, C, ks, ts, groups=groups)
        idx = _t(big)
        assert torch.equal(got[:, :, idx], exact[:, :, idx])
        b200knn.set_default_mode("bf16")
        _assert_equals_deletion(got, bank, lab, C, ks, ts, groups, others)
    else:
        _assert_equals_deletion(got, bank, lab, C, ks, ts, groups, np.concatenate([in_big, others]))


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_k_up_to_n_minus_largest_group(mode, mode_guard):
    N = 300
    bank, lab = _bank(N, 128, 9, 19)
    g_np = np.arange(N) // 10
    g_np[:3] = 1000  # sizes 7, 10, ..., and 3
    groups = _t(g_np)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_loo(bank, lab, 9, (N - 10, 4), (0.1,), groups=groups)
    _assert_equals_deletion(got, bank, lab, 9, (N - 10, 4), (0.1,), groups, [0, 5, 17, N - 1])
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        b200knn.knn_predict_loo(bank, lab, 9, (4, N - 9), (0.1,), groups=groups)


@pytest.mark.parametrize("mode", ["fp32", "bf16", "exact"])
def test_logo_independent_of_batch(mode, mode_guard):
    N = 9000
    g_np = _random_size_groups(N, 20)
    bank, lab = _lot_bank(N, 512, 9, 20, g_np)
    groups = _t(g_np)
    b200knn.set_default_mode(mode)
    ks, ts = (5, 20, 200), (0.1, 0.07)
    ref = b200knn.knn_predict_loo(bank, lab, 9, ks, ts, batch=N, groups=groups)
    for batch in (1000, 333, 4099, N + 5):  # cuts through buckets and groups
        assert torch.equal(b200knn.knn_predict_loo(bank, lab, 9, ks, ts, batch=batch, groups=groups), ref), batch


def test_logo_repair_levels(mode_guard):
    """Rows the cascade's first level leaves uncertified are repaired at the bucket's depth."""
    c = datagen.make_case("absgauss_small")
    bank, lab, C = _t(c["bank"]), _t(c["labels"]), c["C"]
    N = bank.shape[1]
    groups = torch.arange(N, device=DEV) // 8
    reached = []
    for mode in ("fp32", "fp32_bf16"):
        b200knn.set_default_mode(mode)
        got = b200knn.knn_predict_loo(bank, lab, C, KS, TS, groups=groups)
        reached.append(len(K.last_rescore_stats["levels"]) > 1)
        _assert_equals_deletion(got, bank, lab, C, KS, TS, groups, _rows(N, 12, 3))
    assert any(reached), K.last_rescore_stats


@pytest.mark.parametrize("mode", ["exact", "fp32"])
def test_logo_equals_seq_oracle_on_golden(mode, golden_dir, mode_guard):
    g = np.load(os.path.join(golden_dir, "real_FastSiam.npz"))
    b = g["bank_rows_f16"].astype(np.float32)
    b = b / np.maximum(np.linalg.norm(b, axis=1, keepdims=True), 1e-12)
    bank, labels, C = np.ascontiguousarray(b.T), g["bank_labels"].astype(np.int64), 9
    groups = np.arange(3000) // 25
    sims = O.sims_seqfma(b, bank)
    sims[groups[:, None] == groups[None, :]] = -np.inf  # every column of the row's own group
    ss, si = O.canonical_topk_c(sims, max(KS))
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_loo(_t(bank), _t(labels), C, KS, TS, groups=_t(groups)).cpu().numpy()
    assert got.shape == (len(KS), len(TS), 3000, C)
    for i, k in enumerate(KS):
        for j, t in enumerate(TS):
            assert np.array_equal(got[i, j], O.vote_o64(ss[:, :k], si[:, :k], labels, C, t)[0]), (k, t)


def _drop_group_np(keys, row_ids, gids, k_out):
    N = gids.size
    _, idx = O.decode_keys(keys)
    out = np.zeros((keys.shape[0], k_out), dtype=np.uint64)
    bad = False
    for b in range(keys.shape[0]):
        own_ok = 0 <= row_ids[b] < N
        bad |= not own_ok
        nonempty = keys[b] != 0
        in_range = (idx[b] >= 0) & (idx[b] < N)
        bad |= bool((nonempty & ~in_range).any())
        member = nonempty & in_range & own_ok
        member[member] = gids[idx[b][member]] == (gids[row_ids[b]] if own_ok else 0)
        kept = keys[b][~member][:k_out]
        out[b, :kept.size] = kept
    return out, bad


@pytest.mark.parametrize("k_in", [2, 31, 32, 33, 201, 1001])
def test_drop_group_against_numpy(k_in):
    rng = np.random.default_rng(k_in)
    B, N = 777, 50000
    gids = rng.integers(0, 400, N).astype(np.int32)
    members = [np.flatnonzero(gids == g) for g in range(400)]
    row_ids = rng.integers(0, N, B)
    sims = -np.sort(-rng.standard_normal((B, k_in)).astype(np.float32), axis=1)
    idx = rng.integers(0, N, (B, k_in))
    heavy = rng.random(B) < 0.3  # rows whose lists are mostly their own group: fewer than k_out survive
    for b in np.flatnonzero(heavy):
        pick = rng.random(k_in) < 0.8
        idx[b, pick] = rng.choice(members[gids[row_ids[b]]], int(pick.sum()))
    keys = O.make_keys(sims, idx)
    empty = rng.random(B) < 0.2  # trailing empty slots
    cut = rng.integers(0, k_in, B)
    for b in np.flatnonzero(empty):
        keys[b, cut[b]:] = 0
    keys_t, rows_t, gids_t = _t(keys.view(np.int64)), _t(row_ids), _t(gids)
    for k_out in sorted({1, max(1, k_in // 2), max(1, k_in - 33), k_in}):
        flag = torch.zeros((1,), dtype=torch.int32, device=DEV)
        got = K.drop_group(keys_t, rows_t, gids_t, k_out, flag).cpu().numpy().view(np.uint64)
        want, bad = _drop_group_np(keys, row_ids, gids, k_out)
        assert not bad and int(flag.item()) == 0
        assert np.array_equal(got, want), k_out
    # a key index and row ids outside [0, N): flagged, the key kept, the row drops nothing
    keys_bad, rows_bad = keys.copy(), row_ids.copy()
    keys_bad[5, 0] = O.make_keys(sims[5:6, :1], np.array([[N + 3]]))[0, 0]
    rows_bad[7], rows_bad[8] = -1, N
    k_out = max(1, k_in - 1)
    flag = torch.zeros((1,), dtype=torch.int32, device=DEV)
    got = K.drop_group(_t(keys_bad.view(np.int64)), _t(rows_bad), gids_t, k_out, flag).cpu().numpy().view(np.uint64)
    want, bad = _drop_group_np(keys_bad, rows_bad, gids, k_out)
    assert bad and int(flag.item()) == 2
    assert np.array_equal(got, want)
    with pytest.raises(RuntimeError, match="outside the group ids"):
        K.drop_group(_t(keys_bad.view(np.int64)), _t(rows_bad), gids_t, k_out)
    with pytest.raises(RuntimeError, match=f"row_ids has {B - 1} entries for {B} rows"):
        K.drop_group(keys_t, rows_t[1:], gids_t, 1)
    with pytest.raises(RuntimeError, match="same device"):
        K.drop_group(keys_t, rows_t, gids_t.cpu(), 1)


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_knn_graph_leaves_the_group_out(mode):
    N, k = 4000, 12
    g_np = _random_size_groups(N, 21)
    gen = torch.Generator(device=DEV).manual_seed(21)
    x = torch.randn(N, 256, generator=gen, device=DEV)
    _, lot = np.unique(g_np, return_inverse=True)
    x += 3 * torch.randn(int(lot.max()) + 1, 256, generator=gen, device=DEV)[_t(lot)]  # lot-mates near each other
    groups = _t(g_np)
    sims, idx = b200knn.knn_graph(x, k, normalize=False, mode=mode, batch=1500, groups=groups)
    assert not bool((groups[idx] == groups.view(-1, 1)).any())
    g_max = int(np.bincount(lot).max())
    keys = K.topk_keys(x, x.t().contiguous(), k + g_max, mode)  # deeper than any row's search
    s_all, i_all = K.decode_keys(keys)
    keep = groups[i_all] != groups.view(-1, 1)
    keep &= keep.cumsum(1) <= k
    assert torch.equal(idx, i_all[keep].view(N, k)) and torch.equal(sims, s_all[keep].view(N, k))
    # singleton groups: the plain graph
    plain = b200knn.knn_graph(x, k, normalize=False, mode=mode, batch=1500)
    got = b200knn.knn_graph(x, k, normalize=False, mode=mode, batch=1500, groups=torch.arange(N, device=DEV))
    assert torch.equal(got[0], plain[0]) and torch.equal(got[1], plain[1])


def test_feature_bank_and_fp16_bank(mode_guard):
    rng = np.random.default_rng(4)
    C, N = 9, 8000
    g_np = np.arange(N) // 25
    rows = _t(rng.standard_normal((N, 512)).astype(np.float32) * 3)
    lab = _t(datagen.labels(N, C, 4))
    groups = _t(g_np)
    fb = b200knn.FeatureBank.from_rows(rows, lab)
    b200knn.set_default_mode("fp32")
    got = fb.knn_predict_loo(C, KS, TS, groups=groups)
    assert torch.equal(got, b200knn.knn_predict_loo(fb.bank, fb.labels, C, KS, TS, groups=groups))
    _assert_equals_deletion(got, fb.bank, fb.labels, C, KS, TS, groups, [0, 4321, 7999])
    bank16 = fb.bank.half().contiguous()
    for mode in ("fp32", "bf16"):
        b200knn.set_default_mode(mode)
        got16 = b200knn.knn_predict_loo(bank16, lab, C, (5, 20), (0.1,), groups=groups)
        _assert_equals_deletion(got16, bank16, lab, C, (5, 20), (0.1,), groups, [1, 2500, 7998])


def test_unsigned_group_ids(mode_guard):
    N = 3000
    bank, lab = _bank(N, 128, 9, 6)
    g = torch.arange(N, device=DEV) // 12  # 250 groups: ids fit every unsigned width
    b200knn.set_default_mode("fp32")
    want = b200knn.knn_predict_loo(bank, lab, 9, (5, 20), (0.1,), groups=g)
    for dt in (torch.uint8, torch.uint16, torch.uint32, torch.uint64):
        assert torch.equal(b200knn.knn_predict_loo(bank, lab, 9, (5, 20), (0.1,), groups=g.to(dt)), want), dt


def test_logo_label_and_device_errors(mode_guard):
    bank, lab = _bank(3000, 128, 9, 5)
    groups = torch.arange(3000, device=DEV) // 10
    bad = lab.clone()
    bad[:] = 9
    for mode in ("fp32", "exact"):
        b200knn.set_default_mode(mode)
        with pytest.raises(RuntimeError, match="num_classes=9"):
            b200knn.knn_predict_loo(bank, bad, 9, (5, 20), (0.1,), groups=groups)
    with pytest.raises(RuntimeError, match="Expected all tensors to be on the same device"):
        b200knn.knn_predict_loo(bank, lab, 9, (5,), groups=groups.cpu())
