"""GPU: group exclusion inside the neighbour search.  topk_keys(exclude=(query ids, bank ids)) skips
every bank column whose id equals the query row's id, so its keys are bitwise those of a search of
the bank with those columns deleted, indices mapped back to the full bank — in every mode, for single
CTAs and CTA pairs, both tile widths, every list capacity, bank splits, the chunk-major order, ragged
N, duplicates, exactly k eligible rows, excluded peeling and the cascade's later levels.  Then the
public surface: knn_predict_multi / knn_topk with query and bank groups, k-fold cross-validation
through knn_predict_loo(groups=folds) (also against the SEQ oracle on the real golden table) and
knn_graph(groups=) with a group deeper than the streaming lists."""
import os

import numpy as np
import pytest
import torch

import b200knn
import datagen
from b200knn import _lib
from b200knn import knn as K
from oracle import knn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
MODES = ["fp32", "exact", "fp32_f16x2", "f16", "bf16", "bf16x3", "tf32x3"]


@pytest.fixture()
def mode_guard():
    yield
    b200knn.set_default_mode("exact")
    K.GRAPHS["enabled"] = True
    _lib.load().b200knn_set_l2_chunk_bytes(40 << 20)


def _lots(N, B, D, seed, lot=25):
    """A bank of lots (N // lot groups of `lot` rows, each a tight cluster) and B queries that are
    perturbed copies of random bank rows carrying that row's lot id: a query's own lot fills the top
    of its unrestricted list, so the exclusion changes every list."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    bg = (torch.arange(N, device=DEV) // lot).to(torch.int32)
    centre = torch.randn((N + lot - 1) // lot, D, generator=g, device=DEV)
    rows = centre[bg.long()] + 0.15 * torch.randn(N, D, generator=g, device=DEV)
    rows = torch.nn.functional.normalize(rows, dim=1)
    src = torch.randint(0, N, (B,), generator=g, device=DEV)
    q = torch.nn.functional.normalize(rows[src] + 0.05 * torch.randn(B, D, generator=g, device=DEV), dim=1)
    return q.contiguous(), rows.t().contiguous(), bg[src].contiguous(), bg


def _deleted_keys(q, bank, k, mode, qg, bg, b):
    """(sims, full-bank idx) of query b searched against the bank without its group's columns."""
    keep = (bg != qg[b]).nonzero(as_tuple=False).view(-1)
    s, i = K.decode_keys(K.topk_keys(q[b:b + 1].contiguous(), bank[:, keep].contiguous(), k, mode))
    return s[0], keep[i[0]]


def _assert_rows_equal_deletion(keys, q, bank, k, mode, qg, bg, rows):
    sims, idx = K.decode_keys(keys)
    for b in rows:
        b = int(b)
        ws, wi = _deleted_keys(q, bank, k, mode, qg, bg, b)
        assert torch.equal(sims[b].view(torch.int32), ws.view(torch.int32)) and torch.equal(idx[b], wi), (mode, b)


def _check_rows(B, n=24, seed=0):
    rng = np.random.default_rng(seed)
    return np.unique(np.concatenate([[0, B - 1], rng.choice(B, min(B, n), replace=False)]))


# name: (B, N, D, k, what the plan must show)
CONFIGS = {
    "single_cta_splits_ragged": (100, 20011, 256, 200, "single"),
    "pair": (300, 12000, 256, 100, "pair"),
    "tile128_d768": (300, 6000, 768, 100, "tile128"),  # resident-query modes: 128-wide bank tiles
    "wide_d800": (300, 6000, 800, 100, "wide"),         # no resident query tile: CASCADE_WIDE / bf16x3
    "cap64": (200, 8000, 128, 5, 64),
    "cap128": (200, 8000, 128, 40, 128),
    "cap1024_k500": (200, 8000, 128, 500, 1024),
    "cap1024_k992": (200, 8000, 128, 992, 1024),
    "chunks": (37883, 20011, 128, 50, "chunks"),
}


def _kernel_mode(mode, D):
    if mode in K.RESCORED_MODES:
        return None
    return mode if mode == "exact" else K.effective_mode(mode, D)


@pytest.mark.parametrize("cfg", list(CONFIGS))
@pytest.mark.parametrize("mode", MODES)
def test_topk_keys_exclude_equals_column_deletion(mode, cfg, mode_guard):
    B, N, D, k, what = CONFIGS[cfg]
    lib = _lib.load()
    q, bank, qg, bg = _lots(N, B, D, seed=list(CONFIGS).index(cfg))
    km = _kernel_mode(mode, D)
    if what == "chunks":
        assert lib.b200knn_set_l2_chunk_bytes(1 << 20) == 0
    if km is not None:  # the plan the search runs under reaches what the case is for
        plan = K.plan_info(B, N, D, k, km)
        if what == "single":
            assert plan["splits"] > 1 and plan["n_qtiles"] == 1 and N % 128, plan
        elif what == "pair" and km in ("bf16", "f16", "f16x2"):
            assert plan["n_qtiles"] == -(-B // 256), plan  # 256-row tiles: CTA pairs
        elif what == "chunks" and km != "exact":
            assert plan["chunks"] > 1 and plan["splits"] == 1, plan
        elif what == "tile128" and km in ("bf16", "f16", "f16x2"):
            assert K.padded_dim(D) == K.MAX_BF16_DIM > 512, D  # tc_tile_n: 128-wide tiles above 512
        elif what == "wide" and mode in ("bf16", "f16", "f16x2"):  # the resident-query modes
            assert km == "bf16x3", km
        elif isinstance(what, int):
            assert plan["list_capacity"] == what, plan
    keys = K.topk_keys(q, bank, k, mode, exclude=(qg, bg))
    if what == "wide" and mode == "fp32":
        assert K.last_rescore_stats["level"].startswith(K.CASCADE_WIDE[0].partition("@")[0])
    assert keys.shape == (B, k)
    _assert_rows_equal_deletion(keys, q, bank, k, mode, qg, bg, _check_rows(B, seed=B))
    if mode in ("fp32", "fp32_f16x2"):  # the cascade's keys are the exact mode's
        rows = torch.from_numpy(_check_rows(B, 8, seed=1)).to(DEV)
        assert torch.equal(keys[rows], K.topk_keys(q[rows].contiguous(), bank, k, "exact",
                                                   exclude=(qg[rows].contiguous(), bg)))


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16", "f16x2"])
def test_duplicates_inside_and_outside_the_group(mode, mode_guard):
    """Exact copies of a query in its own group are all skipped; copies in other groups are kept,
    lowest index first."""
    N, D, k = 4000, 128, 20
    g = torch.Generator(device=DEV).manual_seed(5)
    rows = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=DEV), dim=1)
    bg = (torch.arange(N, device=DEV) // 10).to(torch.int32)
    q = rows[[15, 2300]].clone()
    rows[[11, 17, 19]] = q[0]        # group 1, query 0's own group
    rows[[3000, 1234]] = q[0]        # groups 300 and 123
    rows[[2301, 2305]] = q[1]        # group 230, query 1's own group
    rows[[77, 3999]] = q[1]          # groups 7 and 399
    bank = rows.t().contiguous()
    qg = torch.tensor([1, 230], dtype=torch.int32, device=DEV)
    keys = K.topk_keys(q, bank, k, mode, exclude=(qg, bg))
    sims, idx = K.decode_keys(keys)
    for b, own, other in ((0, [11, 15, 17, 19], [1234, 3000]), (1, [2300, 2301, 2305], [77, 3999])):
        got = idx[b].tolist()
        assert not set(own) & set(got), (b, got)
        pos = [got.index(i) for i in other]
        assert pos[1] == pos[0] + 1 and sims[b, pos[0]] == sims[b, pos[1]], (b, got)
    _assert_rows_equal_deletion(keys, q, bank, k, mode, qg, bg, [0, 1])


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16", "tf32x3"])
def test_query_id_without_bank_rows_is_the_plain_search(mode, mode_guard):
    q, bank, qg, bg = _lots(9000, 300, 256, 8)
    none = torch.full_like(qg, 10 ** 6)  # no bank row has this id
    K.query_cache.clear()
    assert torch.equal(K.topk_keys(q, bank, 50, mode, exclude=(none, bg)), K.topk_keys(q, bank, 50, mode))


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16", "f16x2"])
def test_exactly_k_eligible_rows(mode, mode_guard):
    N, k = 1200, 150
    q, bank, _, _ = _lots(N, 64, 128, 9)
    bg = torch.zeros(N, dtype=torch.int32, device=DEV)
    bg[torch.randperm(N, generator=torch.Generator().manual_seed(9))[:k].to(DEV)] = 1  # k rows outside group 0
    qg = torch.zeros(64, dtype=torch.int32, device=DEV)
    keys = K.topk_keys(q, bank, k, mode, exclude=(qg, bg))
    assert bool((keys != 0).all())
    _, idx = K.decode_keys(keys)
    assert torch.equal(idx.sort(dim=1).values[0], (bg == 1).nonzero().view(-1))
    _assert_rows_equal_deletion(keys, q, bank, k, mode, qg, bg, [0, 31, 63])
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        K.topk_keys(q, bank, k + 1, mode, exclude=(qg, bg))


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_k_beyond_max_k_takes_excluded_peeling(mode, mode_guard):
    q, bank, qg, bg = _lots(6000, 40, 128, 10, lot=600)
    keys = K.topk_keys(q, bank, 1500, mode, exclude=(qg, bg))
    _assert_rows_equal_deletion(keys, q, bank, 1500, "exact", qg, bg, [0, 7, 39])


def test_cascade_levels_and_exact_fallback_with_exclusion(mode_guard):
    c = datagen.make_case("absgauss_small")
    bank = torch.from_numpy(np.ascontiguousarray(c["bank"])).to(DEV)
    N = bank.shape[1]
    bg = (torch.arange(N, device=DEV) // 8).to(torch.int32)
    q = bank.t()[::3].contiguous()  # bank rows as queries: their own group holds the row itself
    qg = bg[::3].contiguous()
    rows = _check_rows(q.shape[0], 12, seed=3)
    reached = []
    for mode in ("fp32", "fp32_bf16"):
        keys = K.topk_keys(q, bank, c["k"], mode, exclude=(qg, bg))
        levels = K.last_rescore_stats["levels"]
        reached.append(len(levels) > 1)
        idx = torch.from_numpy(rows).to(DEV)
        assert torch.equal(keys[idx], K.topk_keys(q[idx].contiguous(), bank, c["k"], "exact",
                                                  exclude=(qg[idx].contiguous(), bg))), levels
        _assert_rows_equal_deletion(keys, q, bank, c["k"], "exact", qg, bg, rows)
    assert any(reached), K.last_rescore_stats


# ------------------------------------------------------------------ public surface
def _lot_labels(bg, C, seed):
    rng = np.random.default_rng(seed)
    n_lots = int(bg.max()) + 1
    lot_lab = torch.from_numpy(rng.integers(0, C, n_lots)).to(DEV)
    lab = lot_lab[bg.long()].clone()
    flip = torch.from_numpy(rng.random(bg.numel()) < 0.2).to(DEV)
    lab[flip] = torch.from_numpy(rng.integers(0, C, int(flip.sum()))).to(DEV)
    return lab


@pytest.mark.parametrize("B", [300, 700])
@pytest.mark.parametrize("C", [9, 38])
@pytest.mark.parametrize("mode", ["fp32", "bf16"])
def test_knn_predict_multi_with_groups_equals_per_row_deletion(mode, C, B, mode_guard):
    N = 12000
    q, bank, qg, bg = _lots(N, B, 256, 40 + C)
    lab = _lot_labels(bg, C, C)
    qgroups, bgroups = (qg.long() * 7 - 3), (bg.long() * 7 - 3).to(torch.int16)  # any values and dtypes
    ks, ts = (20, 1, 200, 5), (0.1, 0.5, 0.07)
    b200knn.set_default_mode(mode)
    before = dict(K.graph_stats)
    got = b200knn.knn_predict_multi(q, bank, lab, C, ks, ts, query_groups=qgroups, bank_groups=bgroups)
    assert K.graph_stats == before  # calls with groups never capture or replay a graph
    assert got.shape == (4, 3, B, C)
    K.GRAPHS["enabled"] = False  # the per-row references below: one bank each, nothing to replay
    plain = b200knn.knn_predict_multi(q, bank, lab, C, ks, ts)
    rows = _check_rows(B, 30, seed=C)
    differ = 0
    for b in rows:
        b = int(b)
        keep = bg != qg[b]
        want = b200knn.knn_predict_multi(q[b:b + 1], bank[:, keep].contiguous(), lab[keep].contiguous(), C, ks, ts)
        assert torch.equal(got[:, :, b], want[:, :, 0]), b
        differ += not torch.equal(got[:, :, b], plain[:, :, b])
    assert differ >= len(rows) // 2, differ  # the leakage the groups remove
    # knn_topk and FeatureBank take the same groups
    s, i = b200knn.knn_topk(q, bank, 20, query_groups=qgroups, bank_groups=bgroups)
    assert not bool((bg[i] == qg[:, None]).any())
    fb = b200knn.FeatureBank(torch.nn.functional.pad(bank.t(), (0, 0)).contiguous(), 256, lab)
    assert torch.equal(fb.knn_predict_multi(q, C, ks, ts, query_groups=qgroups, bank_groups=bgroups), got)
    s2, i2 = fb.knn_topk(q, 20, query_groups=qgroups, bank_groups=bgroups)
    assert torch.equal(i2, i) and torch.equal(s2, s)


def _folds(N, n_folds, seed, labels=None):
    """Stratified fold ids when labels are given (as sklearn's StratifiedKFold), else shuffled."""
    rng = np.random.default_rng(seed)
    f = np.empty(N, dtype=np.int64)
    if labels is None:
        f[rng.permutation(N)] = np.arange(N) % n_folds
        return f
    for c in np.unique(labels):
        rows = rng.permutation(np.flatnonzero(labels == c))
        f[rows] = np.arange(rows.size) % n_folds
    return f


@pytest.mark.parametrize("mode", ["fp32", "exact", "bf16"])
def test_five_fold_cross_validation_equals_per_row_deletion(mode, mode_guard):
    N, C = 20000, 9
    lab_np = datagen.labels(N, C, 61)
    bank = torch.from_numpy(np.ascontiguousarray(datagen.clustered(N, 256, C, 62, lab_np).T)).to(DEV)
    lab = torch.from_numpy(lab_np).to(DEV)
    folds = torch.from_numpy(_folds(N, 5, 63, lab_np)).to(DEV)
    ks, ts = (5, 20, 200), (0.07, 0.1)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_loo(bank, lab, C, ks, ts, groups=folds)
    assert got.shape == (3, 2, N, C)
    if mode == "bf16":  # every fold row searches deeper than MAX_K: the exact mode's result
        b200knn.set_default_mode("exact")
        assert torch.equal(got, b200knn.knn_predict_loo(bank, lab, C, ks, ts, groups=folds))
    for r in _check_rows(N, 30, seed=64):
        r = int(r)
        keep = folds != folds[r]
        want = b200knn.knn_predict_multi(bank[:, r:r + 1].t(), bank[:, keep].contiguous(), lab[keep].contiguous(),
                                         C, ks, ts)
        assert torch.equal(got[:, :, r], want[:, :, 0]), r


@pytest.mark.parametrize("mode", ["exact", "fp32"])
def test_five_fold_equals_seq_oracle_on_golden(mode, golden_dir, mode_guard):
    g = np.load(os.path.join(golden_dir, "real_FastSiam.npz"))
    b = g["bank_rows_f16"].astype(np.float32)
    b = b / np.maximum(np.linalg.norm(b, axis=1, keepdims=True), 1e-12)
    bank, labels, C = np.ascontiguousarray(b.T), g["bank_labels"].astype(np.int64), 9
    folds = _folds(3000, 5, 7, labels)
    ks, ts = (1, 5, 20, 200), (0.07, 0.1, 0.5)
    sims = O.sims_seqfma(b, bank)
    sims[folds[:, None] == folds[None, :]] = -np.inf  # every column of the row's own fold
    ss, si = O.canonical_topk_c(sims, max(ks))
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_loo(torch.from_numpy(bank).to(DEV), torch.from_numpy(labels).to(DEV), C, ks, ts,
                                  groups=torch.from_numpy(folds).to(DEV)).cpu().numpy()
    for i, k in enumerate(ks):
        for j, t in enumerate(ts):
            assert np.array_equal(got[i, j], O.vote_o64(ss[:, :k], si[:, :k], labels, C, t)[0]), (k, t)


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_knn_graph_group_beyond_max_k(mode, mode_guard):
    N, k = 6000, 10
    rng = np.random.default_rng(71)
    rows = torch.from_numpy(rng.standard_normal((N, 96)).astype(np.float32)).to(DEV)
    g_np = np.arange(N, dtype=np.int64)
    big = np.sort(rng.choice(N, 1500, replace=False))
    g_np[big] = -1  # one group of 1,500 rows: its search skips the group inside the kernel
    groups = torch.from_numpy(g_np).to(DEV)
    sims, idx = b200knn.knn_graph(rows, k, mode=mode, groups=groups)
    fb = b200knn.FeatureBank.from_rows(rows)
    want_mode = "exact" if mode == "bf16" else mode
    for r in np.concatenate([big[:4], [0, 1, N - 1]]):
        r = int(r)
        keep = (groups != groups[r]).nonzero().view(-1)
        ws, wi = b200knn.knn_topk(fb.rows[r:r + 1, :96], fb.bank[:, keep].contiguous(), k,
                                  mode=want_mode if r in set(big.tolist()) else mode)
        assert torch.equal(sims[r].view(torch.int32), ws[0].view(torch.int32)) and torch.equal(idx[r], keep[wi[0]]), r
