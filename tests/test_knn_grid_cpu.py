"""CPU: knn_predict_multi — the (k, t) grid from one neighbour search.  The C ABI's argument checks,
the Python argument errors, the sharded driver under gloo (compute served by the oracle, as in
test_dist_gloo.py) and the opt-in grid of the validation hooks (reference module with stubbed
imports, as in test_hooks_cpu.py)."""
import ctypes
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import datagen
from oracle import knn_oracle as O
from test_dist_gloo import OracleOps, _free_port
from test_hooks_cpu import _Loader, _OracleBank, _oracle_metrics, reference_module  # noqa: F401

import b200knn
from b200knn import _lib


def _grid_args(ks, ts):
    return (ctypes.c_int * max(1, len(ks)))(*ks), len(ks), (ctypes.c_double * max(1, len(ts)))(*ts), len(ts)


def test_vote_multi_abi_refuses_bad_grids_without_gpu():
    lib = _lib.load()

    def call(ks, ts, k_max=None, C=5, pred_ld=None, status_col=-1):
        k_max = ks[-1] if k_max is None and ks else (k_max or 1)
        ka, nk, ta, nt = _grid_args(ks, ts)
        ld = pred_ld if pred_ld is not None else max(1, nk * nt * C)
        return lib.b200knn_vote_multi(1, 1, 4, k_max, 10, 0, C, ka, nk, ta, nt, 1, ld, status_col, 1, None)

    for ks, ts, k_max, what in [((5, 3, 8), (0.1,), None, b"strictly increasing"),
                                ((3, 3), (0.1,), None, b"strictly increasing"),
                                ((0, 3), (0.1,), None, b"strictly increasing"),
                                ((3, 5), (0.1,), 6, b"k_max"),
                                ((3, 5), (0.1, 0.0), None, b"non-zero"),
                                ((), (0.1,), 5, b"n_k"),
                                (tuple(range(1, 18)), (0.1,), None, b"n_k"),
                                ((5,), (), None, b"n_k"),
                                ((5,), tuple(0.1 * i for i in range(1, 10)), None, b"n_k")]:
        assert call(ks, ts, k_max) == -1, (ks, ts)
        assert what in lib.b200knn_last_error(), (ks, ts, lib.b200knn_last_error())
    # output too narrow for n_k*n_t*C, status column inside the rankings
    assert call((3, 5), (0.1, 0.2), pred_ld=19) == -1
    assert call((3, 5), (0.1, 0.2), pred_ld=21, status_col=19) == -1


@pytest.mark.parametrize("ks,ts,match", [
    ((), (0.1,), "empty"), ((5,), (), "empty"), ((5, 5), (0.1,), "duplicate"), ((5,), (0.1, 0.1), "duplicate"),
    ((0, 5), (0.1,), "positive"), ((-3,), (0.1,), "positive"), ((5,), (0.0,), "non-zero"),
    (tuple(range(1, 18)), (0.1,), "at most"), ((5,), tuple(range(1, 10)), "at most"), ((2.5,), (0.1,), "integers"),
])
def test_python_argument_errors(ks, ts, match):
    c = datagen.make_case("ragged")
    f, bank, lab = (torch.from_numpy(c[n]) for n in ("feature", "bank", "labels"))
    with pytest.raises(ValueError, match=match):
        b200knn.knn_predict_multi(f, bank, lab, c["C"], ks, ts)
    with pytest.raises(ValueError, match=match):
        b200knn.ShardedBank(bank, lab, bank.shape[1], ops=_GridOps).knn_predict_multi(f, c["C"], ks, ts)


@pytest.mark.parametrize("k", [1, 200, 1023, 1024, 5000])
def test_vote_class_bound_without_gpu(k):
    """One class past vote_max_classes: B200KNN_E_UNSUPPORTED from the C ABI (refused before any CUDA
    call), a ValueError naming the bound from Python before any tensor reaches the device."""
    from b200knn import knn as K

    lib = _lib.load()
    for grid in (False, True):
        C = K.vote_max_classes(k, grid) + 1
        if grid:
            rc = lib.b200knn_vote_multi(1, 1, 4, k, 10, 0, C, *_grid_args((k,), (0.1,)), 1, C, -1, 1, None)
        else:
            rc = lib.b200knn_vote(1, 1, 4, k, 10, 0, C, 0.1, 1, None, 1, None)
        assert rc == -4 and b"num_classes too large" in lib.b200knn_last_error(), (grid, rc)
    # the figures include/b200knn.h and DESIGN.md quote
    assert [K.vote_max_classes(kk, g) for g in (False, True) for kk in (200, 5000)] == [6100, 4864, 6000, 4352]
    c = datagen.make_case("ragged")
    f, bank, lab = (torch.from_numpy(c[n]) for n in ("feature", "bank", "labels"))
    g1 = K.vote_max_classes(k, True) + 1
    if k < bank.shape[1]:
        with pytest.raises(ValueError, match=f"at most {g1 - 1} classes"):
            b200knn.knn_predict_multi(f, bank, lab, g1, (k,), (0.1,))
        with pytest.raises(ValueError, match=f"at most {g1 - 1} classes"):
            b200knn.knn_predict_loo(bank, lab, g1, (k,), (0.1,))


def test_cpu_tensors_raise():
    c = datagen.make_case("ragged")
    f, bank, lab = (torch.from_numpy(c[n]) for n in ("feature", "bank", "labels"))
    with pytest.raises(RuntimeError, match="CPU fallback|cuda|sm_100a"):
        b200knn.knn_predict_multi(f, bank, lab, c["C"], (1, 5), (0.1,))


def test_grid_view_restores_caller_order():
    B, C, n_t = 3, 4, 2
    order = [2, 0, 1]  # ascending ks sit at caller positions 2, 0, 1
    pred = torch.arange(B * 3 * n_t * C).view(B, 3 * n_t * C)
    g = b200knn.knn.grid_view(pred, order, n_t, C)
    blocks = pred.view(B, 3, n_t, C)
    for pos, i in enumerate(order):
        assert torch.equal(g[i], blocks[:, pos].permute(1, 0, 2))


class _GridOps(OracleOps):
    """OracleOps + the grid vote: O.vote_o64 on each prefix of the key lists."""

    @classmethod
    def vote_multi_packed(cls, keys, labels, num_classes, knn_ks, knn_ts, n_rows_out):
        W = len(knn_ks) * len(knn_ts) * num_classes
        out = torch.zeros((n_rows_out, W + 1), dtype=torch.int64)
        n = keys.shape[0]
        if n:
            blocks = [cls.vote(keys[:, :k], labels, num_classes, t) for k in knn_ks for t in knn_ts]
            out[:n, :W] = torch.cat(blocks, dim=1)
            out[:n, W] = (keys[:, -1] == 0).to(torch.int64)
        return out


def _case_grid(c):
    ks = tuple(dict.fromkeys((c["k"], 1, 5, 3)))  # k_max first: the caller's order is not ascending
    return ks, (0.5, 0.07, 0.1)


def _want_grid(c):
    ks, ts = _case_grid(c)
    s, i = O.topk_seqfma(c["feature"], c["bank"], max(ks))
    return np.stack([np.stack([O.vote_o64(s[:, :k], i[:, :k], c["labels"], c["C"], t)[0] for t in ts]) for k in ks])


def _worker(rank, world, port, case, out_dir, stride, poison, mode, force_uncertified, l2_fail_rank):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        from b200knn import ShardedBank

        _GridOps.sample_stride, _GridOps.poison_threshold = stride, poison
        _GridOps.force_uncertified = force_uncertified
        _GridOps.l2_fail_rank = l2_fail_rank
        c = datagen.make_case(case)
        sb = ShardedBank.from_full(torch.from_numpy(c["bank"]), torch.from_numpy(c["labels"]), ops=_GridOps,
                                   mode=mode)
        q = torch.from_numpy(c["feature"])
        ks, ts = _case_grid(c)
        pred = sb.knn_predict_multi(q, c["C"], ks, ts)
        assert torch.equal(pred, sb.knn_predict_multi(q, c["C"], ks, ts, exchange="allgather"))
        np.save(os.path.join(out_dir, f"grid_{rank}.npy"), pred.numpy())
        dist.barrier()
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("world,case,stride,poison,mode,force,fail_rank", [
    (2, "clustered_small", 0, False, "bf16", False, -1),   # no pre-pass
    (3, "gauss_small", 4, True, "bf16", False, -1),        # a row's sampled threshold poisoned -> recomputed
    (3, "ragged", 0, False, "fp32", False, -1),            # fp32 path, ragged shards
    (2, "mixed38", 4, False, "fp32", True, -1),            # certificates forced to fail -> device level 2
    (3, "clustered_small", 4, True, "fp32", False, -1),    # starved row -> uncertified -> fallback
    (3, "mixed38", 4, False, "fp32", True, 2),             # one shard fails its local certificate -> host path
])
def test_sharded_grid_equals_oracle(world, case, stride, poison, mode, force, fail_rank, tmp_path):
    mp.spawn(_worker, args=(world, _free_port(), case, str(tmp_path), stride, poison, mode, force, fail_rank),
             nprocs=world, join=True)
    want = _want_grid(datagen.make_case(case))
    for r in range(world):
        got = np.load(tmp_path / f"grid_{r}.npy")
        assert got.shape == want.shape and np.array_equal(got, want), r


class _GridOracleBank(_OracleBank):
    def knn_predict_multi(self, feature, num_classes, knn_ks, knn_ts, normalize=False):
        return torch.stack([torch.stack([self.knn_predict(feature, num_classes, k, t, normalize) for t in knn_ts])
                            for k in knn_ks])


def test_hooks_with_grid_keep_own_setting_and_log_grid(reference_module, monkeypatch):
    ref = reference_module
    C, D, n_bank, n_val, bs = 9, 64, 700, 200, 64
    rng = np.random.default_rng(11)
    lab = datagen.labels(n_bank, C, 1)
    emb = (datagen.clustered(n_bank, D, C, 2, lab) * rng.uniform(0.5, 9, (n_bank, 1))).astype(np.float32)
    vlab = datagen.labels(n_val, C, 3)
    vemb = datagen.clustered(n_val, D, C, 4, vlab)
    loader = _Loader([(torch.from_numpy(emb[i:i + bs]), torch.from_numpy(lab[i:i + bs]))
                      for i in range(0, n_bank, bs)], n_bank)
    val = [(torch.from_numpy(vemb[i:i + bs]), torch.from_numpy(vlab[i:i + bs])) for i in range(0, n_val, bs)]
    b200knn.install(hooks=True)
    monkeypatch.setattr(b200knn.hooks._bank, "FeatureBank", _GridOracleBank)
    monkeypatch.setattr(b200knn.hooks._metrics, "knn_metrics", _oracle_metrics)

    def epoch(grid):
        m = ref.KNNBenchmarkModule(loader, C, knn_k=5, knn_t=0.1)
        if grid is not None:
            m.b200knn_knn_grid = grid
        m.backbone = torch.nn.Identity()
        m.on_validation_epoch_start()
        for i, b in enumerate(val):
            m.validation_step(b, i)
        preds = torch.cat(m.all_preds).clone()
        m.on_validation_epoch_end()
        return m, preds

    plain, p0 = epoch(None)
    gridded, p1 = epoch(((20, 1), (0.07,)))
    assert torch.equal(p0, p1)
    assert gridded.max_accuracy == plain.max_accuracy and gridded.max_f1 == plain.max_f1
    assert np.array_equal(gridded.confusion_matrix[0], plain.confusion_matrix[0])
    for key in ("knn_accuracy", "knn_f1"):
        assert gridded.logged[key] == plain.logged[key]
    assert set(plain.logged) == {"knn_accuracy", "knn_f1"}
    grid_keys = {f"knn_{m}_k{k}_t{t}" for m in ("accuracy", "f1") for k in (20, 1, 5) for t in ("0.07", "0.1")}
    assert set(gridded.logged) == {"knn_accuracy", "knn_f1"} | grid_keys
    assert gridded.logged["knn_accuracy_k5_t0.1"] == plain.logged["knn_accuracy"]
    s, i = O.topk_seqfma(O.normalize_rows_ref(vemb), np.ascontiguousarray(O.normalize_rows_ref(emb).T), 20)
    want = O.metrics_ref(O.vote_o64(s, i, lab, C, 0.07)[0][:, 0], vlab, C)
    assert abs(gridded.logged["knn_accuracy_k20_t0.07"] - want["accuracy"]) < 1e-12
    assert gridded.all_preds == [] and "_b200knn_grid_preds" not in gridded.__dict__
