"""GPU: knn_predict_multi — every (k, t) of a grid from one neighbour search is bitwise the separate
knn_predict call: across modes, batch sizes (graph path and eager), C = 38 and C = 1, the peeling
path (k > MAX_K), the cascade's repair levels, tie floods, FeatureBank's fused normalise, the
validation hooks' opt-in grid and the sharded bank over 2 GPUs."""
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


def _separate(q, bank, lab, C, ks, ts):
    return torch.stack([torch.stack([b200knn.knn_predict(q, bank, lab, C, k, t) for t in ts]) for k in ks])


def _bank(N, D, C, B, seed):
    lab = datagen.labels(N, C, seed)
    bank = datagen.clustered(N, D, C, seed + 1, lab).T
    q = datagen.clustered(B, D, C, seed + 2)
    return _t(q), _t(bank), _t(lab)


@pytest.fixture()
def mode_guard():
    yield
    b200knn.set_default_mode("exact")
    K.GRAPHS["enabled"] = True


@pytest.mark.parametrize("mode", ["fp32", "exact", "fp32_f16x2", "f16", "bf16", "bf16x3"])
@pytest.mark.parametrize("B,C", [(64, 9), (1000, 38), (5000, 1), (64, 38)])
def test_grid_bitwise_equals_separate_calls(mode, B, C, mode_guard):
    q, bank, lab = _bank(20000, 512, C, B, 100 + B + C)
    b200knn.set_default_mode(mode)
    ks, ts = (20, 1, 200, 5), (0.1, 0.5, 0.07)  # not ascending: output follows the caller's order
    got = b200knn.knn_predict_multi(q, bank, lab, C, ks, ts)
    assert got.shape == (4, 3, B, C) and got.dtype == torch.int64
    assert torch.equal(got, _separate(q, bank, lab, C, ks, ts))


@pytest.mark.parametrize("golden,name", [("real_FastSiam", "norm_k200"), ("synth_nonneg", "relu_small"),
                                         ("synth_nonneg", "absgauss_small")])
@pytest.mark.parametrize("mode", ["exact", "fp32"])
def test_grid_equals_seq_oracle_on_golden(golden, name, mode, golden_dir, mode_guard):
    g = np.load(os.path.join(golden_dir, f"{golden}.npz"))
    if golden == "real_FastSiam":
        b = g["bank_rows_f16"].astype(np.float32)
        qq = g["query_rows_f16"].astype(np.float32)
        b = b / np.maximum(np.linalg.norm(b, axis=1, keepdims=True), 1e-12)
        qq = qq / np.maximum(np.linalg.norm(qq, axis=1, keepdims=True), 1e-12)
        bank, labels, C = np.ascontiguousarray(b.T), g["bank_labels"].astype(np.int64), 9
    else:
        c = datagen.make_case(name)
        qq, bank, labels, C = c["feature"], c["bank"], c["labels"], c["C"]
    ss, si = g[f"{name}_seq_sims"], g[f"{name}_seq_idx"].astype(np.int64)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_multi(_t(qq), _t(bank), _t(labels), C, KS, TS).cpu().numpy()
    for i, k in enumerate(KS):
        for j, t in enumerate(TS):
            assert np.array_equal(got[i, j], O.vote_o64(ss[:, :k], si[:, :k], labels, C, t)[0]), (k, t)


@pytest.mark.parametrize("mode", ["exact", "fp32", "bf16"])
def test_grid_beyond_max_k_takes_peeling_path(mode, mode_guard):
    q, bank, lab = _bank(6000, 256, 9, 70, 7)
    b200knn.set_default_mode(mode)
    ks, ts = (5, 1000), (0.1, 0.07)
    got = b200knn.knn_predict_multi(q, bank, lab, 9, ks, ts)
    assert torch.equal(got, _separate(q, bank, lab, 9, ks, ts))
    with pytest.raises(RuntimeError, match="k out of range"):
        b200knn.knn_predict_multi(q, bank, lab, 9, (5, 6001), ts)


def test_grid_repair_levels(mode_guard):
    """Rows the cascade's first level leaves uncertified are repaired at k_max by the later levels."""
    c = datagen.make_case("absgauss_small")
    q, bank, lab = _t(c["feature"]), _t(c["bank"]), _t(c["labels"])
    K.GRAPHS["enabled"] = False  # the eager path records the cascade statistics of the call
    reached = []
    for mode in ("fp32", "fp32_bf16"):
        b200knn.set_default_mode(mode)
        got = b200knn.knn_predict_multi(q, bank, lab, c["C"], KS, TS)
        reached.append(len(K.last_rescore_stats["levels"]) > 1)
        K.GRAPHS["enabled"] = True
        assert torch.equal(got, _separate(q, bank, lab, c["C"], KS, TS)), mode
        K.GRAPHS["enabled"] = False
    assert any(reached), K.last_rescore_stats


@pytest.mark.parametrize("mode", ["fp32", "bf16", "exact"])
def test_grid_tie_flood(mode, mode_guard):
    D, N = 512, 70000
    g = torch.Generator(device=DEV).manual_seed(3)
    row = torch.nn.functional.normalize(torch.randn(1, D, generator=g, device=DEV), dim=1)
    bank = row.repeat(N, 1).t().contiguous()
    q = torch.nn.functional.normalize(torch.randn(130, D, generator=g, device=DEV), dim=1)
    q[5] = 0
    lab = torch.randint(0, 9, (N,), generator=g, device=DEV)
    b200knn.set_default_mode(mode)
    got = b200knn.knn_predict_multi(q, bank, lab, 9, KS, TS)
    assert torch.equal(got, _separate(q, bank, lab, 9, KS, TS))


def test_grid_graph_path(mode_guard):
    q, bank, lab = _bank(37348, 512, 9, 64, 21)
    b200knn.set_default_mode("fp32")
    K.clear_call_graphs()
    b200knn.knn_predict_multi(q, bank, lab, 9, (5, 20, 200), (0.1,))  # first call captures
    before = dict(K.graph_stats)
    outs = [b200knn.knn_predict_multi(q, bank, lab, 9, (5, 20, 200), (0.1,)) for _ in range(3)]
    assert K.graph_stats["captures"] == before["captures"]
    assert K.graph_stats["replays"] == before["replays"] + 3
    K.GRAPHS["enabled"] = False
    eager = b200knn.knn_predict_multi(q, bank, lab, 9, (5, 20, 200), (0.1,))
    for o in outs:
        assert torch.equal(o, eager)
    assert torch.equal(eager, _separate(q, bank, lab, 9, (5, 20, 200), (0.1,)))


def test_grid_label_errors(mode_guard):
    q, bank, lab = _bank(3000, 128, 9, 64, 5)
    bad = lab.clone()
    bad[:] = 9
    for mode in ("fp32", "exact"):
        b200knn.set_default_mode(mode)
        with pytest.raises(RuntimeError, match="num_classes=9"):
            b200knn.knn_predict_multi(q, bank, bad, 9, (5, 20), (0.1,))


def test_feature_bank_grid_fused_normalize(mode_guard):
    rng = np.random.default_rng(4)
    C = 9
    rows = _t(rng.standard_normal((8000, 512)).astype(np.float32) * 3)
    lab = _t(datagen.labels(8000, C, 4))
    raw = _t(rng.standard_normal((300, 512)).astype(np.float32) * 7)
    fb = b200knn.FeatureBank.from_rows(rows, lab)
    b200knn.set_default_mode("fp32")
    got = fb.knn_predict_multi(raw, C, KS, TS, normalize=True)
    assert torch.equal(got, fb.knn_predict_multi(K.normalize_rows(raw), C, KS, TS))
    assert torch.equal(got[1, 1], fb.knn_predict(raw, C, 5, 0.1, normalize=True))


def test_hooks_grid_on_device(mode_guard):
    import standin_module as S
    from test_gpu_round2 import _loaders

    C = 9
    bank_loader, val_batches = _loaders(3000, 500, 512, C, 17)
    b200knn.set_default_mode("fp32")
    b200knn.install(hook_classes=(S.StandInKNNModule,))
    try:
        plain = S.StandInKNNModule(bank_loader, C, knn_k=5, knn_t=0.1)
        plain._device = torch.device(DEV)
        p0 = S.run_validation_epoch(plain, val_batches)
        gridded = S.StandInKNNModule(bank_loader, C, knn_k=5, knn_t=0.1)
        gridded._device = torch.device(DEV)
        gridded.b200knn_knn_grid = ((20, 200), (0.07,))
        gridded.on_validation_epoch_start()
        for i, b in enumerate(val_batches):
            gridded.validation_step(b, i)
        p1 = torch.cat(gridded.all_preds).clone()
        targets = torch.cat(gridded.all_targets).clone()
        fb = gridded._b200knn_bank
        gridded.on_validation_epoch_end()
    finally:
        b200knn.uninstall()
    assert torch.equal(p0, p1)
    assert gridded.max_accuracy == plain.max_accuracy and gridded.max_f1 == plain.max_f1
    assert gridded.logged["knn_accuracy"] == plain.logged["knn_accuracy"]
    assert np.array_equal(gridded.confusion_matrix[0], plain.confusion_matrix[0])
    for k in (20, 200, 5):
        for t in (0.07, 0.1):
            sep = torch.cat([fb.knn_predict(b[0], C, k, t, normalize=True)[:, 0] for b in val_batches])
            m = b200knn.knn_metrics(sep, targets, C)
            assert gridded.logged[f"knn_accuracy_k{k}_t{t:g}"] == float(m["accuracy"]), (k, t)
            assert gridded.logged[f"knn_f1_k{k}_t{t:g}"] == float(m["f1"]), (k, t)


def _sharded_worker(rank, world, port, out_dir):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    failures = []
    try:
        for (N, D, B, C) in [(200000, 512, 300, 9), (30000, 512, 130, 38)]:
            g = torch.Generator(device=dev).manual_seed(811)
            bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=dev), dim=1).t().contiguous()
            q = torch.nn.functional.normalize(torch.randn(B, D, generator=g, device=dev), dim=1)
            lab = torch.randint(0, C, (N,), generator=g, device=dev)
            for mode in ("exact", "fp32", "bf16"):
                b200knn.set_default_mode(mode)
                single = b200knn.knn_predict_multi(q, bank, lab, C, KS, TS)
                sb = b200knn.ShardedBank.from_full(bank, lab, mode=mode)
                for exchange in ("alltoall", "allgather"):
                    if not torch.equal(single, sb.knn_predict_multi(q, C, KS, TS, exchange=exchange)):
                        failures.append((N, B, C, mode, exchange))
        flag = torch.tensor([len(failures)], device=dev)
        dist.all_reduce(flag)
        with open(os.path.join(out_dir, f"rank{rank}.txt"), "w") as f:
            f.write(repr(failures))
        assert int(flag.item()) == 0, failures
    finally:
        b200knn.set_default_mode("exact")
        dist.destroy_process_group()


def test_sharded_grid_equals_single_gpu(tmp_path):
    world = min(2, torch.cuda.device_count())
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    import torch.multiprocessing as mp
    from test_gpu_multi import _free_port

    mp.spawn(_sharded_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert open(tmp_path / f"rank{r}.txt").read() == "[]"
