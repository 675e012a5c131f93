"""GPU parity tests proper (run with -m gpu on a B200): the CUDA path through the C ABI
against the oracle on the same seeded inputs and against the committed goldens.
Bar: bit-exact indices / class rankings / similarities in the fp32 "exact" mode."""
import os

import numpy as np
import pytest
import torch

import b200knn
import datagen
from oracle import knn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


@pytest.fixture(scope="module")
def synth(golden_dir):
    both = dict(np.load(os.path.join(golden_dir, "synth.npz")))
    both.update(np.load(os.path.join(golden_dir, "synth_nonneg.npz")))  # non-negative cases (round 2)
    return both


@pytest.mark.parametrize("name", datagen.CASE_NAMES + datagen.RELU_CASE_NAMES)
def test_exact_topk_bitwise_vs_seq_oracle_and_golden(name, synth):
    c = datagen.make_case(name)
    sims, idx = b200knn.knn_topk(_t(c["feature"]), _t(c["bank"]), c["k"], mode="exact")
    sims, idx = sims.cpu().numpy(), idx.cpu().numpy()
    ss, si = O.topk_seqfma(c["feature"], c["bank"], c["k"])
    assert np.array_equal(idx, si)
    assert np.array_equal(sims.view(np.uint32), ss.view(np.uint32))
    assert np.array_equal(idx, synth[name + "_seq_idx"].astype(np.int64))
    assert np.array_equal(sims.view(np.uint32), synth[name + "_seq_sims"].view(np.uint32))
    # positions whose fp64 neighbours are closer than eps * max|s| are ambiguous in fp32.  Same-sign
    # products (non-negative rows) do not cancel, so fp32 rounding of ANY summation order reaches
    # 1.6e-6 relative there (measured: sequential fma vs fp64 on absgauss_small) against 6e-7 on
    # sign-symmetric rows: the ambiguity window of those cases is 2e-6 instead of 4e-7
    eps = 2e-6 if name in datagen.RELU_CASE_NAMES else 4e-7
    r = O.compare_topk(sims, idx, c["feature"], c["bank"], c["k"], eps_scale=eps)
    assert r["idx_mismatch_unambiguous"] == 0 and r["set_mismatch_rows_unambiguous"] == 0
    assert r["max_rel_err"] <= 1e-5  # north-star: similarities within 1e-5 relative of fp64


@pytest.mark.parametrize("name", datagen.CASE_NAMES + datagen.RELU_CASE_NAMES)
def test_knn_predict_vs_goldens(name, synth):
    c = datagen.make_case(name)
    b200knn.set_default_mode("exact")
    pred = b200knn.knn_predict(_t(c["feature"]), _t(c["bank"]), _t(c["labels"]), c["C"], c["k"], c["t"])
    assert pred.dtype == torch.int64 and tuple(pred.shape) == (c["feature"].shape[0], c["C"])
    pred = pred.cpu().numpy()
    assert np.array_equal(pred, synth[name + "_seq_pred"].astype(np.int64))  # bit-exact class ranking
    # against the fp64 canonical oracle and the reference algorithm (R32) under the margin rule
    assert O.compare_pred(pred, synth[name + "_o64_scores"])["rank_mismatch_unambiguous"] == 0
    r32 = synth[name + "_r32_pred"].astype(np.int64)
    sc = synth[name + "_o64_scores"]
    order = np.argsort(-sc, axis=1, kind="stable")
    top2 = np.take_along_axis(sc, order[:, :2], axis=1)
    clear = (top2[:, 0] - top2[:, 1]) > 1e-5 * np.abs(top2[:, 0])
    assert np.array_equal(pred[clear, 0], r32[clear, 0])  # the column the reference consumes (knn.py:99)


@pytest.mark.parametrize("model", ["FastSiam", "SimSiam"])
@pytest.mark.parametrize("tag,k", [("norm_", 5), ("norm_", 200), ("raw_", 5), ("raw_", 200)])
def test_real_banks(model, tag, k, golden_dir):
    g = np.load(os.path.join(golden_dir, f"real_{model}.npz"))
    b = g["bank_rows_f16"].astype(np.float32)
    q = g["query_rows_f16"].astype(np.float32)
    if tag == "norm_":
        b = b / np.maximum(np.linalg.norm(b, axis=1, keepdims=True), 1e-12)
        q = q / np.maximum(np.linalg.norm(q, axis=1, keepdims=True), 1e-12)
    bank = np.ascontiguousarray(b.T)
    t = 0.1 if tag == "norm_" else 1.0e4
    keys = b200knn.topk_keys(_t(q), _t(bank), k, mode="exact")
    sims, idx = b200knn.decode_keys(keys)
    assert np.array_equal(idx.cpu().numpy(), g[f"{tag}k{k}_seq_idx"].astype(np.int64))
    assert np.array_equal(sims.cpu().numpy().view(np.uint32), g[f"{tag}k{k}_seq_sims"].view(np.uint32))
    pred = b200knn.vote(keys, _t(g["bank_labels"].astype(np.int64)), 9, t).cpu().numpy()
    assert np.array_equal(pred, g[f"{tag}k{k}_seq_pred"].astype(np.int64))


def test_fp16_inputs_and_nd_bank_layout():
    """notebook-style bank: (N,D) fp16 rows (3.0-Embeddings-inference.ipynb:493-507) passed as a
    transposed view; fp16 values are exact in fp32, so the result equals the fp32 oracle's."""
    c = datagen.make_case("k5")
    bank16 = c["bank"].T.astype(np.float16)  # (N,D)
    q16 = c["feature"].astype(np.float16)
    sims, idx = b200knn.knn_topk(_t(q16), _t(bank16).t(), 5, mode="exact")
    ss, si = O.topk_seqfma(q16.astype(np.float32), np.ascontiguousarray(bank16.T.astype(np.float32)), 5)
    assert np.array_equal(idx.cpu().numpy(), si)
    assert np.array_equal(sims.cpu().numpy().view(np.uint32), ss.view(np.uint32))


def test_batch_and_split_invariance():
    """sim(q,n) and the selected neighbours do not depend on batch size or on how the bank is
    split over CTAs (B=1 -> many bank splits + merge; B=300 -> few)."""
    N, D, k = 20000, 512, 200
    bank = datagen.clustered(N, D, 9, 5)
    q = datagen.clustered(300, D, 9, 6)
    tb = _t(np.ascontiguousarray(bank.T))
    full = b200knn.topk_keys(_t(q), tb, k, mode="exact").cpu().numpy()
    one = b200knn.topk_keys(_t(q[:1]), tb, k, mode="exact").cpu().numpy()
    some = b200knn.topk_keys(_t(q[:130]), tb, k, mode="exact").cpu().numpy()
    assert np.array_equal(one, full[:1]) and np.array_equal(some, full[:130])
    assert b200knn.plan_info(1, N, D, k, "exact")["splits"] > 1
    ss, si = O.topk_seqfma(q[:8], np.ascontiguousarray(bank.T), k)
    assert np.array_equal(full[:8].view(np.uint64), O.make_keys(ss, si))


def test_ties_duplicates_break_by_lowest_index():
    D = 64
    base = datagen.gauss(50, D, 1)
    bank = np.concatenate([base, base, base], axis=0)  # every vector three times
    q = base[:10]
    sims, idx = b200knn.knn_topk(_t(q), _t(np.ascontiguousarray(bank.T)), 6, mode="exact")
    idx = idx.cpu().numpy()
    for r in range(10):
        assert idx[r, :3].tolist() == [r, r + 50, r + 100]  # self-matches, ascending index


def test_merge_kernel_matches_oracle():
    rng = np.random.default_rng(0)
    # small batches with many lists run several warps per row (select.cu); ragged: lists cut short
    # by a shared admission threshold (empty tails), as bank splits and shards return them
    for (G, B, k_in, k_out, ragged) in [(2, 37, 200, 200, False), (8, 5, 200, 200, False), (3, 9, 20, 20, False),
                                        (5, 4, 10, 37, False), (37, 3, 200, 200, False), (74, 64, 216, 216, True),
                                        (16, 70, 16, 16, False), (9, 1300, 50, 50, True), (16, 6, 992, 992, True),
                                        (52, 64, 16, 16, True)]:
        sims = rng.standard_normal((G, B, k_in)).astype(np.float32)
        sims[0, 0, :5] = 0.25
        idx = rng.permutation(G * B * k_in).reshape(G, B, k_in)
        keys = np.sort(O.make_keys(sims, idx), axis=2)[:, :, ::-1].copy()
        if ragged:
            keep = rng.integers(0, k_in + 1, size=(G, B))
            keep[0] = k_in  # at least k_out keys survive in every row
            keys[np.arange(k_in)[None, None, :] >= keep[:, :, None]] = 0
        got = b200knn.merge_keys(_t(keys.view(np.int64)), k_out).cpu().numpy().view(np.uint64)
        assert np.array_equal(got, O.merge_keys_np(keys, k_out))


def test_vote_matches_oracle_and_reference_tie_rule():
    rng = np.random.default_rng(1)
    for (B, k, C, N) in [(33, 200, 9, 5000), (17, 20, 38, 3000), (5, 5, 9, 100), (3, 7, 1000, 50)]:
        sims = np.sort(rng.uniform(-0.2, 1.0, (B, k)).astype(np.float32), axis=1)[:, ::-1].copy()
        idx = np.stack([rng.choice(N, k, replace=False) for _ in range(B)])
        labels = rng.integers(0, C, N)
        keys = O.make_keys(sims, idx)
        pred, scores = b200knn.vote(_t(keys.view(np.int64)), _t(labels), C, 0.1, return_scores=True)
        want_pred, want_scores = O.vote_o64(sims, idx, labels, C, 0.1)
        np.testing.assert_allclose(scores.cpu().numpy(), want_scores, rtol=1e-13, atol=0)
        r = O.compare_pred(pred.cpu().numpy(), want_scores, rel_margin=1e-12)
        assert r["rank_mismatch_unambiguous"] == 0
        zero = want_scores == 0  # zero-vote classes: ascending class id after all voted classes
        for b in range(B):
            nz = int((~zero[b]).sum())
            assert pred[b, nz:].cpu().tolist() == sorted(np.nonzero(zero[b])[0].tolist())


def test_error_behaviour_mirrors_torch():
    c = datagen.make_case("ragged")
    f, bank, lab = _t(c["feature"]), _t(c["bank"]), _t(c["labels"])
    with pytest.raises(RuntimeError, match="out of range"):  # Tensor.topk
        b200knn.knn_predict(f, bank, lab, c["C"], bank.shape[1] + 1, 0.1)
    with pytest.raises(RuntimeError, match="cannot be multiplied"):  # torch.mm
        b200knn.knn_predict(f[:, :-1], bank, lab, c["C"], 5, 0.1)
    with pytest.raises(RuntimeError, match="must be a matrix"):  # knn.py:89 .squeeze() with B == 1
        b200knn.knn_predict(f[0], bank, lab, c["C"], 5, 0.1)
    bad = lab.clone()
    bad[:] = c["C"]  # label == num_classes: the reference's scatter raises
    with pytest.raises(RuntimeError, match="out of bounds"):
        b200knn.knn_predict(f, bank, bad, c["C"], 5, 0.1)
    empty = b200knn.knn_predict(f[:0], bank, lab, c["C"], 5, 0.1)
    assert tuple(empty.shape) == (0, c["C"])
    k_eq_n = b200knn.knn_topk(f, bank[:, :10].contiguous(), 10, mode="exact")[1].cpu().numpy()
    assert all(sorted(r.tolist()) == list(range(10)) for r in k_eq_n)  # k == N: a permutation


def test_bank_cache_tracks_inplace_updates():
    c = datagen.make_case("k5")
    f, bank = _t(c["feature"]), _t(c["bank"])
    p1 = b200knn.bank_cache.get(bank, "bf16")
    assert b200knn.bank_cache.get(bank, "bf16") is p1
    bank.mul_(1.0)  # bumps _version: the epoch's bank was rebuilt in place
    assert b200knn.bank_cache.get(bank, "bf16") is not p1


def test_north_star_shape_properties():
    """811,457 x 512 bank (BASELINE.json): properties that need no CPU oracle at this size —
    self-retrieval (queries = bank rows, notebooks/2.0-Figures-nearest-neighbors.ipynb:54 where
    rank 0 is the query itself), descending order, index range, and agreement of a sharded
    2-way split + merge with the unsharded result (bitwise)."""
    N, D, k = 811457, 512, 200
    g = torch.Generator(device=DEV).manual_seed(811)
    bank_nd = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=DEV), dim=1)
    bank = bank_nd.t().contiguous()
    rows = torch.arange(0, N, N // 96, device=DEV)[:96]
    q = bank_nd[rows].contiguous()
    keys = b200knn.topk_keys(q, bank, k, mode="exact")
    sims, idx = b200knn.decode_keys(keys)
    assert torch.equal(idx[:, 0], rows)
    assert bool((sims[:, :-1] >= sims[:, 1:]).all()) and int(idx.min()) >= 0 and int(idx.max()) < N
    half = (N + 1) // 2
    k0 = b200knn.topk_keys(q, bank[:, :half].contiguous(), k, mode="exact", idx_offset=0)
    k1 = b200knn.topk_keys(q, bank[:, half:].contiguous(), k, mode="exact", idx_offset=half)
    merged = b200knn.merge_keys(torch.stack([k0, k1]), k)
    assert torch.equal(merged, keys)
    lab = torch.randint(0, 9, (N,), device=DEV)
    pred = b200knn.vote(keys, lab, 9, 0.1)
    assert sorted(pred[0].tolist()) == list(range(9))


def test_exact_at_north_star_size_against_seq_oracle():
    """The large-bank tests take mode "exact" as their reference at N = 811,457 (test_gpu_tc.py's
    test_large_bank_against_exact_mode draws the same bank and queries); here it meets the
    sequential-fma oracle at that size, for 16 of those queries."""
    N, D, k, B = 811457, 512, 200, 256
    g = torch.Generator(device=DEV).manual_seed(811)
    bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=DEV), dim=1).t().contiguous()
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g, device=DEV), dim=1)[:16].contiguous()
    sims, idx = b200knn.knn_topk(q, bank, k, mode="exact")
    ss, si = O.topk_seqfma(q.cpu().numpy(), bank.cpu().numpy(), k)
    assert np.array_equal(idx.cpu().numpy(), si)
    assert np.array_equal(sims.cpu().numpy().view(np.uint32), ss.view(np.uint32))


@pytest.mark.parametrize("k", [49, 112])
@pytest.mark.parametrize("B,N,D", [(64, 30011, 200), (300, 5003, 128)])
def test_exact_list_capacity_256_against_seq_oracle(B, N, D, k):
    from b200knn import knn as K

    plan = K.plan_info(B, N, D, k, "exact")
    assert plan["list_capacity"] == 256 and plan["splits"] > 1, plan
    g = torch.Generator(device=DEV).manual_seed(B + k)
    bank = torch.randn(D, N, generator=g, device=DEV)
    bank[:, N // 2:N // 2 + 40] = bank[:, :40]  # exact duplicates: ties broken by the lower index
    q = torch.randn(B, D, generator=g, device=DEV)
    sims, idx = b200knn.knn_topk(q, bank, k, mode="exact")
    ss, si = O.topk_seqfma(q.cpu().numpy(), bank.cpu().numpy(), k)
    assert np.array_equal(idx.cpu().numpy(), si)
    assert np.array_equal(sims.cpu().numpy().view(np.uint32), ss.view(np.uint32))
