"""GPU: the tcgen05 tensor-core modes (bf16, tf32x3) through the C ABI.
1. the raw similarity tiles (debug dump) against a plain fp32/fp64 GEMM of the SAME prepared
   operands — validates TMA/UMMA descriptors and TMEM addressing;
2. the fused selection against the canonical top-k of those dumped tiles — bit-exact;
3. tf32x3 against the fp64 oracle under the §7.3 contract (1e-5 relative);
4. bf16 recall@k against the fp64 oracle (stated, asserted >= 0.98 on these inputs)."""
import ctypes

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


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def run_dump(q: np.ndarray, bank_dn: np.ndarray, k: int, mode: str):
    lib = _lib.load()
    tq, tb = _t(q), _t(bank_dn)
    pq = b200knn.prepare_rows(tq, mode, vectors_are_columns=False)
    pb = b200knn.prepare_rows(tb, mode, vectors_are_columns=True)
    B, D = q.shape
    N = bank_dn.shape[1]
    keys = torch.zeros((B, k), dtype=torch.int64, device=DEV)
    dump = torch.full((B, N), float("nan"), dtype=torch.float32, device=DEV)
    diag = torch.zeros(4, dtype=torch.int32, device=DEV)
    ws_bytes = lib.b200knn_topk_workspace_bytes(B, N, D, k, _lib.MODES[mode])
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    rc = lib.b200knn_debug_topk_dump(_lib.MODES[mode], pq.hi.data_ptr(), None if pq.lo is None else pq.lo.data_ptr(),
                                     pb.hi.data_ptr(), None if pb.lo is None else pb.lo.data_ptr(),
                                     B, N, D, k, keys.data_ptr(), ws.data_ptr(), ws_bytes, dump.data_ptr(),
                                     diag.data_ptr(), 0, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "debug_topk_dump")
    torch.cuda.synchronize()
    assert diag.cpu().tolist()[0] == 0, f"pipeline wait timed out: {diag.cpu().tolist()}"
    return keys.cpu().numpy().view(np.uint64), dump.cpu().numpy(), pq, pb


CASES = [
    ("ragged", None),            # D=72 (padded to 128), N=1001, B=7: OOB rows/cols everywhere
    ("k5", None),                # B=64, k=5
    ("mixed38", None),           # k=20
    ("clustered_d384", None),    # D=384, k=200
    ("clustered_small", None),   # D=512, k=200, N=4096
]


@pytest.mark.parametrize("mode", ["bf16", "tf32x3", "bf16x3", "f16x2", "f16"])
@pytest.mark.parametrize("name,_", CASES)
def test_tiles_and_selection(name, _, mode):
    c = datagen.make_case(name)
    q, bank, k = c["feature"], c["bank"], c["k"]
    keys, dump, pq, pb = run_dump(q, bank, k, mode)
    D = q.shape[1]
    assert not np.isnan(dump).any(), "some similarity tile was never written"
    if mode == "bf16":
        qh = pq.hi.float().cpu().numpy()[:, :D].astype(np.float64)
        bh = pb.hi.float().cpu().numpy()[:, :D].astype(np.float64)
        ref = qh @ bh.T
        tol = 2e-6  # fp32 accumulation of exact bf16 products
    elif mode == "f16":
        # fp16 x fp16 (one array each): exact products, fp32 accumulation
        assert pq.lo is None and pb.lo is None
        qh = pq.hi.double().cpu().numpy()[:, :D]
        bh = pb.hi.double().cpu().numpy()[:, :D]
        assert (np.abs(qh - q) <= 2.0 ** -11 * np.abs(q) + 2.0 ** -25).all()
        assert (np.abs(bh - bank.T) <= 2.0 ** -11 * np.abs(bank.T) + 2.0 ** -25).all()
        ref = qh @ bh.T
        qn, bn = np.linalg.norm(q, axis=1).max(), np.linalg.norm(bank, axis=0).max()
        tol = 2e-6 * max(1.0, qn * bn)
        lv = K.level_config("fp32_f16", D)  # and against the true similarities: the certificate bound
        bound = lv["err_coef"] * qn * bn + lv["err_abs"] * np.sqrt(K.padded_dim(D)) * (qn + bn)
        assert np.abs(dump.astype(np.float64) - q.astype(np.float64) @ bank.astype(np.float64)).max() <= bound
    elif mode == "f16x2":
        # fp16 queries (one array) x fp16 hi + lo bank: products are exact in fp32, 2 MMAs per k-step
        assert pq.lo is None
        qh = pq.hi.double().cpu().numpy()[:, :D]
        bf = (pb.hi.double() + pb.lo.double()).cpu().numpy()[:, :D]
        assert (np.abs(qh - q) <= 2.0 ** -11 * np.abs(q) + 2.0 ** -25).all()
        assert (np.abs(bf - bank.T) <= 2.0 ** -22 * np.abs(bank.T) + 2.0 ** -25).all()
        ref = qh @ bf.T
        qn, bn = np.linalg.norm(q, axis=1).max(), np.linalg.norm(bank, axis=0).max()
        tol = 4e-6 * max(1.0, qn * bn)
        # and against the true similarities: the certificate bound of level fp32_f16x2
        lv = K.level_config("fp32_f16x2", D)
        bound = lv["err_coef"] * qn * bn + lv["err_abs"] * np.sqrt(K.padded_dim(D)) * (qn + bn)
        assert np.abs(dump.astype(np.float64) - q.astype(np.float64) @ bank.astype(np.float64)).max() <= bound
    elif mode == "bf16x3":
        # hi + lo carries 16 mantissa bits: |x - hi - lo| <= 2^-16 |x|; the kernel drops lo*lo
        qf = (pq.hi.double() + pq.lo.double()).cpu().numpy()[:, :D]
        bf = (pb.hi.double() + pb.lo.double()).cpu().numpy()[:, :D]
        assert np.abs(qf - q).max() <= 2.0 ** -16 * np.abs(q).max() * 1.01
        ref = q.astype(np.float64) @ bank.astype(np.float64)
        scale = np.linalg.norm(q, axis=1).max() * np.linalg.norm(bank, axis=0).max()
        tol = 6e-5 * max(scale, 1e-30)  # the certificate coefficient of level fp32_bf16x3
    else:
        qf = (pq.hi.double() + pq.lo.double()).cpu().numpy()[:, :D]
        bf = (pb.hi.double() + pb.lo.double()).cpu().numpy()[:, :D]
        assert np.array_equal(qf.astype(np.float32), q) and np.array_equal(bf.astype(np.float32), bank.T)
        ref = qf @ bf.T
        tol = 1e-5 * max(1.0, np.abs(ref).max())
    err = np.abs(dump.astype(np.float64) - ref).max()
    assert err <= tol, f"{mode} tile error {err}"
    # selection is exact w.r.t. the tiles it saw
    want_s, want_i = O.canonical_topk_c(dump, k)
    assert np.array_equal(keys, O.make_keys(want_s, want_i))
    # and the product entry point gives the same keys as the debug hook
    again = b200knn.topk_keys(_t(q), _t(bank), k, mode=mode).cpu().numpy().view(np.uint64)
    assert np.array_equal(again, keys)


@pytest.mark.parametrize("name", ["clustered_small", "gauss_small", "mixed38"])
def test_tf32x3_raw_accuracy(name):
    """Raw 3xTF32 similarities: within 1e-5 relative of fp64 (north-star tolerance).  Their ORDER is
    only guaranteed where fp64 neighbours differ by more than the mode's error (2e-5*max|s|: dropped
    lo*lo terms and non-IEEE fp32 accumulation in TMEM) — bit-exact order is the job of mode "fp32"."""
    c = datagen.make_case(name)
    sims, idx = b200knn.knn_topk(_t(c["feature"]), _t(c["bank"]), c["k"], mode="tf32x3")
    r = O.compare_topk(sims.cpu().numpy(), idx.cpu().numpy(), c["feature"], c["bank"], c["k"], eps_scale=2e-5)
    print(f"tf32x3 {name}: max rel err {r['max_rel_err']:.2e}, idx mismatches {r['idx_mismatch_total']:.0f}")
    assert r["max_rel_err"] <= 1e-5  # tolerance stated by BASELINE.json north_star
    assert r["idx_mismatch_unambiguous"] == 0 and r["set_mismatch_rows_unambiguous"] == 0
    assert r["recall_at_k"] >= 0.999


@pytest.mark.parametrize("mode", ["fp32", "fp32_f16", "fp32_f16x2", "fp32_bf16x3", "fp32_bf16", "fp32_tf32"])
@pytest.mark.parametrize("name", datagen.CASE_NAMES)
def test_fp32_modes_bitwise_equal_exact_and_oracle(name, mode):
    """The fp32-matching modes (tensor-core candidates + exact re-scoring + certificate) must give
    bit for bit the neighbours, similarities and class ranking of the sequential-fma oracle."""
    c = datagen.make_case(name)
    f, bank, lab = _t(c["feature"]), _t(c["bank"]), _t(c["labels"])
    keys = b200knn.topk_keys(f, bank, c["k"], mode=mode)
    stats = dict(K.last_rescore_stats)
    sims, idx = b200knn.decode_keys(keys)
    ss, si = O.topk_seqfma(c["feature"], c["bank"], c["k"])
    assert np.array_equal(idx.cpu().numpy(), si)
    assert np.array_equal(sims.cpu().numpy().view(np.uint32), ss.view(np.uint32))
    assert torch.equal(keys, b200knn.topk_keys(f, bank, c["k"], mode="exact"))
    b200knn.set_default_mode(mode)
    try:
        pred = b200knn.knn_predict(f, bank, lab, c["C"], c["k"], c["t"]).cpu().numpy()
    finally:
        b200knn.set_default_mode("exact")
    assert np.array_equal(pred, O.vote_o64(ss, si, c["labels"], c["C"], c["t"])[0])
    print(f"{mode} {name}: first level {stats['level']}, uncertified rows {stats['uncertified']}/{stats['rows']}")
    if mode == "fp32_tf32":
        assert stats["uncertified"] <= max(1, stats["rows"] // 10)


@pytest.mark.parametrize("mode", ["fp32", "fp32_f16", "fp32_f16x2", "fp32_bf16x3", "fp32_bf16", "fp32_tf32"])
@pytest.mark.parametrize("model", ["FastSiam", "SimSiam"])
def test_fp32_modes_real_banks(model, mode, golden_dir):
    """Duplicates, 80 % exact zeros, row norms up to 277 (un-normalised): certificate + fallback
    must still reproduce the golden sequential-fma result exactly."""
    import os

    g = np.load(os.path.join(golden_dir, f"real_{model}.npz"))
    for tag in ("norm_", "raw_"):
        b = g["bank_rows_f16"].astype(np.float32)
        q = g["query_rows_f16"].astype(np.float32)
        if tag == "norm_":
            b = b / np.maximum(np.linalg.norm(b, axis=1, keepdims=True), 1e-12)
            q = q / np.maximum(np.linalg.norm(q, axis=1, keepdims=True), 1e-12)
        bank = np.ascontiguousarray(b.T)
        for k in (5, 200):
            keys = b200knn.topk_keys(_t(q), _t(bank), k, mode=mode)
            sims, idx = b200knn.decode_keys(keys)
            assert np.array_equal(idx.cpu().numpy(), g[f"{tag}k{k}_seq_idx"].astype(np.int64)), (tag, k)
            assert np.array_equal(sims.cpu().numpy().view(np.uint32), g[f"{tag}k{k}_seq_sims"].view(np.uint32))
            print(f"{mode} {model} {tag}k{k}: uncertified {K.last_rescore_stats['uncertified']}/{K.last_rescore_stats['rows']}")


@pytest.mark.parametrize("name", ["clustered_small", "gauss_small"])
def test_bf16_recall(name):
    c = datagen.make_case(name)
    sims, idx = b200knn.knn_topk(_t(c["feature"]), _t(c["bank"]), c["k"], mode="bf16")
    r = O.compare_topk(sims.cpu().numpy(), idx.cpu().numpy(), c["feature"], c["bank"], c["k"])
    print(f"bf16 recall@{c['k']} on {name}: {r['recall_at_k']:.4f}, max rel err {r['max_rel_err']:.2e}")
    assert r["recall_at_k"] >= 0.98 and r["max_rel_err"] <= 2e-2


@pytest.mark.parametrize("mode", ["bf16", "tf32x3", "bf16x3", "f16x2", "f16", "fp32", "fp32_f16", "fp32_f16x2", "fp32_bf16x3", "fp32_bf16", "fp32_tf32"])
def test_large_bank_against_exact_mode(mode):
    """Sizes the CPU oracle cannot cover: tensor-core modes against the on-device exact mode
    (itself bit-checked against the oracle in test_gpu_exact.py) on a 811,457 x 512 bank."""
    N, D, k, B = 811457, 512, 200, 256
    g = torch.Generator(device=DEV).manual_seed(811)
    bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=DEV), dim=1).t().contiguous()
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g, device=DEV), dim=1)
    ek = b200knn.topk_keys(q, bank, k, mode="exact")
    tk = b200knn.topk_keys(q, bank, k, mode=mode)
    es, ei = b200knn.decode_keys(ek)
    ts, ti = b200knn.decode_keys(tk)
    ei, ti = ei.cpu().numpy(), ti.cpu().numpy()
    recall = np.mean([len(set(ei[b]) & set(ti[b])) / k for b in range(B)])
    print(f"{mode} recall@{k} vs exact at N={N}: {recall:.5f}")
    if mode in K.RESCORED_MODES:
        print(f"   uncertified rows {K.last_rescore_stats['uncertified']}/{K.last_rescore_stats['rows']}")
        assert torch.equal(ek, tk)  # bitwise: indices, similarities, order
    elif mode in ("tf32x3", "bf16x3"):
        assert recall >= (0.9995 if mode == "tf32x3" else 0.998) and float((es - ts).abs().max()) <= (1e-5 if mode == "tf32x3" else 6e-5)
        # batch invariance of the tensor-core path: same rows, smaller batch, identical keys
        tk2 = b200knn.topk_keys(q[:64].contiguous(), bank, k, mode=mode)
        assert torch.equal(tk2, tk[:64])
    elif mode == "f16x2":
        assert recall >= 0.99 and float((es - ts).abs().max()) <= 5.2e-4
    elif mode == "f16":
        assert recall >= 0.99 and float((es - ts).abs().max()) <= 1.0e-3
    else:
        assert recall >= 0.98


@pytest.mark.parametrize("mode", ["bf16", "tf32x3", "bf16x3", "f16x2", "f16"])
def test_prepass_threshold_does_not_change_results(mode):
    """The sampling pre-pass only supplies a starting threshold: keys with it on and off must be
    bitwise identical (and the repair path must be a no-op or fix every row)."""
    N, D, k, B = 300000, 512, 200, 200
    g = torch.Generator(device=DEV).manual_seed(5)
    bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=DEV), dim=1).t().contiguous()
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g, device=DEV), dim=1)
    assert K.prepass_stride(N, k) > 0
    on = b200knn.topk_keys(q, bank, k, mode=mode)
    repaired = K.last_prepass_stats["repaired"]
    K.PREPASS["enabled"] = False
    try:
        off = b200knn.topk_keys(q, bank, k, mode=mode)
    finally:
        K.PREPASS["enabled"] = True
    assert torch.equal(on, off)
    print(f"{mode}: pre-pass repaired rows {repaired}/{B}")
    # a threshold that is too high for some rows must be repaired, not returned
    sk = K.sample_keys(q, bank, k, mode)
    tau = K.kth_sim(sk)
    tau[:7] = 5.0
    raw = b200knn.topk_keys(q, bank, k, mode=mode, tau0=tau)
    assert bool((raw[:7] == 0).all()) and torch.equal(raw[7:], off[7:])


@pytest.mark.parametrize("mode", ["bf16", "tf32x3"])
@pytest.mark.parametrize("B,N,stride", [(200, 300000, 62), (513, 40000, 8), (64, 811457, 62), (3, 4096, 1)])
def test_sample_option_is_a_valid_threshold(mode, B, N, stride):
    """The sample option of b200knn_topk_opt keeps, per row, the 16 best 32-column chunk maxima in registers.  Every
    value it returns must be one of the row's sampled similarities (bit for bit), the best one is
    the row maximum, the list is sorted, and its 16-th value is <= the true 16-th best sampled
    similarity (so it is a valid admission threshold) without being much weaker."""
    D = 512
    g = torch.Generator(device=DEV).manual_seed(11)
    bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=DEV), dim=1).t().contiguous()
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g, device=DEV), dim=1)
    pb = K.bank_cache.get(bank, mode)
    pq = K.prepare_rows(q, mode, vectors_are_columns=False)
    n_visit = (N + stride - 1) // stride
    kk = min(64, n_visit)
    lists = K._search(mode, pq, pb, B, n_visit, D, kk, stride=stride)
    regs = K._search(mode, pq, pb, B, n_visit, D, 16, stride=stride, sample=True)
    s_list, _ = b200knn.decode_keys(lists)
    s_reg, i_reg = b200knn.decode_keys(regs)
    assert bool((i_reg == 0).all())
    assert bool((s_reg[:, :-1] >= s_reg[:, 1:]).all())
    assert torch.equal(s_reg[:, 0].view(torch.int32), s_list[:, 0].view(torch.int32))
    assert bool((s_reg[:, 15] <= s_list[:, 15]).all())
    # every returned value above the 64-th best sampled similarity must be one of the top-64
    for b in range(0, B, max(1, B // 16)):
        ref = set(s_list[b].view(torch.int32).tolist())
        floor = float(s_list[b, kk - 1])
        for v, bits in zip(s_reg[b].tolist(), s_reg[b].view(torch.int32).tolist()):
            assert v <= floor or bits in ref
    # not much weaker than the exact 16-th best: at worst the 40-th best sampled value
    if kk >= 40:
        assert bool((s_reg[:, 15] >= s_list[:, 39]).all())
    assert torch.equal(K.kth_sim(regs), s_reg[:, 15].contiguous())


@pytest.mark.parametrize("D", [200, 768, 1024])
@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "tf32x3", "f16x2", "f16", "fp32"])
def test_other_vector_dims(D, mode):
    """D=768 is config c5 (BASELINE.json), D=200 exercises the zero-padded last k-block, D=1024 the
    route around the resident query tile; checked against the on-device exact mode."""
    N, B, k = 20000, 150, 200
    g = torch.Generator(device=DEV).manual_seed(D)
    bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=DEV), dim=1).t().contiguous()
    q = torch.nn.functional.normalize(torch.randn(B, D, generator=g, device=DEV), dim=1)
    ek = b200knn.topk_keys(q, bank, k, mode="exact")
    tk = b200knn.topk_keys(q, bank, k, mode=mode)
    if mode == "fp32":
        assert torch.equal(ek, tk)
        return
    es, ei = b200knn.decode_keys(ek)
    ts, ti = b200knn.decode_keys(tk)
    ei, ti = ei.cpu().numpy(), ti.cpu().numpy()
    recall = np.mean([len(set(ei[b]) & set(ti[b])) / k for b in range(B)])
    err = float((torch.sort(es, dim=1).values - torch.sort(ts, dim=1).values).abs().max())
    print(f"D={D} {mode}: recall@{k} {recall:.4f}, max |sim - exact| {err:.2e}")
    if mode == "bf16" and D <= 768:
        assert recall >= 0.95 and err <= 1e-2
    elif mode in ("f16x2", "f16") and D <= 768:  # wider vectors are routed to bf16x3
        assert recall >= (0.99 if mode == "f16x2" else 0.98) and err <= (5.2e-4 if mode == "f16x2" else 1.0e-3)
    else:
        assert recall >= 0.995 and err <= 6e-5


@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "tf32x3", "f16x2", "f16", "fp32"])
def test_tie_flood_and_degenerate_banks(mode):
    """All similarities equal (identical bank rows, or a zero query): the radix-select prune cannot
    separate anything and must hand over to the exact sort; order is then by lowest index."""
    D, N, k = 512, 70000, 200
    g = torch.Generator(device=DEV).manual_seed(3)
    row = torch.nn.functional.normalize(torch.randn(1, D, generator=g, device=DEV), dim=1)
    bank = row.repeat(N, 1).t().contiguous()                      # N identical rows
    q = torch.nn.functional.normalize(torch.randn(130, D, generator=g, device=DEV), dim=1)
    q[5] = 0                                                      # zero query: every sim is +0
    q[6] = -q[7]
    sims, idx = b200knn.knn_topk(q, bank, k, mode=mode)
    want = torch.arange(k, device=DEV).expand(130, k)
    assert torch.equal(idx, want)
    assert bool((sims[5] == 0).all())
    assert bool((sims == sims[:, :1]).all())
    # a bank whose first half duplicates its second half: every neighbour appears twice, low index first
    half = torch.nn.functional.normalize(torch.randn(4000, D, generator=g, device=DEV), dim=1)
    bank2 = torch.cat([half, half], 0).t().contiguous()
    s2, i2 = b200knn.knn_topk(q[8:72].contiguous(), bank2, 20, mode=mode)  # (not the zero query)
    assert torch.equal(i2[:, 0::2] + 4000, i2[:, 1::2])
    assert torch.equal(s2[:, 0::2], s2[:, 1::2])


@pytest.mark.parametrize("mode", ["bf16", "bf16x3", "tf32x3", "f16x2", "f16", "fp32", "exact"])
@pytest.mark.parametrize("B,N,k", [(1, 200, 200), (3, 257, 1), (129, 300, 300), (64, 1500, 992), (2, 17, 5)])
def test_small_and_extreme_shapes(mode, B, N, k):
    """k = N (every row is a neighbour), one query, banks smaller than one tile, the largest k."""
    D = 128
    g = torch.Generator(device=DEV).manual_seed(B * 1000 + N)
    bank = torch.randn(N, D, generator=g, device=DEV).t().contiguous()
    q = torch.randn(B, D, generator=g, device=DEV)
    ek = b200knn.topk_keys(q, bank, k, mode="exact")
    ss, si = O.topk_seqfma(q.cpu().numpy(), bank.cpu().numpy(), k)
    es, ei = b200knn.decode_keys(ek)
    assert np.array_equal(ei.cpu().numpy(), si) and np.array_equal(es.cpu().numpy().view(np.uint32), ss.view(np.uint32))
    tk = b200knn.topk_keys(q, bank, k, mode=mode)
    if mode in ("fp32", "exact"):
        assert torch.equal(tk, ek)
    else:
        ts, ti = b200knn.decode_keys(tk)
        assert bool((ti >= 0).all()) and bool((ti < N).all())
        if k == N:  # every row must appear exactly once
            assert torch.equal(torch.sort(ti, dim=1).values, torch.arange(N, device=DEV).expand(B, N))
        tol = {"bf16": 0.3, "bf16x3": 2e-3, "tf32x3": 5e-4, "f16x2": 0.1, "f16": 0.1}[mode]
        assert float((ts[:, 0] - es[:, 0]).abs().max()) <= tol


def test_k_limits_and_empty_batch():
    D, N = 64, 2000
    bank = torch.randn(N, D, device=DEV).t().contiguous()
    q = torch.randn(4, D, device=DEV)
    for mode in ("exact", "bf16", "fp32"):
        with pytest.raises(RuntimeError, match="out of range"):
            b200knn.topk_keys(q, bank, N + 1, mode=mode)
        empty = b200knn.topk_keys(q[:0], bank, 10, mode=mode)
        assert empty.shape == (0, 10)
        b200knn.set_default_mode(mode)
        try:
            assert b200knn.knn_predict(q[:0], bank, torch.zeros(N, dtype=torch.int64, device=DEV), 3, 10).shape == (0, 3)
        finally:
            b200knn.set_default_mode("exact")


def test_north_star_size_against_reference_ops_on_device():
    """BASELINE.json's full size (811,457 x 512, k=200, t=0.1, 9 classes): the fp32-matching mode
    against the reference's own op sequence (oracle R32: torch.mm -> topk -> gather -> exp ->
    scatter -> sum -> argsort, here executed by torch on the GPU with TF32 off) wherever fp64 says
    the answer is unambiguous; similarities within 1e-5 relative (north-star tolerance)."""
    N, D, k, B, C, t = 811457, 512, 200, 256, 9, 0.1
    g = torch.Generator(device=DEV).manual_seed(2026)
    cent = torch.nn.functional.normalize(torch.randn(C, D, generator=g, device=DEV), dim=1)
    lab = torch.randint(0, C, (N,), generator=g, device=DEV)
    bank_nd = torch.nn.functional.normalize(cent[lab] + 1.4 * torch.randn(N, D, generator=g, device=DEV) / D ** 0.5, dim=1)
    ql = torch.randint(0, C, (B,), generator=g, device=DEV)
    q = torch.nn.functional.normalize(cent[ql] + 1.4 * torch.randn(B, D, generator=g, device=DEV) / D ** 0.5, dim=1)
    bank = bank_nd.t().contiguous()
    del bank_nd
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False
    try:
        ref_pred, ref_sims, ref_idx, _ = O.knn_predict_r32_full(q, bank, lab, C, k, t)
        s64 = q.double() @ bank.double()
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    top64, _ = s64.topk(k + 1, dim=1)
    del s64
    b200knn.set_default_mode("fp32")
    try:
        pred = b200knn.knn_predict(q, bank, lab, C, k, t)
        sims, idx = b200knn.knn_topk(q, bank, k, mode="fp32")
    finally:
        b200knn.set_default_mode("exact")
    # similarities: rank by rank within 1e-5 relative of the reference's
    assert float(((sims - ref_sims).abs() / ref_sims.abs().clamp_min(1e-3)).max()) <= 1e-5
    # neighbour SETS equal wherever rank k and k+1 are further apart than fp32 rounding can bridge
    clear = (top64[:, k - 1] - top64[:, k]) > 1e-5
    same_set = (torch.sort(idx, dim=1).values == torch.sort(ref_idx, dim=1).values).all(dim=1)
    assert int(clear.sum()) >= B // 2 and bool(same_set[clear].all())
    # neighbour ORDER equal at every rank whose fp64 neighbours are separated on both sides
    sep = (top64[:, :-1] - top64[:, 1:]) > 1e-5                      # (B, k): rank j vs j+1
    pos_ok = sep.clone()
    pos_ok[:, 1:] &= sep[:, :-1]
    assert bool((idx == ref_idx)[pos_ok].all())
    # the class the reference consumes (knn.py:99): equal wherever the fp64 vote is not a near-tie
    w = (ref_sims.double() / t).exp()
    sc = torch.zeros(B, C, dtype=torch.float64, device=DEV).scatter_add_(1, lab[ref_idx], w)
    two = sc.topk(2, dim=1).values
    decided = (two[:, 0] - two[:, 1]) > 1e-4 * two[:, 0]
    assert int(decided.sum()) >= B // 2 and bool((pred[:, 0] == ref_pred[:, 0])[decided].all())
    print(f"north-star vs reference ops: {int(clear.sum())}/{B} rows with unambiguous sets, "
          f"{int(pos_ok.sum())}/{B * k} unambiguous ranks, {int(decided.sum())}/{B} decided votes")
