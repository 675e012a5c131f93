"""GPU: the certified vote's per-query bound from measured fp16 residuals (LEVELS residual_bound,
rescore.cu cert_bound, DESIGN §4.1c / §5).
 * b200knn_row_f16_residual_max against an fp64 restatement;
 * the E that band_kernel computes covers |tensor-core tile - exact-mode similarity| for every
   pair, on the raw TMEM tiles of all-positive and adversarial operands at D = 512 / 768;
 * knn_predict in fp32 mode is bitwise the exact mode on the benchmark's four data kinds at the full
   811,457-row bank, in one large batch and through the CUDA-graph path, and the band it re-scores
   is smaller than under the worst-case bound."""
import numpy as np
import pytest
import torch

import bench
import datagen
from b200knn import _lib
from b200knn import knn as K
from test_gpu_round2 import _adversarial
from test_gpu_tc import run_dump
from test_residual_bound_cpu import bank_residuals, e_new, e_old

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _residuals_gpu(X):
    rows = K.prepare_rows(_t(X), "f32rows", vectors_are_columns=False).hi
    out = torch.zeros(2, dtype=torch.float32, device=DEV)
    _lib.check(_lib.load().b200knn_row_f16_residual_max(rows.data_ptr(), rows.shape[0], rows.shape[1],
                                                        out.data_ptr(), torch.cuda.current_stream().cuda_stream),
               "row_f16_residual_max")
    return out.cpu().numpy().astype(np.float64)


def test_residual_max_matches_fp64():
    rng = np.random.default_rng(4)
    for D in (72, 512, 768):
        for X in (datagen.gauss(3001, D, 1), datagen.absgauss(3001, D, 2) * np.float32(300.0),
                  rng.uniform(2.0 ** -26, 2.0 ** -14, size=(513, D)).astype(np.float32)):
            got, want = _residuals_gpu(X), np.array(bank_residuals(X))
            assert (got >= want).all() and (got <= want * (1 + 2.0 ** -20)).all(), (D, got, want)
    X = datagen.gauss(100, 64, 3)
    X[17, 5] = np.nan
    assert np.isinf(_residuals_gpu(X)).all()


def _band_E(q, bank_dn):
    """E per query as band_kernel computes it (info.z of the certified vote, level fp32_f16)."""
    lab = torch.zeros(bank_dn.shape[1], dtype=torch.int64, device=DEV)
    old = K.GRAPHS["enabled"], K.CERTIFIED_VOTE["enabled"]
    K.GRAPHS["enabled"], K.CERTIFIED_VOTE["enabled"] = False, True
    try:
        K._predict(_t(q), _t(bank_dn), lab, 2, 5, 0.1, "fp32_f16")
    finally:
        K.GRAPHS["enabled"], K.CERTIFIED_VOTE["enabled"] = old
    return K.last_rescore_stats["band_info"][:, 2].contiguous().view(torch.float32).double().cpu().numpy()


@pytest.mark.parametrize("D", [512, 768])
def test_tmem_tiles_within_band_bound(D):
    """|a - s| <= E(q) for every (query, bank row): a the raw TMEM tile of the fp16 pass, s the exact
    mode's similarity, E what band_kernel stored for the query."""
    rng = np.random.default_rng(D)
    h = 2.0 ** rng.integers(-8, 0, size=(8 + 1024, D))
    mid = (h * (1 + 2.0 ** -11)).astype(np.float32)  # fp16 rounding midpoints, all positive
    cases = [("absgauss", datagen.absgauss(16, D, 1), datagen.absgauss(1024, D, 2)),
             ("fp16_midpoints", mid[:8], mid[8:])]
    for p in ("big_first_half_ulp", "big_first_just_under_2ulp", "big_last", "ramp"):
        q, x_dn = _adversarial(D, p, rng)
        cases.append((p, q, np.tile(x_dn.T, (4, 1))))  # >= 993 rows: the certified vote's k_in < N
    for name, q, X in cases:
        bank_dn = np.ascontiguousarray(X.T)
        _, dump, _, _ = run_dump(q, bank_dn, 5, "f16")
        s = K.knn_topk(_t(q), _t(bank_dn), X.shape[0], mode="exact")
        sims = np.empty((q.shape[0], X.shape[0]))
        np.put_along_axis(sims, s[1].cpu().numpy(), s[0].double().cpu().numpy(), axis=1)
        E = _band_E(q, bank_dn)
        err = np.abs(dump.astype(np.float64) - sims).max(axis=1)
        print(f"D={D} {name}: max |a - s| / E = {float((err / E).max()):.3f}, E / old E = "
              f"{float((E / e_old(q, X)).mean()):.3f}")
        assert (err <= E).all(), name
        assert (E >= e_new(q, X) * (1 - 1e-4)).all(), name  # the kernel's E is the restated one


def _bench_inputs(kind, n_query):
    bank_nd, labels, q = bench.make_inputs(DEV, bench.N_BANK, n_query, bench.DIM, seed=0, kind=kind)
    bank = bank_nd.t().contiguous()
    del bank_nd
    return bank, labels, q


def _fp32(q, bank, labels):
    return K._predict(q, bank, labels, bench.N_CLASSES, bench.KNN_K, bench.KNN_T, "fp32")


@pytest.mark.parametrize("kind", ["clustered", "gauss", "relu", "absgauss"])
def test_full_bank_equals_exact_mode(kind):
    bank, labels, q = _bench_inputs(kind, 4096)
    want = K._predict(q, bank, labels, bench.N_CLASSES, bench.KNN_K, bench.KNN_T, "exact")
    flag = K.LEVELS["fp32_f16"]["residual_bound"]
    bands = {}
    try:
        for residual in (False, True):
            K.LEVELS["fp32_f16"]["residual_bound"] = residual
            K.clear_call_graphs()
            got = _fp32(q, bank, labels)
            assert torch.equal(got, want), (kind, residual)
            bands[residual] = K.band_stats()
            graphed = _fp32(q[:384].contiguous(), bank, labels)  # B <= 512: the captured call
            assert torch.equal(graphed, want[:384]), (kind, residual)
    finally:
        K.LEVELS["fp32_f16"]["residual_bound"] = flag
        K.clear_call_graphs()
    print(f"{kind}: band old {bands[False]} new {bands[True]}")
    assert bands[True]["mean"] < bands[False]["mean"]
    del bank, labels, q
    K.bank_cache.clear()
    torch.cuda.empty_cache()
