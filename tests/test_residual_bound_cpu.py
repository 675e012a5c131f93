"""CPU: the per-query certificate bound of knn_predict's certified vote from measured fp16 residuals
(b200knn/knn.py LEVELS residual_bound, csrc/rescore.cu cert_bound, DESIGN §4.1c / §5), restated in
numpy / fp64.  Its operand terms must dominate |q.x - f16(q).f16(x)| and its gamma_D term the
rounding of the exact mode's sequential fma chain (oracle/seqfma.c), on random and adversarial
inputs; on the benchmark's data it must be at most, and about half of, the worst-case bound."""
import math

import numpy as np
import pytest

from b200knn import knn as K
from oracle import knn_oracle as O

INFL = 1.001  # the kernels' inflation of fp32-evaluated norms


def f16(x):
    """f16_operand: rn(sat(x)) to fp16, as fp64."""
    return np.clip(x.astype(np.float32), -65504.0, 65504.0).astype(np.float16).astype(np.float64)


def nrm(x):
    return np.linalg.norm(x.astype(np.float64), axis=-1)


def bank_residuals(X):
    """b200knn_row_f16_residual_max: R = max ||x - f16(x)||, M~ = max ||f16(x)||."""
    Xt = f16(X)
    return float(nrm(X.astype(np.float64) - Xt).max()), float(nrm(Xt).max())


def operand_terms(Q, R, Mt):
    """||f16(q)|| R + rho M~ + rho R per query (rho = ||q - f16(q)||)."""
    Qt = f16(Q)
    qtn, rho = nrm(Qt), nrm(Q.astype(np.float64) - Qt)
    return qtn * R + rho * Mt + rho * R


def gamma(D):
    u = D * 2.0 ** -24
    return u / (1.0 - u)


def e_new(Q, X):
    """The bound band_kernel computes for the fp32_f16 level (norms inflated as the kernel does)."""
    D = Q.shape[1]
    R, Mt = bank_residuals(X)
    Qt = f16(Q)
    qtn, rho = nrm(Qt) * INFL, nrm(Q.astype(np.float64) - Qt) * INFL
    qn, M = nrm(Q) * INFL, float(nrm(X).max()) * INFL
    acc = 1.01 * K.LEVELS["fp32_f16"]["acc_c"] * K.padded_dim(D) * K.ACC_ULP
    return qtn * R + rho * Mt + rho * R + acc * qtn * Mt + gamma(D) * qn * M


def e_old(Q, X):
    """Today's worst-case certificate bound of the fp32_f16 level."""
    D = Q.shape[1]
    lv = K.level_config("fp32_f16", D)
    qn, M = nrm(Q) * INFL, float(nrm(X).max()) * INFL
    return lv["err_coef"] * qn * M + lv["err_abs"] * math.sqrt(K.padded_dim(D)) * (qn + M)


def _patterns(D, rng):
    """(name, queries (B, D), bank rows (N, D)) float32: random and adversarial for fp16 rounding."""
    out = []
    g = lambda n: rng.standard_normal((n, D)).astype(np.float32)  # noqa: E731
    unit = lambda x: (x / np.linalg.norm(x, axis=1, keepdims=True)).astype(np.float32)  # noqa: E731
    out.append(("gauss", unit(g(16)), unit(g(300))))
    out.append(("all_positive", unit(np.abs(g(16))), unit(np.abs(g(300)))))
    out.append(("unnormalised", g(16) * 37.0, g(300) * np.float32(0.013)))
    # midpoints between adjacent fp16 values (rounding error exactly half a unit), just above powers
    # of two where the relative error 2^-11 is largest; both signs
    h = np.float16(1.0) * (2.0 ** rng.integers(-12, 3, size=(316, D)))
    mid = (h.astype(np.float32) * np.float32(1 + 2.0 ** -11)) * rng.choice([-1, 1], size=(316, D)).astype(np.float32)
    out.append(("fp16_midpoints", mid[:16], mid[16:]))
    out.append(("fp16_midpoints_positive", np.abs(mid[:16]), np.abs(mid[16:])))
    # fp16 subnormal range (|x| < 2^-14): absolute rounding 2^-25, relative up to 1
    sub = rng.uniform(2.0 ** -26, 2.0 ** -14, size=(316, D)).astype(np.float32)
    out.append(("fp16_subnormal", sub[:16], sub[16:]))
    mixed = np.where(rng.random((316, D)) < 0.5, sub, np.abs(g(316)) * np.float32(0.05))
    out.append(("subnormal_mixed", mixed[:16].astype(np.float32), mixed[16:].astype(np.float32)))
    # near the fp16 limit: elements up to 6e4 (the max_abs refusal of the level concerns norms)
    big = rng.uniform(3.0e4, 6.0e4, size=(316, D)).astype(np.float32)
    big[:, 1::2] *= np.float32(2.0 ** -20)
    out.append(("near_6e4", big[:16], big[16:]))
    return out


@pytest.mark.parametrize("D", [128, 512, 768])
def test_operand_terms_dominate_operand_rounding(D):
    rng = np.random.default_rng(D)
    for name, Q, X in _patterns(D, rng):
        R, Mt = bank_residuals(X)
        exact = Q.astype(np.float64) @ X.astype(np.float64).T
        rounded = f16(Q) @ f16(X).T
        err = np.abs(exact - rounded)
        bound = operand_terms(Q, R, Mt)[:, None]
        assert (err <= bound).all(), (name, float((err / bound).max()))
        # and every term is needed no more than the residuals say: the bound is far below today's
        # 2^-10 ||q|| M wherever the rows are not adversarial
        if name in ("gauss", "all_positive", "unnormalised"):
            assert (bound[:, 0] < 0.75 * 2.0 ** -10 * nrm(Q) * nrm(X).max()).all(), name


@pytest.mark.parametrize("D", [128, 512, 768])
def test_gamma_term_dominates_the_exact_chain(D):
    rng = np.random.default_rng(100 + D)
    for name, Q, X in _patterns(D, rng):
        s = O.sims_seqfma(Q, np.ascontiguousarray(X.T)).astype(np.float64)
        exact = Q.astype(np.float64) @ X.astype(np.float64).T
        bound = gamma(D) * nrm(Q)[:, None] * nrm(X)[None, :]
        assert (np.abs(s - exact) <= bound).all(), name


def test_gamma_term_on_a_worst_ordered_chain():
    """One large product first, then D - 1 products of just under half a unit of it: every fma of the
    chain rounds by nearly half a unit in the same direction."""
    for D in (128, 512, 768):
        q = np.full((1, D), 2.0 ** -12 * (1 - 2.0 ** -20), dtype=np.float32)
        x = np.full((1, D), 2.0 ** -12, dtype=np.float32)
        q[0, 0], x[0, 0] = 1.0, 1.0
        s = float(O.sims_seqfma(q, np.ascontiguousarray(x.T))[0, 0])
        exact = float((q.astype(np.float64) @ x.astype(np.float64).T)[0, 0])
        assert abs(s - exact) > 0.25 * (D - 1) * 2.0 ** -24  # the chain really loses its rounding
        assert abs(s - exact) <= gamma(D) * float(nrm(q)[0] * nrm(x)[0])


@pytest.mark.parametrize("kind", ["clustered", "gauss", "relu", "absgauss"])
def test_new_bound_halves_the_worst_case_on_benchmark_data(kind):
    import bench

    X, _, Q = bench.make_inputs("cpu", 20000, 256, bench.DIM, seed=0, kind=kind)
    X, Q = X.numpy(), Q.numpy()
    new, old = e_new(Q, X), e_old(Q, X)
    assert (new <= old).all()
    ratio = new / old
    assert 0.4 < float(ratio.mean()) < 0.6, float(ratio.mean())
    # the bound still holds with room on the tensor-core operands (exact fp16 products here)
    exact = Q.astype(np.float64) @ X.astype(np.float64).T
    rounded = f16(Q) @ f16(X).T
    assert float((np.abs(exact - rounded).max(axis=1) / new).max()) < 0.5


def test_new_bound_at_most_old_on_ordinary_rows():
    rng = np.random.default_rng(7)
    for D in (128, 512, 768):
        for scale in (1e-3, 1.0, 30.0):
            Q = (rng.standard_normal((64, D)) * scale).astype(np.float32)
            X = (rng.standard_normal((2000, D)) * scale).astype(np.float32)
            assert (e_new(Q, X) <= e_old(Q, X)).all(), (D, scale)
