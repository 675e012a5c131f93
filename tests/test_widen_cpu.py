"""CPU: oracle pieces and host logic of the SURVEY.md §8(f) rows (bank build, L2 retrieval,
metrics, embedding-table reader)."""
import os

import numpy as np
import torch

import datagen
from oracle import knn_oracle as O


def test_normalize_ref_matches_numpy_and_torch():
    rng = np.random.default_rng(3)
    for d in (72, 384, 512):
        x = (rng.standard_normal((50, d)) * rng.uniform(0.1, 40, (50, 1))).astype(np.float32)
        x[7] = 0.0  # zero row: F.normalize leaves it zero (eps clamp)
        y = O.normalize_rows_ref(x)
        want = torch.nn.functional.normalize(torch.from_numpy(x), dim=1).numpy()
        assert np.all(y[7] == 0)
        # the fp64 norm is at least as accurate as torch's fp32 reduction: results agree to 2 ulp
        assert np.max(np.abs(y - want)) <= 2.5e-7
        n64 = np.sqrt((x.astype(np.float64) ** 2).sum(1))
        assert np.allclose(O.row_sqnorms_ref(x), (n64 ** 2).astype(np.float32), rtol=2e-7)


def test_l2_ranking_is_dot_product_ranking_of_augmented_vectors():
    rng = np.random.default_rng(4)
    data = rng.standard_normal((700, 40)).astype(np.float32) * 3
    q = data[:9] + 0.01 * rng.standard_normal((9, 40)).astype(np.float32)
    qa, bank = O.l2_augment(data, q)
    s, i = O.topk_o64(qa, bank, 6)
    d64, i64 = O.l2_topk_o64(data, q, 6)
    assert np.array_equal(i, i64)
    # and the similarity encodes the distance: s = 2 q.x - ||x||^2  ->  d^2 = ||q||^2 - s
    qq = (q.astype(np.float64) ** 2).sum(1)[:, None]
    # (d^2 carries the fp32 rounding of ||x||^2: absolute error ~ ulp(||x||^2), not relative)
    assert np.allclose(qq - s, d64 ** 2, atol=4e-5 * float(qq.max()))
    # the notebook's own expression (rank 0 = the nearest, here the perturbed source row)
    nb = np.argsort(np.linalg.norm(data.astype(np.float64) - q[3].astype(np.float64), axis=1))[:6]
    assert np.array_equal(nb, i64[3])


def test_metrics_ref_against_sklearn():
    from sklearn.metrics import confusion_matrix, f1_score, recall_score

    rng = np.random.default_rng(5)
    C = 9
    target = rng.choice(C - 1, size=4000, p=np.array([0.05, 0.02, 0.1, 0.2, 0.08, 0.01, 0.04, 0.5]))  # class 8 absent
    pred = np.where(rng.random(4000) < 0.7, target, rng.integers(0, C - 1, 4000))
    m = O.metrics_ref(pred, target, C)
    assert np.array_equal(m["counts"], confusion_matrix(target, pred, labels=np.arange(C)))
    assert abs(m["accuracy"] - recall_score(target, pred, average="macro")) < 1e-12
    assert abs(m["f1"] - f1_score(target, pred, average="macro")) < 1e-12
    want = confusion_matrix(target, pred, labels=np.arange(C), normalize="true")
    assert np.allclose(m["confusion"], want)


def test_metrics_from_counts_on_cpu_tensors():
    from b200knn.metrics import metrics_from_counts

    rng = np.random.default_rng(6)
    target = rng.integers(0, 38, 3000)
    pred = np.where(rng.random(3000) < 0.5, target, rng.integers(0, 38, 3000))
    ref = O.metrics_ref(pred, target, 38)
    got = metrics_from_counts(torch.from_numpy(ref["counts"]))
    assert abs(float(got["accuracy"]) - ref["accuracy"]) < 1e-12
    assert abs(float(got["f1"]) - ref["f1"]) < 1e-12
    assert np.allclose(got["confusion"].numpy(), ref["confusion"])


def test_load_embedding_table_roundtrip(tmp_path):
    """The layout of the reference's tables (notebooks/3.0-Embeddings-inference.ipynb:493-507):
    integer columns 0..511 hold the fp16 embedding, then waferMap, failureType, failureCode."""
    import pandas as pd

    from b200knn.retrieval import load_embedding_table

    rng = np.random.default_rng(7)
    emb = rng.standard_normal((30, 512)).astype(np.float16)
    df = pd.DataFrame(emb, columns=list(range(512)))
    df["waferMap"] = [rng.integers(0, 3, (26, 26), dtype=np.uint8) for _ in range(30)]
    df["failureType"] = ["none"] * 30
    df["failureCode"] = rng.integers(0, 9, 30)
    path = os.path.join(tmp_path, "Demo_preds_subset.pkl.xz")
    df.to_pickle(path)
    got, meta = load_embedding_table(path)
    assert got.shape == (30, 512) and got.dtype == np.float16 and np.array_equal(got, emb)
    assert list(meta.columns) == ["waferMap", "failureType", "failureCode"]
