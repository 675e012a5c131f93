"""CPU: host logic added in round 2 — certificate coefficients that scale with D, level specs with
margins, the margin boost, the pre-pass policy for small batches, the chunk-major work plan (the
planner runs on the host: b200knn_plan_info_ex needs no GPU), wide-vector mode resolution, the
non-negative generators."""
import numpy as np
import pytest
import torch

import datagen
from b200knn import _lib
from b200knn import knn as K


def test_level_config_scales_with_dimension_and_parses_margins():
    a, b = K.level_config("fp32_f16", 512), K.level_config("fp32_f16", 1024)
    assert a["margin"] == 40 and a["cand"] == "f16" and a["name"] == "fp32_f16"
    # err_coef = op_coef + acc_c * D_pad * 2^-23 (x1.01): the accumulation term doubles with D
    acc_a, acc_b = a["err_coef"] - a["op_coef"], b["err_coef"] - b["op_coef"]
    assert abs(acc_b / acc_a - 2.0) < 1e-12
    assert acc_a >= 1.125 * 512 * 2.0 ** -23 and acc_a <= 1.02 * 1.125 * 512 * 2.0 ** -23
    assert K.level_config("fp32_f16", 500)["err_coef"] == a["err_coef"]  # padded to 512
    w = K.level_config("fp32_f16x2@160", 512)
    assert w["margin"] == 160 and w["cand"] == "f16x2" and w["name"] == "fp32_f16x2@160"
    # (MMAs per k-step) * (K + 2) / K
    assert [K.LEVELS[n]["acc_c"] for n in ("fp32_f16", "fp32_f16x2", "fp32_bf16x3", "fp32_tf32")] == [1.125, 2.25, 3.375, 3.75]
    for spec in K.CASCADES["fp32"] + K.CASCADE_WIDE:
        K.level_config(spec, 512)


def test_margin_boost_state_machine():
    nb = K.next_boost
    assert nb(1, 0, 1000, 31) == (2, 0)            # > 3 % uncertified: widen
    assert nb(2, 0, 1000, 31) == (4, 0)
    assert nb(4, 0, 1000, 900) == (4, 0)           # capped
    assert nb(1, 0, 64, 64) == (1, 0)              # small batches never move it
    assert nb(2, 0, 1000, 10) == (2, 0)            # between the thresholds: stay, calm counter reset
    b, c = 2, 0
    for _ in range(K.CASCADE_CALM_CALLS - 1):
        b, c = nb(b, c, 1000, 0)
        assert b == 2
    assert nb(b, c, 1000, 0) == (1, 0)             # calm for CASCADE_CALM_CALLS calls: narrow again


def test_prepass_policy_for_small_batches():
    assert K.prepass_stride(811457, 240) == 75 and K.prepass_stride(811457, 240, 151552) == 75
    assert K.prepass_stride(37348, 45) == 0            # large batches: only for k >= 64
    assert K.prepass_stride(37348, 45, 64) == 14       # the reference-shaped call: any k
    assert K.prepass_stride(37348, 45, 513) == 0
    assert K.prepass_stride(5000, 45, 64) == 0         # too few rows to sample
    s = K.prepass_stride(811457, 5, 64)
    assert s == 8 and (1 - 1 / s) ** 5 > 0             # k = 5: stride floor


def test_chunk_major_plan():
    lib = _lib.load()
    assert lib.b200knn_set_l2_chunk_bytes(40 << 20) == 0
    p = K.plan_info(151552, 811457, 512, 240, "f16")
    assert p["splits"] == 1 and p["grid"] == 74 and p["n_qtiles"] == 592
    assert p["chunks"] > 1 and p["slots"] == 8 and p["chunk_rows"] % 256 == 0
    assert p["chunks"] * p["chunk_rows"] >= 811457 > (p["chunks"] - 1) * p["chunk_rows"]
    assert p["chunk_rows"] * 512 * 2 <= (40 << 20) * 1.05
    # two bank arrays per row: half the rows per chunk
    assert K.plan_info(151552, 811457, 512, 240, "f16x2")["chunk_rows"] * 2 <= p["chunk_rows"] + 512
    # one tile per worker, small banks, bank splits: no chunks
    assert K.plan_info(34590, 138360, 512, 240, "f16")["chunks"] == 1
    small = K.plan_info(64, 811457, 512, 240, "f16")
    assert small["chunks"] == 1 and small["splits"] > 100 and small["grid"] == small["n_items"] <= 148  # single CTAs
    assert K.plan_info(811457, 811457, 512, 50, "bf16")["slots"] == 16  # capped
    try:
        assert lib.b200knn_set_l2_chunk_bytes(0) == 0
        assert K.plan_info(151552, 811457, 512, 240, "f16")["chunks"] == 1
        assert lib.b200knn_set_l2_chunk_bytes(-1) != 0
    finally:
        lib.b200knn_set_l2_chunk_bytes(40 << 20)


def test_wide_vectors_resolve_one_effective_mode():
    for m in ("bf16", "f16", "f16x2"):
        assert K.effective_mode(m, 768) == m and K.effective_mode(m, 769) == "bf16x3" and K.effective_mode(m, 1024) == "bf16x3"
    assert K.effective_mode("tf32x3", 2048) == "tf32x3" and K.effective_mode("exact", 4096) == "exact"
    bank = torch.zeros((1024, 10))
    assert K._cascade_levels(bank, "fp32", track=False) == list(K.CASCADE_WIDE)
    assert K._cascade_levels(torch.zeros((512, 10)), "fp32", track=False, boost=2)[0] == "fp32_f16@80"
    assert K._cascade_levels(torch.zeros((512, 10)), "fp32_f16x2", track=False, boost=4) == ["fp32_f16x2"]


@pytest.mark.parametrize("name", datagen.RELU_CASE_NAMES)
def test_nonnegative_cases_are_nonnegative_and_unit_norm(name):
    c = datagen.make_case(name)
    assert (c["feature"] >= 0).all() and (c["bank"] >= 0).all()
    assert np.allclose(np.linalg.norm(c["bank"], axis=0), 1.0, atol=1e-5)
    sims = c["feature"] @ c["bank"]
    assert sims.min() >= 0 and sims.mean() > 0.3  # every pair of rows is similar: the bunched regime


def test_bench_generators_cover_the_reference_distribution():
    import bench

    for kind in ("clustered", "gauss", "relu", "absgauss"):
        bank, lab, q = bench.make_inputs(torch.device("cpu"), 3000, 50, 64, seed=1, kind=kind)
        assert bank.shape == (3000, 64) and q.shape == (50, 64) and lab.shape == (3000,)
        assert torch.allclose(bank.norm(dim=1), torch.ones(3000), atol=1e-5)
        if kind in ("relu", "absgauss"):
            assert bool((bank >= 0).all()) and bool((q >= 0).all())
    a = bench.make_inputs(torch.device("cpu"), 3000, 50, 64, seed=1, kind="relu", row_range=(1000, 2000))[0]
    b = bench.make_inputs(torch.device("cpu"), 3000, 50, 64, seed=1, kind="relu")[0]
    assert torch.equal(a, b[1000:2000])  # shard-reproducible


def test_bench_library_bar_is_the_reference_op_sequence():
    """bench.py's `gpu_library_baseline` restates lightly's knn_predict inline (it may not import the
    oracle for that leg): on CPU it must give exactly what the oracle's R32 gives."""
    import bench
    from oracle import knn_oracle as O

    c = datagen.make_case("mixed38")
    f, bank, lab = (torch.from_numpy(c[n]) for n in ("feature", "bank", "labels"))
    got = bench.library_knn_predict(f, bank, lab, c["C"], c["k"], c["t"])
    assert torch.equal(got, O.knn_predict_r32(f, bank, lab, c["C"], c["k"], c["t"]))


def test_bench_dump_outputs_full_and_sampled(tmp_path, monkeypatch):
    """--dump-outputs: the whole (Q, C) ranking as float64 while it fits the budget, else the same
    seeded sample of rows on every run, with their indices."""
    import bench

    pred = torch.stack([torch.randperm(9, generator=torch.Generator().manual_seed(r)) for r in range(500)])
    bench.dump_outputs(str(tmp_path / "full"), pred)
    got = np.load(tmp_path / "full" / "pred_labels.npy")
    assert got.dtype == np.float64 and np.array_equal(got, pred.numpy())
    assert not (tmp_path / "full" / "pred_labels_rows.npy").exists()
    monkeypatch.setattr(bench, "DUMP_BYTES", 8 * 10 * 100)
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), pred)
    rows = np.load(tmp_path / "a" / "pred_labels_rows.npy")
    assert rows.dtype == np.float64 and len(rows) == 100 and np.all(np.diff(rows) > 0)
    assert np.array_equal(np.load(tmp_path / "a" / "pred_labels.npy"), pred.numpy()[rows.astype(np.int64)])
    for name in ("pred_labels.npy", "pred_labels_rows.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name))
