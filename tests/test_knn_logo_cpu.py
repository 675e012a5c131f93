"""CPU: leave-one-group-out kNN (knn_predict_loo(groups=...), knn_graph(groups=...)).  The C ABI's
argument checks of b200knn_drop_group, the Python argument errors (raised before any search, so they
need no GPU), CPU tensors raising, and the rule that splits the ks of a bucket into searches."""
import pytest
import torch

import datagen

import b200knn
from b200knn import _lib
from b200knn import knn as K


def test_drop_group_abi_refuses_bad_arguments_without_gpu():
    lib = _lib.load()
    # (keys_in, B, k_in, row_ids, group_ids, N, k_out, keys_out, err_flag, stream)
    for args, what in [((1, -1, 5, 1, 1, 10, 4, 1, 1, None), b"B < 0"),
                       ((1, 4, 5, 1, 1, -1, 4, 1, 1, None), b"N < 0"),
                       ((None, 4, 5, 1, 1, 10, 4, 1, 1, None), b"null pointer"),
                       ((1, 4, 5, None, 1, 10, 4, 1, 1, None), b"null pointer"),
                       ((1, 4, 5, 1, None, 10, 4, 1, 1, None), b"null pointer"),
                       ((1, 4, 5, 1, 1, 10, 4, None, 1, None), b"null pointer"),
                       ((1, 4, 5, 1, 1, 10, 4, 1, None, None), b"null pointer"),
                       ((1, 4, 5, 1, 1, 10, 0, 1, 1, None), b"1 <= k_out <= k_in"),
                       ((1, 4, 5, 1, 1, 10, -2, 1, 1, None), b"1 <= k_out <= k_in"),
                       ((1, 4, 5, 1, 1, 10, 6, 1, 1, None), b"1 <= k_out <= k_in")]:
        assert lib.b200knn_drop_group(*args) == -1, args  # B200KNN_E_ARG
        assert what in lib.b200knn_last_error(), (args, lib.b200knn_last_error())
    # no rows: nothing to launch, accepted without a device; k_out == k_in is allowed
    assert lib.b200knn_drop_group(1, 0, 5, 1, 1, 10, 5, 1, 1, None) == 0


def _ragged():
    c = datagen.make_case("ragged")  # N = 1001, D = 72, C = 5
    return torch.from_numpy(c["bank"]), torch.from_numpy(c["labels"]), c["C"]


def _one_group_of_7(N):
    g = torch.arange(N, dtype=torch.int64) * 3 - 100  # any values: non-contiguous, negative
    g[[4, 90, 91, 300, 512, 700, 1000]] = 12345
    return g


def test_group_errors_before_device_work():
    bank, lab, C = _ragged()
    N = bank.shape[1]
    groups = _one_group_of_7(N)
    with pytest.raises(RuntimeError, match=f"groups has {N - 1} entries for a bank of {N}"):
        b200knn.knn_predict_loo(bank, lab, C, (5,), groups=groups[1:])
    for dt in (torch.float32, torch.float64, torch.bool):
        with pytest.raises(ValueError, match="integer"):
            b200knn.knn_predict_loo(bank, lab, C, (5,), groups=groups.to(dt))
    # the bank without the group of 7 has N - 7 rows
    for ks in ((N - 6,), (5, N - 3), (N,)):
        with pytest.raises(RuntimeError, match="selected index k out of range"):
            b200knn.knn_predict_loo(bank, lab, C, ks, groups=groups)
    # k = N - 7 passes the range check; the CPU tensors raise next
    with pytest.raises(RuntimeError, match="CPU fallback"):
        b200knn.knn_predict_loo(bank, lab, C, (N - 7,), groups=groups)
    # the errors of knn_predict_loo without groups are unchanged with them
    with pytest.raises(ValueError, match="duplicate"):
        b200knn.knn_predict_loo(bank, lab, C, (5, 5), groups=groups)
    with pytest.raises(RuntimeError, match=f"feature_labels has {N - 1} entries for a bank of {N}"):
        b200knn.knn_predict_loo(bank, lab[:-1], C, (5,), groups=groups)
    with pytest.raises(ValueError, match="batch"):
        b200knn.knn_predict_loo(bank, lab, C, (5,), batch=0, groups=groups)
    with pytest.raises(ValueError, match="at most"):
        b200knn.knn_predict_loo(bank, lab, 10 ** 5, (5,), groups=groups)


@pytest.mark.parametrize("dtype", [torch.int8, torch.uint8, torch.int16, torch.int32, torch.int64, torch.uint16,
                                   torch.uint32, torch.uint64])
def test_cpu_tensors_raise(dtype):
    bank, lab, C = _ragged()
    groups = (torch.arange(bank.shape[1]) // 25).to(dtype)
    with pytest.raises(RuntimeError, match="CPU fallback"):
        b200knn.knn_predict_loo(bank, lab, C, (1, 5), (0.1,), groups=groups)


def test_knn_graph_group_errors():
    rows = torch.zeros((100, 8))
    groups = torch.arange(100) // 10  # groups of 10
    with pytest.raises(ValueError, match="include_self"):
        b200knn.knn_graph(rows, 5, include_self=True, groups=groups)
    with pytest.raises(RuntimeError, match="k must be smaller than the number of rows"):
        b200knn.knn_graph(rows, 91, groups=groups)
    with pytest.raises(RuntimeError, match="groups has 99 entries for a bank of 100"):
        b200knn.knn_graph(rows, 5, groups=groups[1:])
    with pytest.raises(ValueError, match="integer"):
        b200knn.knn_graph(rows, 5, groups=groups.float())


def test_group_plan_buckets_rows_by_power_of_two():
    groups = torch.tensor([7, 7, -1, 3, 7, 3, 9, 7, 7, 4, 4, 4], dtype=torch.int32)
    gid, g_max, rows, buckets = K._group_plan(groups, 12, groups.device)
    assert g_max == 5 and gid.dtype == torch.int32
    assert torch.equal(gid, torch.tensor([3, 3, 0, 1, 3, 1, 4, 3, 3, 2, 2, 2], dtype=torch.int32))
    # sizes: group 7 -> 5 (p = 8), 3 -> 2 (p = 2), 4 -> 3 (p = 4), -1 and 9 -> 1 (p = 1)
    assert buckets == [(1, 0, 2), (2, 2, 4), (4, 4, 7), (8, 7, 12)]
    assert rows.tolist() == [2, 6, 3, 5, 9, 10, 11, 0, 1, 4, 7, 8]
    # the same groups: no id is minus another
    _, _, rows_abs, buckets_abs = K._group_plan(groups.abs(), 12, groups.device)
    rows_abs = rows_abs.tolist()
    _, g_max, rows, buckets = K._group_plan(torch.arange(12), 12, groups.device)
    assert g_max == 1 and buckets == [(1, 0, 12)] and rows.tolist() == list(range(12))
    # unsigned ids: the same groups whatever the width, also above 2**63 for uint64
    for dt in (torch.uint16, torch.uint32, torch.uint64):
        u = groups.to(torch.int64).abs().to(dt)
        if dt == torch.uint64:
            u = u.view(torch.int64).add(2 ** 62).add(2 ** 62).view(torch.uint64)  # ids >= 2**63
        _, g_max, rows_u, buckets_u = K._group_plan(u, 12, groups.device)
        assert g_max == 5 and buckets_u == buckets_abs and rows_u.tolist() == rows_abs, dt


KS = (1, 5, 20, 200, 500, 900, 960, 961, 991, 992, 1000, 3000)


@pytest.mark.parametrize("mode", ["bf16", "f16", "f16x2", "bf16x3", "tf32x3", "exact", "fp32", "fp32_f16x2"])
def test_logo_parts_p1_is_loo_parts(mode):
    for i in range(len(KS)):
        for j in range(i + 1, len(KS) + 1):
            assert K.logo_parts(KS[i:j], 1, 10 ** 6, mode) == K.loo_parts(KS[i:j], mode), KS[i:j]


@pytest.mark.parametrize("mode", ["bf16", "f16", "f16x2", "bf16x3", "tf32x3"])
def test_logo_parts_split_raw_modes_on_k_plus_p(mode):
    n = 10 ** 6
    assert K.logo_parts((5, 960), 32, n, mode) == [(5, 960)]  # 960 + 32 = 992 = MAX_K
    assert K.logo_parts((5, 961), 32, n, mode) == [(5,), (961,)]
    assert K.logo_parts((5, 20, 200), 1024, n, mode) == [(5, 20, 200)]  # every search beyond MAX_K
    assert K.logo_parts((5, 20, 900), 128, n, mode) == [(5, 20), (900,)]
    # depths are capped at n: a bank of 992 rows never leaves the raw kernel
    assert K.logo_parts((5, 961), 32, 992, mode) == [(5, 961)]
    assert K.logo_parts((5, 961), 32, 993, mode) == [(5,), (961,)]


@pytest.mark.parametrize("mode", ["exact", "fp32", "fp32_f16x2", "fp32_bf16"])
def test_logo_parts_one_search_per_bucket_in_bit_exact_modes(mode):
    for p in (1, 2, 32, 1024, 2048):
        assert K.logo_parts((5, 20, 200, 961, 3000), p, 10 ** 6, mode) == [(5, 20, 200, 961, 3000)]
