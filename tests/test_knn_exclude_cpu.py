"""CPU: group exclusion inside the neighbour search (topk_keys(exclude=...), knn_predict_multi /
knn_topk(query_groups=, bank_groups=)).  The C ABI's argument checks of the group-excluding
options, the Python argument errors and the k bound (raised before any search, so they need no
GPU), and the rule that picks which leave-one-group-out searches skip the group inside the search."""
import pytest
import torch

import b200knn
from b200knn import _lib
from b200knn import knn as K


def test_topk_opt_refuses_null_group_ids_without_gpu():
    lib = _lib.load()

    def topk_opt(mode, k, qg, bg):
        # (mode, q_hi, q_lo, q_dtype, q_ld, bank_hi, bank_lo, bank_dtype, bank_layout, bank_ld, B, N, dim, k,
        #  idx_offset, out_keys, workspace, workspace_bytes, opts, stream)
        return lib.b200knn_topk_opt(mode, 1, None, 0, 64, 1, None, 0, 1, 64, 4, 100, 64, k, 0, 1, 1, 1 << 20,
                                    _lib.TopkOptions(q_groups=qg, bank_groups=bg), None)

    for mode in (_lib.MODE_BF16, _lib.MODE_EXACT):
        for qg, bg in ((None, 1), (1, None)):
            assert topk_opt(mode, 5, qg, bg) == -1
            assert b"null group ids" in lib.b200knn_last_error()
        # the shape checks of b200knn_topk apply as they are
        assert topk_opt(mode, 101, 1, 1) == -1
        assert b"k out of range" in lib.b200knn_last_error()


def _case(B=4, N=50):
    f = torch.randn(B, 8)
    bank = torch.randn(8, N)
    lab = torch.zeros(N, dtype=torch.int64)
    qg = torch.tensor([0, 1, 2, 3], dtype=torch.int64)[:B]
    bg = torch.arange(N) % 4  # query 0's group has 13 of the 50 bank rows, the others 12
    return f, bank, lab, qg, bg


@pytest.mark.parametrize("call", ["multi", "topk"])
def test_argument_errors_before_any_search(call):
    f, bank, lab, qg, bg = _case()

    def run(k=5, **kw):
        if call == "multi":
            return b200knn.knn_predict_multi(f, bank, lab, 3, (k, 1), (0.1,), **kw)
        return b200knn.knn_topk(f, bank, k, **kw)

    with pytest.raises(ValueError, match="pass both or neither"):
        run(query_groups=qg)
    with pytest.raises(ValueError, match="pass both or neither"):
        run(bank_groups=bg)
    with pytest.raises(RuntimeError, match="query_groups has 3 entries for 4 queries"):
        run(query_groups=qg[:3], bank_groups=bg)
    with pytest.raises(RuntimeError, match="bank_groups has 49 entries for 50 bank rows"):
        run(query_groups=qg, bank_groups=bg[1:])
    for dt in (torch.float32, torch.float64, torch.bool):
        with pytest.raises(ValueError, match="bank_groups must be an integer tensor"):
            run(query_groups=qg, bank_groups=bg.to(dt))
        with pytest.raises(ValueError, match="query_groups must be an integer tensor"):
            run(query_groups=qg.to(dt), bank_groups=bg)
    with pytest.raises(TypeError, match="query_groups must be a torch.Tensor"):
        run(query_groups=[0, 1, 2, 3], bank_groups=bg)
    # ids pass their checks: the CPU tensors raise next (no CPU fallback)
    with pytest.raises(RuntimeError, match="CPU fallback"):
        run(query_groups=qg, bank_groups=bg)


@pytest.mark.parametrize("call", ["multi", "topk"])
def test_k_bound_is_the_smallest_number_of_eligible_rows(call):
    f, bank, lab, qg, bg = _case()

    def run(k, qg=qg, bg=bg):
        if call == "multi":
            return b200knn.knn_predict_multi(f, bank, lab, 3, (1, k), (0.1,), query_groups=qg, bank_groups=bg)
        return b200knn.knn_topk(f, bank, k, query_groups=qg, bank_groups=bg)

    # query 0 keeps 50 - 13 = 37 bank rows
    for k in (38, 50, 51):
        with pytest.raises(RuntimeError, match="selected index k out of range"):
            run(k)
    with pytest.raises(RuntimeError, match="CPU fallback"):
        run(37)
    # ids compared by value across dtypes; a query id with no bank rows leaves the whole bank
    with pytest.raises(RuntimeError, match="CPU fallback"):
        run(50, qg=torch.tensor([7, 8, 9, 10], dtype=torch.uint8), bg=bg.to(torch.int16))
    with pytest.raises(RuntimeError, match="selected index k out of range"):
        run(38, qg=qg.to(torch.uint64), bg=bg.to(torch.int32))


def test_class_bound_checked_with_groups():
    f, bank, lab, qg, bg = _case()
    with pytest.raises(ValueError, match="at most"):
        b200knn.knn_predict_multi(f, bank, lab, 10 ** 5, (5,), (0.1,), query_groups=qg, bank_groups=bg)


def test_feature_bank_passes_the_groups_through():
    import inspect

    for name in ("knn_predict_multi", "knn_topk"):
        params = inspect.signature(getattr(b200knn.FeatureBank, name)).parameters
        assert "query_groups" in params and "bank_groups" in params, name


@pytest.mark.parametrize("k,p,n,deep", [
    (200, 1, 811457, False),     # plain leave-one-out depth 201
    (200, 32, 811457, False),    # lots of 25: depth 232
    (200, 2048, 811457, True),   # one group of 2,000: depth 2,248
    (5, 262144, 811457, True),   # 5-fold cross-validation
    (960, 32, 811457, False),    # depth 992 = MAX_K: still the streaming lists
    (961, 32, 811457, True),     # depth 993
    (200, 2048, 900, False),     # depth min(N, k + p) = 900 <= MAX_K
    (1500, 1, 6000, True),       # k itself beyond MAX_K: excluded peeling
])
def test_logo_excludes_rule(k, p, n, deep):
    assert K.logo_excludes(k, p, n) is deep


def test_deep_parts_follow_the_rule_in_every_mode():
    """The searches of a bucket: a part whose depth min(n, k + p) exceeds MAX_K is exactly the part
    ``logo_excludes`` names; the shallow parts keep the deeper search + drop_group."""
    for mode in ("fp32", "exact", "bf16", "f16"):
        for p in (1, 32, 1024, 2048, 262144):
            for part in K.logo_parts((5, 20, 200), p, 811457, mode):
                assert K.logo_excludes(part[-1], p, 811457) == (min(811457, part[-1] + p) > K.MAX_K)


def test_topk_keys_exclude_checks():
    f, bank, lab, qg, bg = _case()
    with pytest.raises(ValueError, match="int32"):
        K._exclusion((qg, bg), 4, 50, f.device)
    with pytest.raises(RuntimeError, match="have 49 entries for 50 rows"):
        K._exclusion((qg.int(), bg[1:].int()), 4, 50, f.device)
    qg32, bg32, m = K._exclusion((qg.int(), bg.int()), 4, 50, f.device)
    assert m == 13 and qg32.dtype == torch.int32 and bg32.dtype == torch.int32
