"""CPU: knn_predict_loo — leave-one-out kNN of a labelled bank against itself.  The C ABI's argument
checks of b200knn_drop_self, the Python argument errors (raised before any device work, so they
need no GPU), CPU tensors raising, and the rule that splits the ks into searches at k + 1."""
import pytest
import torch

import datagen

import b200knn
from b200knn import _lib
from b200knn import knn as K


def test_drop_self_abi_refuses_bad_arguments_without_gpu():
    lib = _lib.load()
    for args, what in [((1, -1, 5, 0, 1, None), b"B < 0"),
                       ((None, 4, 5, 0, 1, None), b"null pointer"),
                       ((1, 4, 5, 0, None, None), b"null pointer"),
                       ((1, 4, 1, 0, 1, None), b"k_in >= 2"),
                       ((1, 4, 0, 0, 1, None), b"k_in >= 2"),
                       ((1, 4, -3, 0, 1, None), b"k_in >= 2")]:
        assert lib.b200knn_drop_self(*args) == -1, args  # B200KNN_E_ARG
        assert what in lib.b200knn_last_error(), (args, lib.b200knn_last_error())
    # no rows: nothing to launch, accepted without a device
    assert lib.b200knn_drop_self(1, 0, 5, 0, 1, None) == 0


def _ragged():
    c = datagen.make_case("ragged")  # N = 1001, D = 72, C = 5
    return torch.from_numpy(c["bank"]), torch.from_numpy(c["labels"]), c["C"]


@pytest.mark.parametrize("ks,ts,match", [
    ((), (0.1,), "empty"), ((5,), (), "empty"), ((5, 5), (0.1,), "duplicate"), ((5,), (0.1, 0.1), "duplicate"),
    ((0, 5), (0.1,), "positive"), ((5,), (0.0,), "non-zero"), (tuple(range(1, 18)), (0.1,), "at most"),
    ((2.5,), (0.1,), "integers"),
])
def test_grid_errors(ks, ts, match):
    bank, lab, C = _ragged()
    with pytest.raises(ValueError, match=match):
        b200knn.knn_predict_loo(bank, lab, C, ks, ts)


def test_shape_errors_before_device_work():
    bank, lab, C = _ragged()
    N = bank.shape[1]
    for ks in ((N,), (5, N + 3)):  # the bank without the row has N - 1 rows
        with pytest.raises(RuntimeError, match="selected index k out of range"):
            b200knn.knn_predict_loo(bank, lab, C, ks)
    with pytest.raises(RuntimeError, match=f"feature_labels has {N - 1} entries for a bank of {N}"):
        b200knn.knn_predict_loo(bank, lab[:-1], C, (5,))
    with pytest.raises(ValueError, match="batch"):
        b200knn.knn_predict_loo(bank, lab, C, (5,), batch=0)


def test_cpu_tensors_raise():
    bank, lab, C = _ragged()
    with pytest.raises(RuntimeError, match="CPU fallback"):
        b200knn.knn_predict_loo(bank, lab, C, (1, 5), (0.1,))


def test_feature_bank_without_labels_raises():
    fb = b200knn.FeatureBank(torch.zeros((10, 64)), 64)
    with pytest.raises(RuntimeError, match="without labels"):
        fb.knn_predict_loo(5, (3,))


@pytest.mark.parametrize("mode", ["bf16", "f16", "f16x2", "bf16x3", "tf32x3"])
def test_loo_parts_split_raw_modes_on_k_plus_1(mode):
    assert K.loo_parts((5, 991), mode) == [(5, 991)]
    # k = 992 searches at 993 > MAX_K: the exact kernel's side, with the ks beyond it
    assert K.loo_parts((5, 991, 992, 1000), mode) == [(5, 991), (992, 1000)]
    assert K.loo_parts((992,), mode) == [(992,)]
    # knn_predict_multi's own rule splits at k itself
    assert K.grid_parts((5, 992), mode) == [(5, 992)] and K.loo_parts((5, 992), mode) == [(5,), (992,)]


@pytest.mark.parametrize("mode", ["exact", "fp32", "fp32_f16x2", "fp32_bf16"])
def test_loo_parts_one_search_in_bit_exact_modes(mode):
    assert K.loo_parts((5, 991, 992, 1000), mode) == [(5, 991, 992, 1000)]
