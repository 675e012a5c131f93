"""CPU: the C-ABI shared library loads and exports every symbol include/b200knn.h
declares; argument validation that needs no GPU returns the documented codes."""
import ctypes
import os
import re

import pytest

from b200knn import _lib

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "b200knn.h")).read()
    text = re.sub(r"/\*.*?\*/", "", text, flags=re.S)
    return sorted(set(re.findall(r"\b(b200knn_\w+)\s*\(", text)))


def test_header_symbols_all_bound_in_python():
    assert set(declared_symbols()) == set(_lib.SIGNATURES)


def test_library_exports_every_declared_symbol():
    lib = ctypes.CDLL(_lib.lib_path())
    for name in declared_symbols():
        assert hasattr(lib, name), name


def test_abi_version_and_error_string():
    lib = _lib.load()
    assert lib.b200knn_version() == 150
    assert isinstance(lib.b200knn_last_error(), bytes)


def test_argument_validation_without_gpu():
    lib = _lib.load()
    # k > N: Tensor.topk's "selected index k out of range"
    rc = lib.b200knn_topk(_lib.MODE_EXACT, 1, None, 0, 4, 1, None, 0, 0, 8, 2, 8, 4, 9, 0, 1, 1, 1 << 20, None)
    assert rc == -1 and b"k out of range" in lib.b200knn_last_error()
    rc = lib.b200knn_merge(1, 2, 4, 3, 7, 1, None)  # k_out > G*k_in
    assert rc == -1
    rc = lib.b200knn_vote(1, 1, 4, 3, 10, 0, 5, 0.0, 1, None, 1, None)  # t == 0
    assert rc == -1
    rc = lib.b200knn_prepare_rows(1, 7, 0, 4, 8, 4, 1, 1, None, None)  # bad dtype
    assert rc == -1
    assert lib.b200knn_topk_workspace_bytes(64, 1000, 512, 2000, 0) == 0  # k too large


PEERS = dict(peers=[1, 1], n_peers=2, my_rank=0, rows_per_owner=2)  # a valid exchange for B = 4
BF16, EXACT = _lib.MODE_BF16, _lib.MODE_EXACT


@pytest.mark.parametrize("mode,opts,message", [
    (EXACT, dict(bank_row_stride=2), "MODE_EXACT takes no"),
    (EXACT, dict(tau0=1), "MODE_EXACT takes no"),
    (EXACT, dict(sample=1), "MODE_EXACT takes no"),
    (EXACT, dict(PEERS), "MODE_EXACT takes no"),
    (BF16, dict(upper_keys=1), "upper_keys needs MODE_EXACT"),
    (BF16, dict(q_groups=1, bank_groups=1, bank_row_stride=2), "group ids take no"),
    (BF16, dict(q_groups=1, bank_groups=1, tau0=1), "group ids take no"),
    (BF16, dict(q_groups=1, bank_groups=1, sample=1), "group ids take no"),
    (BF16, dict(q_groups=1, bank_groups=1, **PEERS), "group ids take no"),
    (BF16, dict(sample=1, tau0=1), "sample takes no tau0"),
    (BF16, dict(bank_row_stride=2, **PEERS), "visits every row"),
    (BF16, dict(q_groups=1), "null group ids"),
    (EXACT, dict(bank_groups=1), "null group ids"),
    (BF16, dict(bank_row_stride=-1), "bank_row_stride must be >= 0"),
    (BF16, dict(sample=1, k=15), "sample needs k == 16"),
    (BF16, dict(sample=1, N=15), "sample needs k == 16 and at least 16 rows"),
    (BF16, dict(PEERS, n_peers=9, peers=[1] * 9), "1..8 peers"),
    (BF16, dict(PEERS, n_peers=0), "1..8 peers"),
    (BF16, dict(PEERS, peers=None), "1..8 peers"),
    (BF16, dict(PEERS, my_rank=2), "1..8 peers"),
    (BF16, dict(PEERS, my_rank=-1), "1..8 peers"),
    (BF16, dict(PEERS, rows_per_owner=1), "must cover B"),
    (BF16, dict(PEERS, peers=[1, None]), "null peer buffer"),
    (BF16, dict(PEERS, out_keys=1), "out_keys must be NULL"),
    (BF16, dict(out_keys=None), "null pointer"),
])
def test_topk_options_refused_without_gpu(mode, opts, message):
    """Every combination of b200knn_topk_opt's options that no search implements is refused before
    any planning, including sample or a row stride together with group ids."""
    lib = _lib.load()
    opts = dict(opts)
    k, N, out_keys = opts.pop("k", 16), opts.pop("N", 100), opts.pop("out_keys", None if "peers" in opts else 1)
    peers = opts.pop("peers", None)
    o = _lib.TopkOptions(**opts)
    if peers is not None:
        o.host_peer_out = (ctypes.c_void_p * len(peers))(*peers)
    # (mode, q_hi, q_lo, q_dtype, q_ld, bank_hi, bank_lo, bank_dtype, bank_layout, bank_ld, B, N, dim, k,
    #  idx_offset, out_keys, workspace, workspace_bytes, opts, stream)
    rc = lib.b200knn_topk_opt(mode, 1, 1, 0, 64, 1, 1, 0, 1, 64, 4, N, 64, k, 0, out_keys, 1, 1 << 20, o, None)
    assert rc == -1
    assert message.encode() in lib.b200knn_last_error()


def test_plan_is_deterministic_and_covers_bank():
    from b200knn import plan_info

    for (B, N, D, k) in [(64, 811457, 512, 200), (75776, 811457, 512, 200), (5703, 30000, 512, 20), (1, 5, 8, 5)]:
        for mode in ("exact", "bf16", "tf32x3"):
            p = plan_info(B, N, D, k, mode)
            assert p == plan_info(B, N, D, k, mode)
            assert p["splits"] * p["split_rows"] >= N > (p["splits"] - 1) * p["split_rows"]
            assert p["n_items"] == p["n_qtiles"] * p["splits"] and 1 <= p["grid"] <= p["n_items"]
            assert p["list_capacity"] >= k + 32


def test_missing_library_fails_loudly(monkeypatch):
    monkeypatch.setenv("B200KNN_LIB", "/nonexistent/libb200knn.so")
    monkeypatch.setattr(_lib, "_lib", None)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        _lib.load()


def test_graft_entry_build_runs():
    """The driver's build check: compiles whatever is stale, builds the oracle's C restatement and
    verifies the loaded library against include/b200knn.h."""
    import __graft_entry__

    __graft_entry__.build()
