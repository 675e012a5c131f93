"""ctypes binding of libb200knn.so (the C ABI declared in include/b200knn.h).

There is deliberately no fallback: if the shared library is missing or the
device is not an sm_100 GPU the product path raises.  The library is looked up
in-tree (``self-supervised-wafermaps_b200/lib/libb200knn.so``, built by
``csrc/build.sh`` / ``__graft_entry__.build()``) or at ``$B200KNN_LIB``.
"""
from __future__ import annotations

import ctypes
import os
from ctypes import c_char_p, c_double, c_int, c_int32, c_int64, c_size_t, c_void_p

_HERE = os.path.dirname(os.path.abspath(__file__))
_DEFAULT = os.path.normpath(os.path.join(_HERE, "..", "lib", "libb200knn.so"))

# mirrors of the #defines in include/b200knn.h
F32, F16, BF16 = 0, 1, 2
LAYOUT_DN, LAYOUT_ND = 0, 1
MODE_EXACT, MODE_BF16, MODE_TF32X3, MODE_F32ROWS, MODE_BF16X3, MODE_F16X2, MODE_F16 = 0, 1, 2, 3, 4, 5, 6
SAMPLE_R = 16  # B200KNN_SAMPLE_R
MODES = {"exact": MODE_EXACT, "bf16": MODE_BF16, "tf32x3": MODE_TF32X3, "bf16x3": MODE_BF16X3, "f16x2": MODE_F16X2, "f16": MODE_F16}


class TopkOptions(ctypes.Structure):
    """b200knn_topk_options: all zero is a plain b200knn_topk."""
    _fields_ = [("bank_row_stride", c_int64), ("tau0", c_void_p), ("upper_keys", c_void_p),
                ("q_groups", c_void_p), ("bank_groups", c_void_p), ("sample", c_int),
                ("host_peer_out", ctypes.POINTER(c_void_p)), ("n_peers", c_int), ("my_rank", c_int),
                ("rows_per_owner", c_int64)]


# every symbol include/b200knn.h declares: (restype, argtypes)
SIGNATURES = {
    "b200knn_version": (c_int, []),
    "b200knn_last_error": (c_char_p, []),
    "b200knn_device_ok": (c_int, []),
    "b200knn_prepare_rows": (
        c_int,
        [c_void_p, c_int, c_int, c_int64, c_int, c_int64, c_int, c_void_p, c_void_p, c_void_p],
    ),
    "b200knn_topk_workspace_bytes": (c_size_t, [c_int64, c_int64, c_int, c_int, c_int]),
    "b200knn_topk": (
        c_int,
        [c_int, c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int, c_int, c_int64,
         c_int64, c_int64, c_int, c_int, c_int64, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "b200knn_topk_opt": (
        c_int,
        [c_int, c_void_p, c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int, c_int, c_int64,
         c_int64, c_int64, c_int, c_int, c_int64, c_void_p, c_void_p, c_size_t, ctypes.POINTER(TopkOptions),
         c_void_p],
    ),
    "b200knn_broadcast_f32": (c_int, [c_void_p, c_int64, ctypes.POINTER(c_void_p), c_int, c_int64, c_void_p]),
    "b200knn_merge": (c_int, [c_void_p, c_int, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "b200knn_decode_keys": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_void_p]),
    "b200knn_drop_self": (c_int, [c_void_p, c_int64, c_int, c_int64, c_void_p, c_void_p]),
    "b200knn_drop_group": (
        c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "b200knn_vote": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64, c_int, c_double, c_void_p, c_void_p,
         c_void_p, c_void_p],
    ),
    "b200knn_vote_ex": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64, c_int, c_double, c_void_p, c_int64, c_int,
         c_void_p, c_void_p, c_void_p],
    ),
    "b200knn_vote_multi": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64, c_int, ctypes.POINTER(c_int), c_int,
         ctypes.POINTER(c_double), c_int, c_void_p, c_int64, c_int, c_void_p, c_void_p],
    ),
    "b200knn_vote_multilabel": (
        c_int,
        [c_void_p, c_void_p, c_int64, c_int, c_int64, c_int64, c_int, ctypes.POINTER(c_int), c_int,
         ctypes.POINTER(c_double), c_int, c_void_p, c_int64, c_void_p, c_void_p],
    ),
    "b200knn_key_sim_column": (c_int, [c_void_p, c_int64, c_int, c_int, c_void_p, c_void_p]),
    "b200knn_radius_compact": (
        c_int, [c_void_p, c_int64, c_int, c_void_p, ctypes.c_float, c_int64, c_int64, c_void_p, c_void_p, c_void_p,
                c_void_p, c_void_p, c_void_p]),
    "b200knn_radius_tau0": (
        c_int, [c_void_p, c_int64, c_int64, c_int, ctypes.c_float, ctypes.c_float, ctypes.c_float, ctypes.c_float,
                c_void_p, c_void_p, ctypes.c_float, c_void_p, c_void_p, c_void_p, c_void_p]),
    "b200knn_union_edges": (c_int, [c_void_p, c_int64, c_void_p, c_void_p, c_int64, c_int64, c_void_p, c_void_p]),
    "b200knn_components": (c_int, [c_void_p, c_int64, c_void_p, c_void_p]),
    "b200knn_normalize_rows": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, ctypes.c_float, c_void_p, c_void_p]),
    "b200knn_row_sqnorms": (c_int, [c_void_p, c_int, c_int64, c_int, c_int64, c_void_p, c_void_p]),
    "b200knn_confusion": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p, c_void_p]),
    "b200knn_row_norm_max": (c_int, [c_void_p, c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "b200knn_row_f16_residual_max": (c_int, [c_void_p, c_int64, c_int, c_void_p, c_void_p]),
    "b200knn_rescore": (
        c_int,
        [c_void_p, c_int, c_int64, c_void_p, c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_int,
         c_int64, ctypes.c_float, ctypes.c_float, ctypes.c_float, c_void_p, c_void_p, c_void_p, c_void_p,
         c_void_p, c_size_t, c_void_p],
    ),
    "b200knn_rescore_workspace_bytes": (c_size_t, [c_int64, c_int]),
    "b200knn_rescore_vote": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_int, ctypes.c_float,
         ctypes.c_float, ctypes.c_float, c_void_p, c_void_p, ctypes.c_float, c_void_p, c_int64, c_int, c_double,
         c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_void_p, c_size_t, c_void_p],
    ),
    "b200knn_route_keys": (c_int, [c_void_p, c_int64, c_int, c_int64, c_int, c_void_p, c_void_p]),
    "b200knn_route_scatter": (
        c_int, [c_void_p, c_int64, c_int, c_int64, c_int, ctypes.POINTER(c_void_p), c_int64, c_void_p]),
    "b200knn_rescore_scatter": (
        c_int,
        [c_void_p, c_int64, c_void_p, c_int64, c_int, c_void_p, c_int64, c_int, c_int64,
         ctypes.POINTER(c_void_p), c_int, c_int, c_int64, c_void_p, c_size_t, c_void_p],
    ),
    "b200knn_compact_rows": (c_int, [c_void_p, c_int64, c_int64, c_int64, c_void_p, c_int, c_void_p, c_void_p]),
    "b200knn_scatter_rows": (
        c_int, [c_void_p, c_int64, c_void_p, c_int64, c_void_p, c_int, c_void_p, c_int, c_void_p]),
    "b200knn_certify": (
        c_int,
        [c_void_p, c_int, c_int64, c_int, c_void_p, c_int, c_void_p, c_int, c_int64, c_int, ctypes.c_float,
         ctypes.c_float, ctypes.c_float, c_void_p, c_void_p, c_void_p, c_void_p],
    ),
    "b200knn_set_l2_chunk_bytes": (c_int, [c_int64]),
    "b200knn_plan_info_ex": (c_int, [c_int, c_int64, c_int64, c_int, c_int, ctypes.POINTER(c_int64)]),
    "b200knn_debug_topk_dump": (
        c_int,
        [c_int, c_void_p, c_void_p, c_void_p, c_void_p, c_int64, c_int64, c_int, c_int, c_void_p,
         c_void_p, c_size_t, c_void_p, c_void_p, c_int, c_void_p],
    ),
}

_lib = None

# kernels each C entry point launches (bench.py's gpu_launches; a b200knn_topk* call whose plan
# splits the bank launches one more, the split merge — bench.py adds those from plan_info)
KERNELS_PER_CALL = {
    "b200knn_prepare_rows": 1, "b200knn_topk": 1, "b200knn_topk_opt": 1,
    "b200knn_merge": 1, "b200knn_decode_keys": 1, "b200knn_drop_self": 1, "b200knn_drop_group": 1, "b200knn_vote": 1, "b200knn_vote_ex": 1, "b200knn_vote_multi": 1,
    "b200knn_vote_multilabel": 1,
    "b200knn_key_sim_column": 1, "b200knn_normalize_rows": 1, "b200knn_confusion": 1, "b200knn_row_sqnorms": 1, "b200knn_rescore": 2, "b200knn_rescore_vote": 3, "b200knn_route_keys": 1, "b200knn_certify": 1,
    "b200knn_row_norm_max": 1, "b200knn_row_f16_residual_max": 1, "b200knn_debug_topk_dump": 1, "b200knn_broadcast_f32": 1,
    "b200knn_route_scatter": 1, "b200knn_rescore_scatter": 2, "b200knn_compact_rows": 1, "b200knn_scatter_rows": 1,
    "b200knn_radius_compact": 1, "b200knn_radius_tau0": 1, "b200knn_union_edges": 1, "b200knn_components": 1,
}
launch_counter = {"kernels": 0}


class _CountingLib:
    """Thin proxy over the CDLL that counts kernel launches made through the C ABI."""

    def __init__(self, cdll):
        self._cdll = cdll
        self._cache = {}

    def __getattr__(self, name):
        fn = self._cache.get(name)
        if fn is None:
            raw = getattr(self._cdll, name)
            n = KERNELS_PER_CALL.get(name, 0)
            if n:
                def fn(*args, _raw=raw, _n=n):
                    launch_counter["kernels"] += _n
                    return _raw(*args)
            else:
                fn = raw
            self._cache[name] = fn
        return fn


def lib_path() -> str:
    return os.environ.get("B200KNN_LIB", _DEFAULT)


def load() -> ctypes.CDLL:
    """Load the shared library once; raise (never fall back) if it is absent."""
    global _lib
    if _lib is not None:
        return _lib
    path = lib_path()
    if not os.path.exists(path):
        raise RuntimeError(
            f"b200knn: CUDA extension not found at {path}; build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` "
            "(self-supervised-wafermaps_b200/csrc/build.sh). There is no CPU fallback."
        )
    lib = ctypes.CDLL(path)
    for name, (restype, argtypes) in SIGNATURES.items():
        fn = getattr(lib, name)
        fn.restype = restype
        fn.argtypes = argtypes
    _lib = _CountingLib(lib)
    return _lib


def check(rc: int, what: str) -> None:
    if rc != 0:
        msg = load().b200knn_last_error().decode("utf-8", "replace")
        raise RuntimeError(f"b200knn {what} failed ({rc}): {msg}")
