"""Host-side mirror of the reference interface for the kNN hot path.

``knn_predict`` keeps the exact signature, defaults, tensor layouts and return
type of ``lightly.utils.benchmarking.knn_predict`` as the reference binds and
calls it (``src/ssl_wafermap/models/knn.py:16`` import, ``:91-98`` and
``:205-212`` calls): ``feature`` (B,D), ``feature_bank`` (D,N) — the
``.t().contiguous()`` layout of ``knn.py:80`` — ``feature_labels`` (N,) int64,
returning (B, num_classes) int64 class rankings whose column 0 the caller
consumes (``knn.py:99``).  No normalisation happens inside (the caller does it,
``knn.py:77`` / ``:90``).

``knn_topk`` is the additive retrieval entry point (``torch.mm(...).topk(k)``
with the canonical (sim desc, index asc) order) that generalises the
notebooks' brute-force search
(``notebooks/2.0-Figures-nearest-neighbors.ipynb:54``).

Everything here is plumbing: argument checks that mirror torch's errors,
operand-preparation caching, workspace allocation through the PyTorch caching
allocator, and calls through the C ABI on the current CUDA stream.
"""
from __future__ import annotations

import ctypes
import math
import os
import weakref
from typing import Optional, Tuple

import torch

from . import _lib

_DTYPES = {torch.float32: _lib.F32, torch.float16: _lib.F16, torch.bfloat16: _lib.BF16}

TC_MODES = ("bf16", "tf32x3", "bf16x3", "f16x2", "f16")  # raw tensor-core similarity modes
MAX_K = 992  # largest k of the streaming candidate lists (capacity 1024, include/b200knn.h)
MAX_BF16_DIM = 768  # widest (padded) vector whose query tile the BF16 kernel can keep resident

_default_mode = os.environ.get("B200KNN_MODE", "fp32")

# Measurement hook (bench.py): when set to a dict, the similarity + top-k C calls ("topk") and the
# exact re-scoring calls ("rescore") are bracketed by CUDA events recorded on the launching stream
# and the (start, end) pairs are appended to the list under that name.
profile_events = None


class _Timed:
    """with _Timed("topk"): <C call>  — no-op unless bench.py switched profile_events on."""

    __slots__ = ("name", "ev")

    def __init__(self, name: str, on: bool = True):
        self.name = name
        self.ev = None
        if on and profile_events is not None and not torch.cuda.is_current_stream_capturing():
            self.ev = (torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True))

    def __enter__(self):
        if self.ev is not None:
            self.ev[0].record()
        return self

    def __exit__(self, *exc):
        if self.ev is not None:
            self.ev[1].record()
            profile_events.setdefault(self.name, []).append(self.ev)
        return False


# "fp32" modes: tensor-core candidate generation + exact re-scoring (csrc/rescore.cu) + a per-row
# certificate; uncertified rows fall through to the next level and finally to the exact kernel, so
# every one of these modes returns bit for bit the "exact" keys.
#
# Certificate bound of a level: |approx - exact| <= err_coef * ||q|| * max||bank row||
#                                                   + err_abs * sqrt(D_pad) * (||q|| + max||bank row||)
# with err_coef = op_coef + acc_c * D_pad * 2^-23.
#
# op_coef — operand rounding, RIGOROUS (Cauchy-Schwarz on the element-wise rounding errors; checked
# element by element in tests/test_host.py::test_fp16_operand_rounding_bounds):
#   f16   : both operands rounded to fp16: 2^-10 (1 + 2^-12), + err_abs 2^-25 per element for
#           fp16's subnormal range; operands at or beyond max_abs are refused (saturation);
#   f16x2 : fp16 queries x (fp16 hi + fp16 lo) bank: 2^-11 + 2^-22 (only the query keeps 11 bits);
#   bf16  : 2^-7 (two roundings of unit roundoff 2^-8) x 1.02 for their product term;
#   bf16x3: hi + lo operands, |x - hi - lo| <= 2^-16 |x| each + the dropped lo*lo term: 3 * 2^-16;
#   tf32x3: 2^-20 (dropped lo*lo, truncated lo).
# acc_c * D_pad * 2^-23 — accumulation in the tensor core, WORST CASE under this model of
# tcgen05.mma (validated by tests/test_gpu_tc.py::test_tmem_accumulation_error_bound on all-positive
# and adversarial operands at D = 512 / 768 / 1024): the K products of one instruction (K = 16 for
# kind::f16, 8 for kind::tf32) are exact; they and the fp32 accumulator are aligned to the largest
# exponent among them, each addend loses less than one unit in the last place of that binade
# (truncation, no guard bits assumed), and the normalised result loses less than one more.  One
# instruction therefore errs by at most (K + 2) * 2^-23 * A, A = sum_i |q_i x_i| <= ||q|| ||x||,
# and a similarity is n_mma = (MMAs per k-step) * D_pad / K chained instructions:
#       acc error <= n_mma * (K + 2) * 2^-23 * ||q|| ||x||  =  acc_c * D_pad * 2^-23 * ||q|| ||x||,
#   acc_c = (MMAs per k-step) * (K + 2) / K:  f16, bf16 1.125;  f16x2 2.25;  bf16x3 3.375;  tf32x3 3.75.
# Unlike round 1's flat 2e-5 this grows with D and holds for same-sign products (the reference's
# live embeddings are non-negative: timm ResNet-18 pooled post-ReLU, knn.py:322), where truncation
# errors do not cancel: 6.9e-5 (f16) ... 2.3e-4 (tf32x3) at D = 512.
#
# residual_bound — knn_predict's certified vote (b200knn_rescore_vote) replaces op_coef's worst case by
# the rounding residuals the operands really have (DESIGN §4.1c, §5): per query
#   E = ||f16(q)|| R + rho M~ + rho R + acc_c D_pad 2^-23 ||f16(q)|| M~ + gamma_D ||q|| M,
# R = max ||x - f16(x)||, M~ = max ||f16(x)|| over the bank (PreparedRows.f16_residuals), rho =
# ||q - f16(q)||, gamma_D = D 2^-24 / (1 - D 2^-24) for the exact side's own fma chain.  Real rows use
# about half of the 2^-11 a rounding may cost, so E halves and fewer candidates are re-scored.  The
# full re-scoring of the rows the vote leaves, topk_keys and the sharded path keep op_coef.
ACC_ULP = 2.0 ** -23
LEVELS = {
    "fp32_f16": dict(cand="f16", margin=40, op_coef=1.001 * 2.0 ** -10, acc_c=1.125,
                     err_abs=1.01 * 2.0 ** -25, max_abs=6.0e4, residual_bound=True),
    "fp32_f16x2": dict(cand="f16x2", margin=40, op_coef=1.001 * (2.0 ** -11 + 2.0 ** -22), acc_c=2.25,
                       err_abs=1.01 * 2.0 ** -25, max_abs=6.0e4),
    "fp32_bf16": dict(cand="bf16", margin=128, op_coef=1.02 * 2.0 ** -7, acc_c=1.125),
    "fp32_bf16x3": dict(cand="bf16x3", margin=16, op_coef=1.001 * 3 * 2.0 ** -16, acc_c=3.375),
    "fp32_tf32": dict(cand="tf32x3", margin=8, op_coef=1.001 * 2.0 ** -20, acc_c=3.75),
}


def level_config(spec: str, dim: int) -> dict:
    """The level `spec` = "<LEVELS name>" or "<LEVELS name>@<margin>" (a wider candidate margin than
    the level's default) with the certificate's err_coef resolved for vectors of dimension `dim`."""
    name, _, margin = spec.partition("@")
    cfg = dict(LEVELS[name], name=spec)
    if margin:
        cfg["margin"] = int(margin)
    cfg["err_coef"] = cfg["op_coef"] + 1.01 * cfg["acc_c"] * padded_dim(dim) * ACC_ULP
    return cfg


# mode -> levels tried in order (then "exact").  What decides whether a row certifies is the
# candidate margin against the level's error bound E: the exact k-th similarity must beat the
# approximate (k + margin)-th by E, i.e. the row's similarities must spread by E over `margin`
# ranks.  Embeddings whose similarities are bunched (dense non-negative rows: every pair of rows is
# similar) need a wider margin, not more MMAs — re-scoring 80 more candidates costs a few percent,
# a second MMA per k-step doubles the pass.  So "fp32" runs
#   fp16 (1 MMA, margin 40 x boost)  ->  fp16 x split-fp16 (2 MMAs) with margin 160
#   ->  the same with the widest margin the lists allow (k_in = 992)  ->  exact kernel,
# where boost in {1, 2, 4} follows the fraction of rows the first level left uncertified on this
# bank (CASCADE_WIDEN / CASCADE_NARROW), and the first level is skipped for CASCADE_RETRY_CALLS
# calls if even the widest boost leaves more than CASCADE_GIVE_UP.  Vectors wider than the resident
# query tile (D_pad > 768) use the split-BF16 kernel at every level.  These statistics are
# per-process state of the single-GPU path; the sharded driver keeps its own, derived from
# all-gathered counts only, so that every rank takes the same decisions.
CASCADES = {"fp32": ("fp32_f16", "fp32_f16x2@160", "fp32_f16x2@992"), "fp32_f16": ("fp32_f16",),
            "fp32_f16x2": ("fp32_f16x2",),
            "fp32_bf16x3": ("fp32_bf16x3",),
            "fp32_bf16": ("fp32_bf16",), "fp32_tf32": ("fp32_tf32",)}
CASCADE_WIDE = ("fp32_bf16x3@64", "fp32_bf16x3@992")  # "fp32" when D_pad > MAX_BF16_DIM
CASCADE_GIVE_UP = 0.25
CASCADE_RETRY_CALLS = 64
CASCADE_WIDEN = 0.03     # more than this fraction uncertified: double the first level's margin (up to x4)
CASCADE_NARROW = 0.003   # less than this for CASCADE_CALM_CALLS calls in a row: halve it again
CASCADE_CALM_CALLS = 16
CASCADE_MAX_BOOST = 4


def next_boost(boost: int, calm: int, rows: int, uncertified: int):
    """(boost, calm) after a call that left `uncertified` of `rows` rows uncertified at the first level."""
    if rows < 128:
        return boost, calm
    frac = uncertified / rows
    if frac > CASCADE_WIDEN and boost < CASCADE_MAX_BOOST:
        return boost * 2, 0
    if frac < CASCADE_NARROW and boost > 1:
        return (boost // 2, 0) if calm + 1 >= CASCADE_CALM_CALLS else (boost, calm + 1)
    return boost, 0


# first level of each mode (bench / docs)
RESCORED_MODES = {m: LEVELS[c[0].partition("@")[0]] for m, c in CASCADES.items()}
ALL_MODES = tuple(_lib.MODES) + tuple(RESCORED_MODES)

# statistics of the last rescored call (bench / tests): rows that failed the certificate
last_rescore_stats = {"rows": 0, "uncertified": 0, "level": None, "levels": []}


def set_default_mode(mode: str) -> None:
    """Select the similarity mode ``knn_predict``/``knn_topk`` use when none is passed.

    ``"exact"``     fp32 CUDA-core contraction, sequential-fma similarities (bitwise reproducible);
    ``"fp32"``      tensor-core candidates + exact re-scoring + certificate, cascading fp16 (1 MMA per
                    k-step, k + 40..160 candidates, the margin following how bunched the bank's
                    similarities are) -> fp16 x split-fp16 (2 MMAs, k + 160) -> the same with the widest
                    margin the lists allow (k_in = 992) -> exact, for the rows each level cannot certify:
                    bitwise the ``"exact"`` result at tensor-core speed (the fp32-matching mode);
    ``"fp32_f16"`` / ``"fp32_f16x2"`` / ``"fp32_bf16x3"`` / ``"fp32_tf32"`` / ``"fp32_bf16"``  a single level
                    (then exact);
    ``"f16"``       raw tcgen05 fp16 similarities (2^-10 relative to ||q|| ||x||; BF16 mode's speed);
    ``"f16x2"``     raw tcgen05 fp16 x (fp16 hi + lo) similarities (~2.5e-4 relative to ||q|| ||x||);
    ``"bf16x3"``    raw tcgen05 bf16 hi/lo-split similarities (~1e-5 relative);
    ``"tf32x3"``    raw tcgen05 hi/lo-split TF32 similarities (fp32-class accuracy, ~1e-6);
    ``"bf16"``      raw tcgen05 BF16 operands / fp32 accumulate (fastest; recall@k reported by bench).
    """
    global _default_mode
    if mode not in ALL_MODES:
        raise ValueError(f"unknown mode {mode!r}; expected one of {sorted(ALL_MODES)}")
    _default_mode = mode


def get_default_mode() -> str:
    return _default_mode


def _stream() -> int:
    return torch.cuda.current_stream().cuda_stream


def _ptr(t: Optional[torch.Tensor]) -> Optional[int]:
    return None if t is None else t.data_ptr()


def _require_cuda(name: str, t: torch.Tensor) -> None:
    if not isinstance(t, torch.Tensor):
        raise TypeError(f"{name} must be a torch.Tensor, got {type(t).__name__}")
    if not t.is_cuda:
        raise RuntimeError(
            f"b200knn: {name} is on {t.device}; this path runs on sm_100a CUDA tensors only "
            "(no CPU fallback by design)"
        )


def padded_dim(dim: int) -> int:
    return (dim + 63) // 64 * 64


def effective_mode(mode: str, dim: int) -> str:
    """The kernel mode a raw tensor-core mode runs as for vectors of dimension `dim`: bf16 / f16 /
    f16x2 keep a 128-row query tile resident in shared memory (D_pad * 256 B), so wider vectors
    go through the split-BF16 kernel, which streams both operands (and is more accurate)."""
    if mode in ("bf16", "f16x2", "f16") and padded_dim(dim) > MAX_BF16_DIM:
        return "bf16x3"
    return mode


# ----------------------------------------------------------------------------
# operand preparation (+ cache for the bank, which the reference rebuilds once
# per validation epoch and then reuses for every validation step, knn.py:67-98)
# ----------------------------------------------------------------------------
class PreparedRows:
    """K-major rows in the layout the tensor-core kernel streams with TMA."""

    __slots__ = ("mode", "n", "dim", "hi", "lo", "_f32", "_max_norm", "_f16_resid", "_src", "_delegate")

    def __init__(self, mode: str, n: int, dim: int, hi: torch.Tensor, lo: Optional[torch.Tensor]):
        self.mode, self.n, self.dim, self.hi, self.lo = mode, n, dim, hi, lo
        self._f32 = None       # (n, dim_pad) fp32 shadow rows for the exact re-scoring (bf16 candidates)
        self._max_norm = None  # device scalar: max row norm (certificate)
        self._f16_resid = None  # device [R, M~]: fp16 residual statistics (certified vote)
        self._src = None       # (tensor, vectors_are_columns) to build the shadow lazily
        self._delegate = None  # another preparation of the same bank that owns the shadow rows / norm

    def rescore_rows(self):
        """(rows_a, rows_b) fp32 row-major operands whose sum is the caller's exact value."""
        if self._delegate is not None:
            return self._delegate.rescore_rows()
        if self.mode == "tf32x3":  # hi + lo is exactly the caller's fp32 value
            return self.hi, self.lo
        if self._f32 is None:
            src, cols = self._src
            # a FeatureBank already holds its rows as zero-padded (N, D_pad) fp32: no second copy
            own = _padded_rows.get((src.data_ptr(), tuple(src.shape), tuple(src.stride())))
            own = own() if own is not None else None
            self._f32 = own if own is not None else prepare_rows(src, "f32rows", cols).hi
        return self._f32, None

    def max_norm(self) -> torch.Tensor:
        if self._delegate is not None:
            return self._delegate.max_norm()
        if self._max_norm is None:
            a, b = self.rescore_rows()
            out = torch.zeros((1,), dtype=torch.float32, device=a.device)
            with torch.cuda.device(a.device):
                _lib.check(_lib.load().b200knn_row_norm_max(a.data_ptr(), _ptr(b), self.n, a.shape[1],
                                                            out.data_ptr(), _stream()), "row_norm_max")
            self._max_norm = out
        return self._max_norm

    def f16_residuals(self) -> torch.Tensor:
        """Device float32[2]: max ||x - f16(x)|| and max ||f16(x)|| over the rows, f16 the rounding of
        the fp16 candidate pass.  Computed once and kept as long as the preparation: captured call
        graphs read it by pointer."""
        if self._delegate is not None:
            return self._delegate.f16_residuals()
        if self._f16_resid is None:
            a, b = self.rescore_rows()
            if b is not None:
                raise RuntimeError("f16_residuals needs one fp32 row array")
            out = torch.zeros((2,), dtype=torch.float32, device=a.device)
            with torch.cuda.device(a.device):
                _lib.check(_lib.load().b200knn_row_f16_residual_max(a.data_ptr(), self.n, a.shape[1], out.data_ptr(),
                                                                    _stream()), "row_f16_residual_max")
            self._f16_resid = out
        return self._f16_resid


# (D,N) bank views backed by zero-padded (N, D_pad) fp32 rows (b200knn.bank.FeatureBank)
_padded_rows = {}


def register_padded_rows(bank_view: torch.Tensor, rows_padded: torch.Tensor) -> None:
    if len(_padded_rows) > 64:
        for key in [k for k, ref in _padded_rows.items() if ref() is None]:
            _padded_rows.pop(key)
    _padded_rows[(bank_view.data_ptr(), tuple(bank_view.shape), tuple(bank_view.stride()))] = weakref.ref(rows_padded)


def normalize_rows(x: torch.Tensor, eps: float = 1e-12, out: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``F.normalize(x, dim=1)`` of (n, D) rows (reference ``knn.py:77`` / ``:90``) into zero-padded
    fp32 rows; returns the (n, D) view of the (n, D_pad) result.  fp64 norm in a fixed order.
    out: optional contiguous (n, D_pad) fp32 destination (a slice of a preallocated bank)."""
    _require_cuda("x", x)
    if x.dim() != 2:
        raise RuntimeError("normalize_rows expects (n, D) row vectors")
    if x.dtype not in _DTYPES:
        x = x.float()
    if x.stride(1) != 1:
        x = x.contiguous()
    n, dim = x.shape
    if out is None:
        out = torch.empty((n, padded_dim(dim)), dtype=torch.float32, device=x.device)
    elif out.shape != (n, padded_dim(dim)) or out.dtype != torch.float32 or not out.is_contiguous() \
            or out.device != x.device:
        raise ValueError("out must be a contiguous (n, padded_dim(D)) fp32 tensor on the rows' device")
    if n:
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().b200knn_normalize_rows(x.data_ptr(), _DTYPES[x.dtype], n, dim, x.stride(0),
                                                          float(eps), out.data_ptr(), _stream()), "normalize_rows")
    return out[:, :dim]


def row_sqnorms(x: torch.Tensor) -> torch.Tensor:
    """(n,) fp32 squared L2 norms of (n, D) rows, fp64 accumulation in a fixed order."""
    _require_cuda("x", x)
    if x.dtype not in _DTYPES:
        x = x.float()
    if x.stride(1) != 1:
        x = x.contiguous()
    n, dim = x.shape
    out = torch.empty((n,), dtype=torch.float32, device=x.device)
    if n:
        with torch.cuda.device(x.device):
            _lib.check(_lib.load().b200knn_row_sqnorms(x.data_ptr(), _DTYPES[x.dtype], n, dim, x.stride(0),
                                                       out.data_ptr(), _stream()), "row_sqnorms")
    return out


def _layout_of(x: torch.Tensor, vectors_are_columns: bool) -> Tuple[torch.Tensor, int, int]:
    """Return (tensor, layout, ld) describing n vectors of dimension dim without copying
    when the strides allow it.  vectors_are_columns: x is (D, N) (bank); else (N, D)."""
    if vectors_are_columns:
        if x.stride(1) == 1 and x.stride(0) >= max(1, x.shape[1]):
            return x, _lib.LAYOUT_DN, x.stride(0)
        if x.stride(0) == 1 and x.stride(1) >= max(1, x.shape[0]):  # a .t() view of an (N, D) tensor
            return x, _lib.LAYOUT_ND, x.stride(1)
        x = x.contiguous()
        return x, _lib.LAYOUT_DN, x.stride(0)
    if x.stride(1) == 1 and x.stride(0) >= max(1, x.shape[1]):
        return x, _lib.LAYOUT_ND, x.stride(0)
    if x.stride(0) == 1 and x.stride(1) >= max(1, x.shape[0]):
        return x, _lib.LAYOUT_DN, x.stride(1)
    x = x.contiguous()
    return x, _lib.LAYOUT_ND, x.stride(0)


def prepare_rows(x: torch.Tensor, mode: str, vectors_are_columns: bool) -> PreparedRows:
    lib = _lib.load()
    if x.dtype not in _DTYPES:
        x = x.float()
    n, dim = (x.shape[1], x.shape[0]) if vectors_are_columns else (x.shape[0], x.shape[1])
    x, layout, ld = _layout_of(x, vectors_are_columns)
    dpad = padded_dim(dim)
    if mode == "bf16":
        hi = torch.empty((n, dpad), dtype=torch.bfloat16, device=x.device)
        lo = None
    elif mode == "tf32x3":
        hi = torch.empty((n, dpad), dtype=torch.float32, device=x.device)
        lo = torch.empty((n, dpad), dtype=torch.float32, device=x.device)
    elif mode == "bf16x3":
        hi = torch.empty((n, dpad), dtype=torch.bfloat16, device=x.device)
        lo = torch.empty((n, dpad), dtype=torch.bfloat16, device=x.device)
    elif mode == "f16":
        hi = torch.empty((n, dpad), dtype=torch.float16, device=x.device)
        lo = None
    elif mode == "f16x2":  # queries: one fp16 array; bank: hi + lo
        hi = torch.empty((n, dpad), dtype=torch.float16, device=x.device)
        lo = torch.empty((n, dpad), dtype=torch.float16, device=x.device) if vectors_are_columns else None
    elif mode == "f32rows":
        hi = torch.empty((n, dpad), dtype=torch.float32, device=x.device)
        lo = None
    else:
        raise ValueError(f"mode {mode!r} takes caller tensors directly")
    code = _lib.MODE_F32ROWS if mode == "f32rows" else _lib.MODES[mode]
    if n > 0:
        with torch.cuda.device(x.device):
            _lib.check(
                lib.b200knn_prepare_rows(x.data_ptr(), _DTYPES[x.dtype], layout, n, dim, ld,
                                         code, hi.data_ptr(), _ptr(lo), _stream()),
                "prepare_rows",
            )
    prep = PreparedRows(mode, n, dim, hi, lo)
    prep._src = (x, vectors_are_columns)
    return prep


class _BankCache:
    """Prepared banks keyed on the identity *and version* of the caller's tensor, so an
    in-place update or a rebuilt bank (new validation epoch) is re-prepared."""

    def __init__(self, capacity: int = 6):
        self.capacity = capacity
        self._entries = {}
        self._state = {}

    def get(self, bank: torch.Tensor, mode: str) -> PreparedRows:
        key = (bank.data_ptr(), bank._version, tuple(bank.shape), tuple(bank.stride()), bank.dtype,
               bank.device.index, mode)
        hit = self._entries.get(key)
        if hit is not None and hit[0]() is not None:
            return hit[1]
        # the reference rebuilds its bank every validation epoch (knn.py:80): drop the prepared
        # copies (several GB at 811k x 512) of banks that no longer exist before preparing a new one
        for dead in [k_ for k_, v in self._entries.items() if v[0]() is None]:
            self._entries.pop(dead)
        if mode == "f16":
            # fp16(x) is the hi array of the f16x2 split (the next cascade level): share it
            both = self.get(bank, "f16x2")
            prep = PreparedRows("f16", both.n, both.dim, both.hi, None)
            prep._src, prep._delegate = both._src, both
        else:
            prep = prepare_rows(bank, mode, vectors_are_columns=True)
        if len(self._entries) >= self.capacity:
            self._entries.pop(next(iter(self._entries)))
        try:
            ref = weakref.ref(bank)
        except TypeError:  # pragma: no cover
            ref = lambda: bank  # noqa: E731
        self._entries[key] = (ref, prep)
        return prep

    def state(self, bank: torch.Tensor) -> dict:
        """Mutable per-bank notes (cascade statistics), dropped with the bank's cache entries."""
        key = (bank.data_ptr(), bank._version, tuple(bank.shape))
        st = self._state.get(key)
        if st is None:
            if len(self._state) >= 4 * self.capacity:
                self._state.pop(next(iter(self._state)))
            st = self._state[key] = {}
        return st

    def clear(self) -> None:
        self._entries.clear()
        self._state.clear()


bank_cache = _BankCache()


class _QueryCache:
    """The prepared copy of the last query batch (used twice per call: pre-pass and main pass)."""

    def __init__(self):
        self._key = None
        self._val = None

    def get(self, feature: torch.Tensor, mode: str) -> PreparedRows:
        key = (feature.data_ptr(), feature._version, tuple(feature.shape), tuple(feature.stride()),
               feature.dtype, feature.device.index, mode)
        if key != self._key or self._val is None or self._val[0]() is None:
            prep = prepare_rows(feature, mode, vectors_are_columns=False)
            self._key, self._val = key, (weakref.ref(feature), prep)
        return self._val[1]

    def clear(self) -> None:
        self._key = self._val = None


query_cache = _QueryCache()


# ----------------------------------------------------------------------------
# selection keys
# ----------------------------------------------------------------------------
def _check_feature_bank(feature: torch.Tensor, feature_bank: torch.Tensor) -> None:
    _require_cuda("feature", feature)
    _require_cuda("feature_bank", feature_bank)
    if feature.device != feature_bank.device:
        raise RuntimeError("Expected all tensors to be on the same device, but found "
                           f"{feature.device} and {feature_bank.device}")
    if feature.dim() != 2:
        raise RuntimeError("self must be a matrix")  # torch.mm's message (knn.py:89 .squeeze() hazard)
    if feature_bank.dim() != 2:
        raise RuntimeError("mat2 must be a matrix")
    if feature.shape[1] != feature_bank.shape[0]:
        raise RuntimeError(
            f"mat1 and mat2 shapes cannot be multiplied ({feature.shape[0]}x{feature.shape[1]} and "
            f"{feature_bank.shape[0]}x{feature_bank.shape[1]})"
        )


# Sampling pre-pass (tensor-core modes): the r-th best similarity of every s-th bank row is,
# except with probability P[Binomial(k, 1/s) >= r] (2e-7 for the defaults), below the true k-th
# best, so it is a valid starting threshold for the streaming selection.  It removes the list
# warm-up (the first ~k*ln(N/k) insertions), which is what a (query tile, bank shard) work item
# otherwise pays as a fixed cost; rows where the bound fails end with an empty k-th slot and are
# recomputed without it.
PREPASS = {"enabled": os.environ.get("B200KNN_PREPASS", "1") == "1", "r": 16, "rank_factor": 5.0,
           "min_k": 64, "min_sample_rows": 1024, "small_batch": 512,
           # r == 16: use the values-only kernel variant (row top-16 in registers) for the sample
           "register_sample": os.environ.get("B200KNN_REGISTER_SAMPLE", "1") == "1"}


def prepass_stride(n_rows: int, k: int, batch: Optional[int] = None) -> int:
    """Row stride of the sampling pre-pass, or 0 when it does not pay.  Large batches: only for
    k >= min_k (short lists warm up quickly).  Small batches (the reference-shaped B = 64 call) are
    planned with one bank split per SM, every split pays the list warm-up and its merge handles
    `splits` lists per row: there the threshold pays for any k (measured at N = 37,348, k = 5+40:
    125 us of warm-up prunes + 60 us of merge without it)."""
    if not PREPASS["enabled"]:
        return 0
    if k < PREPASS["min_k"] and (batch is None or batch > PREPASS["small_batch"]):
        return 0
    s = max(8, min(256, int(round(PREPASS["rank_factor"] * k / PREPASS["r"]))))
    return s if n_rows // s >= PREPASS["min_sample_rows"] else 0


def _search(mode, q, bank, B, n_visit, D, k, idx_offset=0, *, stride=1, tau0=None, upper=None, groups=None,
            sample=False, peers=None, out=None, timed=False) -> Optional[torch.Tensor]:
    """One b200knn_topk_opt call: the (B, k) keys of queries q among n_visit bank rows.
    q, bank: the caller tensors of ``_exact_operands`` in mode "exact", PreparedRows otherwise.
    Options (include/b200knn.h): row stride, (B,) thresholds tau0, (B,) peeling bound `upper`,
    groups = (query ids, bank ids, ...), the values-only sample, and peers = (device pointers,
    rank, rows_per_owner), which stores the keys into the peers' buffers and returns None."""
    lib = _lib.load()
    if mode == "exact":
        bank, layout, ld = bank
        args = (q.data_ptr(), None, _DTYPES[q.dtype], q.stride(0), bank.data_ptr(), None, _DTYPES[bank.dtype],
                layout, ld)
        dev = q.device
    else:
        args = (q.hi.data_ptr(), _ptr(q.lo), 0, 0, bank.hi.data_ptr(), _ptr(bank.lo), 0, 0, 0)
        dev = q.hi.device
    opts = _lib.TopkOptions(bank_row_stride=stride, tau0=_ptr(tau0), upper_keys=_ptr(upper), sample=sample)
    if groups is not None:
        opts.q_groups, opts.bank_groups = groups[0].data_ptr(), groups[1].data_ptr()
    keys = None
    if peers is not None:
        ptrs, opts.my_rank, opts.rows_per_owner = peers
        opts.host_peer_out, opts.n_peers = _ptr_array(ptrs), len(ptrs)
    elif out is not None:
        assert out.shape == (B, k) and out.dtype == torch.int64 and out.is_contiguous()
        keys = out
    else:
        keys = torch.empty((B, k), dtype=torch.int64, device=dev)
    ws_bytes = lib.b200knn_topk_workspace_bytes(B, n_visit, D, k, _lib.MODES[mode])
    if ws_bytes == 0:
        raise RuntimeError(f"b200knn: unsupported problem (B={B}, N={n_visit}, D={D}, k={k})")
    ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
    with _Timed("topk", timed):
        rc = lib.b200knn_topk_opt(_lib.MODES[mode], *args, B, n_visit, D, k, idx_offset, _ptr(keys), ws.data_ptr(),
                                  ws_bytes, opts, _stream())
    _lib.check(rc, "topk")
    return keys


def _exact_operands(feature: torch.Tensor, feature_bank: torch.Tensor):
    """(q, (bank, layout, ld)): the caller tensors as MODE_EXACT reads them, copied only when needed."""
    q = feature if feature.dtype in _DTYPES else feature.float()
    if q.stride(1) != 1:
        q = q.contiguous()
    bank = feature_bank if feature_bank.dtype in _DTYPES else feature_bank.float()
    return q, _layout_of(bank, vectors_are_columns=True)


def kth_sim(keys: torch.Tensor) -> torch.Tensor:
    """Similarity of the last key of every row (-inf for an empty slot): a (B,) fp32 tensor."""
    B, k = keys.shape
    out = torch.empty((B,), dtype=torch.float32, device=keys.device)
    if B:
        keys = keys.contiguous()
        with torch.cuda.device(keys.device):
            _lib.check(_lib.load().b200knn_key_sim_column(keys.data_ptr(), B, k, k - 1, out.data_ptr(),
                                                          _stream()), "key_sim_column")
    return out


def vote_packed(keys: torch.Tensor, feature_labels: torch.Tensor, num_classes: int, knn_t: float,
                n_rows_out: int) -> torch.Tensor:
    """(n_rows_out, C+1) int64: class rankings of keys' rows in columns [0,C) and the per-row
    status word of b200knn_vote_ex in column C; rows past keys.shape[0] are zero."""
    lib = _lib.load()
    B, k = keys.shape
    C = int(num_classes)
    check_vote_classes(C, k)
    labels = feature_labels if feature_labels.dtype == torch.int64 else feature_labels.long()
    labels = labels.contiguous().view(-1)
    dev = keys.device
    out = torch.zeros((n_rows_out, C + 1), dtype=torch.int64, device=dev) if n_rows_out > B \
        else torch.empty((n_rows_out, C + 1), dtype=torch.int64, device=dev)
    if B:
        with torch.cuda.device(dev):
            flag = torch.zeros((1,), dtype=torch.int32, device=dev)
            _lib.check(lib.b200knn_vote_ex(keys.data_ptr(), labels.data_ptr(), B, k, labels.numel(), 0, C,
                                           float(knn_t), out.data_ptr(), C + 1, C, None, flag.data_ptr(),
                                           _stream()), "vote_ex")
    return out


def sample_keys(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: str,
                n_rows_for_decision: Optional[int] = None) -> Optional[torch.Tensor]:
    """Pre-pass: (B, r) best keys among every s-th bank row, or None when the pre-pass is off."""
    N = feature_bank.shape[1]
    B, D = feature.shape
    s = prepass_stride(n_rows_for_decision if n_rows_for_decision is not None else N, k, B)
    if s == 0 or mode not in TC_MODES:
        return None
    mode = effective_mode(mode, D)
    r = PREPASS["r"]
    n_visit = (N + s - 1) // s
    if n_visit < r:
        return None
    with torch.cuda.device(feature.device):
        pb = bank_cache.get(feature_bank, mode)
        pq = query_cache.get(feature, mode)
        return _search(mode, pq, pb, B, n_visit, D, r, stride=s,
                       sample=(r == _lib.SAMPLE_R and PREPASS["register_sample"]))


def sample_scatter_supported(B: int, n_rows: int, D: int, k: int, mode: str, n_rows_for_decision: int) -> bool:
    """Whether sample_scatter applies to a shard of n_rows rows (pre-pass on, sample planned without splits)."""
    s = prepass_stride(n_rows_for_decision, k, B)
    if s == 0 or mode not in TC_MODES or PREPASS["r"] != _lib.SAMPLE_R or not PREPASS["register_sample"]:
        return False
    n_visit = (n_rows + s - 1) // s
    if n_visit < PREPASS["r"]:
        return False
    try:
        return plan_info(B, n_visit, D, PREPASS["r"], effective_mode(mode, D))["splits"] == 1
    except RuntimeError:
        return False


def sample_scatter(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: str, n_rows_for_decision: int,
                   peer_ptrs, rank: int, rows_per_owner: int) -> None:
    """sample_keys whose (B, 16) sample of query row b is stored straight into the exchange buffer of
    the GPU that owns b (the sharded threshold exchange over NVLink peer memory)."""
    N = feature_bank.shape[1]
    B, D = feature.shape
    s = prepass_stride(n_rows_for_decision, k, B)
    mode = effective_mode(mode, D)
    n_visit = (N + s - 1) // s
    with torch.cuda.device(feature.device):
        pb = bank_cache.get(feature_bank, mode)
        pq = query_cache.get(feature, mode)
        _search(mode, pq, pb, B, n_visit, D, PREPASS["r"], stride=s, sample=True,
                peers=(peer_ptrs, rank, rows_per_owner))


def broadcast_f32(src: torch.Tensor, peer_ptrs, dst_offset: int) -> None:
    """dst[g][dst_offset + i] = src[i] on every peer g (device pointers of every rank's fp32 buffer)."""
    src = src.contiguous()
    assert src.dtype == torch.float32
    if src.numel():
        with torch.cuda.device(src.device):
            _lib.check(_lib.load().b200knn_broadcast_f32(src.data_ptr(), src.numel(), _ptr_array(peer_ptrs),
                                                         len(peer_ptrs), dst_offset, _stream()), "broadcast_f32")


def _exclusion(exclude, B: int, N: int, device: torch.device):
    """``topk_keys``' exclude argument -> (query ids (B,) int32, bank ids (N,) int32, m) with m the
    largest number of bank rows that share one query row's id.  A 3-tuple is taken as already
    checked (the internal form: callers that know m pass it and save the host read here)."""
    if len(exclude) == 3:
        return exclude
    qg, bg = exclude
    for name, t, n in (("query group ids", qg, B), ("bank group ids", bg, N)):
        if not isinstance(t, torch.Tensor) or t.dtype != torch.int32:
            raise ValueError(f"{name} must be an int32 tensor of dense ids")
        if t.numel() != n:
            raise RuntimeError(f"{name} have {t.numel()} entries for {n} rows")
        if t.device != device:
            raise RuntimeError(f"Expected all tensors to be on the same device, but found {device} and {t.device}")
    qg, bg = qg.contiguous().view(-1), bg.contiguous().view(-1)
    m = 0
    if B and N:
        n_ids = max(int(qg.max()), int(bg.max())) + 1
        m = int(torch.bincount(bg, minlength=n_ids)[qg.long()].max())
    return qg, bg, m


def topk_keys(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: Optional[str] = None,
              idx_offset: int = 0, tau0: Optional[torch.Tensor] = None, repair: bool = True,
              out: Optional[torch.Tensor] = None, exclude=None) -> torch.Tensor:
    """(B,k) selection keys (uint64 bit patterns in an int64 tensor), sorted descending under
    the canonical (sim desc, bank index asc) order; bank indices are offset by idx_offset.

    tau0 (tensor-core modes): caller-supplied (B,) admission thresholds — then no pre-pass and
    no validation happen here and rows may come back with empty (0) slots (sharded driver).
    repair=False (tensor-core modes): skip the host-synchronising check for rows the sampled
    threshold starved (empty k-th slot); the caller detects and repairs them (``repair_rows``).
    exclude: optional (query_gids (B,), bank_gids (N,)), dense non-negative int32 ids on the device:
    bank row n is left out of query row b's search when bank_gids[n] == query_gids[b], in every mode
    and path (no sampling pre-pass then).  Keys keep the full bank's indices; k must not exceed
    N minus the largest number of bank rows sharing one query row's id."""
    _lib.load()
    mode = mode or _default_mode
    if mode not in _lib.MODES and mode not in RESCORED_MODES:
        raise ValueError(f"unknown mode {mode!r}")
    if exclude is not None:
        _check_feature_bank(feature, feature_bank)
        if tau0 is not None:
            raise ValueError("topk_keys: exclude runs without an admission threshold (tau0)")
        exclude = _exclusion(exclude, feature.shape[0], feature_bank.shape[1], feature.device)
        if int(k) > feature_bank.shape[1] - exclude[2]:
            raise RuntimeError("selected index k out of range")
    if int(k) > MAX_K:
        # Tensor.topk takes any k <= N; the streaming lists hold MAX_K keys.  Larger k is served by
        # the exact kernel in passes of <= MAX_K (a completeness path, whatever the mode).
        _check_feature_bank(feature, feature_bank)
        return _topk_keys_exact(feature, feature_bank, int(k), idx_offset, exclude)
    if mode in RESCORED_MODES:
        return _topk_keys_rescored(feature, feature_bank, k, mode, idx_offset, exclude=exclude)
    _check_feature_bank(feature, feature_bank)
    B, D = feature.shape
    mode = effective_mode(mode, D)
    N = feature_bank.shape[1]
    k = int(k)
    if k <= 0 or k > N:
        raise RuntimeError("selected index k out of range")  # Tensor.topk's message
    dev = feature.device
    with torch.cuda.device(dev):
        if B == 0:
            return torch.empty((B, k), dtype=torch.int64, device=dev)
        if mode == "exact":
            return _topk_keys_exact(feature, feature_bank, k, idx_offset, exclude)
        pb = bank_cache.get(feature_bank, mode)
        pq = query_cache.get(feature, mode)
        if exclude is not None:
            # no sampling pre-pass: a threshold sampled from the whole bank may come from the row's
            # own group and would starve the row
            return _search(mode, pq, pb, B, N, D, k, idx_offset, groups=exclude, timed=True)
        if tau0 is not None:  # `out`: write the keys straight into a caller buffer (sharded exchange)
            return _search(mode, pq, pb, B, N, D, k, idx_offset, tau0=tau0.contiguous(), out=out, timed=True)
        sk = sample_keys(feature, feature_bank, k, mode)
        if sk is None:
            return _search(mode, pq, pb, B, N, D, k, idx_offset, timed=True)
        keys = _search(mode, pq, pb, B, N, D, k, idx_offset, tau0=kth_sim(sk), timed=True)
        if not repair:
            return keys
        return _repair_rows(keys, lambda rows: _search(mode, _rows_of(pq, rows), pb, rows.numel(), N, D, k,
                                                       idx_offset))


def _topk_keys_exact(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, idx_offset: int,
                     exclude=None) -> torch.Tensor:
    """MODE_EXACT keys, with ``topk_keys``' checked exclusion.  Tensor.topk takes any k <= N and the
    streaming lists hold MAX_K keys: pass i selects the best min(MAX_K, remaining) keys strictly
    below the last key of pass i-1, so k <= MAX_K is one pass without a bound and larger k takes
    ceil(k / MAX_K) scans of the bank."""
    B, D = feature.shape
    N = feature_bank.shape[1]
    if k > N:
        raise RuntimeError("selected index k out of range")
    dev = feature.device
    keys = torch.empty((B, k), dtype=torch.int64, device=dev)
    if B == 0:
        return keys
    q, bank = _exact_operands(feature, feature_bank)
    upper = None
    done = 0
    with torch.cuda.device(dev):
        while done < k:
            kp = min(MAX_K, k - done)
            if kp == k:  # one pass: straight into keys, recorded as the "topk" event
                return _search("exact", q, bank, B, N, D, k, idx_offset, groups=exclude, out=keys, timed=True)
            part = _search("exact", q, bank, B, N, D, kp, idx_offset, upper=upper, groups=exclude)
            keys[:, done:done + kp] = part
            upper = part[:, -1].contiguous()
            done += kp
    return keys


def topk_scatter(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: str, idx_offset: int,
                 tau0: Optional[torch.Tensor], peer_ptrs, rank: int, rows_per_owner: int) -> bool:
    """Fused top-k + exchange (b200knn_topk_opt with peers): this shard's keys of query row b are stored
    into peer_ptrs[b // rows_per_owner] (device pointers of every rank's (G, rows_per_owner, k)
    exchange buffer, mapped in this process).  Returns False when the problem is planned with
    bank splits (caller falls back to the NCCL exchange)."""
    if mode not in TC_MODES:
        return False
    _check_feature_bank(feature, feature_bank)
    B, D = feature.shape
    mode = effective_mode(mode, D)
    N = feature_bank.shape[1]
    if B == 0 or k <= 0 or k > N or len(peer_ptrs) > 8:
        return False
    if plan_info(B, N, D, k, mode)["splits"] != 1:
        return False
    with torch.cuda.device(feature.device):
        pb = bank_cache.get(feature_bank, mode)
        pq = query_cache.get(feature, mode)
        _search(mode, pq, pb, B, N, D, k, idx_offset, tau0=None if tau0 is None else tau0.contiguous(),
                peers=(peer_ptrs, rank, rows_per_owner), timed=True)
    return True


def recompute_rows(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: str, rows: torch.Tensor,
                   idx_offset: int = 0, exclude=None) -> torch.Tensor:
    """Keys of the given query rows computed without any admission threshold."""
    sub = feature[rows].contiguous()
    if exclude is not None:
        exclude = _exclusion(exclude, feature.shape[0], feature_bank.shape[1], feature.device)
        return topk_keys(sub, feature_bank, k, "exact" if mode in RESCORED_MODES else mode, idx_offset,
                         exclude=(exclude[0][rows], exclude[1], exclude[2]))
    if mode == "exact" or mode in RESCORED_MODES:
        return topk_keys(sub, feature_bank, k, "exact", idx_offset)
    B, D = sub.shape
    mode = effective_mode(mode, D)
    with torch.cuda.device(feature.device):
        pb = bank_cache.get(feature_bank, mode)
        pq = prepare_rows(sub, mode, vectors_are_columns=False)
        return _search(mode, pq, pb, B, feature_bank.shape[1], D, k, idx_offset)


def _rows_of(pq: "PreparedRows", rows: torch.Tensor) -> "PreparedRows":
    return PreparedRows(pq.mode, rows.numel(), pq.dim, pq.hi[rows].contiguous(),
                        None if pq.lo is None else pq.lo[rows].contiguous())


def _repair_rows(keys: torch.Tensor, recompute) -> torch.Tensor:
    """Rows whose k-th slot is empty were selected under a threshold that was too high (the
    ~1e-7 tail of the sampling pre-pass): recompute them without a threshold."""
    bad = keys[:, -1] == 0
    last_prepass_stats["rows"] = keys.shape[0]
    n_bad = int(bad.sum().item())
    last_prepass_stats["repaired"] = n_bad
    if n_bad:
        rows = bad.nonzero(as_tuple=False).view(-1)
        keys[rows] = recompute(rows)
    return keys


last_prepass_stats = {"rows": 0, "repaired": 0}


def _rescored_level(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, level: str, idx_offset: int,
                    n_bad: Optional[torch.Tensor] = None, exclude=None):
    """One cascade level, nothing synchronises: (keys (B,k), uncertified flags (B,) int32, count int32[1]).
    n_bad: optional zeroed int32[1] the count is accumulated into (the caller's status word).
    exclude: ``topk_keys``' checked (query ids, bank ids, m) for these rows."""
    B, D = feature.shape
    cfg = level_config(level, D)
    N = feature_bank.shape[1]
    # the streaming lists hold at most MAX_K keys: near that limit the margin shrinks (and with it
    # the chance to certify; uncertified rows still end up exact through the next level)
    k_in = min(N, k + cfg["margin"], max(k, MAX_K))
    if exclude is not None:
        # every row keeps at least k_in eligible bank rows, so no candidate slot stays empty (the
        # re-scoring kernel would read an empty k_in-th slot as uncertified).  The certificate's
        # max row norm of the whole bank still bounds the reduced bank's.
        k_in = min(k_in, N - exclude[2])
    # no repair pass on the candidates: a row its sampled threshold starved has an empty k_in-th
    # slot, which the re-scoring kernel reports as uncertified
    cand = topk_keys(feature, feature_bank, k_in, cfg["cand"], idx_offset, repair=False, exclude=exclude)
    return _rescore_candidates(feature, feature_bank, cand, k, cfg, idx_offset, n_bad)


def _rescore_candidates(feature: torch.Tensor, feature_bank: torch.Tensor, cand: torch.Tensor, k: int, cfg: dict,
                        idx_offset: int, n_bad: Optional[torch.Tensor] = None):
    """The re-scoring and certificate of a level on its candidates cand (B, k_in): ``_rescored_level``'s result."""
    lib = _lib.load()
    B, D = feature.shape
    N = feature_bank.shape[1]
    k_in = cand.shape[1]
    dev = feature.device
    pb = bank_cache.get(feature_bank, cfg["cand"])
    rows_a, rows_b = pb.rescore_rows()
    max_norm = pb.max_norm()
    # fp32 queries select the TMA-pipelined re-scoring kernels (fp16/bf16 -> fp32 is exact)
    q = feature if feature.dtype == torch.float32 else feature.float()
    if q.stride(1) != 1:
        q = q.contiguous()
    out = torch.empty((B, k), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        flags = torch.empty((B,), dtype=torch.int32, device=dev)
        if n_bad is None:
            n_bad = torch.zeros((1,), dtype=torch.int32, device=dev)
        ws_bytes = int(lib.b200knn_rescore_workspace_bytes(B, k_in)) if rows_b is None else 0
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
        with _Timed("rescore"):
            rc = lib.b200knn_rescore(q.data_ptr(), _DTYPES[q.dtype], q.stride(0), rows_a.data_ptr(),
                                     _ptr(rows_b), N, D, cand.data_ptr(), B, k_in, k, idx_offset,
                                     float(cfg["err_coef"]), float(cfg.get("err_abs", 0.0)) * math.sqrt(padded_dim(D)),
                                     float(cfg.get("max_abs", 0.0)), max_norm.data_ptr(), out.data_ptr(),
                                     flags.data_ptr(), n_bad.data_ptr(), _ptr(ws), ws_bytes, _stream())
        _lib.check(rc, "rescore")
    return out, flags, n_bad


# ---- pieces of the sharded fp32 mode (b200knn/sharded.py): candidates are merged by the owner of
# a query, re-scored by the shard that owns each candidate's bank row, merged again and certified
def cascade_levels(feature_bank: torch.Tensor, mode: str, boost: int = 1) -> list:
    """The candidate levels a rescored mode tries in order on this bank (LEVELS entries + names)."""
    return [level_config(name, feature_bank.shape[0])
            for name in _cascade_levels(feature_bank, mode, track=False, boost=boost)]


def route_keys(keys: torch.Tensor, rows_per_shard: int, n_shards: int) -> torch.Tensor:
    """(n, k) keys -> (n_shards, n, k): block g keeps the keys whose bank row shard g owns."""
    n, k = keys.shape
    out = torch.empty((n_shards, n, k), dtype=torch.int64, device=keys.device)
    if n:
        keys = keys.contiguous()
        with torch.cuda.device(keys.device):
            _lib.check(_lib.load().b200knn_route_keys(keys.data_ptr(), n, k, rows_per_shard, n_shards,
                                                      out.data_ptr(), _stream()), "route_keys")
    return out


def rescore_sparse(feature: torch.Tensor, feature_bank: torch.Tensor, cand: torch.Tensor, cand_mode: str,
                   idx_offset: int) -> torch.Tensor:
    """Exact (sequential-fma) keys of the candidates in `cand` (B, k_in; lists filled from the front, empty slots only behind the last candidate;
    indices offset by idx_offset into this bank), sorted descending, zero-padded: (B, k_in)."""
    lib = _lib.load()
    B, D = feature.shape
    N = feature_bank.shape[1]
    k_in = cand.shape[1]
    dev = feature.device
    pb = bank_cache.get(feature_bank, cand_mode)
    rows_a, rows_b = pb.rescore_rows()
    q = feature if feature.dtype == torch.float32 else feature.float()
    if q.stride(1) != 1:
        q = q.contiguous()
    out = torch.empty((B, k_in), dtype=torch.int64, device=dev)
    if B == 0:
        return out
    cand = cand.contiguous()
    with torch.cuda.device(dev):
        flags = torch.empty((B,), dtype=torch.int32, device=dev)
        n_bad = torch.zeros((1,), dtype=torch.int32, device=dev)
        ws_bytes = int(lib.b200knn_rescore_workspace_bytes(B, k_in)) if rows_b is None else 0
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev) if ws_bytes else None
        _lib.check(lib.b200knn_rescore(q.data_ptr(), _DTYPES[q.dtype], q.stride(0), rows_a.data_ptr(),
                                       _ptr(rows_b), N, D, cand.data_ptr(), B, k_in, k_in, idx_offset,
                                       0.0, 0.0, 0.0, pb.max_norm().data_ptr(), out.data_ptr(),
                                       flags.data_ptr(), n_bad.data_ptr(), _ptr(ws), ws_bytes, _stream()),
                   "rescore")
    return out


def _ptr_array(ptrs):
    return (ctypes.c_void_p * len(ptrs))(*[int(p) for p in ptrs])


def route_scatter(keys: torch.Tensor, rows_per_shard: int, n_shards: int, inbox_ptrs, row_offset: int) -> None:
    """route_keys fused with its exchange: the keys of row r that shard g owns go, compacted, into
    row (row_offset + r) of shard g's inbox (device pointers of every rank's (Q_pad, k) inbox)."""
    n, k = keys.shape
    if n:
        keys = keys.contiguous()
        with torch.cuda.device(keys.device):
            _lib.check(_lib.load().b200knn_route_scatter(keys.data_ptr(), n, k, rows_per_shard, n_shards,
                                                         _ptr_array(inbox_ptrs), row_offset, _stream()),
                       "route_scatter")


def rescore_scatter(feature: torch.Tensor, feature_bank: torch.Tensor, cand: torch.Tensor, cand_mode: str,
                    idx_offset: int, peer_ptrs, rank: int, rows_per_owner: int) -> None:
    """rescore_sparse whose sorted exact keys of query row b are stored straight into the exchange
    buffer of the GPU that owns b (peer memory; the owners zero their buffers beforehand)."""
    lib = _lib.load()
    B, D = feature.shape
    if B == 0:
        return
    N = feature_bank.shape[1]
    k_in = cand.shape[1]
    dev = feature.device
    pb = bank_cache.get(feature_bank, effective_mode(cand_mode, D))
    rows_a, rows_b = pb.rescore_rows()
    if rows_b is not None:  # tf32x3 operands (hi + lo): reassemble once
        rows_a = rows_a + rows_b
    q = feature if feature.dtype == torch.float32 else feature.float()
    if q.stride(1) != 1:
        q = q.contiguous()
    cand = cand.contiguous()
    with torch.cuda.device(dev):
        ws_bytes = int(lib.b200knn_rescore_workspace_bytes(B, k_in))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        with _Timed("rescore"):
            rc = lib.b200knn_rescore_scatter(q.data_ptr(), q.stride(0), rows_a.data_ptr(), N, D, cand.data_ptr(),
                                             B, k_in, idx_offset, _ptr_array(peer_ptrs), len(peer_ptrs), rank,
                                             rows_per_owner, ws.data_ptr(), ws_bytes, _stream())
        _lib.check(rc, "rescore_scatter")


def compact_rows(packed: torch.Tensor, col: int, mask: int, cap: int):
    """(rows int64 (cap,), count int32 (1,)): ascending numbers of the rows of `packed` (n, ld) int64
    whose column `col` has a bit of `mask` set, zero-padded; count may exceed cap (overflow)."""
    n, ld = packed.shape
    assert packed.dtype == torch.int64 and packed.stride(1) == 1
    rows = torch.empty((cap,), dtype=torch.int64, device=packed.device)
    count = torch.empty((1,), dtype=torch.int32, device=packed.device)
    with torch.cuda.device(packed.device):
        _lib.check(_lib.load().b200knn_compact_rows(packed.data_ptr() + 8 * col, packed.stride(0), n, mask,
                                                    rows.data_ptr(), cap, count.data_ptr(), _stream()),
                   "compact_rows")
    return rows, count


def scatter_rows(dst: torch.Tensor, src: torch.Tensor, rows: torch.Tensor, count: torch.Tensor) -> None:
    """dst[rows[i]] = src[i] for i < min(len(rows), count) — (n, w) int64 row-major tensors."""
    assert dst.dtype == torch.int64 and src.dtype == torch.int64 and dst.stride(1) == 1 and src.stride(1) == 1
    assert dst.shape[1] == src.shape[1] and src.shape[0] == rows.numel()
    with torch.cuda.device(dst.device):
        _lib.check(_lib.load().b200knn_scatter_rows(dst.data_ptr(), dst.stride(0), src.data_ptr(), src.stride(0),
                                                    rows.data_ptr(), rows.numel(), count.data_ptr(), dst.shape[1],
                                                    _stream()), "scatter_rows")


def local_exact_keys(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: str,
                     idx_offset: int, n_shards: int = 1) -> torch.Tensor:
    """(B, k+1) int64, nothing synchronises: columns [0, k) the exact top-min(k, N) keys of this bank
    shard (zero-padded), column k = 1 where the certificate failed.  One level of `mode`'s cascade at
    its base margin: a shard holds 1/G of the bank, so its rank gaps are G times wider than the
    global ones the first level failed on.  With G >= 4 shards the FIRST level (fp16, 1 MMA per
    k-step) is therefore tried again on the shard; below that the second (fp16 x split-fp16)."""
    B = feature.shape[0]
    N = feature_bank.shape[1]
    levels = _cascade_levels(feature_bank, mode, track=False)
    level = (levels[0] if n_shards >= 4 or len(levels) == 1 else levels[1]).partition("@")[0]
    k_loc = min(int(k), N)
    out = torch.zeros((B, k + 1), dtype=torch.int64, device=feature.device)
    if B and k_loc:
        keys, flags, _ = _rescored_level(feature, feature_bank, k_loc, level, idx_offset)
        out[:, :k_loc] = keys
        out[:, k] = flags
    return out


def certify(exact: torch.Tensor, approx: torch.Tensor, feature: torch.Tensor, level: dict,
            max_norm: torch.Tensor, all_rows: bool) -> torch.Tensor:
    """(n,) int32 flags: 1 where the exact k-th key does not beat the approximate k_in-th by the
    level's error bound (see b200knn_rescore)."""
    n, k = exact.shape
    k_in = approx.shape[1]
    D = feature.shape[1]
    dev = exact.device
    flags = torch.zeros((n,), dtype=torch.int32, device=dev)
    if n == 0:
        return flags
    q = feature if feature.dtype in _DTYPES else feature.float()
    if q.stride(1) != 1:
        q = q.contiguous()
    exact, approx = exact.contiguous(), approx.contiguous()
    with torch.cuda.device(dev):
        n_bad = torch.zeros((1,), dtype=torch.int32, device=dev)
        _lib.check(_lib.load().b200knn_certify(
            q.data_ptr(), _DTYPES[q.dtype], q.stride(0), D, exact.data_ptr(), k, approx.data_ptr(), k_in, n,
            1 if all_rows else 0, float(level["err_coef"]),
            float(level.get("err_abs", 0.0)) * math.sqrt(padded_dim(D)), float(level.get("max_abs", 0.0)),
            max_norm.data_ptr(), flags.data_ptr(), n_bad.data_ptr(), _stream()), "certify")
    return flags


def bank_max_norm(feature_bank: torch.Tensor, cand_mode: str) -> torch.Tensor:
    """Device scalar: max row norm of this bank (x1.001), as the certificate uses it."""
    return bank_cache.get(feature_bank, cand_mode).max_norm()


def _cascade_levels(feature_bank: torch.Tensor, mode: str, track: bool = True, boost: int = 1):
    """The level specs `mode` tries in order on this bank.  track=False (sharded driver, captured
    graphs): the per-process statistics (margin boost, "skip the first level") are neither read nor
    updated — the caller passes its own `boost` — so every rank of a process group derives the
    same list (ranks that disagreed would mismatch their collectives)."""
    levels = list(CASCADES[mode])
    if len(levels) > 1 and padded_dim(feature_bank.shape[0]) > MAX_BF16_DIM:
        levels = list(CASCADE_WIDE)  # no resident query tile at this width
    if len(levels) > 1:
        skip = False
        if track:
            st = bank_cache.state(feature_bank)
            boost = st.get("boost", 1)
            if st.get("skip_first", 0) > 0:
                st["skip_first"] -= 1
                skip = True
        if skip:
            levels = levels[1:]
        elif boost > 1:
            name = levels[0].partition("@")[0]
            levels[0] = f"{name}@{level_config(levels[0], 1)['margin'] * boost}"
    return levels


def _cascade_fix(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, levels, rows: torch.Tensor,
                 idx_offset: int, exclude=None) -> torch.Tensor:
    """Keys of `rows` (uncertified at the previous level) from the remaining levels, then exact.
    exclude: ``topk_keys``' checked (query ids, bank ids, m) of `feature`'s rows."""
    sub = feature[rows].contiguous()
    if exclude is not None:
        exclude = (exclude[0][rows], exclude[1], exclude[2])
    for level in levels:
        out, flags, n_bad = _rescored_level(sub, feature_bank, k, level, idx_offset, exclude=exclude)
        last_rescore_stats["levels"].append((level, int(rows.numel()), int(n_bad.item())))
        if int(n_bad.item()) == 0:
            return out
        left = flags.nonzero(as_tuple=False).view(-1)
        out[left] = _cascade_fix(sub, feature_bank, k, levels[levels.index(level) + 1:], left, idx_offset, exclude)
        return out
    last_rescore_stats["levels"].append(("exact", int(rows.numel()), 0))
    return topk_keys(sub, feature_bank, k, "exact", idx_offset, exclude=exclude)


def _note_first_level(feature_bank: torch.Tensor, mode: str, levels, rows: int, uncertified: int,
                      track: bool = True) -> None:
    last_rescore_stats["rows"], last_rescore_stats["uncertified"] = rows, uncertified
    last_rescore_stats["level"] = levels[0]
    last_rescore_stats["levels"] = [(levels[0], rows, uncertified)]  # (level, rows in, rows left uncertified)
    first = CASCADES[mode][0].partition("@")[0]
    if track and len(CASCADES[mode]) > 1 and levels[0].partition("@")[0] in (first, CASCADE_WIDE[0].partition("@")[0]) \
            and rows > 0:
        st = bank_cache.state(feature_bank)
        boost = st.get("boost", 1)
        if boost >= CASCADE_MAX_BOOST and rows >= 128 and uncertified > CASCADE_GIVE_UP * rows:
            st["skip_first"] = CASCADE_RETRY_CALLS
        st["boost"], st["calm"] = next_boost(boost, st.get("calm", 0), rows, uncertified)


def _topk_keys_rescored(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: str,
                        idx_offset: int = 0, defer: bool = False, track: bool = True, boost: int = 1,
                        n_bad: Optional[torch.Tensor] = None, exclude=None):
    """Tensor-core candidates -> exact sequential-fma re-scoring -> best k, with a per-row
    certificate; rows a level cannot certify go to the next level and finally to the "exact"
    kernel, so the keys are bitwise those of mode "exact".
    defer=True: nothing synchronises; returns (keys, flags, n_bad, fix) and the caller, after
    reading n_bad in its own synchronisation, replaces keys[rows] by fix(rows)."""
    _check_feature_bank(feature, feature_bank)
    B, D = feature.shape
    N = feature_bank.shape[1]
    k = int(k)
    if k <= 0 or k > N:
        raise RuntimeError("selected index k out of range")
    dev = feature.device
    if B == 0:
        out = torch.empty((B, k), dtype=torch.int64, device=dev)
        return (out, None, None, None) if defer else out
    levels = _cascade_levels(feature_bank, mode, track, boost)
    if exclude is not None:
        exclude = _exclusion(exclude, B, N, dev)
    out, flags, n_bad = _rescored_level(feature, feature_bank, k, levels[0], idx_offset, n_bad, exclude)

    def fix(rows, n_rows_bad):
        _note_first_level(feature_bank, mode, levels, B, n_rows_bad, track)
        if rows is None:
            return None
        return _cascade_fix(feature, feature_bank, k, levels[1:], rows, idx_offset, exclude)

    if defer:
        return out, flags, n_bad, fix
    bad = int(n_bad.item())
    if bad:
        rows = flags.nonzero(as_tuple=False).view(-1)
        out[rows] = fix(rows, bad)
    else:
        _note_first_level(feature_bank, mode, levels, B, 0, track)
    return out


def decode_keys(keys: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    lib = _lib.load()
    sims = torch.empty(keys.shape, dtype=torch.float32, device=keys.device)
    idx = torch.empty(keys.shape, dtype=torch.int64, device=keys.device)
    if keys.numel():
        with torch.cuda.device(keys.device):
            _lib.check(lib.b200knn_decode_keys(keys.data_ptr(), keys.numel(), sims.data_ptr(),
                                               idx.data_ptr(), _stream()), "decode_keys")
    return sims, idx


def drop_self(keys: torch.Tensor, self_offset: int) -> torch.Tensor:
    """(B, k_in) sorted keys of bank rows [self_offset, self_offset + B) searched against their own
    bank -> (B, k_in - 1): row b without the key of bank row b + self_offset, or without its last
    key when that row is not in the list (``b200knn_drop_self``)."""
    _require_cuda("keys", keys)
    B, k_in = keys.shape
    keys = keys.contiguous()
    out = torch.empty((B, max(k_in - 1, 0)), dtype=torch.int64, device=keys.device)
    with torch.cuda.device(keys.device):
        _lib.check(_lib.load().b200knn_drop_self(keys.data_ptr(), B, k_in, int(self_offset), out.data_ptr(),
                                                 _stream()), "drop_self")
    return out


def drop_group(keys: torch.Tensor, row_ids: torch.Tensor, group_ids: torch.Tensor, k_out: int,
               flag: Optional[torch.Tensor] = None) -> torch.Tensor:
    """(B, k_in) sorted keys of bank rows row_ids (B,) searched against their own bank, group_ids
    (N,) int32 the group of every bank row -> (B, k_out): the first k_out keys of row b outside the
    group of bank row row_ids[b], zero-filled when fewer survive (``b200knn_drop_group``).  A key
    index or row id outside [0, N) sets the device int32[1] `flag` to 2; without a flag it raises."""
    _require_cuda("keys", keys)
    if group_ids.dtype != torch.int32:
        raise ValueError(f"group_ids must be int32, got {group_ids.dtype}")
    B, k_in = keys.shape
    if row_ids.numel() != B:
        raise RuntimeError(f"row_ids has {row_ids.numel()} entries for {B} rows of keys")
    if flag is not None and (flag.dtype != torch.int32 or flag.numel() < 1):
        raise ValueError("flag must be a device int32 tensor of at least one element")
    for t in (row_ids, group_ids) + (() if flag is None else (flag,)):
        if t.device != keys.device:
            raise RuntimeError(f"Expected all tensors to be on the same device, but found {keys.device} and {t.device}")
    keys = keys.contiguous()
    row_ids = row_ids.to(torch.int64).contiguous().view(-1)
    group_ids = group_ids.contiguous().view(-1)
    out = torch.empty((B, int(k_out)), dtype=torch.int64, device=keys.device)
    check = flag is None
    with torch.cuda.device(keys.device):
        if check:
            flag = torch.zeros((1,), dtype=torch.int32, device=keys.device)
        _lib.check(_lib.load().b200knn_drop_group(keys.data_ptr(), B, k_in, row_ids.data_ptr(), group_ids.data_ptr(),
                                                  group_ids.numel(), int(k_out), out.data_ptr(), flag.data_ptr(),
                                                  _stream()), "drop_group")
        if check and int(flag.item()):
            raise RuntimeError("drop_group: a key index or row id is outside the group ids")
    return out


def radius_tau0(feature: torch.Tensor, feature_bank: torch.Tensor, tau: float, cfg: dict, cand_mode: str,
                return_e: bool = False):
    """(tau0 (B,) fp32, refused (B,) int32) of a radius search at similarity >= tau (fp32) whose
    candidates come from `cand_mode` under the bound of level `cfg` (``b200knn_radius_tau0``); the
    residual form of the bound where the level has it and the candidates really are fp16.
    return_e: also the (B,) fp32 bound E of every row (tests)."""
    B, D = feature.shape
    pb = bank_cache.get(feature_bank, cand_mode)
    err_coef, err_abs, acc_coef, resid = _bound_terms(cfg, pb, D, cfg.get("residual_bound", False) and
                                                      cand_mode == "f16")
    q = feature if feature.dtype == torch.float32 else feature.float()
    if q.stride(1) != 1:
        q = q.contiguous()
    tau0 = torch.empty((B,), dtype=torch.float32, device=q.device)
    refused = torch.empty((B,), dtype=torch.int32, device=q.device)
    e = torch.empty((B,), dtype=torch.float32, device=q.device) if return_e else None
    with torch.cuda.device(q.device):
        _lib.check(_lib.load().b200knn_radius_tau0(q.data_ptr(), q.stride(0), B, D, float(tau), float(err_coef),
                                                   float(err_abs), float(cfg.get("max_abs", 0.0)),
                                                   pb.max_norm().data_ptr(), _ptr(resid), float(acc_coef),
                                                   tau0.data_ptr(), refused.data_ptr(), _ptr(e), _stream()),
                   "radius_tau0")
    return (tau0, refused, e) if return_e else (tau0, refused)


def radius_count(keys: torch.Tensor, rows: Optional[torch.Tensor], tau: float, self_offset: int, cap: int,
                 counts: torch.Tensor) -> torch.Tensor:
    """Count pass of ``b200knn_radius_compact``: counts[rows[i]] (rows None: i) = the keys of list
    row i with sim >= tau, not the row's own, at most cap; returns the (n,) int32 `full` bits
    (1: last slot non-empty, 2: and its sim >= tau)."""
    n, m = keys.shape
    full = torch.zeros((n,), dtype=torch.int32, device=keys.device)
    if n:
        keys = keys.contiguous()
        with torch.cuda.device(keys.device):
            _lib.check(_lib.load().b200knn_radius_compact(keys.data_ptr(), n, m, _ptr(rows), float(tau),
                                                          int(self_offset), int(cap), counts.data_ptr(),
                                                          full.data_ptr(), None, None, None, _stream()),
                       "radius_compact")
    return full


def radius_emit(keys: torch.Tensor, rows: Optional[torch.Tensor], tau: float, self_offset: int,
                offsets: torch.Tensor, indices: torch.Tensor, sims: torch.Tensor) -> None:
    """Emit pass of ``b200knn_radius_compact`` into the CSR arrays (offsets from the count pass)."""
    n, m = keys.shape
    if n and indices.numel():
        keys = keys.contiguous()
        with torch.cuda.device(keys.device):
            _lib.check(_lib.load().b200knn_radius_compact(keys.data_ptr(), n, m, _ptr(rows), float(tau),
                                                          int(self_offset), 1, None, None, offsets.data_ptr(),
                                                          indices.data_ptr(), sims.data_ptr(), _stream()),
                       "radius_compact")


def union_edges(parent: torch.Tensor, offsets: torch.Tensor, indices: torch.Tensor, row_offset: int,
                flag: torch.Tensor) -> None:
    """Union the CSR edges (row_offset + r, indices[j]) into the int32 parent array (``b200knn_union_edges``)."""
    n_rows = offsets.numel() - 1
    if n_rows > 0 and indices.numel():
        with torch.cuda.device(parent.device):
            _lib.check(_lib.load().b200knn_union_edges(parent.data_ptr(), parent.numel(), offsets.data_ptr(),
                                                       indices.data_ptr(), n_rows,
                                                       int(row_offset), flag.data_ptr(), _stream()), "union_edges")


def components(parent: torch.Tensor) -> torch.Tensor:
    """(n,) int64: the smallest node of every node's component (``b200knn_components``)."""
    labels = torch.empty((parent.numel(),), dtype=torch.int64, device=parent.device)
    if parent.numel():
        with torch.cuda.device(parent.device):
            _lib.check(_lib.load().b200knn_components(parent.data_ptr(), parent.numel(), labels.data_ptr(),
                                                      _stream()), "components")
    return labels


def merge_keys(keys_in: torch.Tensor, k_out: int) -> torch.Tensor:
    """(G,B,k_in) sorted candidate lists -> (B,k_out): the shard-merge step."""
    lib = _lib.load()
    _require_cuda("keys_in", keys_in)
    G, B, k_in = keys_in.shape
    keys_in = keys_in.contiguous()
    out = torch.empty((B, k_out), dtype=torch.int64, device=keys_in.device)
    if B:
        with torch.cuda.device(keys_in.device):
            _lib.check(lib.b200knn_merge(keys_in.data_ptr(), G, B, k_in, k_out, out.data_ptr(),
                                         _stream()), "merge")
    return out


def vote(keys: torch.Tensor, feature_labels: torch.Tensor, num_classes: int, knn_t: float,
         label_offset: int = 0, return_scores: bool = False, check_labels: bool = True,
         return_flag: bool = False, flag: Optional[torch.Tensor] = None):
    """keys (B,k) + labels (N,) -> (B,C) int64 class ranking (score desc, class asc)."""
    lib = _lib.load()
    _require_cuda("feature_labels", feature_labels)
    B, k = keys.shape
    labels = feature_labels
    if labels.dtype != torch.int64:
        labels = labels.long()
    labels = labels.contiguous().view(-1)
    C = int(num_classes)
    check_vote_classes(C, k)
    dev = keys.device
    pred = torch.empty((B, C), dtype=torch.int64, device=dev)
    scores = torch.empty((B, C), dtype=torch.float64, device=dev) if return_scores else None
    if B:
        with torch.cuda.device(dev):
            if flag is None:
                flag = torch.zeros((1,), dtype=torch.int32, device=dev)
            _lib.check(lib.b200knn_vote(keys.data_ptr(), labels.data_ptr(), B, k, labels.numel(),
                                        label_offset, C, float(knn_t), pred.data_ptr(), _ptr(scores),
                                        flag.data_ptr(), _stream()), "vote")
            if check_labels:
                _raise_vote_flag(int(flag.item()), C)
    if return_flag:  # device int32[1]: 0 ok, 1 label outside [0,C), 2 neighbour index outside labels
        return pred, (flag if B else torch.zeros((1,), dtype=torch.int32, device=dev))
    return (pred, scores) if return_scores else pred


MAX_GRID_KS, MAX_GRID_TS = 16, 8  # kVoteMaxKs / kVoteMaxTs of csrc/kernels.h
VOTE_CHUNK, VOTE_SMEM_BYTES, VOTE_WARPS = 1024, 200 * 1024, 4  # kVoteChunk / kVoteSmemBytes, kVoteWarps


def vote_max_classes(k: int, grid: bool = False) -> int:
    """The largest num_classes the vote kernel (grid: the grid vote kernel) serves for lists of k
    keys.  Keys pass through shared memory in chunks of at most VOTE_CHUNK, so k itself is not
    bounded; each of the block's VOTE_WARPS rows also keeps C fp64 scores there."""
    kc = min(int(k), VOTE_CHUNK)
    keys_bytes = 16 * kc if grid else (12 * kc + 7) // 8 * 8
    return (VOTE_SMEM_BYTES // VOTE_WARPS - keys_bytes) // 8


def check_vote_classes(num_classes: int, k: int, grid: bool = False) -> None:
    c_max = vote_max_classes(k, grid)
    if int(num_classes) > c_max:
        raise ValueError(f"num_classes={int(num_classes)} is more than the {'grid ' if grid else ''}vote serves "
                         f"at k={int(k)}: at most {c_max} classes")


def _vote_multi_into(keys, feature_labels, num_classes, knn_ks, knn_ts, out, status_col, flag) -> None:
    """b200knn_vote_multi of keys (B, knn_ks[-1]) into the (>= B, ld) int64 tensor `out`."""
    B, k = keys.shape
    check_vote_classes(num_classes, k, grid=True)
    labels = feature_labels if feature_labels.dtype == torch.int64 else feature_labels.long()
    labels = labels.contiguous().view(-1)
    ks = (ctypes.c_int * len(knn_ks))(*[int(x) for x in knn_ks])
    ts = (ctypes.c_double * len(knn_ts))(*[float(x) for x in knn_ts])
    keys = keys.contiguous()
    with torch.cuda.device(keys.device):
        _lib.check(_lib.load().b200knn_vote_multi(keys.data_ptr(), labels.data_ptr(), B, k, labels.numel(), 0,
                                                  int(num_classes), ks, len(knn_ks), ts, len(knn_ts),
                                                  out.data_ptr(), out.stride(0), status_col, flag.data_ptr(),
                                                  _stream()), "vote_multi")


def vote_multi(keys: torch.Tensor, feature_labels: torch.Tensor, num_classes: int, knn_ks, knn_ts,
               check_labels: bool = True, flag: Optional[torch.Tensor] = None) -> torch.Tensor:
    """keys (B, k_max) sorted + labels (N,) -> (B, n_k*n_t*C) int64: block (i, j) of a row is what
    ``vote`` returns for the row's first knn_ks[i] keys at knn_t = knn_ts[j].  knn_ks strictly
    increasing with knn_ks[-1] == k_max.  flag: optional device int32[1] for the label status
    (check_labels=False leaves reading it to the caller)."""
    _require_cuda("feature_labels", feature_labels)
    B = keys.shape[0]
    C = int(num_classes)
    pred = torch.empty((B, len(knn_ks) * len(knn_ts) * C), dtype=torch.int64, device=keys.device)
    if B:
        if flag is None:
            flag = torch.zeros((1,), dtype=torch.int32, device=keys.device)
        _vote_multi_into(keys, feature_labels, C, knn_ks, knn_ts, pred, -1, flag)
        if check_labels:
            _raise_vote_flag(int(flag.item()), C)
    return pred


def vote_multi_packed(keys: torch.Tensor, feature_labels: torch.Tensor, num_classes: int, knn_ks, knn_ts,
                      n_rows_out: int) -> torch.Tensor:
    """vote_packed for a grid: (n_rows_out, W+1) int64, W = n_k*n_t*C, the rankings of vote_multi in
    columns [0, W) and vote_packed's status word in column W; rows past keys.shape[0] are zero."""
    B = keys.shape[0]
    W = len(knn_ks) * len(knn_ts) * int(num_classes)
    dev = keys.device
    out = torch.zeros((n_rows_out, W + 1), dtype=torch.int64, device=dev) if n_rows_out > B \
        else torch.empty((n_rows_out, W + 1), dtype=torch.int64, device=dev)
    if B:
        flag = torch.zeros((1,), dtype=torch.int32, device=dev)
        _vote_multi_into(keys, feature_labels, num_classes, knn_ks, knn_ts, out, W, flag)
    return out


MAX_LABELS = 64  # label sets are 64-bit masks (include/b200knn.h b200knn_vote_multilabel)


def pack_label_bits(label_matrix: torch.Tensor) -> torch.Tensor:
    """(N, L) 0/1 label matrix (bool or integer dtype, 1 <= L <= 64) -> (N,) int64 bitmasks, bit l set
    when row n carries label l.  Bit 63 is the sign bit: the int64 view of the uint64 mask the vote
    kernel reads."""
    _check_label_matrix(label_matrix)
    return _label_bits(label_matrix)


def _label_bits(m: torch.Tensor) -> torch.Tensor:
    weight = torch.tensor([1 << b if b < 63 else -(1 << 63) for b in range(m.shape[1])], dtype=torch.int64,
                          device=m.device)
    # distinct powers of two: the sum is the bitwise or, and bit 63's -2^63 cannot overflow it
    return (m.to(torch.int64) * weight).sum(1)


def _check_label_matrix(m: torch.Tensor, n_rows: Optional[int] = None) -> None:
    if not isinstance(m, torch.Tensor):
        raise TypeError(f"label_matrix must be a torch.Tensor, got {type(m).__name__}")
    if m.dim() != 2:
        raise ValueError(f"label_matrix must be (N, L), got shape {tuple(m.shape)}")
    if m.dtype.is_floating_point or m.dtype.is_complex:
        raise ValueError(f"label_matrix must be bool or integer 0/1 entries, got {m.dtype}")
    if n_rows is not None and m.shape[0] != n_rows:
        raise ValueError(f"label_matrix has {m.shape[0]} rows for a bank of {n_rows}")
    if not 1 <= m.shape[1] <= MAX_LABELS:
        raise ValueError(f"label_matrix must have 1 to {MAX_LABELS} labels, got {m.shape[1]}")
    if m.dtype != torch.bool and bool(((m != 0) & (m != 1)).any()):
        raise ValueError("label_matrix entries must be 0 or 1")


class _MultiLabelVote:
    """knn_t of a multi-label call: per-label scores over the (ks, ts) grid, ks ascending, from
    (N,) label bitmasks (``vote_multilabel``).  Not a tuple: a tuple knn_t is the class-ranking grid."""

    __slots__ = ("ks", "ts")

    def __init__(self, ks, ts):
        self.ks, self.ts = tuple(ks), tuple(ts)


def vote_multilabel(keys: torch.Tensor, label_bits: torch.Tensor, n_labels: int, knn_ks, knn_ts,
                    check_labels: bool = True, flag: Optional[torch.Tensor] = None) -> torch.Tensor:
    """keys (B, k_max) sorted + label_bits (N,) int64 (``pack_label_bits``) -> (B, n_k*n_t*L) fp64: block
    (i, j) of a row holds, for every label l < n_labels, S_l / W over the row's first knn_ks[i] keys at
    knn_t = knn_ts[j] (b200knn_vote_multilabel, include/b200knn.h).  knn_ks strictly increasing with
    knn_ks[-1] == k_max; knn_ts finite and > 0.  flag: as ``vote_multi`` (2: neighbour index outside
    the labels)."""
    _require_cuda("label_bits", label_bits)
    if label_bits.dtype != torch.int64:
        raise TypeError(f"label_bits must be int64 bitmasks, got {label_bits.dtype}")
    B, k = keys.shape
    L = int(n_labels)
    scores = torch.empty((B, len(knn_ks) * len(knn_ts) * L), dtype=torch.float64, device=keys.device)
    if B:
        if flag is None:
            flag = torch.zeros((1,), dtype=torch.int32, device=keys.device)
        bits = label_bits.contiguous().view(-1)
        ks = (ctypes.c_int * len(knn_ks))(*[int(x) for x in knn_ks])
        ts = (ctypes.c_double * len(knn_ts))(*[float(x) for x in knn_ts])
        keys = keys.contiguous()
        with torch.cuda.device(keys.device):
            _lib.check(_lib.load().b200knn_vote_multilabel(keys.data_ptr(), bits.data_ptr(), B, k, bits.numel(), 0,
                                                           L, ks, len(knn_ks), ts, len(knn_ts), scores.data_ptr(),
                                                           scores.stride(0), flag.data_ptr(), _stream()),
                       "vote_multilabel")
        if check_labels:
            _raise_vote_flag(int(flag.item()), L)
    return scores


def _raise_vote_flag(f: int, C: int) -> None:
    if f == 1:
        # the reference raises here from zeros(...).scatter(...) (lightly knn_predict)
        raise RuntimeError("index out of bounds: a feature_labels entry is outside "
                           f"[0, num_classes={C})")
    if f == 2:
        raise RuntimeError("index out of bounds: neighbour index outside feature_labels")


def check_grid(knn_ks, knn_ts):
    """Validate a (knn_ks, knn_ts) grid: (ks as ints, ts as floats, ascending order of ks)."""
    ks, ts = list(knn_ks), list(knn_ts)
    if not ks or not ts:
        raise ValueError("knn_ks and knn_ts must not be empty")
    if len(ks) > MAX_GRID_KS or len(ts) > MAX_GRID_TS:
        raise ValueError(f"at most {MAX_GRID_KS} values of knn_k and {MAX_GRID_TS} of knn_t per call")
    if any(int(k) != k for k in ks):
        raise ValueError(f"knn_ks must be integers, got {ks}")
    ks, ts = [int(k) for k in ks], [float(t) for t in ts]
    if min(ks) <= 0:
        raise ValueError(f"every knn_k must be positive, got {ks}")
    if any(t == 0.0 for t in ts):
        raise ValueError("knn_t must be non-zero")
    if len(set(ks)) != len(ks) or len(set(ts)) != len(ts):
        raise ValueError(f"duplicate values in knn_ks {ks} or knn_ts {ts}")
    return ks, ts, sorted(range(len(ks)), key=ks.__getitem__)


# ----------------------------------------------------------------------------
# the reference's public symbols for this path
# ----------------------------------------------------------------------------
def _vote_step(keys, feature_labels, num_classes, knn_t, flag):
    """The vote of a call, label status into the device int32[1] `flag`: knn_t a temperature ->
    (B, C) rankings (``vote``); knn_t a (ks, ts) grid, ks ascending and ks[-1] == keys.shape[1] ->
    (B, n_k*n_t*C) rankings (``vote_multi``); knn_t a ``_MultiLabelVote`` (feature_labels the (N,)
    bitmasks, num_classes the label count L) -> (B, n_k*n_t*L) fp64 scores (``vote_multilabel``)."""
    if isinstance(knn_t, _MultiLabelVote):
        return vote_multilabel(keys, feature_labels, num_classes, knn_t.ks, knn_t.ts, check_labels=False, flag=flag)
    if isinstance(knn_t, tuple):
        return vote_multi(keys, feature_labels, num_classes, knn_t[0], knn_t[1], check_labels=False, flag=flag)
    return vote(keys, feature_labels, num_classes, knn_t, check_labels=False, return_flag=True, flag=flag)[0]


# knn_predict returns the class ranking only, so a rescored-mode call re-scores only the candidates
# near rank k and certifies the ranking from intervals on the others (b200knn_rescore_vote,
# DESIGN §4.1c).  Rows it cannot certify are re-scored in full and voted as before.  The switch
# exists for A/B measurements (scripts/bench_vote_certificate.py) and tests; results are the same.
CERTIFIED_VOTE = {"enabled": os.environ.get("B200KNN_CERTIFIED_VOTE", "1") == "1"}
CERTIFIED_VOTE_MAX_CLASSES = 256  # B200KNN_RESCORE_VOTE_MAX_CLASSES


def _certified_vote_applies(feature, feature_bank, num_classes, knn_k, knn_t, mode, exclude) -> bool:
    """Whether a knn_predict call takes the certified vote: a rescored mode with one fp32 row array,
    a single temperature, no group exclusion, and k_in < N at every margin (k_in <= max(k, MAX_K))."""
    return (CERTIFIED_VOTE["enabled"] and mode in RESCORED_MODES and mode != "fp32_tf32"
            and not isinstance(knn_t, (tuple, _MultiLabelVote)) and float(knn_t) != 0.0 and exclude is None
            and int(num_classes) <= CERTIFIED_VOTE_MAX_CLASSES
            and feature_bank.shape[1] > max(int(knn_k), MAX_K))


def _bound_terms(cfg: dict, pb: "PreparedRows", D: int, residual: bool):
    """(err_coef, err_abs, acc_coef, bank_resid) of the bound E of a level (the arguments of
    b200knn_rescore_vote and b200knn_radius_tau0): with residual, the measured fp16 residuals of the
    bank pb (err_coef = the exact chain's gamma_D), else the level's worst-case model."""
    if residual:
        u = D * 2.0 ** -24
        return u / (1.0 - u), 0.0, 1.01 * cfg["acc_c"] * padded_dim(D) * ACC_ULP, pb.f16_residuals()
    return cfg["err_coef"], cfg.get("err_abs", 0.0) * math.sqrt(padded_dim(D)), 0.0, None


def _predict_certified(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t, mode, track, boost, status):
    """The certified vote of a rescored-mode call, nothing synchronises: (pred (B,C), flags (B,) int32, fix).
    status[1] counts the rows it leaves uncertified; fix(rows, n) returns their exact keys: their full
    candidate lists re-scored under the first level's certificate, then the rest of the cascade."""
    lib = _lib.load()
    _check_feature_bank(feature, feature_bank)
    B, D = feature.shape
    N = feature_bank.shape[1]
    k, C = int(knn_k), int(num_classes)
    dev = feature.device
    levels = _cascade_levels(feature_bank, mode, track, boost)
    cfg = level_config(levels[0], D)
    k_in = min(N, k + cfg["margin"], max(k, MAX_K))
    cand = topk_keys(feature, feature_bank, k_in, cfg["cand"], repair=False)
    pb = bank_cache.get(feature_bank, cfg["cand"])
    rows, _ = pb.rescore_rows()
    max_norm = pb.max_norm()
    err_coef, err_abs, acc_coef, resid = _bound_terms(cfg, pb, D, cfg.get("residual_bound", False))
    q = feature if feature.dtype == torch.float32 else feature.float()
    if q.stride(1) != 1:
        q = q.contiguous()
    labels = (feature_labels if feature_labels.dtype == torch.int64 else feature_labels.long()).contiguous().view(-1)
    pred = torch.empty((B, C), dtype=torch.int64, device=dev)
    with torch.cuda.device(dev):
        flags = torch.empty((B,), dtype=torch.int32, device=dev)
        band = torch.empty((B, k_in), dtype=torch.int64, device=dev)
        info = torch.empty((B, 4), dtype=torch.int32, device=dev)
        ws_bytes = int(lib.b200knn_rescore_workspace_bytes(B, k_in))
        ws = torch.empty((ws_bytes,), dtype=torch.uint8, device=dev)
        with _Timed("rescore"):
            rc = lib.b200knn_rescore_vote(q.data_ptr(), q.stride(0), rows.data_ptr(), N, D, cand.data_ptr(), B, k_in, k,
                                          float(err_coef), float(err_abs), float(cfg.get("max_abs", 0.0)),
                                          max_norm.data_ptr(), _ptr(resid), float(acc_coef), labels.data_ptr(),
                                          labels.numel(), C, float(knn_t), band.data_ptr(), info.data_ptr(),
                                          pred.data_ptr(), flags.data_ptr(), status.data_ptr(), ws.data_ptr(),
                                          ws_bytes, _stream())
        _lib.check(rc, "rescore_vote")

    def fix(rows_bad, n_rows_bad):
        last_rescore_stats["band_info"] = info  # (B, 4): p, r per row (band_stats)
        if rows_bad is None:
            _note_first_level(feature_bank, mode, levels, B, 0, track)
            last_rescore_stats["vote_fallback"] = 0
            return None
        sub = feature[rows_bad].contiguous()
        keys, left_flags, n_left = _rescore_candidates(sub, feature_bank, cand[rows_bad].contiguous(), k, cfg, 0)
        n_left = int(n_left.item())
        _note_first_level(feature_bank, mode, levels, B, n_left, track)
        last_rescore_stats["vote_fallback"] = n_rows_bad
        if n_left:
            left = left_flags.nonzero(as_tuple=False).view(-1)
            keys[left] = _cascade_fix(sub, feature_bank, k, levels[1:], left, 0)
        return keys

    return pred, flags, fix


def band_stats() -> dict:
    """Band sizes (candidates re-scored per row) of the last certified-vote call: mean, max, and the
    rows it left to the full re-scoring.  Synchronises; for measurements."""
    info = last_rescore_stats.get("band_info")
    if info is None:
        return {}
    served = info[:, 0] >= 0
    size = (info[:, 1] - info[:, 0])[served].double()
    return {"rows": int(info.shape[0]), "mean": float(size.mean()) if size.numel() else 0.0,
            "max": int(size.max()) if size.numel() else 0, "sure_mean": float(info[served, 0].double().mean())
            if size.numel() else 0.0, "fallback_rows": int(last_rescore_stats.get("vote_fallback", 0))}


def _predict_enqueue(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t, mode, track=True, boost=1,
                     exclude=None):
    """Everything of one tensor-core-mode call, enqueued without a host synchronisation (so it can
    be captured into a CUDA graph): (pred (B,C), status int32[2] = [vote flag, rows to recompute],
    bad_rows (B,) mask/flags, fix).  status[0]: 1 label / 2 neighbour index out of range;
    status[1]: rows a sampled threshold starved, or rows whose re-scoring could not be certified.
    knn_t: a temperature, or a (ks, ts) grid (``_vote_step``; pred is then (B, n_k*n_t*C))."""
    # one zeroed status word per call: [vote flag, rows to recompute] — the kernels write into it
    status = torch.zeros((2,), dtype=torch.int32, device=feature.device)
    if _certified_vote_applies(feature, feature_bank, num_classes, knn_k, knn_t, mode, exclude):
        pred, bad_rows, fix = _predict_certified(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t,
                                                 mode, track, boost, status)
        return pred, status, bad_rows, fix
    if mode in RESCORED_MODES:
        keys, bad_rows, _, fix = _topk_keys_rescored(feature, feature_bank, knn_k, mode, defer=True,
                                                     track=track, boost=boost, n_bad=status[1:2], exclude=exclude)
    else:
        keys = topk_keys(feature, feature_bank, knn_k, mode, repair=False, exclude=exclude)
        bad_rows = keys[:, -1] == 0
        status[1:2] = bad_rows.sum().to(torch.int32)
        fix = None
    pred = _vote_step(keys, feature_labels, num_classes, knn_t, status[0:1])
    return pred, status, bad_rows, fix


def _predict_finish(pred, status, bad_rows, fix, feature, feature_bank, feature_labels, num_classes, knn_k,
                    knn_t, mode, exclude=None):
    """The host side of a call after its one synchronisation (`status` is a host list here)."""
    n_fix = int(status[1])
    if mode not in RESCORED_MODES:
        last_prepass_stats["rows"], last_prepass_stats["repaired"] = pred.shape[0], n_fix
    elif n_fix == 0:
        fix(None, 0)  # records the statistics of a fully certified call
    if n_fix:
        rows = bad_rows.nonzero(as_tuple=False).view(-1)
        fixed = fix(rows, n_fix) if mode in RESCORED_MODES else \
            recompute_rows(feature, feature_bank, knn_k, mode, rows, exclude=exclude)
        flag2 = torch.zeros((1,), dtype=torch.int32, device=pred.device)
        pred[rows] = _vote_step(fixed, feature_labels, num_classes, knn_t, flag2)
        status[0] = max(int(status[0]), int(flag2.item()))
    _raise_vote_flag(int(status[0]), int(num_classes))
    return pred


# ---- the reference-shaped call (B = 64 per validation_step, knn.py:87-99; scripts/WM811k_benchmark.py:71)
# is launch-latency bound: a dozen small kernels and as many Python -> C transitions per call.  For
# batches of at most GRAPH_MAX_BATCH rows the enqueued part of a call is captured ONCE per
# (bank, batch shape, k, C, t or (ks, ts) grid, mode) into a CUDA graph and replayed: one copy of the queries into
# the graph's static input, one graph launch, one read of the status word.  A non-zero status (rows
# to recompute, label errors — rare) re-runs the call on the ordinary path, so results and errors
# are exactly those of the un-captured call.
GRAPH_MAX_BATCH = 512
GRAPHS = {"enabled": os.environ.get("B200KNN_GRAPHS", "1") == "1", "capacity": 4}
graph_stats = {"captures": 0, "replays": 0, "fallbacks": 0}


class _CallGraph:
    __slots__ = ("graph", "q_static", "pred", "status_host", "bad_rows", "fix", "bank_ref", "keep")


_call_graphs = {}


def _graph_boost(feature_bank, mode) -> int:
    """The first level's margin boost a captured call of this bank uses (part of the graph key)."""
    if mode in RESCORED_MODES and len(CASCADES[mode]) > 1:
        return bank_cache.state(feature_bank).get("boost", 1)
    return 1


def _graph_key(feature, feature_bank, labels, num_classes, knn_k, knn_t, mode):
    return (_graph_boost(feature_bank, mode), feature_bank.data_ptr(), feature_bank._version, tuple(feature_bank.shape), tuple(feature_bank.stride()),
            feature_bank.dtype, feature_bank.device.index, labels.data_ptr(), labels._version,
            tuple(feature.shape), feature.dtype, int(num_classes), int(knn_k),
            knn_t if isinstance(knn_t, tuple) else float(knn_t), mode, CERTIFIED_VOTE["enabled"])


def _graph_for(feature, feature_bank, labels, num_classes, knn_k, knn_t, mode):
    for dead in [k_ for k_, g in _call_graphs.items() if g.bank_ref() is None]:
        _call_graphs.pop(dead)
    key = _graph_key(feature, feature_bank, labels, num_classes, knn_k, knn_t, mode)
    hit = _call_graphs.get(key)
    if hit is not None:
        return hit
    dev = feature.device
    entry = _CallGraph()
    entry.q_static = torch.empty_like(feature, memory_format=torch.contiguous_format)
    entry.q_static.copy_(feature)
    entry.status_host = torch.zeros((2,), dtype=torch.int32).pin_memory()
    side = torch.cuda.Stream(device=dev)
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):  # warm-up on a side stream, as graph capture requires
        query_cache.clear()
        _predict_enqueue(entry.q_static, feature_bank, labels, num_classes, knn_k, knn_t, mode, track=False,
                         boost=key[0])
    torch.cuda.current_stream().wait_stream(side)
    torch.cuda.synchronize(dev)
    query_cache.clear()
    entry.graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(entry.graph):
        pred, status, bad_rows, fix = _predict_enqueue(entry.q_static, feature_bank, labels, num_classes, knn_k,
                                                       knn_t, mode, track=False, boost=key[0])
        entry.status_host.copy_(status, non_blocking=True)
    query_cache.clear()  # it now refers to tensors of the graph's private pool
    entry.pred, entry.bad_rows, entry.fix = pred, bad_rows, fix
    entry.bank_ref = weakref.ref(feature_bank)
    # the graph holds raw pointers into the prepared copies of this bank (operands, re-scoring rows,
    # max norm) and into the labels: keep them alive for as long as the graph
    entry.keep = [labels] + [prep for ref, prep in bank_cache._entries.values() if ref() is feature_bank]
    if len(_call_graphs) >= GRAPHS["capacity"]:
        _call_graphs.pop(next(iter(_call_graphs)))
    _call_graphs[key] = entry
    graph_stats["captures"] += 1
    return entry


def clear_call_graphs() -> None:
    _call_graphs.clear()


def knn_predict(feature: torch.Tensor, feature_bank: torch.Tensor, feature_labels: torch.Tensor,
                num_classes: int, knn_k: int = 200, knn_t: float = 0.1) -> torch.Tensor:
    """Drop-in for ``lightly.utils.benchmarking.knn_predict`` (reference call sites
    ``src/ssl_wafermap/models/knn.py:91-98``, ``:205-212``).

    Args and return value are the reference's: feature (B,D), feature_bank (D,N),
    feature_labels (N,), returns (B, num_classes) int64 with the predicted class in
    column 0.  Neighbour order is (similarity desc, bank index asc); class order is
    (score desc, class id asc).
    """
    return _predict(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t, _default_mode)


def _vote_checked(keys, feature_labels, num_classes, knn_t):
    """``_vote_step`` raising the label errors itself (one host synchronisation)."""
    if isinstance(knn_t, _MultiLabelVote):
        return vote_multilabel(keys, feature_labels, num_classes, knn_t.ks, knn_t.ts)
    if isinstance(knn_t, tuple):
        return vote_multi(keys, feature_labels, num_classes, knn_t[0], knn_t[1])
    return vote(keys, feature_labels, num_classes, knn_t)


def _predict(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t, mode, exclude=None):
    """knn_predict in `mode`; knn_t a temperature, or a (ks, ts) grid with ks ascending and
    ks[-1] == knn_k (``_vote_step``).  exclude: ``topk_keys``' group exclusion (such calls are
    never captured into a CUDA graph)."""
    _require_cuda("feature_labels", feature_labels)
    if feature_labels.numel() != feature_bank.shape[1]:
        _check_feature_bank(feature, feature_bank)
        raise RuntimeError(
            f"feature_labels has {feature_labels.numel()} entries for a bank of {feature_bank.shape[1]}")
    multilabel = isinstance(knn_t, _MultiLabelVote)  # per-label scores: no class-count bound, no graph
    if not multilabel:
        check_vote_classes(num_classes, knn_k, grid=isinstance(knn_t, tuple))
    if mode == "exact" or int(knn_k) > MAX_K:
        return _vote_checked(topk_keys(feature, feature_bank, knn_k, mode, exclude=exclude), feature_labels,
                             num_classes, knn_t)
    _check_feature_bank(feature, feature_bank)
    knn_k = int(knn_k)
    if knn_k <= 0 or knn_k > feature_bank.shape[1]:
        raise RuntimeError("selected index k out of range")
    if feature.shape[0] == 0:
        return _vote_checked(torch.empty((0, knn_k), dtype=torch.int64, device=feature.device), feature_labels,
                             num_classes, knn_t)
    # Tensor-core modes: everything is enqueued first and ONE host synchronisation reads the
    # status word (vote flag; rows to recompute: rows a sampled threshold starved, or rows whose
    # exact re-scoring could not be certified).
    if GRAPHS["enabled"] and exclude is None and not multilabel and feature.shape[0] <= GRAPH_MAX_BATCH \
            and feature_labels.dtype == torch.int64 \
            and feature_labels.is_contiguous() and not torch.cuda.is_current_stream_capturing():
        with torch.cuda.device(feature.device):
            g = _graph_for(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t, mode)
            g.q_static.copy_(feature)
            g.graph.replay()
            pred = g.pred.clone()
            torch.cuda.current_stream().synchronize()
            graph_stats["replays"] += 1
            if mode in RESCORED_MODES and len(CASCADES[mode]) > 1:
                st = bank_cache.state(feature_bank)  # the margin boost follows the captured calls too
                st["boost"], st["calm"] = next_boost(st.get("boost", 1), st.get("calm", 0), feature.shape[0],
                                                     int(g.status_host[1]))
            if not g.status_host.any():
                return pred
            # rows to recompute / label errors: the ordinary host side, on the graph's own buffers
            # (q_static still holds this call's queries)
            graph_stats["fallbacks"] += 1
            return _predict_finish(pred, g.status_host.tolist(), g.bad_rows, g.fix, g.q_static, feature_bank,
                                   feature_labels, num_classes, knn_k, knn_t, mode)
    pred, status, bad_rows, fix = _predict_enqueue(feature, feature_bank, feature_labels, num_classes, knn_k,
                                                   knn_t, mode, exclude=exclude)
    return _predict_finish(pred, status.tolist(), bad_rows, fix, feature, feature_bank, feature_labels,
                           num_classes, knn_k, knn_t, mode, exclude)


def knn_predict_multi(feature: torch.Tensor, feature_bank: torch.Tensor, feature_labels: torch.Tensor,
                      num_classes: int, knn_ks=(200,), knn_ts=(0.1,), query_groups: Optional[torch.Tensor] = None,
                      bank_groups: Optional[torch.Tensor] = None) -> torch.Tensor:
    """``knn_predict`` for every (knn_k, knn_t) of a grid from ONE neighbour search at
    k_max = max(knn_ks) and one vote kernel: (len(knn_ks), len(knn_ts), B, num_classes) int64, where
    [i, j] is bitwise ``knn_predict(..., knn_ks[i], knn_ts[j])`` in the default mode.  The top-k list
    is the first k entries of the top-k_max list: the (sim desc, index asc) order and the
    similarities themselves do not depend on k.  At most 16 values of k and 8 of t, no duplicates.

    query_groups (B,) and bank_groups (N,): optional integer ids (any integer dtype, compared by
    value, on the bank's device), both or neither.  [i, j, b] is then the same call for query b
    against the bank without every column c with bank_groups[c] == query_groups[b] (labels
    likewise): a held-out query never votes with rows of its own group (a lot, a wafer's repeats).
    The search skips those columns itself, at depth max(knn_ks); max(knn_ks) must not exceed the
    smallest number of bank rows left to any query."""
    ks, ts, order = check_grid(knn_ks, knn_ts)
    mode = _default_mode
    searches = grid_parts(tuple(ks[i] for i in order), mode)
    for part in searches:  # before the first search
        check_vote_classes(num_classes, part[-1], grid=True)
    exclude = _query_bank_exclusion(feature, feature_bank, query_groups, bank_groups, max(ks))
    parts = [_predict(feature, feature_bank, feature_labels, num_classes, part[-1], (part, tuple(ts)), mode,
                      exclude) for part in searches]
    return grid_view(torch.cat(parts, dim=1) if len(parts) > 1 else parts[0], order, len(ts), num_classes)


def knn_predict_multilabel(feature: torch.Tensor, feature_bank: torch.Tensor, label_matrix: torch.Tensor,
                           knn_ks=(200,), knn_ts=(0.1,)) -> torch.Tensor:
    """Multi-label kNN scores for every (knn_k, knn_t) of a grid from ONE neighbour search at
    k_max = max(knn_ks), as ``knn_predict_multi``: (len(knn_ks), len(knn_ts), B, L) float64, where
    [i, j, b, l] is the exp(sim/t)-weighted share of query b's knn_ks[i] nearest bank rows that carry
    label l, in [0, 1]:  sum_{r<k, row r has l} w_r / sum_{r<k} w_r,  w_r = exp((s_r - s_0) / t), s_0
    the nearest similarity; fp64, added in rank order (b200knn_vote_multilabel, include/b200knn.h).
    A row without labels (a normal wafer) still weighs in W.

    label_matrix: (N, L) 0/1 targets, bool or any integer dtype, 1 <= L <= 64, on the bank's device
    (the torchmetrics / scikit-learn multi-label format).  The neighbour lists are those of
    ``knn_predict`` in the default mode; knn_ts must be finite and > 0.  Single-label banks get
    class probabilities from ``F.one_hot(labels, C)``."""
    ks, ts, order = check_grid(knn_ks, knn_ts)
    if not all(t > 0.0 and math.isfinite(t) for t in ts):
        raise ValueError(f"knn_ts must be finite and > 0 for per-label scores, got {ts}")
    n_bank = feature_bank.shape[1] if feature_bank.dim() == 2 else None
    _check_label_matrix(label_matrix, n_bank)
    if n_bank is not None and max(ks) > n_bank:
        raise RuntimeError("selected index k out of range")
    _check_feature_bank(feature, feature_bank)
    _require_cuda("label_matrix", label_matrix)
    if label_matrix.device != feature_bank.device:
        raise RuntimeError("Expected all tensors to be on the same device, but found "
                           f"{label_matrix.device} and {feature_bank.device}")
    mode = _default_mode
    bits, L = _label_bits(label_matrix), label_matrix.shape[1]
    parts = [_predict(feature, feature_bank, bits, L, part[-1], _MultiLabelVote(part, ts), mode)
             for part in grid_parts(tuple(ks[i] for i in order), mode)]
    return grid_view(torch.cat(parts, dim=1) if len(parts) > 1 else parts[0], order, len(ts), L)


def grid_parts(ks_ascending: tuple, mode: str) -> list:
    """The searches a grid needs: one at k_max, except in a raw tensor-core mode whose ks straddle
    MAX_K — lists longer than MAX_K come from the exact kernel, shorter ones from the mode's own
    similarities, so each side gets its own search."""
    if mode in TC_MODES and ks_ascending[0] <= MAX_K < ks_ascending[-1]:
        n_lo = sum(k <= MAX_K for k in ks_ascending)
        return [ks_ascending[:n_lo], ks_ascending[n_lo:]]
    return [ks_ascending]


def loo_parts(ks_ascending: tuple, mode: str) -> list:
    """``grid_parts`` for leave-one-out ks, whose searches run at k + 1: a raw tensor-core mode
    never asks its kernel for more than MAX_K keys, so its k = MAX_K is served by the exact kernel."""
    return [tuple(k - 1 for k in part) for part in grid_parts(tuple(k + 1 for k in ks_ascending), mode)]


def logo_parts(ks_ascending: tuple, p: int, n: int, mode: str) -> list:
    """The searches of the leave-one-group-out rows whose group size g has p = the smallest power of
    two >= g, in a bank of n rows: k is searched at depth min(n, k + p), and the ks are split by
    ``grid_parts``' rule applied to those depths, so a raw tensor-core mode never asks its kernel for
    more than MAX_K keys.  p = 1 is ``loo_parts``."""
    n_lo = len(grid_parts(tuple(min(n, k + p) for k in ks_ascending), mode)[0])
    return [tuple(ks_ascending)] if n_lo == len(ks_ascending) else [tuple(ks_ascending[:n_lo]),
                                                                    tuple(ks_ascending[n_lo:])]


_GROUP_DTYPES = (torch.uint8, torch.int8, torch.int16, torch.int32, torch.int64)
_GROUP_DTYPES_WIDENED = (torch.uint16, torch.uint32)  # to int64, losslessly


def _query_bank_exclusion(feature, feature_bank, query_groups, bank_groups, k_max: int):
    """``topk_keys``' exclusion (query ids, bank ids, m) for query_groups (B,) / bank_groups (N,) of
    any integer dtype, made dense by one torch.unique over both; None when both are None.  Raises,
    before any search, on one missing id tensor, a length or device mismatch, a non-integer dtype,
    and k_max above the smallest number of bank rows outside a query's group."""
    if query_groups is None and bank_groups is None:
        return None
    if query_groups is None or bank_groups is None:
        raise ValueError("query_groups and bank_groups go together: pass both or neither")
    if feature.dim() != 2 or feature_bank.dim() != 2:
        _check_feature_bank(feature, feature_bank)
    B, N = feature.shape[0], feature_bank.shape[1]
    ids = []
    for name, g, n in (("query_groups", query_groups, B), ("bank_groups", bank_groups, N)):
        if not isinstance(g, torch.Tensor):
            raise TypeError(f"{name} must be a torch.Tensor, got {type(g).__name__}")
        if g.numel() != n:
            raise RuntimeError(f"{name} has {g.numel()} entries for {n} {'queries' if n == B else 'bank rows'}")
        if g.dtype not in _GROUP_DTYPES + _GROUP_DTYPES_WIDENED + (torch.uint64,):
            raise ValueError(f"{name} must be an integer tensor, got {g.dtype}")
        if g.device != feature_bank.device:
            raise RuntimeError("Expected all tensors to be on the same device, but found "
                               f"{feature_bank.device} and {g.device}")
        g = g.reshape(-1)
        if g.dtype in _GROUP_DTYPES_WIDENED:
            g = g.to(torch.int64)
        elif g.dtype == torch.uint64:  # the same bits as int64: equal ids stay equal, distinct ones distinct
            g = g.view(torch.int64)
        ids.append(g.to(torch.int64))
    _, inv = torch.unique(torch.cat(ids), return_inverse=True)
    inv = inv.to(torch.int32)
    qg, bg = inv[:B].contiguous(), inv[B:].contiguous()
    m = int(torch.bincount(bg, minlength=B + N)[qg.long()].max()) if B and N else 0
    if int(k_max) > N - m:  # the bank without the query's group has N - m rows for some query
        raise RuntimeError("selected index k out of range")
    return qg, bg, m


def _group_plan(groups: torch.Tensor, n: int, device: torch.device):
    """The buckets of a leave-one-group-out search: (dense int32 group ids (n,), largest group size,
    rows (n,) int64 in bucket order, [(p, lo, hi)]) where positions [lo, hi) of `rows` hold, in
    ascending order, the rows whose group size g has p = the smallest power of two >= g, p
    ascending.  One torch.unique and one host read of the group statistics."""
    if groups.numel() != n:
        raise RuntimeError(f"groups has {groups.numel()} entries for a bank of {n}")
    if groups.dtype not in _GROUP_DTYPES + _GROUP_DTYPES_WIDENED + (torch.uint64,):
        raise ValueError(f"groups must be an integer tensor, got {groups.dtype}")
    if groups.device != device:
        raise RuntimeError(f"Expected all tensors to be on the same device, but found {device} and {groups.device}")
    groups = groups.reshape(-1)
    if groups.dtype in _GROUP_DTYPES_WIDENED:
        groups = groups.to(torch.int64)
    elif groups.dtype == torch.uint64:  # the same bits as int64: equal ids stay equal, distinct ones distinct
        groups = groups.view(torch.int64)
    _, inv, cnt = torch.unique(groups, return_inverse=True, return_counts=True)
    e_group = torch.frexp((cnt - 1).double()).exponent.long()  # the bit length of g - 1: p = 2**e
    rows = torch.sort(e_group[inv], stable=True).indices
    rows_per_e = torch.zeros((64,), dtype=torch.int64, device=cnt.device).scatter_add_(0, e_group, cnt)
    stats = torch.cat([cnt.max().view(1), rows_per_e]).tolist()
    buckets, lo = [], 0
    for e, m in enumerate(stats[1:]):
        if m:
            buckets.append((1 << e, lo, lo + m))
            lo += m
    return inv.to(torch.int32), stats[0], rows, buckets


def logo_excludes(k: int, p: int, n: int) -> bool:
    """Whether the leave-one-group-out rows of bucket p (group sizes in (p/2, p]) search for a list
    of k neighbours by skipping their group inside the search (at depth k) instead of searching
    deeper and dropping the group's keys afterwards: when that deeper search, min(n, k + p), would
    not fit the streaming lists (MAX_K)."""
    return min(n, int(k) + int(p)) > MAX_K


def _group_searches(feature_bank: torch.Tensor, plan, ks_ascending: tuple, mode: str, batch: int,
                    flag: torch.Tensor):
    """Yields (part, lo, hi, keys) for every search of a leave-one-group-out pass over the bank's own
    rows: keys (hi - lo, part[-1]) are the lists of rows plan[2][lo:hi] without their groups.  Each
    search runs one ``topk_keys`` at depth min(N, part[-1] + p) (every mode, cascade and repair) and
    one ``drop_group``; it takes max(1, min(batch, batch * (part[-1] + 1) // depth)) rows, so its key
    buffer is no larger than that of a leave-one-out search of `batch` rows.  A part deeper than
    MAX_K (``logo_excludes``) instead runs one group-excluding ``topk_keys`` at depth part[-1] on
    `batch` rows: the mode's own path, or in a raw tensor-core mode the exact kernel, whose result
    the deeper search gave such rows."""
    gid, g_max, rows, buckets = plan
    n = feature_bank.shape[1]
    bank_rows = feature_bank.t()
    whole = len(buckets) == 1  # rows is arange(n): the queries are views
    for p, b_lo, b_hi in buckets:
        for part in logo_parts(ks_ascending, p, n, mode):
            excl = logo_excludes(part[-1], p, n)
            depth = part[-1] if excl else min(n, part[-1] + p)
            step = max(1, min(batch, batch * (part[-1] + 1) // depth))
            for lo in range(b_lo, b_hi, step):
                hi = min(b_hi, lo + step)
                q = bank_rows[lo:hi] if whole else bank_rows.index_select(0, rows[lo:hi])
                if q.stride(1) != 1:
                    q = q.contiguous()
                if excl:
                    # a row's own id is its group's, so the row itself is skipped with it
                    qg = gid[lo:hi] if whole else gid.index_select(0, rows[lo:hi])
                    yield part, lo, hi, topk_keys(q, feature_bank, depth, "exact" if mode in TC_MODES else mode,
                                                  exclude=(qg, gid, g_max))
                    continue
                yield part, lo, hi, drop_group(topk_keys(q, feature_bank, depth, mode), rows[lo:hi], gid, part[-1],
                                               flag)


def knn_predict_loo(feature_bank: torch.Tensor, feature_labels: torch.Tensor, num_classes: int,
                    knn_ks=(200,), knn_ts=(0.1,), batch: int = 75776,
                    groups: Optional[torch.Tensor] = None) -> torch.Tensor:
    """Leave-one-out kNN class rankings of a labelled bank against itself:
    (len(knn_ks), len(knn_ts), N, num_classes) int64, where [i, j, r] is bitwise
    ``knn_predict_multi(feature_bank[:, r:r+1].t(), bank without column r, labels without entry r,
    num_classes, knn_ks, knn_ts)[i, j, 0]`` in the default mode.

    Neighbours are ordered by (sim desc, index asc) and a pair's similarity does not depend on the
    other bank rows, so deleting row r leaves the order of the others unchanged: the top-k of the
    bank without r is the full bank's top-(k+1) list with r's own key removed (by index, so an exact
    duplicate of r stays), or its first k entries when r is not in it.  One search of the bank's
    rows at max(knn_ks) + 1 per batch of `batch` rows, one ``drop_self`` and one grid vote; the
    result does not depend on `batch`.  In a raw tensor-core mode a search at k + 1 > MAX_K comes
    from the exact kernel (as ``knn_predict`` serves k > MAX_K), so k = MAX_K gives the "exact"
    mode's leave-one-out result there.  feature_bank (D, N) as ``knn_predict`` takes it;
    max(knn_ks) < N.

    groups: optional (N,) integer ids (any values and integer dtype, on the bank's device) for
    leave-one-group-out: [i, j, r] is then the same call against the bank without every column c
    with groups[c] == groups[r] (``_knn_predict_logo``); groups=None is the path above, and
    groups=torch.arange(N) gives its result bitwise."""
    ks, ts, order = check_grid(knn_ks, knn_ts)
    if feature_bank.dim() != 2:
        raise RuntimeError("mat2 must be a matrix")
    N = feature_bank.shape[1]
    if feature_labels.numel() != N:
        raise RuntimeError(f"feature_labels has {feature_labels.numel()} entries for a bank of {N}")
    if groups is not None:
        return _knn_predict_logo(feature_bank, feature_labels, num_classes, ks, ts, order, batch, groups)
    if max(ks) >= N:  # the bank without the row has N - 1 rows
        raise RuntimeError("selected index k out of range")
    if int(batch) <= 0:
        raise ValueError(f"batch must be positive, got {batch}")
    mode = _default_mode
    parts = loo_parts(tuple(ks[i] for i in order), mode)
    for part in parts:
        check_vote_classes(num_classes, part[-1], grid=True)
    _require_cuda("feature_bank", feature_bank)
    _require_cuda("feature_labels", feature_labels)
    if feature_labels.device != feature_bank.device:
        raise RuntimeError("Expected all tensors to be on the same device, but found "
                           f"{feature_bank.device} and {feature_labels.device}")
    C = int(num_classes)
    labels = feature_labels.long().contiguous().view(-1)
    pred = torch.empty((N, len(ks) * len(ts) * C), dtype=torch.int64, device=feature_bank.device)
    with torch.cuda.device(feature_bank.device):
        flag = torch.zeros((1,), dtype=torch.int32, device=feature_bank.device)
        for lo in range(0, N, int(batch)):
            hi = min(N, lo + int(batch))
            q = feature_bank[:, lo:hi].t()  # bank rows lo..hi-1 as (b, D) queries, values unchanged
            if q.stride(1) != 1:
                q = q.contiguous()
            col = 0
            for part in parts:
                keys = drop_self(topk_keys(q, feature_bank, part[-1] + 1, mode), lo)
                _vote_multi_into(keys, labels, C, part, ts, pred[lo:hi, col:], -1, flag)
                col += len(part) * len(ts) * C
        _raise_vote_flag(int(flag.item()), C)
    return grid_view(pred, order, len(ts), C)


def _knn_predict_logo(feature_bank, feature_labels, num_classes, ks, ts, order, batch, groups) -> torch.Tensor:
    """``knn_predict_loo`` with every row's whole group left out.  Deleting G(r), the rows of r's
    group, leaves the (sim desc, index asc) order of the others unchanged, and at most g(r) = |G(r)|
    keys of a list are in G(r), so the top-k of the bank without G(r) is the full bank's
    top-(k + g(r)) list without the members of G(r), cut to k.  The search depth is min(N, k + p) with p the smallest
    power of two >= g(r), a function of the row alone, so the result does not depend on `batch`:
    rows are searched in buckets of equal p (``logo_parts``, ``_group_searches``) and voted into a
    bucket-ordered buffer that one permutation puts back in row order.  In a raw tensor-core mode a
    search deeper than MAX_K comes from the exact kernel, so such rows get the "exact" mode's
    result.  max(knn_ks) <= N - (largest group size).  One host read of the group statistics after
    torch.unique and one of the label flag."""
    N = feature_bank.shape[1]
    if int(batch) <= 0:
        raise ValueError(f"batch must be positive, got {batch}")
    # the class bound falls with k, so the search ending at max(knn_ks) is the worst part of any bucket
    check_vote_classes(num_classes, max(ks), grid=True)
    plan = _group_plan(groups, N, feature_bank.device)
    if max(ks) > N - plan[1]:  # the bank without the largest group has N - g_max rows
        raise RuntimeError("selected index k out of range")
    mode = _default_mode
    ks_ascending = tuple(ks[i] for i in order)
    _require_cuda("feature_bank", feature_bank)
    _require_cuda("feature_labels", feature_labels)
    if feature_labels.device != feature_bank.device:
        raise RuntimeError("Expected all tensors to be on the same device, but found "
                           f"{feature_bank.device} and {feature_labels.device}")
    C = int(num_classes)
    labels = feature_labels.long().contiguous().view(-1)
    pred = torch.empty((N, len(ks) * len(ts) * C), dtype=torch.int64, device=feature_bank.device)
    with torch.cuda.device(feature_bank.device):
        flag = torch.zeros((1,), dtype=torch.int32, device=feature_bank.device)
        for part, lo, hi, keys in _group_searches(feature_bank, plan, ks_ascending, mode, int(batch), flag):
            col = ks_ascending.index(part[0]) * len(ts) * C
            _vote_multi_into(keys, labels, C, part, ts, pred[lo:hi, col:], -1, flag)
        if len(plan[3]) > 1:  # bucket order -> row order
            pred = torch.empty_like(pred).index_copy_(0, plan[2], pred)
        _raise_vote_flag(int(flag.item()), C)
    return grid_view(pred, order, len(ts), C)


def grid_view(pred: torch.Tensor, order, n_t: int, num_classes: int) -> torch.Tensor:
    """(B, n_k*n_t*C) rankings over ks sorted by `order` -> (n_k, n_t, B, C) in the caller's order."""
    B = pred.shape[0]
    g = pred.view(B, len(order), n_t, int(num_classes)).permute(1, 2, 0, 3)
    inv = [0] * len(order)
    for pos, i in enumerate(order):
        inv[i] = pos
    return g[torch.tensor(inv, device=pred.device)] if inv != list(range(len(order))) else g.contiguous()


def knn_topk(feature: torch.Tensor, feature_bank: torch.Tensor, k: int, mode: Optional[str] = None,
             query_groups: Optional[torch.Tensor] = None,
             bank_groups: Optional[torch.Tensor] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """``torch.mm(feature, feature_bank).topk(k, dim=-1)`` without materialising the
    similarity matrix: (sims fp32 (B,k) sorted desc, idx int64 (B,k)), ties by lowest index.
    query_groups / bank_groups: as ``knn_predict_multi``; query b's list then skips every bank
    column of its group, and the indices are still those of the full bank."""
    exclude = _query_bank_exclusion(feature, feature_bank, query_groups, bank_groups, k)
    return decode_keys(topk_keys(feature, feature_bank, k, mode, exclude=exclude))


def plan_info(B: int, N: int, D: int, k: int, mode: Optional[str] = None) -> dict:
    lib = _lib.load()
    out = (ctypes.c_int64 * 9)()
    _lib.check(lib.b200knn_plan_info_ex(_lib.MODES[mode or _default_mode], B, N, D, k, out), "plan_info")
    names = ("n_qtiles", "splits", "split_rows", "n_items", "grid", "list_capacity", "chunks", "chunk_rows", "slots")
    return dict(zip(names, [int(v) for v in out]))
