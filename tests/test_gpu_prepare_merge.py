"""GPU: operand preparation and the key merge, bit for bit against numpy restatements.

b200knn_prepare_rows: every mode's stated rounding (BF16 round-to-nearest-even; TF32X3 hi rounded to
nearest with ties away from zero, lo = x - hi exactly; BF16X3; F16 / F16X2 round-to-nearest-even after
saturation to +-65504, lo only when a lo array is given; F32ROWS a copy), from fp32, fp16 and bf16
sources, in both layouts with a leading dimension larger than the natural one, with zero pad columns.
The inputs hold exact rounding ties, fp32 subnormals, the fp16 subnormal range and values either side
of 65504.  A rounding slip there (truncation for RNE, say) doubles the operand error and still passes
every tolerance downstream, so only a bitwise check sees it.

b200knn_merge: against oracle.knn_oracle.merge_keys_np with odd and even list lengths, k_out below k_in
and at every list-capacity boundary, 1 to 1,024 lists, both merge kernels, lists of exactly 64 and 65
keys, more than 4,096 staged keys, more identical keys than the sorting network holds, and unsorted
zero-terminated lists as the tensor-core kernel hands them over.  b200knn_key_sim_column on full and
empty slots.
"""
import numpy as np
import pytest
import torch

from b200knn import _lib
from b200knn import knn as K
from oracle import knn_oracle as O

gpu = pytest.mark.gpu
DEV = "cuda:0"


# ------------------------------------------------------------------ numpy restatement of prepare.cu
def bf16_rn(x: np.ndarray) -> np.ndarray:
    """fp32 -> bf16 bits, round to nearest, ties to even (finite inputs)."""
    u = x.astype(np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x7FFF + ((u >> 16) & 1)) >> 16).astype(np.uint16)


def bf16_val(h: np.ndarray) -> np.ndarray:
    return (h.astype(np.uint32) << 16).view(np.float32)


def tf32_rna(x: np.ndarray) -> np.ndarray:
    """fp32 -> tf32 (10 stored mantissa bits) in an fp32 container: round to nearest, ties away."""
    u = x.astype(np.float32).view(np.uint32).astype(np.uint64)
    return ((u + 0x1000) & 0xFFFFE000).astype(np.uint32).view(np.float32)


def f16_sat(x: np.ndarray) -> np.ndarray:
    return np.minimum(np.maximum(x, np.float32(-65504.0)), np.float32(65504.0)).astype(np.float16)


def prepare_ref(x: np.ndarray, mode: str, with_lo: bool, dim_pad: int):
    """(hi, lo) bit patterns of b200knn_prepare_rows for fp32 rows x (n, dim)."""
    n, dim = x.shape
    xp = np.zeros((n, dim_pad), dtype=np.float32)
    xp[:, :dim] = x
    if mode == "bf16":
        return bf16_rn(xp), None
    if mode == "bf16x3":
        hi = bf16_rn(xp)
        return hi, bf16_rn(xp - bf16_val(hi))
    if mode == "tf32x3":
        hi = tf32_rna(xp)
        return hi.view(np.uint32), (xp - hi).view(np.uint32)
    if mode in ("f16", "f16x2"):
        hi = f16_sat(xp)
        lo = f16_sat(xp - hi.astype(np.float32)) if with_lo else None
        return hi.view(np.uint16), None if lo is None else lo.view(np.uint16)
    assert mode == "f32rows"
    return xp.view(np.uint32), None


def special_rows(n: int, dim: int, seed: int) -> np.ndarray:
    """fp32 rows: random values among exact rounding ties of every target format, fp32 subnormals,
    the fp16 subnormal range and values either side of 65504."""
    rng = np.random.default_rng(seed)
    x = (rng.standard_normal((n, dim)) * np.exp2(rng.integers(-8, 8, (n, dim)))).astype(np.float32)
    u = x.view(np.uint32)
    flat = u.reshape(-1)
    m = flat.size
    pick = lambda frac: rng.random(m) < frac  # noqa: E731
    t = pick(0.08)
    flat[t] = (flat[t] & 0xFFFF0000) | 0x8000         # bf16 ties (both parities of the kept bit)
    t = pick(0.08)
    flat[t] = (flat[t] & 0xFFFFE000) | 0x1000         # tf32 ties
    h = rng.standard_normal(m).astype(np.float16)     # fp16 ties: midpoints of adjacent fp16 values
    mid = (h.astype(np.float32) + np.nextafter(h, np.float16(np.inf)).astype(np.float32)) * np.float32(0.5)
    t = pick(0.08) & np.isfinite(mid)
    flat[t] = mid[t].view(np.uint32)
    special = np.array([1e-40, -3e-42, 1.4e-45, -1.1754942e-38,               # fp32 subnormals
                        1e-5, -3e-7, 5.9604645e-08, 2.9802322e-08, -8.9406967e-08, 6.1035156e-05,  # fp16 subnormals
                        65503.9, 65504.0, -65504.0, 65519.996, 65520.0, -65536.0, 70000.0, -1e6,  # around 65504
                        0.0, -0.0, 1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11],
                       dtype=np.float32)
    t = pick(0.15)
    flat[t] = special[rng.integers(0, special.size, int(t.sum()))].view(np.uint32)
    return x


PREP_MODES = [("bf16", False), ("tf32x3", True), ("bf16x3", True), ("f16", False), ("f16", True),
              ("f16x2", False), ("f16x2", True), ("f32rows", False)]
MODE_CODES = dict(_lib.MODES, f32rows=_lib.MODE_F32ROWS)
TORCH_DT = {"f32": torch.float32, "f16": torch.float16, "bf16": torch.bfloat16}
OUT_DT = {"bf16": torch.int16, "bf16x3": torch.int16, "f16": torch.int16, "f16x2": torch.int16,
          "tf32x3": torch.int32, "f32rows": torch.int32}


@gpu
@pytest.mark.parametrize("layout", ["nd", "dn"])
@pytest.mark.parametrize("src_dtype", ["f32", "f16", "bf16"])
@pytest.mark.parametrize("mode,with_lo", PREP_MODES, ids=[f"{m}-{'lo' if lo else 'hi'}" for m, lo in PREP_MODES])
def test_prepare_rows_bitwise_equals_numpy(mode, with_lo, src_dtype, layout):
    n, dim = (131, 72) if layout == "nd" else (133, 200)   # neither D is a multiple of 64
    dim_pad = K.padded_dim(dim)
    xs = special_rows(n, dim, seed=dim + len(mode))
    if src_dtype == "f16":  # finite fp16 sources only (non-finite inputs have no contract)
        xs = np.clip(xs, -65504.0, 65504.0)
    x = torch.from_numpy(xs).to(DEV).to(TORCH_DT[src_dtype])
    want_hi, want_lo = prepare_ref(x.float().cpu().numpy(), mode, with_lo, dim_pad)
    if layout == "nd":   # (n, dim) rows inside an (n, dim + 9) buffer
        buf = torch.full((n, dim + 9), 7.0, dtype=x.dtype, device=DEV)
        buf[:, :dim] = x
        ld, code = dim + 9, _lib.LAYOUT_ND
    else:                # vectors are the columns of a (dim, n + 5) buffer
        buf = torch.full((dim, n + 5), 7.0, dtype=x.dtype, device=DEV)
        buf[:, :n] = x.t()
        ld, code = n + 5, _lib.LAYOUT_DN
    hi = torch.full((n, dim_pad), -1, dtype=OUT_DT[mode], device=DEV)   # pad columns must be written
    lo = torch.full((n, dim_pad), -1, dtype=OUT_DT[mode], device=DEV) if with_lo else None
    rc = _lib.load().b200knn_prepare_rows(buf.data_ptr(), K._DTYPES[x.dtype], code, n, dim, ld, MODE_CODES[mode],
                                          hi.data_ptr(), K._ptr(lo), torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "prepare_rows")
    np_dt = np.uint16 if OUT_DT[mode] == torch.int16 else np.uint32
    got_hi = hi.cpu().numpy().view(np_dt)
    assert not got_hi[:, dim:].any(), "pad columns of hi are not +0"
    bad = np.argwhere(got_hi != want_hi)
    assert bad.size == 0, f"hi: {len(bad)} elements differ, first at {bad[0]}: input {x.float().cpu().numpy()[tuple(bad[0])]!r}, " \
                          f"got {got_hi[tuple(bad[0])]:#x}, want {want_hi[tuple(bad[0])]:#x}"
    if with_lo:
        got_lo = lo.cpu().numpy().view(np_dt)
        assert not got_lo[:, dim:].any(), "pad columns of lo are not +0"
        bad = np.argwhere(got_lo != want_lo)
        assert bad.size == 0, f"lo: {len(bad)} elements differ, first at {bad[0]}: input {x.float().cpu().numpy()[tuple(bad[0])]!r}, " \
                              f"got {got_lo[tuple(bad[0])]:#x}, want {want_lo[tuple(bad[0])]:#x}"


def test_prepare_restatement_cpu():
    """The numpy restatement itself, on values whose rounding is known by hand."""
    x = np.array([[1.0 + 2.0 ** -8, 1.0 + 3 * 2.0 ** -8, 1.0 + 2.0 ** -11, 1.0 + 3 * 2.0 ** -11, 65519.0, 1e6, -2.0 ** -25, 1e-40]],
                 dtype=np.float32)
    hi, _ = prepare_ref(x, "bf16", False, 64)
    assert bf16_val(hi[0, :4]).tolist() == [1.0, 1.0 + 2.0 ** -6, 1.0, 1.0]                # ties to even
    assert bf16_val(hi[0, 7:8])[0] != 0                                                    # subnormal kept
    hi, lo = prepare_ref(x, "tf32x3", True, 64)
    h = hi.view(np.float32)[0]
    assert h[2] == np.float32(1.0 + 2.0 ** -10) and h[3] == np.float32(1.0 + 2.0 ** -9)     # ties away from zero
    assert np.array_equal(h[:8] + lo.view(np.float32)[0, :8], x[0])                         # hi + lo == x
    hi, lo = prepare_ref(x, "f16x2", True, 64)
    f = hi.view(np.float16)[0]
    assert f[2] == np.float16(1.0) and f[3] == np.float16(1.0 + 2.0 ** -9)                 # ties to even
    assert f[4] == np.float16(65504.0) and f[5] == np.float16(65504.0)                      # saturation
    assert lo.view(np.float16)[0, 5] == np.float16(65504.0)
    assert f[6] == 0 and np.signbit(f[6])                                                   # -2^-25: tie to -0


# ------------------------------------------------------------------ merge
def make_lists(rng, G, B, k_in, lengths, ordered, pool=None):
    """(G, B, k_in) uint64: list (g, b) holds lengths[g, b] non-empty keys, then zeros; descending
    when `ordered`, in random order otherwise.  pool: draw keys from it (duplicates across lists)."""
    if pool is None:
        keys = rng.integers(1, 2 ** 64 - 1, size=(G, B, k_in), dtype=np.uint64, endpoint=True)
    else:
        keys = pool[rng.integers(0, pool.size, size=(G, B, k_in))]
    if ordered:
        keys = np.sort(keys, axis=2)[:, :, ::-1]
    return np.where(np.arange(k_in)[None, None, :] < lengths[:, :, None], keys, np.uint64(0))


def run_merge(keys_np, k_out):
    t = torch.from_numpy(np.ascontiguousarray(keys_np).view(np.int64)).to(DEV)
    return K.merge_keys(t, k_out).cpu().numpy().view(np.uint64)


def lengths_of(rng, fill, G, B, k_in):
    if fill == "full":
        return np.full((G, B), k_in)
    if fill == "short":       # lists that ran under a shared threshold: the staged fast path
        return rng.integers(0, min(k_in, 40) + 1, (G, B))
    return rng.integers(0, k_in + 1, (G, B))  # "mixed": long lists take the warp-serial path


# (G, B, k_in, k_out, fill, ordered): k_out at every capacity boundary, odd and even k_in, k_out < k_in,
# merge_small_kernel (B < 1,184 and G >= 8) and merge_kernel (otherwise)
MERGE_CASES = [
    (1, 300, 1, 1, "full", True), (8, 64, 3, 16, "mixed", False), (74, 64, 16, 17, "short", True),
    (1024, 8, 7, 48, "mixed", False), (8, 1300, 49, 49, "full", True), (74, 1300, 20, 112, "short", False),
    (1024, 16, 113, 113, "short", True), (1, 2000, 241, 240, "full", False), (8, 64, 240, 241, "mixed", True),
    (74, 64, 992, 992, "mixed", False), (1024, 4, 992, 992, "short", True), (8, 1200, 500, 992, "full", True),
    (74, 1184, 16, 16, "short", False), (8, 100, 101, 50, "mixed", False), (2, 500, 993, 992, "mixed", True),
    (74, 3, 66, 17, "full", False), (1024, 2, 1, 1, "full", False),
]


@gpu
@pytest.mark.parametrize("G,B,k_in,k_out,fill,ordered", MERGE_CASES,
                         ids=[f"G{c[0]}-B{c[1]}-kin{c[2]}-kout{c[3]}-{c[4]}-{'sorted' if c[5] else 'unsorted'}" for c in MERGE_CASES])
def test_merge_equals_numpy(G, B, k_in, k_out, fill, ordered):
    rng = np.random.default_rng(G * 7919 + k_out)
    keys = make_lists(rng, G, B, k_in, lengths_of(rng, fill, G, B, k_in), ordered)
    assert np.array_equal(run_merge(keys, k_out), O.merge_keys_np(keys, k_out))


@gpu
@pytest.mark.parametrize("long_len", [64, 65])
@pytest.mark.parametrize("k_in", [80, 81])
def test_merge_list_of_64_and_65_keys(long_len, k_in):
    """merge_small_kernel stages lists of up to 64 keys; one of 65 sends the row down the slow path."""
    rng = np.random.default_rng(long_len + k_in)
    G, B = 8, 32
    lengths = rng.integers(0, 11, (G, B))
    lengths[3] = long_len
    for ordered in (True, False):
        keys = make_lists(rng, G, B, k_in, lengths, ordered)
        for k_out in (48, 200):
            assert np.array_equal(run_merge(keys, k_out), O.merge_keys_np(keys, k_out)), (ordered, k_out)


@gpu
def test_merge_more_than_4096_staged_keys():
    rng = np.random.default_rng(3)
    G, B, k_in = 74, 64, 64
    lengths = np.full((G, B), 60)          # 4,440 keys: beyond the 4,096-key staging buffer
    lengths[:, ::2] = rng.integers(50, 64, (G, B // 2))
    for ordered in (True, False):
        keys = make_lists(rng, G, B, k_in, lengths, ordered)
        for k_out in (16, 200, 992):
            assert np.array_equal(run_merge(keys, k_out), O.merge_keys_np(keys, k_out)), (ordered, k_out)


@gpu
@pytest.mark.parametrize("G,B", [(74, 64), (148, 1300), (8, 5)])
def test_merge_identical_keys_beyond_the_network(G, B):
    """The sample's index-0 keys: many lists of the same value — more identical keys than the
    list capacity, which no radix-select threshold can separate."""
    rng = np.random.default_rng(G + B)
    same = O.make_keys(np.array([0.25], np.float32), np.array([0]))
    pool = np.concatenate([np.repeat(same, 50), O.make_keys(rng.standard_normal(6).astype(np.float32), np.zeros(6, np.int64))])
    for k_in, k_out in ((16, 16), (17, 64), (40, 112)):
        lengths = rng.integers(k_in // 2, k_in + 1, (G, B))
        keys = make_lists(rng, G, B, k_in, lengths, True, pool=pool)
        got = run_merge(keys, k_out)
        assert np.array_equal(got, O.merge_keys_np(keys, k_out)), (k_in, k_out)


@gpu
def test_key_sim_column_decodes_full_and_empty_slots():
    rng = np.random.default_rng(11)
    B, k = 1000, 37
    sims = rng.standard_normal((B, k)).astype(np.float32)
    sims[::3, 5] = -0.0
    sims[1::7, 9] = 1e-42
    keys = O.make_keys(sims, rng.integers(0, 2 ** 31, (B, k)))
    keys[::4, 20:] = 0                     # empty slots decode to -inf
    keys[5] = 0
    t = torch.from_numpy(keys.view(np.int64)).to(DEV)
    want, _ = O.decode_keys(keys)
    lib = _lib.load()
    for j in (0, 5, 9, 19, 20, k - 1):
        out = torch.full((B,), float("nan"), dtype=torch.float32, device=DEV)
        _lib.check(lib.b200knn_key_sim_column(t.data_ptr(), B, k, j, out.data_ptr(),
                                              torch.cuda.current_stream().cuda_stream), "key_sim_column")
        assert np.array_equal(out.cpu().numpy().view(np.uint32), want[:, j].view(np.uint32)), j
    assert torch.equal(K.kth_sim(t).cpu().view(torch.int32), torch.from_numpy(want[:, -1].copy()).view(torch.int32))
