"""GPU: the tensor-core top-k (tc_topk_kernel) bit for bit against its own similarity tiles.

The selection of every raw tensor-core mode is meant to be exact: the keys it returns are the
canonical top-k (sim desc, index asc) of the fp32 similarities it computed in TMEM.  The debug entry
point dumps those similarities; the reference here builds the canonical keys from the dumped bits with
torch integer ops and selects with torch.topk — no b200knn kernel takes part in it.  Every case checks
(a) the pipeline diagnostic word is 0 and the dump is within the mode's tolerance of an fp64 GEMM of the
prepared operands, (b) the debug keys equal the reference bitwise, (c) the product build returns the
same keys, and (d) for CTA pairs, every dumped row is bitwise the row of a single-CTA run of the same
queries.  The cases reach every (mode, single / pair, tile width) at every list capacity, bank splits
merged by both merge kernels, the chunk-major order, ragged shapes and the similarity patterns where
selection goes wrong (every column qualifying, ties across the k-th cut and the split and chunk
boundaries, all-equal rows, signed zeros, negative-only similarities).  Then the options of
b200knn_topk_opt against the dump of a plain call: tau0, group ids, bank_row_stride and the sample.
"""
import numpy as np
import pytest
import torch

from b200knn import _lib
from b200knn import knn as K
from oracle import knn_oracle as O

DEV = "cuda:0"
gpu = pytest.mark.gpu
SIGN = -(1 << 63)        # int64 with only the top bit set: flips a uint64 key to a signed-sortable one
CAPS = ((1, 16), (17, 48), (49, 112), (113, 240), (241, 992))  # k range of list capacity 64 .. 1024


# ------------------------------------------------------------------ reference (torch integer ops only)
def sortable_keys(sims: torch.Tensor) -> torch.Tensor:
    """(R, N) fp32 similarities -> (R, N) int64 whose signed order is the canonical key order:
    orderable(sim) << 32 | (0xFFFFFFFF - column), -0 counted as +0, with the top bit flipped so that
    signed int64 compares like the uint64 keys of include/b200knn.h (key == sortable ^ SIGN)."""
    b = sims.contiguous().view(torch.int32).to(torch.int64) & 0xFFFFFFFF
    b = torch.where(b == 0x80000000, torch.zeros_like(b), b)  # -0 -> +0
    o = torch.where(b >= 0x80000000, b ^ 0xFFFFFFFF, b | 0x80000000)
    col = torch.arange(sims.shape[1], device=sims.device, dtype=torch.int64)
    return (o - (1 << 31)) * (1 << 32) + (0xFFFFFFFF - col)


def ref_topk(sims: torch.Tensor, k: int, drop=None, block_elems: int = 1 << 27) -> torch.Tensor:
    """Canonical top-k keys (uint64 bits in int64) of every row of `sims`; columns where
    drop(r0, r1) is True are never selected, and rows with fewer than k others are zero-filled."""
    R, N = sims.shape
    out = torch.empty((R, k), dtype=torch.int64, device=sims.device)
    rows = max(1, block_elems // max(1, N))
    for r0 in range(0, R, rows):
        r1 = min(R, r0 + rows)
        s = sortable_keys(sims[r0:r1])
        if drop is not None:
            s.masked_fill_(drop(r0, r1), SIGN)  # SIGN ^ SIGN == 0: an empty slot
        out[r0:r1] = torch.topk(s, k, dim=1).values ^ SIGN
    return out


def chunk_max_keys(sims: torch.Tensor, r: int = 16) -> torch.Tensor:
    """The sample option's stated result: the r largest 32-column chunk maxima of each row as keys
    with index field 0, sorted descending, 0 for a missing value."""
    R, N = sims.shape
    pad = (-N) % 32
    x = torch.nn.functional.pad(sims, (0, pad), value=float("-inf")).view(R, -1, 32).amax(dim=2)
    top = torch.topk(x, min(r, x.shape[1]), dim=1).values
    top = torch.nn.functional.pad(top, (0, r - top.shape[1]), value=float("-inf"))
    keys = (sortable_keys(top) ^ SIGN) | 0xFFFFFFFF  # index field 0
    return torch.where(torch.isinf(top) & (top < 0), torch.zeros_like(keys), keys)


def test_reference_helper_matches_oracle_cpu():
    """The reference of this file against the oracle's canonical top-k, on the CPU: random values,
    exact ties, signed zeros, negatives, subnormals and infinities."""
    rng = np.random.default_rng(7)
    R, N, k = 40, 777, 50
    s = rng.standard_normal((R, N)).astype(np.float32)
    s[:, ::7] = np.round(s[:, ::7], 1)                       # ties
    s[3] = 0.0
    s[3, ::2] = -0.0                                         # signed zeros only
    s[4] = 1.5                                               # one value
    s[5, :100] = -np.abs(s[5, :100])
    s[6, 10:20] = np.float32(1e-42)                          # subnormals
    s[6, 30] = -np.float32(1e-42)
    s[7, 5], s[7, 6] = np.inf, -np.inf
    s[8] = -np.abs(s[8])                                     # negative only
    want = O.make_keys(*O.canonical_topk_c(s, k))
    got = ref_topk(torch.from_numpy(s), k, block_elems=5 * N).numpy().view(np.uint64)
    assert np.array_equal(got, want)
    # and with dropped columns: the same as the oracle on -inf-free rows restricted by hand
    drop = torch.from_numpy(rng.random((R, N)) < 0.9)
    got = ref_topk(torch.from_numpy(s), k, drop=lambda a, b: drop[a:b]).numpy().view(np.uint64)
    for r in range(R):
        keep = np.flatnonzero(~drop[r].numpy())
        full = O.make_keys(s[r, keep], keep)
        order = np.argsort(full)[::-1][:k]
        w = np.zeros(k, dtype=np.uint64)
        w[:order.size] = full[order]
        assert np.array_equal(got[r], w), r
    # the sample reference: chunk maxima as index-0 keys
    cm = chunk_max_keys(torch.from_numpy(s[:, :100].copy())).numpy().view(np.uint64)
    for r in range(R):
        m = np.concatenate([s[r, :100], np.full(28, -np.inf, np.float32)]).reshape(4, 32).max(axis=1)
        w = np.sort(O.make_keys(m, np.zeros(4, np.int64)))[::-1]
        assert np.array_equal(cm[r, :4], w) and not cm[r, 4:].any(), r


# ------------------------------------------------------------------ GPU plumbing
@pytest.fixture(autouse=True)
def chunk_guard():
    yield
    if torch.cuda.is_available():
        _lib.load().b200knn_set_l2_chunk_bytes(40 << 20)


def set_chunk_bytes(n):
    assert _lib.load().b200knn_set_l2_chunk_bytes(n) == 0


def prepare(q, bank, mode):
    return (K.prepare_rows(q, mode, vectors_are_columns=False), K.prepare_rows(bank, mode, vectors_are_columns=True))


def debug_dump(mode, pq, pb, B, N, D, k):
    """b200knn_debug_topk_dump: (keys (B, k), dump (B, N)) of a plain search."""
    lib = _lib.load()
    keys = torch.zeros((B, k), dtype=torch.int64, device=DEV)
    dump = torch.full((B, N), float("nan"), dtype=torch.float32, device=DEV)
    diag = torch.zeros(4, dtype=torch.int32, device=DEV)
    ws_bytes = lib.b200knn_topk_workspace_bytes(B, N, D, k, _lib.MODES[mode])
    ws = torch.empty(ws_bytes, dtype=torch.uint8, device=DEV)
    rc = lib.b200knn_debug_topk_dump(_lib.MODES[mode], pq.hi.data_ptr(), K._ptr(pq.lo), pb.hi.data_ptr(),
                                     K._ptr(pb.lo), B, N, D, k, keys.data_ptr(), ws.data_ptr(), ws_bytes,
                                     dump.data_ptr(), diag.data_ptr(), 0, torch.cuda.current_stream().cuda_stream)
    _lib.check(rc, "debug_topk_dump")
    torch.cuda.synchronize()
    assert diag.tolist() == [0, 0, 0, 0], f"pipeline wait timed out: {diag.tolist()}"
    assert not bool(dump.isnan().any()), "some similarity tile was never written"
    return keys, dump


def _f64(p, D):
    x = p.hi.double()
    if p.lo is not None:
        x = x + p.lo.double()
    return x[:, :D]


def check_tiles(mode, pq, pb, dump, D, one_sign=False):
    """(a): the dump against an fp64 GEMM of the prepared operands, within the tolerances of
    test_gpu_tc.py::test_tiles_and_selection (scaled by the row norms; widened in proportion to D
    beyond 512, the longest accumulation that test reaches).  Those tolerances hold for operands of
    both signs; when every product has one sign nothing cancels, the fp32 accumulator carries the
    full similarity at every step and its rounding error is larger (measured on a B200: up to 1.4x
    the two-sign tolerance in f16), so one-sign operands are allowed twice the tolerance."""
    qf, bf = _f64(pq, D), _f64(pb, D)
    qn, bn = float(qf.norm(dim=1).max()), float(bf.norm(dim=1).max())
    longer = max(1.0, K.padded_dim(D) / 512) * (2.0 if one_sign else 1.0)
    if mode in ("bf16", "f16"):
        tol = 2e-6 * max(1.0, qn * bn)
    elif mode == "f16x2":
        tol = 4e-6 * max(1.0, qn * bn)
    elif mode == "bf16x3":
        tol = 6e-5 * max(qn * bn, 1e-30)
    else:
        tol = None  # tf32x3: 1e-5 relative to the largest similarity, below
    err, top = 0.0, 0.0
    rows = max(1, (1 << 26) // max(1, dump.shape[1]))
    for r0 in range(0, dump.shape[0], rows):
        ref = qf[r0:r0 + rows] @ bf.t()
        err = max(err, float((dump[r0:r0 + rows].double() - ref).abs().max()))
        top = max(top, float(ref.abs().max()))
    if tol is None:
        tol = 1e-5 * max(1.0, top)
    assert err <= tol * longer, f"{mode} tile error {err} > {tol * longer}"


def plan_of(mode, B, N, D, k):
    return K.plan_info(B, N, D, k, mode)


def uses_pair(mode, B):
    return mode in ("bf16", "f16", "f16x2") and B > 128


def assert_plan(mode, B, N, D, k, plan):
    """The plan reaches the kernel variant the case is for: CTA pairs (256-row query tiles) exactly
    when tc_use_pair says so, and the list capacity of k."""
    tile_m = 256 if uses_pair(mode, B) else 128
    assert plan["n_qtiles"] == -(-B // tile_m), (mode, B, plan)
    assert plan["list_capacity"] == next(c for c, (lo, hi) in zip((64, 128, 256, 512, 1024), CAPS) if lo <= k <= hi)


# ------------------------------------------------------------------ data
def make_data(pattern, B, N, D, seed):
    """(q (B, D), bank (D, N)) fp32 on the GPU."""
    g = torch.Generator(device=DEV).manual_seed(seed)
    nrm = torch.nn.functional.normalize
    if pattern == "unit":
        bank = nrm(torch.randn(N, D, generator=g, device=DEV), dim=1)
        q = nrm(torch.randn(B, D, generator=g, device=DEV), dim=1)
    elif pattern == "rising":
        # integer rows: sim = +-(n + offset), exact in every mode and accumulation order.  Rows with
        # + see every column beat the previous ones (every column qualifies, the list overflows and is
        # pruned after every 32 columns); rows with - see only the first k qualify.
        n = torch.arange(N, device=DEV)
        bank = torch.zeros(N, D, device=DEV)
        bank[:, 0], bank[:, 1], bank[:, 2] = (n // 256).float(), (n % 256).float(), 2.0
        b = torch.arange(B, device=DEV)
        sgn = torch.where(b % 3 == 2, -1.0, 1.0)
        q = torch.zeros(B, D, device=DEV)
        q[:, 0], q[:, 1] = 256.0 * sgn, sgn
        q[:, 2] = torch.where(b % 2 == 1, -32768.0, 0.0)  # odd rows: negative similarities only
    elif pattern == "dup":
        # every row three times, at n, n + M, n + 2M: ties across the k-th cut, splits and chunks
        M = N // 3 + 5
        base = nrm(torch.randn(M, D, generator=g, device=DEV), dim=1)
        bank = base[torch.arange(N, device=DEV) % M]
        src = torch.randint(0, M, (B,), generator=g, device=DEV)
        q = nrm(base[src] + 0.1 * torch.randn(B, D, generator=g, device=DEV), dim=1)
    elif pattern == "equal":
        bank = nrm(torch.randn(1, D, generator=g, device=DEV), dim=1).repeat(N, 1)
        q = nrm(torch.randn(B, D, generator=g, device=DEV), dim=1)
        q[::5] = 0.0  # zero queries
    elif pattern == "zeroq":
        # zero queries against rows of one sign each: +0 and -0 products
        sgn = torch.where(torch.rand(N, generator=g, device=DEV) < 0.5, -1.0, 1.0)
        bank = nrm(torch.randn(N, D, generator=g, device=DEV), dim=1).abs() * sgn[:, None]
        q = nrm(torch.randn(B, D, generator=g, device=DEV), dim=1)
        q[::2] = 0.0
    elif pattern == "neg":
        bank = -nrm(torch.randn(N, D, generator=g, device=DEV), dim=1).abs()
        q = nrm(torch.randn(B, D, generator=g, device=DEV), dim=1).abs()
    else:
        raise ValueError(pattern)
    return q.contiguous(), bank.t().contiguous()


PATTERNS = ("unit", "rising", "dup", "equal", "zeroq", "neg")


def run_case(mode, q, bank, k, pair_check=True, one_sign=False):
    """(a)-(d) for one search; returns (pq, pb, dump) for option checks."""
    B, D = q.shape
    N = bank.shape[1]
    pq, pb = prepare(q, bank, mode)
    keys, dump = debug_dump(mode, pq, pb, B, N, D, k)
    check_tiles(mode, pq, pb, dump, D, one_sign)                               # (a)
    ref = ref_topk(dump, k)
    bad = (keys != ref).any(dim=1).nonzero().view(-1)
    assert bad.numel() == 0, f"{mode}: {bad.numel()} rows differ from the tiles' top-{k}, first {bad[:8].tolist()}"  # (b)
    assert torch.equal(K._search(mode, pq, pb, B, N, D, k), keys)              # (c)
    if pair_check and uses_pair(mode, B):                                      # (d)
        for r0 in (0, 128):
            r1 = min(B, r0 + 128)
            sq = K.prepare_rows(q[r0:r1].contiguous(), mode, vectors_are_columns=False)
            _, single = debug_dump(mode, sq, pb, r1 - r0, N, D, k)
            same = (single.view(torch.int32) == dump[r0:r1].view(torch.int32)).all(dim=1)
            assert bool(same.all()), f"{mode}: pair rows {(~same).nonzero().view(-1)[:8].tolist()} (+{r0}) differ from a single-CTA run"
    return pq, pb, dump


# ------------------------------------------------------------------ 1. every kernel variant x capacity
# (mode, B, D): single CTAs at B <= 128, CTA pairs above; resident-query modes with 256-wide bank tiles
# (D_pad <= 512) and 128-wide ones (D_pad 576..768); the streamed-query modes at D = 64, 200, 1024
VARIANTS = [(m, B, D) for m in ("bf16", "f16", "f16x2") for B, D in ((100, 72), (300, 512), (77, 640), (300, 768))]
VARIANTS += [(m, B, D) for m in ("bf16x3", "tf32x3") for B, D in ((100, 64), (300, 200), (64, 1024))]
MATRIX = []
for _i, (_m, _B, _D) in enumerate(VARIANTS):
    for _c, (_lo, _hi) in enumerate(CAPS):
        _k = (_lo, _hi)[(_i + _c) % 2]
        MATRIX.append((_m, _B, _D, _k, 1500 + 37 * _i + 11 * _c, PATTERNS[(_i + _c) % len(PATTERNS)]))
# k = N and banks smaller than one tile
MATRIX += [("bf16", 100, 72, 100, 100, "unit"), ("f16x2", 300, 128, 200, 200, "dup"), ("f16", 129, 640, 97, 97, "neg"),
           ("tf32x3", 5, 200, 33, 33, "rising"), ("bf16x3", 300, 64, 992, 992, "equal"), ("bf16", 2, 16, 1, 17, "zeroq")]


@gpu
@pytest.mark.parametrize("mode,B,D,k,N,pattern", MATRIX, ids=[f"{m}-B{B}-D{D}-k{k}-N{N}-{p}" for m, B, D, k, N, p in MATRIX])
def test_selection_equals_tiles(mode, B, D, k, N, pattern):
    assert_plan(mode, B, N, D, k, plan_of(mode, B, N, D, k))
    if K.padded_dim(D) > 512 and mode in ("bf16", "f16", "f16x2"):
        assert K.padded_dim(D) <= K.MAX_BF16_DIM  # 128-wide bank tiles (tc_tile_n)
    q, bank = make_data(pattern, B, N, D, seed=sum(map(ord, mode)) + B + D + k + N)
    run_case(mode, q, bank, k, one_sign=(pattern == "neg"))


# ------------------------------------------------------------------ 2. plans: splits, both merges, chunks
# (mode, B, N, D, k, pattern, chunk bytes or None, what the plan must show)
PLANS = [
    ("bf16", 64, 200003, 128, 200, "unit", None, "merge_small"),      # splits >= 8, B < 1,184
    ("f16x2", 100, 150001, 256, 17, "dup", None, "merge_small"),
    ("tf32x3", 64, 80011, 64, 992, "rising", None, "merge_small"),
    ("bf16", 1300, 100003, 128, 100, "dup", None, "merge_kernel"),    # splits > 1, B >= 1,184
    ("bf16x3", 1200, 60001, 200, 240, "unit", None, "merge_kernel"),
    ("f16", 1250, 90001, 72, 5, "rising", None, "merge_kernel"),
    ("bf16", 37800, 9001, 128, 100, "dup", 1 << 20, "chunks"),       # chunk-major, ragged last chunk
    ("f16", 37800, 9001, 72, 300, "rising", 300 << 10, "chunks"),
    ("f16x2", 37800, 7001, 128, 48, "unit", 300 << 10, "chunks"),
    ("tf32x3", 37800, 5003, 64, 200, "dup", 1 << 20, "chunks"),
    ("bf16x3", 37800, 6007, 128, 16, "neg", 300 << 10, "chunks"),
]


def assert_plan_kind(plan, B, what):
    if what == "merge_small":
        assert plan["splits"] >= 8 and B < 1184, plan   # launch_merge_t: merge_small_kernel
    elif what == "merge_kernel":
        assert plan["splits"] > 1 and B >= 1184, plan   # merge_kernel
    elif what == "chunks":
        assert plan["chunks"] > 1 and plan["splits"] == 1, plan


@gpu
@pytest.mark.parametrize("mode,B,N,D,k,pattern,chunk,what", PLANS, ids=[f"{p[0]}-{p[7]}-B{p[1]}-k{p[4]}" for p in PLANS])
def test_selection_equals_tiles_plans(mode, B, N, D, k, pattern, chunk, what):
    if chunk is not None:
        set_chunk_bytes(chunk)
    plan = plan_of(mode, B, N, D, k)
    assert_plan(mode, B, N, D, k, plan)
    assert_plan_kind(plan, B, what)
    if what == "chunks":
        assert N % plan["chunk_rows"] % 32, plan  # the last chunk ends inside a 32-column group
    q, bank = make_data(pattern, B, N, D, seed=B + N)
    run_case(mode, q, bank, k, pair_check=(what != "chunks"), one_sign=(pattern == "neg"))


# ------------------------------------------------------------------ 3. options of b200knn_topk_opt
def _thresholds(dump, k):
    """Per-row tau0 at several ranks of the row (each exactly one of its similarities), -inf, and one
    above every similarity (an all-empty row)."""
    B, N = dump.shape
    srt = torch.sort(dump, dim=1, descending=True).values
    ranks = [r for r in (1, max(1, k // 2), k, min(N, 2 * k), min(N, 5 * k)) if r <= N]
    tau = torch.empty(B, dtype=torch.float32, device=DEV)
    b = torch.arange(B, device=DEV)
    n_kind = len(ranks) + 2
    for j, r in enumerate(ranks):
        sel = b % n_kind == j
        tau[sel] = srt[sel, r - 1]
    tau[b % n_kind == len(ranks)] = float("-inf")
    top = b % n_kind == len(ranks) + 1
    tau[top] = torch.nextafter(srt[top, 0], torch.tensor(float("inf"), device=DEV))
    return tau


# (mode, B, N, D, k, pattern, chunk bytes or None, what the plan must show or None)
TAU_CASES = [
    ("bf16", 100, 3001, 128, 50, "unit", None, None),
    ("f16", 300, 2999, 256, 200, "dup", None, None),              # CTA pair
    ("bf16x3", 64, 100003, 128, 100, "unit", None, "merge_small"),
    ("f16x2", 1300, 80001, 128, 20, "rising", None, "merge_kernel"),
    ("bf16", 37800, 9001, 128, 64, "dup", 300 << 10, "chunks"),
    ("tf32x3", 100, 4001, 200, 992, "equal", None, None),
]


@gpu
@pytest.mark.parametrize("mode,B,N,D,k,pattern,chunk,what", TAU_CASES, ids=[f"{c[0]}-B{c[1]}-k{c[4]}-{c[5]}" for c in TAU_CASES])
def test_tau0_option_equals_filtered_tiles(mode, B, N, D, k, pattern, chunk, what):
    """tau0: the top-k of the columns with sim > tau0[b] (strict), zero-filled."""
    if chunk is not None:
        set_chunk_bytes(chunk)
    plan = plan_of(mode, B, N, D, k)
    assert_plan(mode, B, N, D, k, plan)
    if what:
        assert_plan_kind(plan, B, what)
    q, bank = make_data(pattern, B, N, D, seed=k + N)
    pq, pb = prepare(q, bank, mode)
    _, dump = debug_dump(mode, pq, pb, B, N, D, k)
    tau = _thresholds(dump, k)
    got = K._search(mode, pq, pb, B, N, D, k, tau0=tau)
    want = ref_topk(dump, k, drop=lambda r0, r1: dump[r0:r1] <= tau[r0:r1, None])
    bad = (got != want).any(dim=1).nonzero().view(-1)
    assert bad.numel() == 0, f"{bad.numel()} rows differ, first {bad[:8].tolist()}"
    assert bool((got[tau > dump.amax(dim=1)] == 0).all())


GROUP_CASES = [(m, B, k, p) for i, (m, B) in enumerate([("bf16", 100), ("f16x2", 300), ("tf32x3", 64), ("f16", 200)])
               for j, (lo, hi) in enumerate(CAPS) for k, p in [((lo, hi)[(i + j) % 2], PATTERNS[(i + j) % len(PATTERNS)])]]


@gpu
@pytest.mark.parametrize("mode,B,k,pattern", GROUP_CASES, ids=[f"{m}-B{B}-k{k}-{p}" for m, B, k, p in GROUP_CASES])
def test_group_option_equals_masked_tiles(mode, B, k, pattern):
    """Group ids (the EXCL kernels): the top-k of the dump with the row's own group masked,
    zero-filled when fewer than k columns remain."""
    N, D = 2011, 128
    assert_plan(mode, B, N, D, k, plan_of(mode, B, N, D, k))
    q, bank = make_data(pattern, B, N, D, seed=7 * k + B)
    g = torch.Generator(device=DEV).manual_seed(k)
    bg = (torch.arange(N, device=DEV) // 25).to(torch.int32)
    bg[N // 4:N // 4 + 1200] = 1000       # one group of 1,200 rows: its queries keep 811 < k columns at k = 992
    qg = bg[torch.randint(0, N, (B,), generator=g, device=DEV)].contiguous()
    qg[::4] = 1000
    qg[1::9] = -5                         # no bank row has this id
    pq, pb = prepare(q, bank, mode)
    _, dump = debug_dump(mode, pq, pb, B, N, D, k)
    got = K._search(mode, pq, pb, B, N, D, k, groups=(qg, bg))
    want = ref_topk(dump, k, drop=lambda r0, r1: bg[None, :] == qg[r0:r1, None])
    bad = (got != want).any(dim=1).nonzero().view(-1)
    assert bad.numel() == 0, f"{bad.numel()} rows differ, first {bad[:8].tolist()}"


STRIDE_CASES = [("bf16", 100, 30011, 128, 40, 3, True), ("f16x2", 300, 40001, 256, 150, 8, True),
                ("tf32x3", 64, 200003, 64, 100, 62, True), ("bf16x3", 130, 20001, 200, 300, 5, False)]


@gpu
@pytest.mark.parametrize("mode,B,N,D,k,stride,with_tau", STRIDE_CASES, ids=[f"{c[0]}-s{c[5]}-k{c[4]}" for c in STRIDE_CASES])
def test_row_stride_option_equals_tiles_of_the_strided_bank(mode, B, N, D, k, stride, with_tau):
    """bank_row_stride s (with tau0): the reference is the dump of bank[:, ::s] prepared contiguously;
    indices are visit indices."""
    q, bank = make_data("unit", B, N, D, seed=stride)
    sub = bank[:, ::stride].contiguous()
    n_visit = sub.shape[1]
    assert n_visit == -(-N // stride)
    pq, pb = prepare(q, bank, mode)
    ps = K.prepare_rows(sub, mode, vectors_are_columns=True)
    _, dump = debug_dump(mode, pq, ps, B, n_visit, D, k)
    tau = _thresholds(dump, k) if with_tau else None
    got = K._search(mode, pq, pb, B, n_visit, D, k, stride=stride, tau0=tau)
    drop = (lambda r0, r1: dump[r0:r1] <= tau[r0:r1, None]) if with_tau else None
    want = ref_topk(dump, k, drop=drop)
    bad = (got != want).any(dim=1).nonzero().view(-1)
    assert bad.numel() == 0, f"{bad.numel()} rows differ, first {bad[:8].tolist()}"


SAMPLE_CASES = [("bf16", 200, 300000, 512, 62, "unit"), ("tf32x3", 513, 40000, 128, 8, "dup"),
                ("f16x2", 64, 811457, 128, 62, "unit"), ("f16", 3, 4096, 128, 1, "rising"),
                ("bf16", 64, 200003, 128, 1, "equal"), ("bf16x3", 100, 1000, 64, 1, "neg")]


@gpu
@pytest.mark.parametrize("mode,B,N,D,stride,pattern", SAMPLE_CASES, ids=[f"{c[0]}-B{c[1]}-s{c[4]}-{c[5]}" for c in SAMPLE_CASES])
def test_sample_option_is_the_top16_chunk_maxima(mode, B, N, D, stride, pattern):
    """sample: the 16 largest 32-column chunk maxima of the visited columns, as keys with index 0
    (bank splits merged; on the all-equal bank every split returns 16 identical keys, more than the
    merge's network holds)."""
    q, bank = make_data(pattern, B, N, D, seed=N + stride)
    sub = bank[:, ::stride].contiguous()
    n_visit = sub.shape[1]
    pq, pb = prepare(q, bank, mode)
    ps = K.prepare_rows(sub, mode, vectors_are_columns=True)
    plan = plan_of(mode, B, n_visit, D, 16)
    _, dump = debug_dump(mode, pq, ps, B, n_visit, D, 16)
    got = K._search(mode, pq, pb, B, n_visit, D, 16, stride=stride, sample=True)
    want = chunk_max_keys(dump)
    bad = (got != want).any(dim=1).nonzero().view(-1)
    assert bad.numel() == 0, f"splits {plan['splits']}: {bad.numel()} rows differ, first {bad[:8].tolist()}"
    if pattern == "equal":
        assert plan["splits"] * 16 > 64, plan  # > CAP identical keys reach the merge
