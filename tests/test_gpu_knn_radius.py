"""GPU: knn_radius / radius_graph / near_duplicate_groups (b200knn/retrieval.py).
 * "exact" equals sims_seqfma(q, bank) >= tau32 of the CPU oracle, in canonical order, on both real
   golden banks (raw and normalised) and a synthetic 37,348-row bank;
 * the fp32 modes are bitwise "exact" on the four data kinds with planted near-duplicate groups of 2,
   5, 40 and 1,500 rows (every ladder level), at D = 384 / 512 / 768 / 1024 (the wide first level),
   and on 256 rows of the 811,457-row bank; the other fp32 levels (f16x2, bf16, tf32); thresholds
   at an exact pair similarity; fp16 rounding-midpoint rows (the residual terms of E) and
   fp16-exact adversarial rows, with tau just below the pair the fp16 pass underestimates most;
 * b200knn_radius_tau0 against the host restatement at the E it reports, and its refusal path
   (query norms beyond the fp16 range);
 * raw tensor-core modes equal their own topk_keys(..., 992, mode) cut at tau32;
 * max_per_row, saturation, peeling past 992, nnz = 0, B = 0, N < 32, argument errors;
 * radius_graph's self removal by index and batch invariance, and its rows at the default cap
   (993 keys with their own) searched with their own row left out instead of peeled; near_duplicate_groups against scipy's
   components of the exact edge set; knn_predict_loo(groups=near_duplicate_groups(...)[0])."""
import os

import numpy as np
import pytest
import torch
from scipy.sparse import csr_matrix
from scipy.sparse.csgraph import connected_components

import b200knn
import bench
import datagen
from b200knn import _lib
from b200knn import knn as K
from b200knn import retrieval as R
from oracle import knn_oracle as O
from test_gpu_round2 import _adversarial
from test_gpu_tc import run_dump
from test_residual_bound_cpu import e_new

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
F32 = np.float32
GOLDEN = os.path.join(os.path.dirname(__file__), "golden")


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _ref(q, bank_dn, tau, self_offset=-1, cap=None):
    """CSR rows of the oracle: columns with seqfma sim >= fp32(tau), (sim desc, index asc)."""
    s = O.sims_seqfma(np.ascontiguousarray(q, dtype=np.float32), np.ascontiguousarray(bank_dn, dtype=np.float32))
    t = F32(tau)
    offs, idx, sims = [0], [], []
    for b in range(s.shape[0]):
        c = np.nonzero(s[b] >= t)[0]
        if self_offset >= 0:
            c = c[c != b + self_offset]
        c = c[np.lexsort((c, -s[b, c].astype(np.float64)))]
        if cap is not None:
            c = c[:cap]
        idx.append(c)
        sims.append(s[b, c])
        offs.append(offs[-1] + c.size)
    return np.array(offs), np.concatenate(idx), np.concatenate(sims).astype(np.float32)


def _np(r):
    return r.offsets.cpu().numpy(), r.indices.cpu().numpy(), r.sims.cpu().numpy(), r.saturated.cpu().numpy()


def _same(a, b):
    for x, y in zip(_np(a), _np(b)):
        assert x.shape == y.shape and (x.view(np.uint8) == y.view(np.uint8)).all() if x.size else x.shape == y.shape


def _planted(kind, N, D, seed, sizes=(2, 5, 40, 1500)):
    """(N, D) normalised rows of a data kind with planted near-duplicate groups (members are tiny
    perturbations of one row, a few exact copies); returns rows and the planted row numbers."""
    rng = np.random.default_rng(seed)
    if kind == "gauss":
        x = datagen.gauss(N, D, seed)
    elif kind == "absgauss":
        x = datagen.absgauss(N, D, seed)
    else:
        x = getattr(datagen, kind)(N, D, 9, seed)
    pos = rng.permutation(N)
    planted, at = [], 0
    for g in sizes:
        members = pos[at:at + g]
        at += g
        base = x[members[0]]
        noise = 2e-3 * rng.standard_normal((g, D)).astype(np.float32) / np.sqrt(D)
        noise[: max(1, g // 10)] = 0.0  # exact copies
        m = base + noise
        if kind in ("relu", "absgauss"):
            m = np.abs(m)
        x[members] = m / np.linalg.norm(m, axis=1, keepdims=True)
        planted.append(members)
    return x.astype(np.float32), planted


@pytest.mark.parametrize("name", ["real_FastSiam", "real_SimSiam"])
@pytest.mark.parametrize("norm", [False, True])
def test_exact_equals_oracle_golden(name, norm):
    g = np.load(os.path.join(GOLDEN, name + ".npz"))
    x = g["bank_rows_f16"].astype(np.float32)
    if norm:
        x = x / np.maximum(np.linalg.norm(x, axis=1, keepdims=True), 1e-12)
    sqn = (x.astype(np.float64) ** 2).sum(1)
    for tau in ((0.999, 0.99) if norm else (float(np.quantile(sqn, 0.5)), float(np.quantile(sqn, 0.99)))):
        want = _ref(x, x.T, tau)
        got = b200knn.knn_radius(_t(x), _t(x.T), tau, mode="exact", max_per_row=None)
        o, i, s, sat = _np(got)
        assert (o == want[0]).all() and (i == want[1]).all() and (s.view(np.uint32) == want[2].view(np.uint32)).all()
        assert not sat.any()
        for mode in ("fp32", "fp32_f16", "fp32_bf16x3"):
            _same(b200knn.knn_radius(_t(x), _t(x.T), tau, mode=mode, max_per_row=None), got)


def test_exact_equals_oracle_synthetic():
    x, planted = _planted("clustered", 37348, 512, 3)
    rng = np.random.default_rng(0)
    rows = np.unique(np.concatenate([rng.choice(37348, 400, replace=False)] + [p[:30] for p in planted]))[:512]
    q = x[rows]
    for tau in (0.999, 0.9):
        want = _ref(q, x.T, tau, cap=992)
        got = b200knn.knn_radius(_t(q), _t(x.T), tau, mode="exact")
        o, i, s, _ = _np(got)
        assert (o == want[0]).all() and (i == want[1]).all() and (s.view(np.uint32) == want[2].view(np.uint32)).all()


@pytest.mark.parametrize("kind", ["clustered", "gauss", "relu", "absgauss"])
@pytest.mark.parametrize("D", [384, 512, 768, 1024])
def test_fp32_modes_bitwise_exact(kind, D):
    x, planted = _planted(kind, 37348, D, 11 + D)
    rng = np.random.default_rng(D)
    rows = np.concatenate([rng.choice(37348, 300, replace=False)] + [p[:20] for p in planted])
    q, bank = _t(x[rows]), _t(x.T)
    for tau in (0.999, 0.99):
        for cap in (992, None):
            want = b200knn.knn_radius(q, bank, tau, mode="exact", max_per_row=cap)
            for mode in ("fp32", "fp32_f16", "fp32_bf16x3"):
                _same(b200knn.knn_radius(q, bank, tau, mode=mode, max_per_row=cap), want)
            if cap is None:
                o = want.offsets.cpu().numpy()
                assert (np.diff(o) >= 1400).sum() >= 20  # the 1,500 group's rows peel past 992
    # every ladder level ran on this data
    b200knn.knn_radius(q, bank, 0.999, mode="fp32", max_per_row=None)
    st = R.last_radius_stats
    assert st["first"] == q.shape[0] and st["second"] > 0 and st["peel"] > 0


@pytest.mark.parametrize("kind", ["clustered", "relu"])
def test_fp32_bitwise_exact_full_bank(kind):
    bank_nd, _, _ = bench.make_inputs(DEV, bench.N_BANK, 16, bench.DIM, seed=0, kind=kind)
    rng = np.random.default_rng(1)
    rows = torch.from_numpy(rng.choice(bench.N_BANK, 256, replace=False)).to(DEV)
    # plant: 64 rows become near-copies of row 0 (a group the ladder has to climb for)
    bank_nd[rows[:64]] = bank_nd[rows[0]] + 1e-4 * torch.randn(64, bench.DIM, device=DEV) / bench.DIM ** 0.5
    bank_nd = torch.nn.functional.normalize(bank_nd, dim=1)
    bank = bank_nd.t().contiguous()
    del bank_nd
    q = bank[:, rows].t().contiguous()
    for tau in (0.999, 0.95):
        want = b200knn.knn_radius(q, bank, tau, mode="exact")
        _same(b200knn.knn_radius(q, bank, tau, mode="fp32"), want)
        assert want.indices.numel() >= 64 * 64


def test_threshold_at_exact_pair_similarity():
    x, _ = _planted("clustered", 5000, 512, 5)
    q, bank = _t(x[:64]), _t(x.T)
    ex = b200knn.knn_radius(q, bank, -1.0, mode="exact", max_per_row=None)
    rng = np.random.default_rng(2)
    for b in range(0, 64, 8):
        lo, hi = int(ex.offsets[b]), int(ex.offsets[b + 1])
        j = lo + int(rng.integers(1, min(40, hi - lo)))
        s, n = F32(ex.sims[j].item()), int(ex.indices[j])
        for mode in ("exact", "fp32", "fp32_f16", "fp32_bf16x3"):
            r = b200knn.knn_radius(q[b:b + 1], bank, float(s), mode=mode)
            assert n in r.indices.tolist()
            r = b200knn.knn_radius(q[b:b + 1], bank, float(np.nextafter(s, F32(2))), mode=mode)
            assert n not in r.indices.tolist()


@pytest.mark.parametrize("pattern", ["big_first_half_ulp", "big_first_just_under_2ulp", "big_last", "ramp"])
def test_adversarial_no_pair_lost(pattern):
    rng = np.random.default_rng(7)
    q, x = _adversarial(512, pattern, rng)
    q, bank = _t(q), _t(x)
    exact = K.decode_keys(K.topk_keys(q, bank, bank.shape[1], "exact"))
    approx = K.decode_keys(K.topk_keys(q, bank, bank.shape[1], "f16"))
    for b in range(q.shape[0]):
        s_ex = torch.empty(bank.shape[1], device=DEV).index_copy_(0, exact[1][b], exact[0][b])
        s_ap = torch.empty(bank.shape[1], device=DEV).index_copy_(0, approx[1][b], approx[0][b])
        worst = int(torch.argmin(s_ap.double() - s_ex.double()))
        tau = float(np.nextafter(F32(s_ex[worst].item()), F32(-np.inf)))
        want = b200knn.knn_radius(q[b:b + 1], bank, tau, mode="exact", max_per_row=None)
        assert worst in want.indices.tolist()
        for mode in ("fp32", "fp32_f16"):
            _same(b200knn.knn_radius(q[b:b + 1], bank, tau, mode=mode, max_per_row=None), want)


def _midpoints(n, D, rng):
    """Positive rows whose every element is an fp16 rounding midpoint h (1 + 2^-11): the fp16
    operands lose the most they can, so the residual terms of E are at work."""
    h = 2.0 ** rng.integers(-8, 0, size=(n, D))
    return (h * (1 + 2.0 ** -11)).astype(np.float32)


@pytest.mark.parametrize("D", [512, 768])
def test_fp16_midpoints_no_pair_lost(D):
    """tau just below the pair whose fp16 similarity a falls furthest below the exact s (among each
    row's 500 nearest, so the admission threshold prunes the rest of the 20,000-row bank): that pair
    and every other neighbour are found, bitwise as "exact"."""
    rng = np.random.default_rng(D)
    X = _midpoints(20000, D, rng)
    q = _midpoints(8, D, rng)
    bank_dn = np.ascontiguousarray(X.T)
    _, dump, _, _ = run_dump(q, bank_dn, 5, "f16")  # the fp16 pass's own similarities a
    s = O.sims_seqfma(q, bank_dn)
    qt, bank = _t(q), _t(bank_dn)
    for b in range(q.shape[0]):
        near = np.argsort(-s[b].astype(np.float64), kind="stable")[:500]
        worst = int(near[np.argmin(dump[b, near].astype(np.float64) - s[b, near])])
        tau = float(s[b, worst])
        want = b200knn.knn_radius(qt[b:b + 1], bank, tau, mode="exact", max_per_row=None)
        assert worst in want.indices.tolist() and want.indices.numel() < 1000
        for mode in ("fp32", "fp32_f16"):
            got = b200knn.knn_radius(qt[b:b + 1], bank, tau, mode=mode, max_per_row=None)
            _same(got, want)
            assert R.last_radius_stats["peel"] == 0  # served by the admission threshold, not the exact path
        assert int(K.radius_tau0(qt[b:b + 1], bank, F32(tau), K.level_config("fp32_f16", D), "f16")[1][0]) == 0


@pytest.mark.parametrize("D", [512, 1024])
def test_admission_kernel_matches_restatement(D):
    """tau0[b] is bitwise admission_threshold(tau, E_b) at the E_b the kernel reports; for the
    residual form E_b is at least the restated bound of tests/test_residual_bound_cpu.py."""
    rng = np.random.default_rng(3)
    X = np.concatenate([datagen.absgauss(3000, D, 1), _midpoints(1000, D, rng)])
    Q = np.concatenate([datagen.absgauss(40, D, 2), _midpoints(24, D, rng), X[:8] * F32(3.0)])
    bank, q = _t(np.ascontiguousarray(X.T)), _t(Q)
    for level, cand in (("fp32_f16", "f16"), ("fp32_bf16x3", "bf16x3"), ("fp32_f16x2", "f16x2")):
        cfg = K.level_config(level, D)
        cand = K.effective_mode(cand, D)
        for tau in (0.999, 0.5, -0.25, 3.0, 0.0):
            tau0, refused, e = K.radius_tau0(q, bank, F32(tau), cfg, cand, return_e=True)
            tau0, e = tau0.cpu().numpy(), e.cpu().numpy()
            assert not refused.any()
            for b in range(Q.shape[0]):
                assert tau0[b].view(np.uint32) == R.admission_threshold(F32(tau), e[b]).view(np.uint32)
            if level == "fp32_f16" and cand == "f16":
                assert (e.astype(np.float64) >= e_new(Q, X) * (1 - 1e-4)).all()


def test_refused_rows_take_the_exact_path():
    """Query norms at or beyond the fp16 range (max_abs): the f16 level refuses the rows, which are
    then served exactly; the result is bitwise "exact"."""
    x, _ = _planted("clustered", 6000, 256, 31, sizes=(2, 40))
    bank = _t(np.ascontiguousarray(x.T))
    q = _t(x[:16] * F32(1e5))
    s = b200knn.knn_radius(q, bank, -1e9, mode="exact", max_per_row=None).sims
    tau = float(s[20].item())  # about the 20th neighbour of row 0
    _, refused = K.radius_tau0(q, bank, F32(tau), K.level_config("fp32_f16", 256), "f16")
    assert refused.all()
    want = b200knn.knn_radius(q, bank, tau, mode="exact")
    assert want.indices.numel() > 0
    got = b200knn.knn_radius(q, bank, tau, mode="fp32_f16")
    _same(got, want)
    assert R.last_radius_stats["peel"] == 16


@pytest.mark.parametrize("D", [512, 768])
def test_other_fp32_levels_bitwise_exact(D):
    x, planted = _planted("relu", 37348, D, 41)
    rng = np.random.default_rng(1)
    rows = np.concatenate([rng.choice(37348, 200, replace=False)] + [p[:10] for p in planted])
    q, bank = _t(x[rows]), _t(x.T)
    for tau in (0.999, 0.99):
        for cap in (992, None):
            want = b200knn.knn_radius(q, bank, tau, mode="exact", max_per_row=cap)
            for mode in ("fp32_f16x2", "fp32_bf16", "fp32_tf32"):
                _same(b200knn.knn_radius(q, bank, tau, mode=mode, max_per_row=cap), want)


@pytest.mark.parametrize("mode", ["exact", "fp32", "f16", "bf16x3"])
def test_self_join_at_default_cap_is_not_peeled(mode):
    """radius_graph at max_per_row = 992: a row of a 1,500-row group needs 993 keys with its own, so
    it is searched again with itself left out (no peeling), keeps 992 of its neighbours, in the mode's
    own similarities, and is saturated.  fp32 is bitwise "exact", and "exact" is the oracle."""
    n = 6000
    x, planted = _planted("clustered", n, 256, 43, sizes=(2, 40, 1500))
    rows = _t(x)
    g = b200knn.radius_graph(rows, 0.999, normalize=False, mode=mode)
    st = dict(R.last_radius_stats)
    assert st["peel"] == 0 and st["self_excluded"] >= 1500
    o = g.offsets.cpu().numpy()
    big = planted[2]
    assert (np.diff(o)[big] == 992).all() and g.saturated[torch.from_numpy(big).to(DEV)].all()
    assert int(g.saturated.sum()) == 1500
    if mode == "exact":
        want = _ref(x, x.T, 0.999, self_offset=0, cap=992)
        assert (o == want[0]).all() and (g.indices.cpu().numpy() == want[1]).all()
        assert (g.sims.cpu().numpy().view(np.uint32) == want[2].view(np.uint32)).all()
    elif mode == "fp32":
        _same(g, b200knn.radius_graph(rows, 0.999, normalize=False, mode="exact"))
    else:  # the mode's own keys: its own-row-excluded top 992, cut at tau
        fb = b200knn.FeatureBank.from_rows(rows, normalize=False)
        sub = torch.from_numpy(big[:64]).to(DEV)
        keys = K.topk_keys(fb.rows[sub, :fb.dim].contiguous(), fb.bank, 992, mode,
                           exclude=(sub.to(torch.int32), torch.arange(n, dtype=torch.int32, device=DEV), 1))
        s, i = K.decode_keys(keys)
        for j, r in enumerate(big[:64]):
            keep = s[j] >= float(F32(0.999))
            assert torch.equal(i[j][keep].cpu(), g.indices[o[r]:o[r + 1]].cpu())
            assert torch.equal(s[j][keep].cpu().view(torch.int32), g.sims[o[r]:o[r + 1]].cpu().view(torch.int32))


@pytest.mark.parametrize("mode", ["f16", "bf16", "f16x2", "bf16x3", "tf32x3"])
def test_raw_modes_equal_own_topk(mode):
    x, _ = _planted("clustered", 37348, 512, 9)
    q, bank = _t(x[:384]), _t(x.T)
    for tau in (0.999, 0.95):
        r = b200knn.knn_radius(q, bank, tau, mode=mode)
        s, i = K.decode_keys(K.topk_keys(q, bank, 992, mode))
        o = r.offsets.cpu()
        t = F32(tau)
        for b in range(q.shape[0]):
            if bool(r.saturated[b]):
                continue
            keep = s[b] >= float(t)
            assert torch.equal(i[b][keep].cpu(), r.indices[o[b]:o[b + 1]].cpu())
            assert torch.equal(s[b][keep].cpu().view(torch.int32), r.sims[o[b]:o[b + 1]].cpu().view(torch.int32))


def test_max_per_row_and_edge_cases():
    x, planted = _planted("clustered", 6000, 256, 13, sizes=(2, 5, 40, 1500))
    big = planted[3][:8]
    q, bank = _t(x[big]), _t(x.T)
    full = b200knn.knn_radius(q, bank, 0.999, mode="exact", max_per_row=None)
    assert (np.diff(full.offsets.cpu().numpy()) >= 1500).all() and not full.saturated.any()
    for cap in (1, 32, 100, 992, 993):
        for mode in ("exact", "fp32", "f16"):
            r = b200knn.knn_radius(q, bank, 0.999, mode=mode, max_per_row=cap)
            assert (np.diff(r.offsets.cpu().numpy()) == cap).all() and r.saturated.all()
            if mode != "f16":  # the exact top-cap rows of the full result
                o = full.offsets.cpu().numpy()
                want = np.concatenate([full.indices.cpu().numpy()[o[b]:o[b] + cap] for b in range(8)])
                assert (r.indices.cpu().numpy() == want).all()
    # tau above every similarity; B = 0; N < 32
    r = b200knn.knn_radius(q, bank, 1.5, mode="fp32")
    assert r.indices.numel() == 0 and r.offsets.tolist() == [0] * 9 and not r.saturated.any()
    r = b200knn.knn_radius(q[:0], bank, 0.5)
    assert r.offsets.tolist() == [0] and r.indices.numel() == 0 and r.saturated.numel() == 0
    small = _t(x[:20].T)
    want = _ref(x[:5], x[:20].T, 0.0)
    for mode in ("exact", "fp32", "f16"):
        r = b200knn.knn_radius(_t(x[:5]), small, 0.0, mode=mode)
        if mode != "f16":
            assert (r.offsets.cpu().numpy() == want[0]).all() and (r.indices.cpu().numpy() == want[1]).all()
        assert not r.saturated.any()


def test_radius_graph_self_and_batches():
    x, planted = _planted("clustered", 8000, 512, 17, sizes=(2, 5, 40, 300))
    x[100] = x[7]  # an exact duplicate of lower index
    rows = _t(x)
    g = b200knn.radius_graph(rows, 0.999, mode="exact", max_per_row=None)
    o, i = g.offsets.cpu().numpy(), g.indices.cpu().numpy()
    for r in range(8000):
        assert r not in i[o[r]:o[r + 1]]
    assert 7 in i[o[100]:o[101]] and 100 in i[o[7]:o[8]]
    want = _ref(x, x.T, 0.999, self_offset=0)
    assert (o == want[0]).all() and (i == want[1]).all()
    gs = b200knn.radius_graph(rows, 0.999, mode="exact", max_per_row=None, include_self=True)
    os_, is_ = gs.offsets.cpu().numpy(), gs.indices.cpu().numpy()
    assert all(r in is_[os_[r]:os_[r + 1]] for r in range(0, 8000, 97))
    for mode in ("fp32", "f16"):
        a = b200knn.radius_graph(rows, 0.999, mode=mode)
        for batch in (777, 4096):
            _same(b200knn.radius_graph(rows, 0.999, mode=mode, batch=batch), a)
        if mode == "fp32":
            _same(a, b200knn.radius_graph(rows, 0.999, mode="exact"))


def _scipy_groups(g, n):
    o, i = g.offsets.cpu().numpy(), g.indices.cpu().numpy()
    m = csr_matrix((np.ones(i.size), i, o), shape=(n, n))
    _, lab = connected_components(m, directed=True, connection="weak")
    mins = np.full(lab.max() + 1, n)
    np.minimum.at(mins, lab, np.arange(n))
    return mins[lab]


def test_near_duplicate_groups():
    n = 20000
    x, planted = _planted("relu", n, 512, 23, sizes=(2, 5, 40, 1500))
    rows = _t(x)
    for tau in (0.999, 0.97):
        want = _scipy_groups(b200knn.radius_graph(rows, tau, mode="exact", max_per_row=None), n)
        ids, n_sat = b200knn.near_duplicate_groups(rows, tau, max_per_row=None)
        assert n_sat == 0 and (ids.cpu().numpy() == want).all()
        ids2, _ = b200knn.near_duplicate_groups(rows, tau, max_per_row=None, batch=3001)
        assert torch.equal(ids, ids2)
    for p in planted:
        assert len(set(ids.cpu().numpy()[p].tolist())) == 1
    # saturated rows only drop edges: every returned group lies inside one true group
    true = _scipy_groups(b200knn.radius_graph(rows, 0.999, mode="exact", max_per_row=None), n)
    ids, n_sat = b200knn.near_duplicate_groups(rows, 0.999, max_per_row=16, batch=5000)
    assert n_sat >= 1500
    got = ids.cpu().numpy()
    for gid in np.unique(got):
        assert np.unique(true[got == gid]).size == 1


def test_loo_with_near_duplicate_groups():
    n, C = 12000, 9
    x, planted = _planted("clustered", n, 256, 29, sizes=(2, 5, 40, 300))
    lab = datagen.labels(n, C, 3)
    for p in planted:
        lab[p] = lab[p[0]]
    rows, labels = _t(x), _t(lab)
    fb = b200knn.FeatureBank.from_rows(rows)
    groups, _ = b200knn.near_duplicate_groups(rows, 0.999)
    plain = b200knn.knn_predict_loo(fb.bank, labels, C, (1,), (0.1,))[0, 0, :, 0]
    grouped = b200knn.knn_predict_loo(fb.bank, labels, C, (1,), (0.1,), groups=groups)[0, 0, :, 0]
    members = torch.from_numpy(np.concatenate(planted)).to(DEV)
    assert bool((plain[members] == labels[members]).all())  # a near-copy always votes its own label
    assert bool((plain[members] != grouped[members]).any())


def test_argument_errors_before_any_launch():
    x, _ = _planted("gauss", 1000, 64, 1, sizes=(2,))
    q, bank, rows = _t(x[:4]), _t(x.T), _t(x)
    before = _lib.launch_counter["kernels"]
    for bad in (float("nan"), float("inf"), 1e39):
        with pytest.raises(ValueError):
            b200knn.knn_radius(q, bank, bad)
        with pytest.raises(ValueError):
            b200knn.radius_graph(rows, bad)
    for cap in (0, -3):
        with pytest.raises(ValueError):
            b200knn.knn_radius(q, bank, 0.5, max_per_row=cap)
        with pytest.raises(ValueError):
            b200knn.near_duplicate_groups(rows, 0.5, max_per_row=cap)
    with pytest.raises(ValueError):
        b200knn.knn_radius(q, bank, 0.5, mode="fp64")
    with pytest.raises(ValueError):
        b200knn.radius_graph(rows, 0.5, batch=0)
    with pytest.raises(RuntimeError, match="mat1 and mat2 shapes cannot be multiplied"):
        b200knn.knn_radius(q[:, :32], bank, 0.5)
    with pytest.raises(RuntimeError, match="self must be a matrix"):
        b200knn.knn_radius(q[0], bank, 0.5)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        b200knn.knn_radius(q.cpu(), bank, 0.5)
    with pytest.raises(RuntimeError, match="no CPU fallback"):
        b200knn.near_duplicate_groups(rows.cpu(), 0.5)
    assert _lib.launch_counter["kernels"] == before
