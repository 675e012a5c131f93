"""CPU: the host rules of knn_radius / radius_graph / near_duplicate_groups (b200knn/retrieval.py).
 * the admission threshold: the largest fp32 strictly below tau32 - E, against an exact restatement;
 * the escalation ladder (32 -> 992 -> peeling) and saturation over max_per_row in {1, 32, 992, 993,
   None}, simulated from each row's true neighbour count;
 * the compaction rule on hand-made key lists (ties at tau, the row's own index at any rank, empty
   slots), restated in NumPy as the count / emit kernels apply it;
 * the components rule (hook the larger root under the smaller, path halving) against scipy's
   connected_components, labels = component minima."""
from fractions import Fraction

import numpy as np
import pytest
import torch
from scipy.sparse import coo_matrix
from scipy.sparse.csgraph import connected_components

from b200knn import retrieval as R
from oracle import knn_oracle as O

F32 = np.float32


def _check_admission(t, e):
    got = R.admission_threshold(t, e)
    assert isinstance(got, np.float32)
    exact = Fraction(float(F32(t))) - Fraction(float(F32(e)))
    assert Fraction(float(got)) < exact
    up = np.nextafter(got, F32(np.inf))
    assert Fraction(float(up)) >= exact


@pytest.mark.parametrize("t", [0.999, 0.99, 1.0, 0.5, 2.0 ** -20, 0.0, -0.25, 277.0 ** 2])
@pytest.mark.parametrize("e", [0.0, 2.0 ** -149, 3 * 2.0 ** -149, 2.0 ** -126 * 0.75, 1e-7, 2.0 ** -24,
                               2.0 ** -23, 6.1e-5, 0.01, 1e30])
def test_admission_threshold_is_largest_fp32_below(t, e):
    _check_admission(t, e)


def test_admission_threshold_on_fp32_boundaries():
    rng = np.random.default_rng(0)
    for _ in range(300):
        t = F32(rng.uniform(-1, 1))
        # E equal to an ulp multiple of t (exact difference) and just off it (inexact difference)
        ulp = np.spacing(np.abs(t))
        for e in (ulp, 2 * ulp, ulp * F32(0.5), F32(rng.uniform(0, 1e-3)), np.nextafter(ulp, F32(1))):
            _check_admission(t, e)
    # E = 0: the next fp32 value below tau32, also across a binade edge and at zero
    for t in (F32(1.0), F32(0.5), F32(2.0 ** -126), F32(0.0), F32(-1.0)):
        assert R.admission_threshold(t) == np.nextafter(t, F32(-np.inf))


def _simulate(count, n_bank, max_per_row, drop_self):
    """Level each row's list finally comes from ('first', 'second', 'peel') and its saturated flag,
    for a raw-mode row with `count` admitted columns (its own row among them when drop_self)."""
    cap = n_bank if max_per_row is None else max_per_row
    cap_search = min(n_bank, cap + (1 if drop_self else 0))
    depths = R.radius_ladder(n_bank, cap_search)
    for level, depth in enumerate(depths):
        full = torch.tensor([3 if count >= depth else 0], dtype=torch.int32)
        esc, sat = R.radius_plan(depth, cap_search, n_bank, full, True)
        if not bool(esc[0]):
            return ("first", "second")[level], bool(sat[0])
    return "peel", count >= cap_search and cap_search < n_bank


@pytest.mark.parametrize("max_per_row", [1, 32, 992, 993, None])
def test_escalation_ladder(max_per_row):
    n_bank = 5000
    for count in (0, 1, 2, 31, 32, 33, 500, 991, 992, 993, 994, 1500, 5000):
        level, sat = _simulate(count, n_bank, max_per_row, drop_self=False)
        cap = n_bank if max_per_row is None else max_per_row
        if max_per_row is not None and max_per_row <= 32:
            assert level == "first"
        elif count < 32:
            assert level == "first"
        elif count < 992 or cap <= 992:
            assert level == "second"
        else:
            assert level == "peel"
        # saturated exactly when the row has at least max_per_row columns (the list filled at the cap)
        assert sat == (count >= cap and cap < n_bank), (count, max_per_row)
    # depths: (32, min(992, cap)) or (cap,) for small caps, and N when the bank is small
    assert R.radius_ladder(5000, 1) == (1,)
    assert R.radius_ladder(5000, 32) == (32,)
    assert R.radius_ladder(5000, 993) == (32, 992)
    assert R.radius_ladder(20, 5000) == (20,)
    assert R.radius_ladder(100, 5000) == (32, 100)


def test_plan_order_of_lists():
    """A re-scored candidate list (not the exact order) continues on any filled last slot; an exact
    list only when its last key is a neighbour; a list holding every column never continues."""
    full = torch.tensor([0, 1, 3], dtype=torch.int32)
    esc, sat = R.radius_plan(32, 993, 5000, full, exact_order=False)
    assert esc.tolist() == [False, True, True] and not sat.any()
    esc, sat = R.radius_plan(32, 993, 5000, full, exact_order=True)
    assert esc.tolist() == [False, False, True]
    esc, sat = R.radius_plan(992, 992, 5000, full, exact_order=True)
    assert sat.tolist() == [False, False, True] and not esc.any()
    esc, sat = R.radius_plan(32, 993, 32, full, exact_order=True)
    assert not esc.any() and not sat.any()


def _compact_np(keys, tau, self_idx, cap):
    """The count / emit rule: keys non-empty, sim >= tau, index != self_idx; the first cap of them."""
    sims, idx = O.decode_keys(keys)
    keep = (keys != 0) & (sims >= F32(tau)) & (idx != self_idx)
    return idx[keep][:cap], sims[keep][:cap]


def test_compaction_rule_hand_made():
    tau = F32(0.75)
    s = np.array([0.9, 0.8, 0.75, 0.75, np.nextafter(tau, F32(-1)), 0.5], dtype=np.float32)
    i = np.array([7, 3, 2, 9, 1, 4], dtype=np.int64)
    keys = O.make_keys(s, i)
    assert (np.diff(keys.astype(np.uint64).astype(np.float64)) <= 0).all()  # canonical order
    idx, sims = _compact_np(keys, tau, -1, 10)
    assert idx.tolist() == [7, 3, 2, 9]  # ties at tau are neighbours, the next fp32 below is not
    for self_idx, want in ((7, [3, 2, 9]), (9, [7, 3, 2]), (1, [7, 3, 2, 9]), (4, [7, 3, 2, 9])):
        assert _compact_np(keys, tau, self_idx, 10)[0].tolist() == want  # own index at any rank
    assert _compact_np(keys, tau, 3, 2)[0].tolist() == [7, 2]
    empty = np.concatenate([keys[:3], np.zeros(4, dtype=keys.dtype)])  # front-filled, empty tail
    assert _compact_np(empty, tau, -1, 10)[0].tolist() == [7, 3, 2]
    assert _compact_np(np.zeros(5, dtype=keys.dtype), tau, -1, 10)[0].size == 0


def _components_hooking(n, edges, rng):
    """Union-find as the device does it, with the edges in a random order and retries interleaved:
    hook the larger root under the smaller, path halving in find."""
    parent = np.arange(n)

    def find(x):
        while parent[x] != x:
            if parent[parent[x]] != parent[x]:
                parent[x] = parent[parent[x]]
            x = parent[x]
        return x

    for a, b in edges[rng.permutation(len(edges))]:
        while True:
            ra, rb = find(a), find(b)
            if ra == rb:
                break
            lo, hi = min(ra, rb), max(ra, rb)
            if parent[hi] == hi:  # the CAS
                parent[hi] = lo
                break
        assert (parent <= np.arange(n)).all()
    return np.array([find(x) for x in range(n)])


@pytest.mark.parametrize("seed", range(6))
def test_components_rule_matches_scipy(seed):
    rng = np.random.default_rng(seed)
    n = int(rng.integers(1, 400))
    m = int(rng.integers(0, 3 * n))
    edges = rng.integers(0, n, (m, 2))
    got = _components_hooking(n, edges, rng)
    g = coo_matrix((np.ones(m), (edges[:, 0], edges[:, 1])), shape=(n, n)) if m else coo_matrix((n, n))
    _, lab = connected_components(g, directed=True, connection="weak")
    mins = np.full(lab.max() + 1, n)
    np.minimum.at(mins, lab, np.arange(n))
    assert (got == mins[lab]).all()
