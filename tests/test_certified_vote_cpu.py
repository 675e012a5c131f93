"""The rules of knn_predict's certified class vote (DESIGN §4.1c, csrc/rescore.cu band_kernel +
rescore_vote_kernel) restated in numpy and checked against the exact vote of fp32 similarities:
every case either certifies and equals the exact ranking, or is flagged."""
import numpy as np
import pytest


def exact_ranking(s, idx, labels, k, C, t):
    """vote_kernel on the exact top k: (sim desc, idx asc), fp64 weights summed in rank order."""
    order = np.lexsort((idx, -s.astype(np.float64)))[:k]
    sc = np.zeros(C)
    for j in order:
        sc[labels[idx[j]]] += np.exp(np.float64(s[j]) / t)
    return sorted(range(C), key=lambda c: (-sc[c], c))


def certified_ranking(a, s, idx, labels, k, C, t, E, n_bank):
    """The kernels' rules on candidates sorted by approximate key; None = flagged."""
    m = len(a)
    if m >= n_bank or not np.isfinite(E):
        return None  # k_in >= N: not served by this path
    a64, E = a.astype(np.float64), float(E)
    ak, ak1 = a64[k - 1], a64[k if k < m else m - 1]
    p = int(np.sum(a64[:k] > ak1 + 2 * E))
    r = int(np.sum(a64 + E >= ak - E))
    band = np.arange(p, r)
    bkeys = sorted(band, key=lambda j: (-np.float64(s[j]), idx[j]))[:k - p]
    if k - p > 0:
        bound = a64[r if r < m else m - 1] + E
        if not np.float64(s[bkeys[-1]]) > bound:
            return None
    lo, hi, cnt = np.zeros(C), np.zeros(C), np.zeros(C, int)
    for i in range(p):
        x1, x2 = (a64[i] - E) / t, (a64[i] + E) / t
        pad = (abs(x1) + abs(x2)) * 2.0 ** -48
        with np.errstate(over="ignore", under="ignore"):
            lo[labels[idx[i]]] += np.exp(min(x1, x2) - pad) * (1 - 2.0 ** -48)
            hi[labels[idx[i]]] += np.exp(max(x1, x2) + pad) * (1 + 2.0 ** -48)
        cnt[labels[idx[i]]] += 1
    for j in bkeys:
        with np.errstate(over="ignore"):
            w = np.exp(np.float64(s[j]) / t)
        lo[labels[idx[j]]] += w
        hi[labels[idx[j]]] += w
        cnt[labels[idx[j]]] += 1
    widen = (k + 8) * 2.0 ** -48
    lo, hi = lo * (1 - widen), hi * (1 + widen)
    present = [c for c in range(C) if cnt[c]]
    for c in present:
        if not (lo[c] >= np.finfo(np.float64).tiny and np.isfinite(hi[c])):
            return None
        for o in present:
            if o != c and not (lo[c] > hi[o] or lo[o] > hi[c]):
                return None
    ranked = sorted(present, key=lambda c: -lo[c]) + [c for c in range(C) if not cnt[c]]
    return ranked


def make_case(rng, n_bank, k, m, C, t, E, kind="random", scale=1.0):
    s_all = (rng.standard_normal(n_bank) * 0.2 * scale).astype(np.float32)
    if kind == "dup":  # duplicates straddling rank k
        top = np.sort(s_all)[::-1]
        s_all[rng.choice(n_bank, 3 * k + 3, replace=False)] = top[k]
    if kind == "near":  # near-ties at ranks k and k + 1
        order = np.argsort(-s_all)
        s_all[order[k]] = np.nextafter(s_all[order[k - 1]], -np.inf)
    labels = rng.integers(0, C, n_bank)
    if kind == "close":  # two classes of almost equal weight
        labels = np.arange(n_bank) % 2
    noise = rng.uniform(-E, E, n_bank)
    a_all = (s_all.astype(np.float64) + noise).astype(np.float32)
    # |a - s| <= E after rounding a to fp32: widen E by a few ulps of the largest |a|
    E_cert = E + 4 * np.spacing(np.float32(np.abs(a_all).max()))
    idx_all = np.arange(n_bank)
    cand = np.lexsort((idx_all, -a_all.astype(np.float64)))[:m]
    return a_all[cand], s_all[cand], idx_all[cand], labels, s_all, E_cert


CASES = [
    # (n_bank, k, m, C, t, E, kind, scale)
    (3000, 200, 240, 9, 0.1, 1e-4, "random", 1.0),
    (3000, 200, 240, 9, 0.1, 1e-4, "near", 1.0),
    (3000, 20, 60, 9, 0.1, 1e-4, "dup", 1.0),
    (3000, 200, 240, 2, 0.1, 1e-4, "close", 1.0),
    (3000, 200, 240, 38, -0.1, 1e-4, "random", 1.0),
    (3000, 200, 240, 9, 1e-3, 1e-4, "random", 1.0),       # exp underflow / overflow at small t
    (3000, 200, 240, 9, 0.1, 1e-2, "random", 5000.0),     # unnormalised rows: overflow
    (3000, 1, 41, 9, 0.1, 1e-4, "random", 1.0),
    (3000, 992, 992, 9, 0.1, 1e-4, "random", 1.0),
    (240, 200, 240, 9, 0.1, 1e-4, "random", 1.0),         # k_in >= N
]


@pytest.mark.parametrize("case", CASES, ids=[f"{c[6]}-k{c[1]}-C{c[3]}-t{c[4]}-x{c[7]}-N{c[0]}" for c in CASES])
def test_rules_certify_only_the_exact_ranking(case):
    n_bank, k, m, C, t, E, kind, scale = case
    rng = np.random.default_rng(1234)
    n_cert = 0
    for _ in range(8):
        a, s, idx, labels, s_all, E_cert = make_case(rng, n_bank, k, m, C, t, E, kind, scale)
        got = certified_ranking(a, s, idx, labels, k, C, t, E_cert, n_bank)
        if got is None:
            continue
        n_cert += 1
        with np.errstate(over="ignore"):
            want = exact_ranking(s_all, np.arange(n_bank), labels, k, C, t)
        assert got == want
    if kind == "random" and scale == 1.0 and k < m < n_bank and abs(t) >= 0.1:
        assert n_cert > 0  # the rules do certify ordinary rows (k = m leaves no margin for rule 2)


def test_non_finite_bound_is_flagged():
    # band_kernel does not serve a row whose E is not finite (p = -1), like a starved one
    rng = np.random.default_rng(7)
    a, s, idx, labels, _, E = make_case(rng, 3000, 200, 240, 9, 0.1, 1e-4)
    assert certified_ranking(a, s, idx, labels, 200, 9, 0.1, np.inf, 3000) is None
