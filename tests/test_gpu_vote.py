"""GPU: the class-vote and confusion kernels of csrc/vote.cu driven directly with crafted keys, against a
plain fp64 reference: k across the 32-lane loop, the peeling boundary (992 / 993), the 1024-key chunk
and far beyond it; C with one, two and many classes per lane; B around the 4 rows of a block;
negative, tiny and huge temperatures; ±0 similarities; constructed exact ties; the status word's
bits; the grid vote against the single vote; the class-count bound; confusion counts past the first
pass of the grid-stride loop and above the shared-memory histogram; and knn_predict /
knn_predict_multi / knn_predict_loo at k > 3195 end to end.

Reference (restated here: oracle.vote_o64 maps an empty slot's index -1 to the last label):
weights exp(float64(sim) / t) added per class in rank order j = 0..k-1, an empty key (0) casts no
vote, classes ranked by (score desc, class asc).

Comparison rules.  CUDA's double exp is within 1 ulp but not correctly rounded, so scores are not
compared bit for bit with NumPy's:
  * scores agree within (k + 2) * 2**-52 relative, and exactly where the reference is 0 or inf;
  * rankings are equal on every row where no two class scores lie within that bound; a pair that is
    exactly equal on both sides (no votes, underflow to 0, overflow to inf, a constructed tie) is a
    tie both sides break by class index, not an ambiguity;
  * constructed exact ties (two classes given the same sims in the same rank order) are bitwise
    equal device scores.
"""
import ctypes

import numpy as np
import pytest
import torch

import b200knn
import datagen
from b200knn import _lib
from b200knn import knn as K
from oracle import knn_oracle as O

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
KS = [1, 2, 31, 32, 33, 200, 992, 993, 3195, 3196, 4260, 4261, 8192]
CS = [1, 2, 31, 32, 33, 38, 64, 65, 1000]
BS = [0, 1, 3, 4, 5, 1001]
TS = [0.07, 0.1, 1.0, 1000.0, -0.1]
E_UNSUPPORTED = -4  # B200KNN_E_UNSUPPORTED of include/b200knn.h


def _t(x):
    return torch.from_numpy(np.ascontiguousarray(x)).to(DEV)


def _case(B, k, C, seed, extreme=False):
    """Crafted sorted keys of B rows: (keys uint64 (B, k), labels int64 (B*k,) indexed by the keys'
    bank index b*k + j).  Row kinds by b % 5: 0 random; 1 trailing empty slots; 2 two classes given
    the same sims in the same rank order (an exact tie); 3 many +0.0 / -0.0 and repeated sims;
    4 every slot empty.  extreme: class c's sims lie near level c % 6 of (0.999, 0.95, 0.5, -0.5,
    -0.95, -0.999), so at t = 1e-3 some classes' weights overflow to inf, some underflow to 0."""
    rng = np.random.default_rng(seed)
    lab = rng.integers(0, C, (B, k))
    if extreme:
        level = np.array([0.999, 0.95, 0.5, -0.5, -0.95, -0.999], np.float32)[lab % 6]
        sims = (level + rng.uniform(-1e-3, 1e-3, (B, k))).astype(np.float32)
    else:
        sims = rng.uniform(-1, 1, (B, k)).astype(np.float32)
    for b in range(3, B, 5):
        sims[b, rng.random(k) < 0.3] = 0.0
        sims[b, rng.random(k) < 0.3] = -0.0
        sims[b, rng.random(k) < 0.2] = sims[b, 0]
    order = np.argsort(-sims, axis=1, kind="stable")  # descending; a key's label moves with it
    sims, lab = np.take_along_axis(sims, order, 1), np.take_along_axis(lab, order, 1)
    empty = np.zeros((B, k), bool)
    empty[1::5, :] = np.arange(k)[None, :] >= rng.integers(1, max(k, 2), (len(range(1, B, 5)), 1))
    empty[4::5, :] = True
    for b in range(2, B, 5):
        if C < 2:
            continue
        a, c = rng.choice(C, 2, replace=False)
        for j in range(0, k - 1, 2):
            sims[b, j + 1] = sims[b, j]
            lab[b, j:j + 2] = (a, c) if rng.random() < 0.5 else (c, a)
        empty[b, k - 1] = k % 2 == 1  # an odd last key would break the tie
    idx = np.arange(B * k, dtype=np.int64).reshape(B, k)
    keys = O.make_keys(sims, idx)
    keys[empty] = 0
    return keys, lab.reshape(-1)


def _ref_vote(keys, labels, C, t):
    """(pred (B,C) int64, scores (B,C) f64): the fp64 reference of the module docstring."""
    sims, idx = O.decode_keys(keys)
    B, k = keys.shape
    lab = np.where(idx >= 0, labels[np.maximum(idx, 0)], -1)
    with np.errstate(over="ignore", under="ignore"):
        w = np.exp(sims.astype(np.float64) / np.float64(t))
    scores = np.zeros((B, C))
    rows = np.arange(B)
    for j in range(k):  # one rank at a time: a row adds to one class per j, so no index repeats
        v = lab[:, j] >= 0
        scores[rows[v], lab[v, j]] += w[v, j]
    return np.argsort(-scores, axis=1, kind="stable").astype(np.int64), scores


def _check_vote(pred, scores, keys, labels, C, t):
    """Asserts the comparison rules; returns the number of rows whose ranking was compared."""
    k = keys.shape[1]
    tol = (k + 2) * 2.0 ** -52
    want_pred, want = _ref_vote(keys, labels, C, t)
    exact = (want == 0) | np.isinf(want)
    assert np.array_equal(scores[exact], want[exact])
    assert np.all(np.abs(scores[~exact] - want[~exact]) <= tol * want[~exact])
    a = np.take_along_axis(want, want_pred, axis=1)
    g = np.take_along_axis(scores, want_pred, axis=1)
    tied = (a[:, :-1] == a[:, 1:]) & (g[:, :-1] == g[:, 1:])
    with np.errstate(invalid="ignore"):
        close = ~np.isinf(a[:, :-1]) & (a[:, :-1] - a[:, 1:] <= tol * a[:, :-1]) & ~tied
    unamb = ~close.any(axis=1)
    assert np.array_equal(pred[unamb], want_pred[unamb])
    return int(unamb.sum())


def _check_ties(pred, scores, keys, labels):
    """The constructed ties of _case's rows 2, 7, ...: bitwise equal scores, lower class first."""
    B, k = keys.shape
    for b in range(2, B, 5):
        _, idx = O.decode_keys(keys[b, :2])
        if k < 2 or idx[1] < 0:
            continue
        a, c = sorted(labels[idx[:2]])
        if a == c:
            continue
        assert scores[b, a] == scores[b, c], b
        pos = {int(x): i for i, x in enumerate(pred[b])}
        assert pos[a] < pos[c] and (scores[b, a] == 0 or pos[a] + 1 == pos[c]), b


def _status_ref(keys, labels, C, label_offset=0):
    _, idx = O.decode_keys(keys)
    li = idx - label_offset
    bad_idx = (idx >= 0) & ((li < 0) | (li >= labels.size))
    lab = np.where((idx >= 0) & ~bad_idx, labels[np.clip(li, 0, labels.size - 1)], 0)
    bad_lab = (idx >= 0) & ~bad_idx & ((lab < 0) | (lab >= C))
    return (keys[:, -1] == 0) * 1 | bad_lab.any(1) * 2 | bad_idx.any(1) * 4


def _sweep():
    cases = [(k, 9, 5, 0.1) for k in KS]
    cases += [(k, C, 5 if k < 1000 else 3, 0.1) for C in CS for k in (200, 4261)]
    cases += [(k, 9, B, t) for B in BS for k, t in ((33, 0.1), (3196, 0.07))]
    cases += [(k, 38 if k < 1000 else 9, 5, t) for t in TS for k in (200, 8192)]
    return cases


@pytest.mark.parametrize("k,C,B,t", _sweep())
def test_vote_against_fp64_reference(k, C, B, t):
    keys, labels = _case(B, k, C, seed=k * 7 + C * 13 + B + int(abs(t) * 100))
    kd, ld = _t(keys.view(np.int64)), _t(labels)
    pred, scores = b200knn.vote(kd, ld, C, t, return_scores=True)
    assert pred.shape == (B, C) and scores.shape == (B, C)
    pred, scores = pred.cpu().numpy(), scores.cpu().numpy()
    checked = _check_vote(pred, scores, keys, labels, C, t)
    assert checked >= (B * 3) // 5 - 1 or t == 1000.0  # at t = 1000 every weight is ~1: near ties abound
    _check_ties(pred, scores, keys, labels)
    # the status word and the grid vote of the same keys: the same ranking, bitwise
    packed = K.vote_packed(kd, ld, C, t, B + 2).cpu().numpy()
    assert np.array_equal(packed[:B, :C], pred) and not packed[B:].any()
    assert np.array_equal(packed[:B, C], _status_ref(keys, labels, C))
    grid = K.vote_multi_packed(kd, ld, C, (k,), (t,), B + 1).cpu().numpy()
    assert np.array_equal(grid, packed[:B + 1])


@pytest.mark.parametrize("k", [200, 5000])
@pytest.mark.parametrize("C", [9, 65])
def test_vote_overflow_and_underflow_weights(k, C):
    """t = 1e-3 with sims near ±1: exp(sim / t) overflows to inf (such classes tie, ranked by class
    index) or underflows to 0 (such classes tie with the classes that got no vote)."""
    t = 1e-3
    keys, labels = _case(12, k, C, seed=k + C, extreme=True)
    pred, scores = b200knn.vote(_t(keys.view(np.int64)), _t(labels), C, t, return_scores=True)
    pred, scores = pred.cpu().numpy(), scores.cpu().numpy()
    _, want = _ref_vote(keys, labels, C, t)
    assert np.isinf(want).any() and np.isfinite(want[want > 0]).any()
    _, idx = O.decode_keys(keys)
    voted = np.zeros_like(want, bool)
    for b in range(keys.shape[0]):
        voted[b, labels[idx[b][idx[b] >= 0]]] = True
    assert (voted & (want == 0)).any()  # underflowed votes, tied with the classes without votes
    assert _check_vote(pred, scores, keys, labels, C, t) == keys.shape[0]
    _check_ties(pred, scores, keys, labels)
    for b in range(keys.shape[0]):  # inf block first, then finite, then zeros; class order inside ties
        s = scores[b, pred[b]]
        for v in (np.inf, 0.0):
            assert (np.diff(pred[b][s == v]) > 0).all()


def test_signed_zero_sims():
    """A -0.0 similarity votes exactly as +0.0: the search's key maps both to one key, and a key that
    still carries -0.0 gets the same weight and rank."""
    assert O.make_keys(np.float32([-0.0]), [7])[0] == O.make_keys(np.float32([0.0]), [7])[0]
    sims = np.float32([0.5, 0.0, 0.0, 0.0, -0.25])
    keys = np.stack([O.make_keys(sims, np.arange(5))] * 2)
    keys[1, 3] = (np.uint64(0x7FFFFFFF) << np.uint64(32)) | np.uint64(0xFFFFFFFF - 3)  # raw -0.0
    assert O.decode_keys(keys[1, 3:4])[0].view(np.uint32)[0] == 0x80000000
    labels = np.array([2, 0, 1, 1, 0])
    for t in (0.1, -0.1):
        pred, scores = b200knn.vote(_t(keys.view(np.int64)), _t(labels), 3, t, return_scores=True)
        assert torch.equal(pred[0], pred[1]) and torch.equal(scores[0], scores[1])


def _raw_vote_ex(keys, labels, C, t, label_offset):
    """b200knn_vote_ex with a label offset (the sharded owner's form): (rc, (B, C+1) rankings + status)."""
    B, k = keys.shape
    out = torch.zeros((B, C + 1), dtype=torch.int64, device=DEV)
    flag = torch.zeros((1,), dtype=torch.int32, device=DEV)
    rc = _lib.load().b200knn_vote_ex(keys.data_ptr(), labels.data_ptr(), B, k, labels.numel(), label_offset, C,
                                     float(t), out.data_ptr(), C + 1, C, None, flag.data_ptr(), K._stream())
    torch.cuda.synchronize()
    return rc, out, int(flag.item())


def _raw_vote_multi(keys, labels, C, ks, ts, label_offset, status=True):
    B, k = keys.shape
    W = len(ks) * len(ts) * C
    out = torch.zeros((B, W + 1), dtype=torch.int64, device=DEV)
    flag = torch.zeros((1,), dtype=torch.int32, device=DEV)
    rc = _lib.load().b200knn_vote_multi(keys.data_ptr(), labels.data_ptr(), B, k, labels.numel(), label_offset, C,
                                        (ctypes.c_int * len(ks))(*ks), len(ks), (ctypes.c_double * len(ts))(*ts),
                                        len(ts), out.data_ptr(), W + 1, W if status else -1, flag.data_ptr(),
                                        K._stream())
    torch.cuda.synchronize()
    return rc, out, int(flag.item())


@pytest.mark.parametrize("k", [40, 1500])
def test_status_word_bits(k):
    """Bit 1: slot k-1 empty; bit 2: a label outside [0, C), negative too; bit 4: a neighbour index
    outside [label_offset, label_offset + n_labels).  Each on its own row and together."""
    C, off, n_lab = 9, 1000, 3 * k
    rng = np.random.default_rng(k)
    labels = rng.integers(0, C, n_lab)
    labels[5], labels[6] = C, -3
    sims = -np.sort(-rng.uniform(-1, 1, (9, k)).astype(np.float32), axis=1)
    idx = off + 10 + rng.integers(0, n_lab - 10, (9, k))  # clean rows
    idx[2, k // 2] = off + 5                       # label C
    idx[3, 1] = off + 6                            # label -3
    idx[4, k - 2] = off - 1                        # below the offset
    idx[5, 0] = off + n_lab                        # past the labels
    idx[7, 3], idx[8, 7], idx[8, 9] = off + 6, off + 5, off + n_lab + 9
    keys = O.make_keys(sims, idx)
    keys[1, k - 10:] = 0
    keys[6, k - 1] = 0
    keys[7, k - 1:] = 0
    keys[8, k - 1] = 0
    want = np.array([0, 1, 2, 2, 4, 4, 1, 3, 7])
    assert np.array_equal(_status_ref(keys, labels, C, off), want)
    kd, ld = _t(keys.view(np.int64)), _t(labels)
    rc, out, _ = _raw_vote_ex(kd, ld, C, 0.1, off)
    assert rc == 0 and np.array_equal(out[:, C].cpu().numpy(), want)
    ks, ts = (k // 2, k), (0.1, -0.3)
    rc, out2, _ = _raw_vote_multi(kd, ld, C, ks, ts, off)
    assert rc == 0 and np.array_equal(out2[:, -1].cpu().numpy(), want)
    # rows 0, 1 and 6 are clean apart from empty slots: their rankings are the single vote's
    clean = _t(np.array([0, 1, 6]))
    single = b200knn.vote(kd[clean], ld, C, ts[1], label_offset=off)
    assert torch.equal(out2[clean, 3 * C:4 * C], single)
    assert torch.equal(out[clean, :C], b200knn.vote(kd[clean], ld, C, 0.1, label_offset=off))
    # vote_packed / vote_multi_packed (label offset 0): the same bits
    keys0 = O.make_keys(sims, np.where(idx < off, n_lab + 100, idx - off))
    keys0[keys == 0] = 0
    k0 = _t(keys0.view(np.int64))
    assert np.array_equal(K.vote_packed(k0, ld, C, 0.1, 9)[:, C].cpu().numpy(), want)
    assert np.array_equal(K.vote_multi_packed(k0, ld, C, ks, ts, 9)[:, -1].cpu().numpy(), want)
    # the host flag raises knn_predict's errors
    for rows, msg in (([2, 3], r"outside \[0, num_classes=9\)"), ([4, 5], "neighbour index outside feature_labels")):
        sel = _t(np.array(rows))
        with pytest.raises(RuntimeError, match=msg):
            b200knn.vote(kd[sel], ld, C, 0.1, label_offset=off)
        with pytest.raises(RuntimeError, match=msg):
            K.vote_multi(k0[sel], ld, C, ks, ts)
        with pytest.raises(RuntimeError, match=msg):
            b200knn.vote(k0[sel], ld, C, 0.1)


GRIDS = [
    ((1, 2, 31, 32, 33, 64, 100, 200, 992, 993, 1023, 1024, 1025, 2047, 3196, 5000),
     (0.07, 0.1, 1.0, 1000.0, -0.1, 1e-3, 0.5, -2.0)),  # the largest grid
    ((1, 5), (0.1,)),
    ((32, 64, 96, 1024, 2048), (0.1, 0.07)),          # boundaries on multiples of 32 and of the chunk
    ((31, 65, 97, 1000, 1030, 2049), (0.1, -0.5)),    # ... and off them
    ((1500,), (0.1, 0.2, 0.3)),                      # one k past the chunk, several t
]


@pytest.mark.parametrize("ks,ts", GRIDS)
@pytest.mark.parametrize("C", [9, 65])
def test_vote_multi_equals_vote(ks, ts, C):
    keys, labels = _case(11, ks[-1], C, seed=len(ks) * 31 + C)
    kd, ld = _t(keys.view(np.int64)), _t(labels)
    got = K.vote_multi(kd, ld, C, ks, ts)
    assert got.shape == (11, len(ks) * len(ts) * C)
    for i, k in enumerate(ks):
        for j, t in enumerate(ts):
            want = b200knn.vote(kd[:, :k].contiguous(), ld, C, t)
            blk = (i * len(ts) + j) * C
            assert torch.equal(got[:, blk:blk + C], want), (k, t)


@pytest.mark.parametrize("k", [5, 1023, 1024, 5000])
def test_class_count_bound(k):
    """The largest C of vote_max_classes is served and one more is refused: a ValueError naming the
    bound from Python before any launch, B200KNN_E_UNSUPPORTED from the C ABI."""
    keys, _ = _case(3, k, 9, seed=k)
    kd = _t(keys.view(np.int64))
    for grid in (False, True):
        c_max = K.vote_max_classes(k, grid)
        labels = np.random.default_rng(k).integers(0, c_max, 3 * k)
        ld = _t(labels)
        if grid:
            pred = K.vote_multi(kd, ld, c_max, (k,), (0.1,))
            assert torch.equal(pred, b200knn.vote(kd, ld, c_max, 0.1))
            assert _raw_vote_multi(kd, ld, c_max + 1, (k,), (0.1,), 0)[0] == E_UNSUPPORTED
            with pytest.raises(ValueError, match=f"at most {c_max} classes"):
                K.vote_multi(kd, ld, c_max + 1, (k,), (0.1,))
        else:
            pred, scores = b200knn.vote(kd, ld, c_max, 0.1, return_scores=True)
            _check_vote(pred.cpu().numpy(), scores.cpu().numpy(), keys, labels, c_max, 0.1)
            assert _raw_vote_ex(kd, ld, c_max + 1, 0.1, 0)[0] == E_UNSUPPORTED
            for fn in (lambda C: b200knn.vote(kd, ld, C, 0.1), lambda C: K.vote_packed(kd, ld, C, 0.1, 3)):
                with pytest.raises(ValueError, match=f"at most {c_max} classes"):
                    fn(c_max + 1)
    assert K.vote_max_classes(k, True) <= K.vote_max_classes(k, False)


@pytest.fixture()
def mode_guard():
    yield
    b200knn.set_default_mode("exact")


def test_class_count_bound_before_search(mode_guard):
    rng = np.random.default_rng(0)
    bank = _t(rng.standard_normal((64, 6000)).astype(np.float32))
    q = _t(rng.standard_normal((5, 64)).astype(np.float32))
    lab = _t(datagen.labels(6000, 9, 1))
    for mode in ("exact", "bf16"):
        b200knn.set_default_mode(mode)
        for k in (5, 5000):
            c1 = K.vote_max_classes(k) + 1
            g1 = K.vote_max_classes(k, grid=True) + 1
            before = _lib.launch_counter["kernels"]
            with pytest.raises(ValueError, match=f"at most {c1 - 1} classes"):
                b200knn.knn_predict(q, bank, lab, c1, k, 0.1)
            with pytest.raises(ValueError, match=f"at most {g1 - 1} classes"):
                b200knn.knn_predict_multi(q, bank, lab, g1, (3, k), (0.1,))
            with pytest.raises(ValueError, match=f"at most {g1 - 1} classes"):
                b200knn.knn_predict_loo(bank, lab, g1, (3, k), (0.1,))
            assert _lib.launch_counter["kernels"] == before
        # at the bound: the 9 voted classes lead, the classes without votes follow in order
        c_max = K.vote_max_classes(5000)
        pred = b200knn.knn_predict(q, bank, lab, c_max, 5000, 0.1)
        assert torch.equal(pred[:, :9], b200knn.knn_predict(q, bank, lab, 9, 5000, 0.1))
        assert torch.equal(pred[:, 9:], torch.arange(9, c_max, device=DEV).expand(5, -1))


NS = [1, 255, 256, 257, 151551, 151552, 151553, 10 ** 6]


@pytest.mark.parametrize("C", [1, 2, 63, 64, 65, 200])
def test_confusion_counts_exact(C):
    """151,552 = 592 blocks x 256 threads: the grid-stride loop's first pass ends there."""
    rng = np.random.default_rng(C)
    for n in NS:
        target = rng.integers(0, C, n)
        pred = np.where(rng.random(n) < 0.6, target, rng.integers(0, C, n))
        want = np.zeros((C, C), np.int64)
        np.add.at(want, (target, pred), 1)
        got = b200knn.confusion_counts(_t(pred), _t(target), C)
        assert got.dtype == torch.int64 and np.array_equal(got.cpu().numpy(), want), n
    n = 151553  # a bad entry in the second pass, in either argument
    for bad in (-1, C, -(2 ** 40), 2 ** 40):
        for which in (0, 1):
            p, t = rng.integers(0, C, n), rng.integers(0, C, n)
            (p, t)[which][-1] = bad
            with pytest.raises(RuntimeError, match=f"outside \\[0, num_classes={C}\\)"):
                b200knn.confusion_counts(_t(p), _t(t), C)


def test_confusion_global_path_equals_shared_path():
    rng = np.random.default_rng(3)
    target, pred = rng.integers(0, 64, 300000), rng.integers(0, 64, 300000)
    small = b200knn.confusion_counts(_t(pred), _t(target), 64)
    for C in (65, 200):
        big = b200knn.confusion_counts(_t(pred), _t(target), C)
        assert torch.equal(big[:64, :64], small) and int(big.sum()) == 300000


@pytest.mark.parametrize("C", [65, 200])
def test_knn_metrics_above_64_classes(C):
    rng = np.random.default_rng(C)
    target = rng.integers(0, C - 1, 200000)  # the last class never occurs
    pred = np.where(rng.random(200000) < 0.6, target, rng.integers(0, C - 1, 200000))
    m = b200knn.knn_metrics(_t(pred), _t(target), C)
    ref = O.metrics_ref(pred, target, C)
    assert np.array_equal(m["counts"].cpu().numpy(), ref["counts"])
    assert abs(float(m["accuracy"]) - ref["accuracy"]) < 1e-12
    assert abs(float(m["f1"]) - ref["f1"]) < 1e-12
    assert np.allclose(m["confusion"].cpu().numpy(), ref["confusion"], rtol=1e-15, atol=0)


def _deleted(bank, lab, C, ks, ts, r):
    """knn_predict_multi of bank row r against the bank without column r: (n_k, n_t, C)."""
    keep = torch.ones(bank.shape[1], dtype=torch.bool, device=bank.device)
    keep[r] = False
    q = bank[:, r:r + 1].t()
    return b200knn.knn_predict_multi(q, bank[:, keep].contiguous(), lab[keep].contiguous(), C, ks, ts)[:, :, 0]


def _large_k_case():
    rng = np.random.default_rng(5000)
    N, D, B = 6000, 64, 37
    bank = np.ascontiguousarray(rng.standard_normal((N, D)).astype(np.float32).T)
    q = rng.standard_normal((B, D)).astype(np.float32)
    return q, bank, datagen.labels(N, 9, 6)


@pytest.mark.parametrize("mode", ["exact", "fp32"])
def test_large_k_end_to_end(mode, mode_guard):
    """k = 5000 > 4260 and a grid to 5000 > 3195 at C = 9 (N = 6000, D = 64): the SEQ oracle's lists
    with the reference vote, the grid bitwise the separate calls, LOO bitwise row deletion."""
    q, bank, lab = _large_k_case()
    ss, si = O.topk_seqfma(q, bank, 5000)
    keys = O.make_keys(ss, si)
    b200knn.set_default_mode(mode)
    qd, bd, ld = _t(q), _t(bank), _t(lab)
    pred = b200knn.knn_predict(qd, bd, ld, 9, 5000, 0.5)
    seq_pred, scores = b200knn.vote(_t(keys.view(np.int64)), ld, 9, 0.5, return_scores=True)
    assert torch.equal(pred, seq_pred)
    assert _check_vote(pred.cpu().numpy(), scores.cpu().numpy(), keys, lab, 9, 0.5) == q.shape[0]
    ks, ts = (5, 3500, 5000), (0.1, 0.5)
    grid = b200knn.knn_predict_multi(qd, bd, ld, 9, ks, ts)
    for i, k in enumerate(ks):
        for j, t in enumerate(ts):
            assert torch.equal(grid[i, j], b200knn.knn_predict(qd, bd, ld, 9, k, t)), (k, t)
    loo = b200knn.knn_predict_loo(bd, ld, 9, (3500,), (0.1,))
    for r in (0, 2999, 5999):
        assert torch.equal(loo[:, :, r], _deleted(bd, ld, 9, (3500,), (0.1,), r)), r


def test_large_k_bf16_equals_exact(mode_guard):
    """Lists longer than 992 come from the exact kernel in the raw modes."""
    q, bank, lab = _large_k_case()
    qd, bd, ld = _t(q), _t(bank), _t(lab)
    out = {}
    for mode in ("exact", "bf16"):
        b200knn.set_default_mode(mode)
        out[mode] = (b200knn.knn_predict(qd, bd, ld, 9, 5000, 0.5),
                     b200knn.knn_predict_multi(qd, bd, ld, 9, (3500, 5000), (0.1, 0.5)),
                     b200knn.knn_predict_loo(bd, ld, 9, (3500,), (0.1,)))
    for a, b in zip(out["exact"], out["bf16"]):
        assert torch.equal(a, b)
