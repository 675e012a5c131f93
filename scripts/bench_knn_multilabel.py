"""Cost of knn_predict_multilabel (per-label scores over a (k, t) grid from one neighbour search) against
knn_predict_multi, whose search it shares.

  python scripts/bench_knn_multilabel.py --out DIR [--reps R] [--queries Q]

North star (N = 811,457, D = 512, Q = 151,552, fp32 mode, ks = (10, 20, 100, 200), ts = (0.07, 0.1)):
knn_predict_multilabel with L = 8 labels against knn_predict_multi with 9 classes, timed alternately with
CUDA events (every call ends in its own host synchronisation).  The bank's labels are the benchmark's 9
classes as 8-pattern sets (class c < 8: pattern c; class 8, the most frequent: no pattern); the cost
does not depend on which bits are set.  Then the vote kernels alone on the k = 200 keys (CUDA events over repeated
launches): b200knn_vote_multilabel against b200knn_vote_multi, and the multi-label kernel as bytes/s
against HBM peak (k_max * 8 B of keys in, n_k * n_t * L * 8 B of scores out per query; the label
gather hits L2).  The bank's 1.66 GB of fp32 rows exceed the 126 MB L2, so every search reads it from
HBM.  c3 shape (N = 30,000, Q = 5,703, D = 512, k = 20, L = 8, t = 0.1): the same two calls.  At both
sizes the scores are compared bitwise with b200knn_vote_multilabel on the mode's own top-k keys.
Writes DIR/bench_knn_multilabel.json with the GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import sys

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
for p in (ROOT, os.path.join(ROOT, "self-supervised-wafermaps_b200"), os.path.join(ROOT, "scripts")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import bench  # noqa: E402  (make_inputs: the benchmark's seeded synthetic embeddings)
import b200knn  # noqa: E402
from b200knn import knn as K  # noqa: E402
from bench_knn_grid import event_ms, gpu_info, stats  # noqa: E402

HBM_PEAK = 7.7e12  # B/s, NVIDIA's HGX B200 data sheet, per GPU


def compare(N, Q, ks, ts, reps, seed):
    bank_nd, labels, q = bench.make_inputs("cuda", N, Q, 512, seed=seed)
    bank = bank_nd.t().contiguous()
    del bank_nd
    m = torch.nn.functional.one_hot(labels, 9)[:, :8].to(torch.uint8)
    L = m.shape[1]
    b200knn.set_default_mode("fp32")
    calls = {
        "multilabel": lambda: K.knn_predict_multilabel(q, bank, m, ks, ts),
        "multi_C9": lambda: K.knn_predict_multi(q, bank, labels, 9, ks, ts),
    }
    outs = {name: fn() for name, fn in calls.items()}  # warm-up: bank preparation, first launches
    times = {name: [] for name in calls}
    for _ in range(reps):  # alternate the two so drift and neighbours hit them alike
        for name, fn in calls.items():
            ms, outs[name] = event_ms(fn)
            times[name].append(ms)
    keys = K.topk_keys(q, bank, max(ks), "fp32")
    bits = b200knn.pack_label_bits(m)
    asc = sorted(range(len(ks)), key=ks.__getitem__)
    own = K.grid_view(K.vote_multilabel(keys, bits, L, [ks[i] for i in asc], ts), asc, len(ts), L)
    med = {name: stats(v)["median"] for name, v in times.items()}
    res = {
        "shape": {"N": N, "D": 512, "Q": Q, "mode": "fp32", "knn_ks": ks, "knn_ts": ts, "L": L, "C": 9},
        "ms": {name: stats(v) for name, v in times.items()},
        "multilabel_over_multi": med["multilabel"] / med["multi_C9"],
        "bitwise_equal_to_vote_of_own_keys": bool(torch.equal(outs["multilabel"], own)),
    }
    return res, keys, labels, bits, L


def kernels(keys, labels, bits, L, ks, ts, n=20):
    ks = sorted(ks)
    flag = torch.zeros((1,), dtype=torch.int32, device="cuda")
    out = {}
    for name, fn in (("vote_multilabel", lambda: K.vote_multilabel(keys, bits, L, ks, ts, check_labels=False,
                                                                   flag=flag)),
                     ("vote_multi_C9", lambda: K.vote_multi(keys, labels, 9, ks, ts, check_labels=False, flag=flag))):
        fn()

        def loop():  # outputs are dropped at once: the allocator reuses one block, no allocation in the window
            for _ in range(n):
                fn()

        runs = []
        for _ in range(3):
            ms, _ = event_ms(loop)
            runs.append(ms / n)
        out[name] = stats(runs)
    B, k = keys.shape
    moved = B * k * 8 + B * len(ks) * len(ts) * L * 8
    ms = out["vote_multilabel"]["median"]
    out["vote_multilabel_bytes"] = moved
    out["vote_multilabel_bytes_per_s"] = moved / (ms * 1e-3)
    out["vote_multilabel_share_of_hbm_peak"] = moved / (ms * 1e-3) / HBM_PEAK
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--queries", type=int, default=151552)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_knn_multilabel.py measures on a GPU; none is visible")
    os.makedirs(args.out, exist_ok=True)
    ks, ts = (10, 20, 100, 200), (0.07, 0.1)
    res = {"gpu": gpu_info()}
    ns, keys, labels, bits, L = compare(811457, args.queries, ks, ts, args.reps, seed=0)
    ns["kernel_ms"] = kernels(keys, labels, bits, L, ks, ts)
    res["north_star"] = ns
    del keys, labels, bits
    res["c3"] = compare(30000, 5703, (20,), (0.1,), max(args.reps, 20), seed=3)[0]
    path = os.path.join(args.out, "bench_knn_multilabel.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
