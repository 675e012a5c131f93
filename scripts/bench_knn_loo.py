"""Cost of knn_predict_loo (leave-one-out kNN of a labelled bank against itself) against its search floor.

  python scripts/bench_knn_loo.py --out DIR [--reps R] [--checks C]

Seeded bench.make_inputs banks, D = 512, fp32 mode, ks = (5, 20, 200), ts = (0.07, 0.1), at two sizes:
N = 37,348, C = 9 (the reference's train_data bank) and N = 811,457 (WM-811K).  Timed alternately with
CUDA events, every call ending in a host synchronisation: the LOO call, and the search floor, i.e.
topk_keys of every bank row at k_max + 1 = 201 in the same batches of 75,776 rows.  The 811k bank's
1.66 GB of fp32 rows exceed the 126 MB L2, so every pass reads it from HBM.  drop_self_kernel and
vote_multi_kernel alone: CUDA events over repeated launches on the keys of one batch.  C seeded rows
per size are checked bitwise against knn_predict_multi on the bank with that row deleted (each check
copies and prepares a whole bank).  Writes DIR/bench_knn_loo.json with the GPU's name and power limit
read in the same run.
"""
import argparse
import json
import os
import sys

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
for p in (ROOT, os.path.join(ROOT, "self-supervised-wafermaps_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (make_inputs: the benchmark's seeded synthetic embeddings)
from b200knn import knn as K  # noqa: E402
from bench_knn_grid import event_ms, gpu_info, stats  # noqa: E402

KS, TS, C, D, BATCH = (5, 20, 200), (0.07, 0.1), 9, 512, 75776


def kernel_ms(fn, n=50):
    fn()

    def loop():  # outputs are dropped at once: the allocator reuses one block, no allocation in the window
        for _ in range(n):
            fn()

    ms, _ = event_ms(loop)
    return ms / n


def one_size(N, seed, reps, n_checks):
    bank_nd, labels, _ = bench.make_inputs("cuda", N, 1, D, seed=seed)
    bank = bank_nd.t().contiguous()  # the reference's (D, N) feature_bank
    del bank_nd
    K.set_default_mode("fp32")
    k1 = max(KS) + 1

    def floor():
        for lo in range(0, N, BATCH):
            K.topk_keys(bank[:, lo:lo + BATCH].t().contiguous(), bank, k1, "fp32")

    calls = {"loo": lambda: K.knn_predict_loo(bank, labels, C, KS, TS, batch=BATCH), "search_floor": floor}
    outs = {name: fn() for name, fn in calls.items()}  # warm-up: bank preparation, first launches
    times = {name: [] for name in calls}
    for _ in range(reps):  # alternate the two so drift and neighbours hit them alike
        for name, fn in calls.items():
            ms, outs[name] = event_ms(fn)
            times[name].append(ms)
    loo = outs["loo"]
    # the kernels after the search, alone, on the keys of the first batch
    b = min(N, BATCH)
    keys = K.topk_keys(bank[:, :b].t().contiguous(), bank, k1, "fp32")
    dropped = K.drop_self(keys, 0)
    flag = torch.zeros((1,), dtype=torch.int32, device="cuda")
    kern = {"drop_self_batch": kernel_ms(lambda: K.drop_self(keys, 0)),
            "vote_multi_batch": kernel_ms(lambda: K.vote_multi(dropped, labels, C, KS, TS, check_labels=False,
                                                               flag=flag))}
    n_batches = (N + BATCH - 1) // BATCH
    bytes_drop = b * (2 * k1 - 1) * 8
    # explicit row deletion for seeded rows
    rows = np.sort(np.random.default_rng(seed).choice(N, n_checks, replace=False))
    checks = []
    for r in rows.tolist():
        keep = torch.ones(N, dtype=torch.bool, device="cuda")
        keep[r] = False
        want = K.knn_predict_multi(bank[:, r:r + 1].t(), bank[:, keep].contiguous(), labels[keep].contiguous(), C,
                                   KS, TS)[:, :, 0]
        checks.append(bool(torch.equal(loo[:, :, r], want)))
        del want, keep
        torch.cuda.empty_cache()
    med = {name: stats(v)["median"] for name, v in times.items()}
    after_search = (kern["drop_self_batch"] + kern["vote_multi_batch"]) * N / b
    return {
        "shape": {"N": N, "D": D, "C": C, "mode": "fp32", "knn_ks": KS, "knn_ts": TS, "batch": BATCH,
                  "batches": n_batches, "seed": seed},
        "ms": {name: stats(v) for name, v in times.items()},
        "loo_over_search_floor": med["loo"] / med["search_floor"],
        "kernel_ms": kern,
        "drop_self_GBps": bytes_drop / (kern["drop_self_batch"] * 1e-3) / 1e9,
        "drop_plus_vote_ms_all_rows": after_search,
        "drop_plus_vote_share_of_loo": after_search / med["loo"],
        "rows_checked": rows.tolist(),
        "bitwise_equal_to_row_deletion": checks,
        "all_bitwise_equal": all(checks),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--checks", type=int, default=32)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_knn_loo.py measures on a GPU; none is visible")
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(),
           "train_data_37k": one_size(37348, 1, args.reps, args.checks),
           "wm811k": one_size(811457, 0, args.reps, args.checks)}
    path = os.path.join(args.out, "bench_knn_loo.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
