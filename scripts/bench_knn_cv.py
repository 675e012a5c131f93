"""Cost of group exclusion inside the neighbour search: k-fold cross-validation through
knn_predict_loo(groups=folds), leave-one-group-out with a group deeper than the streaming lists, and
knn_predict_multi with query / bank groups, against plain leave-one-out and the ungrouped call.

  python scripts/bench_knn_cv.py --out DIR [--reps R] [--checks C]

Seeded bench.make_inputs banks, D = 512, fp32 mode, C = 9, ks = (5, 20, 200), ts = (0.07, 0.1), at two
sizes: N = 37,348 (the reference's train_data bank) and N = 811,457 (WM-811K).  Calls, timed
alternately with CUDA events, each ending in a host synchronisation:
  - loo:         plain leave-one-out (groups=None), searches at k + 1 and drops the row;
  - lots_of_25:  groups = arange(N) // 25, searches at k + 32 and drops the group (unchanged path);
  - group_2000:  one group of 2,000 seeded rows plus singletons: those rows search at depth k with
                 their group skipped inside the search (before: k + 2048 through exact peeling);
  - fold5:       5-fold cross-validation, seeded fold ids: every row skips its fold of N/5 rows;
  - multi / multi_groups: knn_predict_multi of Q = 151,552 queries (bank rows plus noise) without
                 and with query / bank groups (lots of 25, a query carrying its source row's lot):
                 the grouped call runs the excluded epilogue and has no sampling pre-pass.
The 811k bank's 1.66 GB of fp32 rows exceed the 126 MB L2, so every pass reads it from HBM.  C seeded
rows per grouped case are checked bitwise against knn_predict_multi on the bank without the row's
group (each check copies and prepares a whole bank).  Writes DIR/bench_knn_cv.json with the GPU's
name and power limit read in the same run.
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

KS, TS, C, D, BATCH, Q = (5, 20, 200), (0.07, 0.1), 9, 512, 75776, 151552


def deletion_checks(bank, labels, bank_groups, got, rows, queries=None, query_groups=None):
    """got[:, :, r] against knn_predict_multi of query r on the bank without its group's columns."""
    out = []
    for r in rows:
        q = bank[:, r:r + 1].t() if queries is None else queries[r:r + 1]
        own = bank_groups[r] if query_groups is None else query_groups[r]
        keep = bank_groups != own
        want = K.knn_predict_multi(q, bank[:, keep].contiguous(), labels[keep].contiguous(), C, KS, TS)[:, :, 0]
        out.append(bool(torch.equal(got[:, :, r], want)))
        del want, keep
        torch.cuda.empty_cache()
    return out


def one_size(N, seed, reps, n_checks):
    bank_nd, labels, _ = bench.make_inputs("cuda", N, 1, D, seed=seed)
    bank = bank_nd.t().contiguous()  # the reference's (D, N) feature_bank
    del bank_nd
    K.set_default_mode("fp32")
    rng = np.random.default_rng(seed)
    big = torch.from_numpy(np.sort(rng.choice(N, 2000, replace=False))).cuda()
    lots = torch.arange(N, device="cuda") // 25
    g2000 = torch.arange(N, device="cuda")
    g2000[big] = -1
    folds = torch.from_numpy(rng.permutation(N) % 5).cuda()
    groups = {"lots_of_25": lots, "group_2000": g2000, "fold5": folds}
    g = torch.Generator(device="cuda").manual_seed(seed)
    src = torch.randint(0, N, (Q,), generator=g, device="cuda")
    queries = torch.nn.functional.normalize(bank.t()[src] + 0.02 * torch.randn(Q, D, generator=g, device="cuda"),
                                            dim=1)
    q_lots = lots[src].contiguous()

    def loo(gr):
        return lambda: K.knn_predict_loo(bank, labels, C, KS, TS, batch=BATCH, groups=gr)

    calls = {"loo": loo(None), **{name: loo(gr) for name, gr in groups.items()},
             "multi": lambda: K.knn_predict_multi(queries, bank, labels, C, KS, TS),
             "multi_groups": lambda: K.knn_predict_multi(queries, bank, labels, C, KS, TS, query_groups=q_lots,
                                                         bank_groups=lots)}
    outs = {name: fn() for name, fn in calls.items()}  # warm-up: bank preparation, first launches
    times = {name: [] for name in calls}
    for _ in range(reps):  # alternate the calls so drift and neighbours hit them alike
        for name, fn in calls.items():
            ms, outs[name] = event_ms(fn)
            times[name].append(ms)
    med = {name: stats(v)["median"] for name, v in times.items()}
    check_rows = np.sort(rng.choice(N, n_checks, replace=False)).tolist()
    in_big = big[torch.randperm(2000, generator=torch.Generator().manual_seed(seed))[:n_checks // 2].cuda()]
    big_rows = sorted(in_big.tolist()) + np.sort(rng.choice(N, n_checks - n_checks // 2, replace=False)).tolist()
    q_rows = np.sort(rng.choice(Q, n_checks, replace=False)).tolist()
    checks = {"lots_of_25": deletion_checks(bank, labels, lots, outs["lots_of_25"], check_rows),
              "group_2000": deletion_checks(bank, labels, g2000, outs["group_2000"], big_rows),
              "fold5": deletion_checks(bank, labels, folds, outs["fold5"], check_rows),
              "multi_groups": deletion_checks(bank, labels, lots, outs["multi_groups"], q_rows, queries, q_lots)}
    return {
        "shape": {"N": N, "D": D, "C": C, "mode": "fp32", "knn_ks": KS, "knn_ts": TS, "batch": BATCH, "Q": Q,
                  "seed": seed},
        "ms": {name: stats(v) for name, v in times.items()},
        "over_loo": {name: med[name] / med["loo"] for name in ("lots_of_25", "group_2000", "fold5")},
        "multi_groups_over_multi": med["multi_groups"] / med["multi"],
        "rows_checked": {"lots_of_25": check_rows, "group_2000": big_rows, "fold5": check_rows,
                         "multi_groups": q_rows},
        "bitwise_equal_to_group_deletion": checks,
        "all_bitwise_equal": all(all(v) for v in checks.values()),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--checks", type=int, default=32)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_knn_cv.py measures on a GPU; none is visible")
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(),
           "train_data_37k": one_size(37348, 1, args.reps, args.checks),
           "wm811k": one_size(811457, 0, args.reps, args.checks)}
    path = os.path.join(args.out, "bench_knn_cv.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
