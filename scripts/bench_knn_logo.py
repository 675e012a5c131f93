"""Cost of knn_predict_loo(groups=...) (leave-one-group-out kNN of a labelled bank against itself)
against plain leave-one-out.

  python scripts/bench_knn_logo.py --out DIR [--reps R] [--checks C]

Seeded bench.make_inputs banks, D = 512, fp32 mode, C = 9, ks = (5, 20, 200), ts = (0.07, 0.1), at two
sizes: N = 37,348 (the reference's train_data bank) and N = 811,457 (WM-811K).  Four calls, timed
alternately with CUDA events, every call ending in a host synchronisation:
  - loo:          plain leave-one-out (groups=None), searches at k + 1;
  - singletons:   groups = arange(N), which must be bitwise `loo` at the same cost;
  - lots_of_25:   groups = arange(N) // 25, searches at k + 32;
  - group_2000:   one group of 2,000 seeded rows plus singletons: those rows search at
                  k + 2048 > MAX_K, i.e. through the exact peeling path.
The 811k bank's 1.66 GB of fp32 rows exceed the 126 MB L2, so every pass reads it from HBM.
drop_group_kernel alone (and drop_self_kernel on the plain search's keys for comparison): CUDA events
over repeated launches on the keys of one search.  C seeded rows per size of lots_of_25, and C / 2 rows
of group_2000 (half of them in the group), are checked bitwise against knn_predict_multi on the bank
without the row's group (each check copies and prepares a whole bank).  Writes DIR/bench_knn_logo.json
with the GPU's name and power limit read in the same run.
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
from bench_knn_loo import kernel_ms  # noqa: E402

KS, TS, C, D, BATCH = (5, 20, 200), (0.07, 0.1), 9, 512, 75776


def deletion_checks(bank, labels, groups, got, rows):
    out = []
    for r in rows:
        keep = groups != groups[r]
        want = K.knn_predict_multi(bank[:, r:r + 1].t(), bank[:, keep].contiguous(), labels[keep].contiguous(), C,
                                   KS, TS)[:, :, 0]
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
    groups = {"singletons": torch.arange(N, device="cuda"), "lots_of_25": torch.arange(N, device="cuda") // 25}
    g2000 = torch.arange(N, device="cuda")
    g2000[big] = -1
    groups["group_2000"] = g2000

    def call(g):
        return lambda: K.knn_predict_loo(bank, labels, C, KS, TS, batch=BATCH, groups=g)

    calls = {"loo": call(None), **{name: call(g) for name, g in groups.items()}}
    outs = {name: fn() for name, fn in calls.items()}  # warm-up: bank preparation, first launches
    times = {name: [] for name in calls}
    for _ in range(reps):  # alternate the calls so drift and neighbours hit them alike
        for name, fn in calls.items():
            ms, outs[name] = event_ms(fn)
            times[name].append(ms)
    med = {name: stats(v)["median"] for name, v in times.items()}
    # the exclusion kernels alone, on the keys of one search each
    k_max = max(KS)
    b1 = min(N, BATCH)
    keys1 = K.topk_keys(bank[:, :b1].t().contiguous(), bank, k_max + 1, "fp32")
    depth = k_max + 32
    b32 = min(N, BATCH * (k_max + 1) // depth)
    keys32 = K.topk_keys(bank[:, :b32].t().contiguous(), bank, depth, "fp32")
    flag = torch.zeros((1,), dtype=torch.int32, device="cuda")
    gid = {name: torch.unique(g, return_inverse=True)[1].to(torch.int32) for name, g in groups.items()}
    rows1, rows32 = torch.arange(b1, device="cuda"), torch.arange(b32, device="cuda")
    kern = {
        "drop_self_k201": kernel_ms(lambda: K.drop_self(keys1, 0)),
        "drop_group_k201_singletons": kernel_ms(lambda: K.drop_group(keys1, rows1, gid["singletons"], k_max, flag)),
        "drop_group_k232_lots_of_25": kernel_ms(lambda: K.drop_group(keys32, rows32, gid["lots_of_25"], k_max, flag)),
    }
    kern_rows = {"drop_self_k201": b1, "drop_group_k201_singletons": b1, "drop_group_k232_lots_of_25": b32}
    # drop_group: 8 B per key read plus its 4 B group-id gather (from L2), 8 B per key written
    kern_bytes = {"drop_self_k201": b1 * (2 * k_max + 1) * 8,
                  "drop_group_k201_singletons": b1 * ((k_max + 1) * 12 + k_max * 8),
                  "drop_group_k232_lots_of_25": b32 * (depth * 12 + k_max * 8)}
    assert int(flag.item()) == 0
    del keys1, keys32
    torch.cuda.empty_cache()
    check_rows = np.sort(rng.choice(N, n_checks, replace=False)).tolist()
    in_big = big[torch.randperm(2000, generator=torch.Generator().manual_seed(seed))[:n_checks // 4].cuda()]
    big_rows = sorted(in_big.tolist()) + np.sort(rng.choice(N, n_checks // 4, replace=False)).tolist()
    checks = {"lots_of_25": deletion_checks(bank, labels, groups["lots_of_25"], outs["lots_of_25"], check_rows),
              "group_2000": deletion_checks(bank, labels, groups["group_2000"], outs["group_2000"], big_rows)}
    return {
        "shape": {"N": N, "D": D, "C": C, "mode": "fp32", "knn_ks": KS, "knn_ts": TS, "batch": BATCH, "seed": seed},
        "ms": {name: stats(v) for name, v in times.items()},
        "over_loo": {name: med[name] / med["loo"] for name in calls if name != "loo"},
        "singletons_bitwise_equal_loo": bool(torch.equal(outs["singletons"], outs["loo"])),
        "kernel_ms": kern,
        "kernel_rows": kern_rows,
        "kernel_GBps": {name: kern_bytes[name] / (kern[name] * 1e-3) / 1e9 for name in kern},
        "drop_group_ms_all_rows_lots_of_25": kern["drop_group_k232_lots_of_25"] * N / b32,
        "rows_checked": {"lots_of_25": check_rows, "group_2000": big_rows},
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
        raise SystemExit("bench_knn_logo.py measures on a GPU; none is visible")
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(),
           "train_data_37k": one_size(37348, 1, args.reps, args.checks),
           "wm811k": one_size(811457, 0, args.reps, args.checks)}
    path = os.path.join(args.out, "bench_knn_logo.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
