"""Cost of the radius self-join (radius_graph) and its parts, beside the closest existing floors.

  python scripts/bench_knn_radius.py --out DIR [--reps R] [--sizes 37348,811457]

Seeded bench.make_inputs rows, D = 512, fp32 mode, normalised, at N = 37,348 (the reference's
train_data bank) and N = 811,457 (WM-811K): "clustered" with planted near-duplicate groups of 2, 5, 40
and 1,500 rows (tiny perturbations of one row, so every ladder level runs), and "relu" / "absgauss"
(dense non-negative rows) as they come, at tau in {0.999, 0.99}.  Per case:
  - time per radius_graph call: the median of R calls, CUDA events, every call ending in the host
    read of its nnz; the cases alternate call by call;
  - its parts, from one more call with the library's event hooks on: admission thresholds, candidate
    pass (first depth), re-scoring, compaction, second depth, certified top-max_per_row, peeling,
    and near_duplicate_groups' union and flatten;
  - rows per ladder level and nnz.
Beside it on the same rows and mode: knn_graph(rows, 10) and topk_keys at k = 32 (all rows against
all rows, in batches of 75,776), the closest existing floors.  The 811k rows (1.66 GB fp32) exceed
the 126 MB L2.  Writes DIR/bench_knn_radius.json with the GPU's name and power limit read in the
same run.
"""
import argparse
import json
import os
import sys

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
for p in (ROOT, os.path.join(ROOT, "self-supervised-wafermaps_b200"), os.path.dirname(os.path.abspath(__file__))):
    if p not in sys.path:
        sys.path.insert(0, p)

import numpy as np  # noqa: E402
import torch  # noqa: E402

import bench  # noqa: E402  (make_inputs: the benchmark's seeded synthetic embeddings)
import b200knn  # noqa: E402
from b200knn import knn as K  # noqa: E402
from b200knn import retrieval as R  # noqa: E402
from bench_knn_grid import event_ms, gpu_info, stats  # noqa: E402

D, BATCH, TAUS = 512, 75776, (0.999, 0.99)
PLANTED = (2, 5, 40, 1500)


def make_rows(N, kind, seed=0):
    rows, _, _ = bench.make_inputs("cuda", N, 1, D, seed=seed, kind=kind)
    if kind == "clustered":
        g = torch.Generator(device="cuda").manual_seed(seed + 1)
        pos = torch.randperm(N, generator=g, device="cuda")
        at = 0
        for size in PLANTED:
            members = pos[at:at + size]
            at += size
            noise = 2e-3 * torch.randn(size, D, generator=g, device="cuda") / D ** 0.5
            rows[members] = rows[members[0]] + noise
    return torch.nn.functional.normalize(rows, dim=1).contiguous()


def floors(rows):
    fb = b200knn.FeatureBank.from_rows(rows)
    n = rows.shape[0]

    def topk32():
        for lo in range(0, n, BATCH):
            K.topk_keys(fb.rows[lo:lo + BATCH, :fb.dim], fb.bank, 32, "fp32")
        return None

    return {"knn_graph_k10": lambda: b200knn.knn_graph(rows, 10, mode="fp32")[1][-1, -1].item(),
            "topk_keys_k32": lambda: (topk32(), torch.cuda.synchronize())}


def parts_of(rows, tau):
    K.profile_events = {}
    r = b200knn.radius_graph(rows, tau, mode="fp32")
    levels = dict(R.last_radius_stats)
    b200knn.near_duplicate_groups(rows, tau, mode="fp32")
    torch.cuda.synchronize()
    ev, K.profile_events = K.profile_events, None
    parts = {name: sum(a.elapsed_time(b) for a, b in pairs) for name, pairs in ev.items()}
    return {"parts_ms": parts, "rows_per_level": levels, "nnz": int(r.indices.numel()),
            "saturated": int(r.saturated.sum()), "note": "parts_ms: one radius_graph call, then one "
            "near_duplicate_groups call (radius_union / radius_flatten and the second call's search parts "
            "add to the same names); topk = every tensor-core search inside the ladder"}


def one_size(N, reps):
    out = {"N": N, "cases": {}}
    for kind in ("clustered", "relu", "absgauss"):
        rows = make_rows(N, kind)
        calls = {f"radius_graph_tau{t}": (lambda t=t: b200knn.radius_graph(rows, t, mode="fp32").indices.numel())
                 for t in TAUS}
        calls.update(floors(rows))
        for fn in calls.values():  # warm-up: every shape, the bank preparations
            fn()
        times = {name: [] for name in calls}
        for _ in range(reps):
            for name, fn in calls.items():
                times[name].append(event_ms(fn)[0])
        case = {name: stats(ts) for name, ts in times.items()}
        for t in TAUS:
            case[f"radius_graph_tau{t}"].update(parts_of(rows, t))
        out["cases"][kind + ("_planted" if kind == "clustered" else "")] = case
        del rows
        K.bank_cache.clear()
        K.query_cache.clear()
        torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sizes", default="37348,811457")
    a = ap.parse_args()
    os.makedirs(a.out, exist_ok=True)
    res = {"gpu": gpu_info(), "mode": "fp32", "D": D, "batch": BATCH, "planted_groups": PLANTED,
           "timing": "CUDA events around each call (ending in a host read), median of --reps, cases alternated",
           "sizes": [one_size(int(n), a.reps) for n in a.sizes.split(",")]}
    path = os.path.join(a.out, "bench_knn_radius.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res)[:4000])


if __name__ == "__main__":
    main()
