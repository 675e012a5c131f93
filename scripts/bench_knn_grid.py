"""Cost of knn_predict_multi (a (k, t) grid from one neighbour search) against knn_predict.

  python scripts/bench_knn_grid.py --out DIR [--reps R] [--queries Q]

North star (N = 811,457, D = 512, Q = 151,552, fp32 mode, ks = (10, 20, 100, 200), ts = (0.07, 0.1)):
one grid call, one knn_predict(k=200) and the 8 separate calls, timed alternately with CUDA events
(every call ends in its own host synchronisation); the vote_multi kernel alone (CUDA events over
repeated launches on the k = 200 keys).  The bank's 1.66 GB of fp32 rows exceed the 126 MB L2, so
every pass reads it from HBM.  Reference shape (B = 64, N = 37,348, ks = (5, 20, 200), ts = (0.1,)):
microseconds per call on the CUDA-graph path next to knn_predict at k = 5 and k = 200.  Outputs are
compared bitwise with the separate calls at the timed sizes.  Writes DIR/bench_knn_grid.json with the
GPU's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
for p in (ROOT, os.path.join(ROOT, "self-supervised-wafermaps_b200")):
    if p not in sys.path:
        sys.path.insert(0, p)

import torch  # noqa: E402

import bench  # noqa: E402  (make_inputs: the benchmark's seeded synthetic embeddings)
import b200knn  # noqa: E402
from b200knn import knn as K  # noqa: E402


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=power.limit,clocks.max.sm",
                              "--format=csv,noheader"], capture_output=True, text=True, timeout=30).stdout
        info["power_limit"], info["max_sm_clock"] = [s.strip() for s in out.strip().split(",")]
    except Exception as e:  # reported, not hidden
        info["nvidia_smi_error"] = repr(e)
    return info


def event_ms(fn):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    out = fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b), out


def stats(xs):
    xs = sorted(xs)
    return {"median": xs[len(xs) // 2], "min": xs[0], "max": xs[-1], "n": len(xs)}


def north_star(reps, n_query):
    ks, ts = (10, 20, 100, 200), (0.07, 0.1)
    bank_nd, labels, q = bench.make_inputs("cuda", 811457, n_query, 512, seed=0)
    bank = bank_nd.t().contiguous()
    del bank_nd
    b200knn.set_default_mode("fp32")
    calls = {
        "grid": lambda: K.knn_predict_multi(q, bank, labels, 9, ks, ts),
        "single_k200": lambda: K.knn_predict(q, bank, labels, 9, 200, 0.1),
        "separate_8": lambda: [K.knn_predict(q, bank, labels, 9, k, t) for k in ks for t in ts],
    }
    outs = {name: fn() for name, fn in calls.items()}  # warm-up: bank preparation, first launches
    times = {name: [] for name in calls}
    for _ in range(reps):  # alternate the three so drift and neighbours hit them alike
        for name, fn in calls.items():
            ms, outs[name] = event_ms(fn)
            times[name].append(ms)
    sep = torch.stack([torch.stack(outs["separate_8"][i * len(ts):(i + 1) * len(ts)]) for i in range(len(ks))])
    equal = bool(torch.equal(outs["grid"], sep))
    # the vote kernels alone, on the k = 200 keys of the same queries
    keys = K.topk_keys(q, bank, 200, "fp32")
    flag = torch.zeros((1,), dtype=torch.int32, device="cuda")
    kern = {}
    for name, fn in (("vote_multi", lambda: K.vote_multi(keys, labels, 9, ks, ts, check_labels=False, flag=flag)),
                     ("vote_k200", lambda: K.vote(keys, labels, 9, 0.1, check_labels=False, flag=flag))):
        fn()
        n = 20

        def loop():  # outputs are dropped at once: the allocator reuses one block, no allocation in the window
            for _ in range(n):
                fn()

        ms, _ = event_ms(loop)
        kern[name] = ms / n
    med = {name: stats(v)["median"] for name, v in times.items()}
    return {
        "shape": {"N": 811457, "D": 512, "Q": n_query, "mode": "fp32", "knn_ks": ks, "knn_ts": ts, "C": 9},
        "ms": {name: stats(v) for name, v in times.items()},
        "grid_over_single_k200": med["grid"] / med["single_k200"],
        "separate_over_grid": med["separate_8"] / med["grid"],
        "kernel_ms": kern,
        "bitwise_equal_to_separate_calls": equal,
    }


def reference_shape(n_calls):
    ks, ts = (5, 20, 200), (0.1,)
    bank_nd, labels, q = bench.make_inputs("cuda", 37348, 64, 512, seed=1)
    bank = bank_nd.t().contiguous()
    b200knn.set_default_mode("fp32")
    calls = {
        "grid": lambda: K.knn_predict_multi(q, bank, labels, 9, ks, ts),
        "single_k5": lambda: K.knn_predict(q, bank, labels, 9, 5, 0.1),
        "single_k200": lambda: K.knn_predict(q, bank, labels, 9, 200, 0.1),
    }
    outs = {}
    for name, fn in calls.items():
        for _ in range(5):  # capture + warm replays
            outs[name] = fn()
    us = {name: [] for name in calls}
    for _ in range(5):
        for name, fn in calls.items():
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for _ in range(n_calls):
                fn()  # each call ends in its one host synchronisation
            us[name].append((time.perf_counter() - t0) / n_calls * 1e6)
    sep = torch.stack([torch.stack([K.knn_predict(q, bank, labels, 9, k, t) for t in ts]) for k in ks])
    return {
        "shape": {"N": 37348, "D": 512, "B": 64, "mode": "fp32", "knn_ks": ks, "knn_ts": ts, "C": 9},
        "us_per_call": {name: stats(v) for name, v in us.items()},
        "graph_stats": dict(K.graph_stats),
        "bitwise_equal_to_separate_calls": bool(torch.equal(outs["grid"], sep)),
    }


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--queries", type=int, default=151552)
    ap.add_argument("--ref-calls", type=int, default=200)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_knn_grid.py measures on a GPU; none is visible")
    os.makedirs(args.out, exist_ok=True)
    res = {"gpu": gpu_info(), "reference_shape": reference_shape(args.ref_calls),
           "north_star": north_star(args.reps, args.queries)}
    path = os.path.join(args.out, "bench_knn_grid.json")
    with open(path, "w") as f:
        json.dump(res, f, indent=1)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
