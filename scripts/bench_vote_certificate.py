"""A/B of knn_predict's certified class vote (DESIGN §4.1c) against the full re-scoring of every candidate.

  python scripts/bench_vote_certificate.py --out DIR [--reps R] [--kinds clustered,gauss,relu,absgauss]

The flagship step (bench.py: fp32 mode, N = 811,457, D = 512, k = 200, t = 0.1, C = 9, Q = 151,552
queries, seeded bench.make_inputs data) with b200knn.knn.CERTIFIED_VOTE switched on and off
alternately in one process, R times each, every step timed with CUDA events and ending in a host
synchronisation.  Per side: median / min / max step, the CUDA-event time of the re-scoring calls
("rescore": the gather kernels and their select / vote), and on the switch-on side the band size
(candidates re-scored per row, mean and max) and the rows the certificate left to the full
re-scoring.  Each data kind's predictions are compared bitwise between the two sides.  The 811k
bank's 1.66 GB of fp32 rows exceed the 126 MB L2, so every step reads them from HBM.  Writes
DIR/bench_vote_certificate.json with the GPU's name and power limit read in the same run.
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

import b200knn  # noqa: E402
import bench  # noqa: E402  (make_inputs: the benchmark's seeded synthetic embeddings)
from b200knn import knn as K  # noqa: E402
from bench_knn_grid import gpu_info, stats  # noqa: E402


def one_step(q, bank, labels):
    K.query_cache.clear()  # a new batch every step in real use: re-prepare (cast) the queries
    K.profile_events = {}
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    pred = K.knn_predict(q, bank, labels, bench.N_CLASSES, bench.KNN_K, bench.KNN_T)
    b.record()
    torch.cuda.synchronize()
    ev, K.profile_events = K.profile_events, None
    rescore = sum(x.elapsed_time(y) for x, y in ev.get("rescore", []))
    return a.elapsed_time(b), rescore, pred


def run_kind(kind, reps, n_query):
    bank_nd, labels, q = bench.make_inputs("cuda", bench.N_BANK, n_query, bench.DIM, seed=0, kind=kind)
    bank = bank_nd.t().contiguous()
    del bank_nd
    b200knn.set_default_mode("fp32")
    side = {True: {"step_ms": [], "rescore_ms": [], "band_mean": [], "band_max": [], "fallback_rows": []},
            False: {"step_ms": [], "rescore_ms": []}}
    preds = {}
    for on in (True, False):  # warm-up: preparation, module loads
        K.CERTIFIED_VOTE["enabled"] = on
        one_step(q, bank, labels)
    for _ in range(reps):
        for on in (True, False):
            K.CERTIFIED_VOTE["enabled"] = on
            ms, rs, preds[on] = one_step(q, bank, labels)
            side[on]["step_ms"].append(ms)
            side[on]["rescore_ms"].append(rs)
            if on:
                st = K.band_stats()
                side[on]["band_mean"].append(st["mean"])
                side[on]["band_max"].append(st["max"])
                side[on]["fallback_rows"].append(st["fallback_rows"])
    K.CERTIFIED_VOTE["enabled"] = True
    out = {"Q": n_query, "predictions_bitwise_equal": bool(torch.equal(preds[True], preds[False]))}
    for on, name in ((True, "on"), (False, "off")):
        d = side[on]
        out[name] = {"step_ms": stats(d["step_ms"]), "rescore_ms": stats(d["rescore_ms"]),
                     "queries_per_s_median_step": n_query / (stats(d["step_ms"])["median"] * 1e-3)}
        if on:
            out[name]["band_mean"] = sum(d["band_mean"]) / len(d["band_mean"])
            out[name]["band_max"] = max(d["band_max"])
            out[name]["fallback_rows"] = d["fallback_rows"]
    out["speedup_median_step"] = out["off"]["step_ms"]["median"] / out["on"]["step_ms"]["median"]
    del bank, labels, q
    K.bank_cache.clear()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=7)
    ap.add_argument("--queries", type=int, default=8 * bench.WAVE)
    ap.add_argument("--kinds", default="clustered,gauss,relu,absgauss")
    args = ap.parse_args()
    if args.reps < 5:
        raise SystemExit("--reps must be at least 5 (the spread of the alternated runs is part of the result)")
    result = {"gpu": gpu_info(), "reps_per_side": args.reps,
              "config": f"knn_predict fp32 N={bench.N_BANK} D={bench.DIM} k={bench.KNN_K} t={bench.KNN_T} "
                        f"C={bench.N_CLASSES}", "kinds": {}}
    for kind in args.kinds.split(","):
        result["kinds"][kind] = run_kind(kind, args.reps, args.queries)
        print(kind, json.dumps(result["kinds"][kind]), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_vote_certificate.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"gpu": result["gpu"]}))


if __name__ == "__main__":
    main()
