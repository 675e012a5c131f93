"""A/B of the certified vote's bound E from measured fp16 residuals (LEVELS["fp32_f16"]["residual_bound"],
DESIGN §4.1c / §5) against the worst-case bound.

  python scripts/bench_residual_bound.py --out DIR [--reps R] [--kinds clustered,gauss,relu,absgauss]

The flagship step (bench.py: fp32 mode, N = 811,457, D = 512, k = 200, t = 0.1, C = 9, Q = 151,552
queries, seeded bench.make_inputs data) with the residual bound switched on and off alternately in one
process (call graphs cleared at every flip), R times each, every step timed with CUDA events and ending
in a host synchronisation.  Per side: median / min / max step, the CUDA-event time of the re-scoring
calls ("rescore"), the band size (candidates re-scored per row, mean and max), the rows the
certificate left to the full re-scoring and the cascade of the last step (level, rows in, rows left
uncertified).  Each data kind's predictions are compared bitwise between the two sides.  The 811k
bank's 1.66 GB of fp32 rows exceed the 126 MB L2, so every step reads them from HBM.  Writes
DIR/bench_residual_bound.json with the GPU's name, power limit and the SM clocks sampled during the
timed steps.
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
import bench  # noqa: E402  (make_inputs: the benchmark's seeded synthetic embeddings; ClockSampler)
from b200knn import knn as K  # noqa: E402
from bench_knn_grid import gpu_info, stats  # noqa: E402
from bench_vote_certificate import one_step  # noqa: E402


def set_bound(residual):
    if K.LEVELS["fp32_f16"]["residual_bound"] != residual:
        K.LEVELS["fp32_f16"]["residual_bound"] = residual
        K.clear_call_graphs()


def run_kind(kind, reps, n_query):
    bank_nd, labels, q = bench.make_inputs("cuda", bench.N_BANK, n_query, bench.DIM, seed=0, kind=kind)
    bank = bank_nd.t().contiguous()
    del bank_nd
    b200knn.set_default_mode("fp32")
    K.CERTIFIED_VOTE["enabled"] = True
    keys = ("step_ms", "rescore_ms", "band_mean", "band_max", "fallback_rows", "cascade_last_step")
    side = {on: {k: [] for k in keys} for on in (True, False)}
    preds = {}
    for on in (True, False):  # warm-up: preparation, residual statistics, module loads
        set_bound(on)
        one_step(q, bank, labels)
    with bench.ClockSampler() as clocks:
        for _ in range(reps):
            for on in (True, False):
                set_bound(on)
                ms, rs, preds[on] = one_step(q, bank, labels)
                st = K.band_stats()
                d = side[on]
                d["step_ms"].append(ms)
                d["rescore_ms"].append(rs)
                d["band_mean"].append(st["mean"])
                d["band_max"].append(st["max"])
                d["fallback_rows"].append(st["fallback_rows"])
                d["cascade_last_step"].append(K.last_rescore_stats["levels"])
    set_bound(True)
    out = {"Q": n_query, "predictions_bitwise_equal": bool(torch.equal(preds[True], preds[False])),
           "clocks": clocks.summary()}
    for on, name in ((True, "residual"), (False, "worst_case")):
        d = side[on]
        out[name] = {"step_ms": stats(d["step_ms"]), "rescore_ms": stats(d["rescore_ms"]),
                     "queries_per_s_median_step": n_query / (stats(d["step_ms"])["median"] * 1e-3),
                     "band_mean": sum(d["band_mean"]) / len(d["band_mean"]), "band_max": max(d["band_max"]),
                     "fallback_rows": d["fallback_rows"], "cascade_last_step": d["cascade_last_step"][-1]}
    out["speedup_median_step"] = out["worst_case"]["step_ms"]["median"] / out["residual"]["step_ms"]["median"]
    out["rescore_ratio_median"] = out["residual"]["rescore_ms"]["median"] / out["worst_case"]["rescore_ms"]["median"]
    del bank, labels, q
    K.bank_cache.clear()
    torch.cuda.empty_cache()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=9)
    ap.add_argument("--queries", type=int, default=8 * bench.WAVE)
    ap.add_argument("--kinds", default="clustered,gauss,relu,absgauss")
    args = ap.parse_args()
    if args.reps < 7:
        raise SystemExit("--reps must be at least 7 (the spread of the alternated runs is part of the result)")
    result = {"gpu": gpu_info(), "reps_per_side": args.reps,
              "config": f"knn_predict fp32 N={bench.N_BANK} D={bench.DIM} k={bench.KNN_K} t={bench.KNN_T} "
                        f"C={bench.N_CLASSES}", "kinds": {}}
    for kind in args.kinds.split(","):
        result["kinds"][kind] = run_kind(kind, args.reps, args.queries)
        print(kind, json.dumps(result["kinds"][kind]), flush=True)
    os.makedirs(args.out, exist_ok=True)
    with open(os.path.join(args.out, "bench_residual_bound.json"), "w") as f:
        json.dump(result, f, indent=1)
    print(json.dumps({"gpu": result["gpu"]}))


if __name__ == "__main__":
    main()
