#!/usr/bin/env python
"""bench.py — kNN queries/s on the north-star workload (BASELINE.json):
knn_predict on an 811,457 x 512 bank, k=200, t=0.1, 9 classes, in the BIT-EXACT `fp32` mode.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--mode fp32|bf16|...] [--data clustered|gauss|relu|absgauss]
                  [--dump-outputs DIR]      # the last timed step's class ranking -> DIR/pred_labels.npy
  python bench.py --impl reference ...      # the reference algorithm on the host CPU cores
  python bench.py --config ref              # the reference-shaped call: N=37,348, B=64 per call, k=5

A step = one knn_predict call over one batch of Q synthetic queries.
  value : queries/s with queries, bank (prepared, cached) and labels resident in HBM
  e2e   : the same through the public API with HOST (pinned) queries: H2D copy of the batch,
          knn_predict, D2H of the predicted class column, all inside the timed region
  N > 1 : the bank is row-sharded over the ranks (north-star mode 4); every rank holds the whole
          query batch.  Fixed total work as N grows -> "scaling": "strong".
Side objects of the default line (1 GPU): `bf16_mode` (the fast approximate mode + recall),
`gpu_library_baseline` (the reference's own ops, torch.mm + topk + ... via cuBLAS/ATen on the SAME
B200, fp32 / TF32 / fp16-autocast as the reference really runs them), `ref_shaped_call` (B=64 per call:
us per call against that library bar), `data_variants` (the bit-exact mode on gauss / relu /
absgauss embeddings), `tf32_peak_measured`.
One JSON line on rank 0 (contract in the task statement).
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
for _p in (ROOT, os.path.join(ROOT, "self-supervised-wafermaps_b200"), os.path.join(ROOT, "tests")):
    if _p not in sys.path:
        sys.path.insert(0, _p)

N_BANK, DIM, KNN_K, KNN_T, N_CLASSES = 811457, 512, 200, 0.1, 9
METRIC = "kNN queries/s @811k×512 bank, k=200"
WAVE = 148 * 128  # queries one resident wave of CTAs covers
L2_BYTES = 126e6


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm=p["hbm_gbs"], bf16=p["bf16_tflops_sustained"], bf16_burst=p["bf16_tflops"], src="measured")
    return dict(hbm=6650.0, bf16=1400.0, bf16_burst=1590.0, src="fallback")


def ncu_traffic(mode, Q, N, world):
    """DRAM bytes (read+write) per launch of the dominant kernel from the committed
    `ncu --set full` capture of this exact configuration (profiles/ncu_traffic.json), else None."""
    path = os.path.join(ROOT, "profiles", "ncu_traffic.json")
    try:
        for e in json.load(open(path)):
            if e["mode"] == mode and e["Q"] == Q and e["N"] == N and e["n_gpus"] == world:
                return e["dram_bytes_per_launch"]
    except Exception:
        pass
    return None


def make_inputs(device, n_bank, n_query, dim, seed, row_range=None, kind="clustered"):
    """Synthetic embeddings generated on the device under test, in chunks of 65,536 rows with one
    generator per chunk, so a rank can generate only the bank rows it owns (row_range) and results
    do not depend on the total size (SURVEY.md §8d).  Labels are generated for all rows (replicated).
      clustered : normalise(centroid[label] + 1.4 N(0,I)/sqrt(D))   (WM-811K class priors)
      gauss     : normalise(N(0,I))
      relu      : normalise(max(0, centroid[label] + 1.4 N(0,I)/sqrt(D))) — non-negative rows, like the
                  reference's post-ReLU ResNet-18 features (src/ssl_wafermap/models/knn.py:322, :77)
      absgauss  : normalise(|N(0,I)|)"""
    import torch

    g0 = torch.Generator(device=device).manual_seed(seed)
    prior = torch.tensor([859, 111, 1037, 1936, 719, 30, 173, 239, 7345], dtype=torch.float64, device=device)
    if N_CLASSES != 9:  # MixedWM38 (config c3): flat prior
        prior = torch.ones(N_CLASSES, dtype=torch.float64, device=device)
    cent = torch.nn.functional.normalize(torch.randn(N_CLASSES, dim, generator=g0, device=device), dim=1)
    lo_own, hi_own = row_range if row_range is not None else (0, n_bank)

    def rows(n, stream_id, lo_want, hi_want):
        out = torch.empty(max(0, hi_want - lo_want), dim, device=device)
        lab = torch.empty(n, dtype=torch.int64, device=device)
        for ci, lo in enumerate(range(0, n, 65536)):
            hi = min(n, lo + 65536)
            g = torch.Generator(device=device).manual_seed(seed * 1000003 + stream_id * 100003 + ci)
            l = torch.multinomial(prior, hi - lo, replacement=True, generator=g)
            lab[lo:hi] = l
            a, b = max(lo, lo_want), min(hi, hi_want)
            if a < b:
                z = torch.randn(hi - lo, dim, generator=g, device=device)
                if kind == "gauss":
                    x = z
                elif kind == "absgauss":
                    x = z.abs()
                else:
                    x = cent[l] + 1.4 * z / dim ** 0.5
                    if kind == "relu":
                        x = x.clamp_min(0.0)
                out[a - lo_want:b - lo_want] = torch.nn.functional.normalize(x, dim=1)[a - lo:b - lo]
        return out, lab

    bank_nd, labels = rows(n_bank, 1, lo_own, hi_own)
    q, _ = rows(n_query, 2, 0, n_query)
    return bank_nd, labels, q


class ClockSampler:
    """Samples SM clocks and throttle reasons with one streaming `nvidia-smi -lms 50` process
    while the timed region runs (a fresh nvidia-smi per sample is too slow for sub-second runs)."""

    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.rows, self.index, self.proc = [], index, None
        self.th = threading.Thread(target=self.run, daemon=True)

    def run(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                parts = [x.strip() for x in line.strip().split(",")]
                if len(parts) >= 6:
                    self.rows.append(parts)
        except Exception:
            pass

    def __enter__(self):
        self.th.start()
        time.sleep(0.15)  # let the first sample land before the timed region starts
        return self

    def __exit__(self, *a):
        if self.proc is not None:
            try:
                self.proc.terminate()
            except Exception:
                pass
        self.th.join(timeout=3)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unsampled"]}
        sm = [float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": float(self.rows[0][1]) if self.rows[0][1].replace(".", "").isdigit() else None,
                "reasons": reasons, "samples": len(self.rows)}


def cpu_reference_rate(batch, n_calls, threads=None):
    """The reference algorithm (oracle R32: lightly's knn_predict restated op for op) on torch
    CPU fp32 with all host threads, on a bounded sample of the SAME workload: `n_calls` calls
    of `batch` queries against the full bank (after one untimed warm-up call)."""
    import torch

    from oracle import knn_oracle as O

    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    g = torch.Generator().manual_seed(811)
    bank = torch.nn.functional.normalize(torch.randn(N_BANK, DIM, generator=g), dim=1).t().contiguous()
    labels = torch.randint(0, N_CLASSES, (N_BANK,), generator=g)
    q = torch.nn.functional.normalize(torch.randn(batch, DIM, generator=g), dim=1)
    O.knn_predict_r32(q, bank, labels, N_CLASSES, KNN_K, KNN_T)
    times = []
    for _ in range(n_calls):
        t0 = time.perf_counter()
        O.knn_predict_r32(q, bank, labels, N_CLASSES, KNN_K, KNN_T)
        times.append(time.perf_counter() - t0)
    return batch * n_calls / sum(times), times, threads


def cpu_name():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    batch = 64 if args.config == "ref" else 1024
    rate, times, threads = cpu_reference_rate(batch, args.warmup + args.steps)
    times = times[args.warmup:]
    rate = batch * len(times) / sum(times)
    sample = f"{len(times)} calls of B={batch} queries against the full {N_BANK}x{DIM} bank, k={KNN_K}"
    line = {
        "impl": "reference", "metric": metric_name(), "value": rate, "unit": "queries/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * sum(times) / len(times), "higher_is_better": True, "scaling": "strong",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"knn_predict N={N_BANK} D={DIM} k={KNN_K} t={KNN_T} C={N_CLASSES}; B={batch} per step",
                   "reference": "lightly knn_predict restated (oracle R32), torch CPU fp32 (MKL), all host threads",
                   "cpu": cpu_name()},
        "cpu_baseline": {"value": rate, "unit": "queries/s", "cores": threads, "kind": "port", "sample": sample},
        "e2e": {"value": rate, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_BYTES = 64 * 10**6 - 1024  # 64 MB less room for two .npy headers


def dump_outputs(out_dir, pred_labels):
    """Writes what knn_predict returned, the (Q, C) class ranking, as float64 (class indices are exact
    in it) to out_dir/pred_labels.npy.  Above DUMP_BYTES in all it keeps a fixed seeded sample of the
    rows, sorted, and writes their indices to out_dir/pred_labels_rows.npy."""
    import numpy as np

    pred = pred_labels.cpu().numpy().astype(np.float64)
    n_rows, n_cols = pred.shape
    if pred.nbytes > DUMP_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(n_rows, DUMP_BYTES // (8 * (n_cols + 1)), replace=False))
        pred = pred[rows]
    else:
        rows = None
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pred_labels.npy"), pred)
    if rows is not None:
        np.save(os.path.join(out_dir, "pred_labels_rows.npy"), rows.astype(np.float64))


def elem_bytes(cand_mode):
    return {"bf16": 2, "f16": 2, "bf16x3": 4, "f16x2": 2, "tf32x3": 8, "exact": 4}[cand_mode]


def metric_name():
    return METRIC if (N_BANK, DIM, KNN_K) == (811457, 512, 200) else f"kNN queries/s @{N_BANK}x{DIM} bank, k={KNN_K}"


# ---------------------------------------------------------------------------------------------
# The library bar (SURVEY.md §2a / §8d): the reference's own op sequence — lightly's knn_predict,
# restated here because lightly is not installable — executed by torch on the SAME GPU, i.e.
# cuBLAS GEMM + ATen topk/gather/exp/scatter/sum/argsort, in the three numeric settings the
# reference can run it in: fp32 (allow_tf32 off), TF32 (set_float32_matmul_precision("high"),
# scripts/WM811k_benchmark.py:35) and fp16 autocast (precision="16-mixed", :57/:1107).
def library_knn_predict(feature, feature_bank, feature_labels, num_classes, knn_k, knn_t):
    import torch

    sim_matrix = torch.mm(feature, feature_bank)
    sim_weight, sim_indices = sim_matrix.topk(k=knn_k, dim=-1)
    sim_labels = torch.gather(feature_labels.expand(feature.size(0), -1), dim=-1, index=sim_indices)
    sim_weight = (sim_weight / knn_t).exp()
    one_hot = torch.zeros(feature.size(0) * knn_k, num_classes, device=sim_labels.device)
    one_hot = one_hot.scatter(dim=-1, index=sim_labels.view(-1, 1), value=1.0)
    pred_scores = torch.sum(one_hot.view(feature.size(0), -1, num_classes) * sim_weight.unsqueeze(dim=-1), dim=1)
    return pred_scores.argsort(dim=-1, descending=True)


def time_calls(fn, n_calls, n_warm=3):
    """Mean milliseconds per call (host-side loop, CUDA events on the current stream, sync on both sides)."""
    import torch

    for _ in range(n_warm):
        fn()
    torch.cuda.synchronize()
    s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    s.record()
    for _ in range(n_calls):
        fn()
    e.record()
    torch.cuda.synchronize()
    return s.elapsed_time(e) / n_calls


def library_settings():
    import torch

    class Setting:
        def __init__(self, name, tf32, autocast):
            self.name, self.tf32, self.autocast = name, tf32, autocast

        def __enter__(self):
            self.old = torch.backends.cuda.matmul.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = self.tf32
            self.ctx = torch.autocast("cuda", dtype=torch.float16) if self.autocast else None
            if self.ctx:
                self.ctx.__enter__()

        def __exit__(self, *a):
            if self.ctx:
                self.ctx.__exit__(*a)
            torch.backends.cuda.matmul.allow_tf32 = self.old

    return [Setting("fp32", False, False), Setting("tf32", True, False), Setting("fp16_autocast", True, True)]


def library_baseline(q, bank, labels, batches=(1024, 64)):
    """queries/s of the library bar per numeric setting and batch size, same bank / k / t / C."""
    out = {"ops": "torch.mm + topk + gather + div/exp + zeros/scatter + mul/sum + argsort (cuBLAS + ATen) on this GPU",
           "bank": f"{bank.shape[1]}x{bank.shape[0]}", "k": KNN_K}
    for st in library_settings():
        for b in sorted({min(b, q.shape[0]) for b in batches}, reverse=True):
            qb = q[:b].contiguous()
            with st:
                ms = time_calls(lambda: library_knn_predict(qb, bank, labels, N_CLASSES, KNN_K, KNN_T), 10 if b > 64 else 30)
            out[f"{st.name}_B{b}"] = {"queries_per_s": b / (ms * 1e-3), "ms_per_call": ms}
    return out


def tf32_peak():
    """In-run TF32 dense peak (SURVEY.md §8d): torch.matmul fp32 8192^3 with allow_tf32, best of 10 and
    the mean of a back-to-back second."""
    import torch

    a = torch.randn(8192, 8192, device="cuda")
    b = torch.randn(8192, 8192, device="cuda")
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        best = 1e9
        for _ in range(10):
            best = min(best, time_calls(lambda: torch.matmul(a, b), 1, 1))
        sustained = time_calls(lambda: torch.matmul(a, b), 40, 2)
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    fl = 2 * 8192 ** 3 / 1e12
    return {"tflops_burst": fl / (best * 1e-3), "tflops_sustained": fl / (sustained * 1e-3),
            "how": "torch.matmul fp32 8192^3, allow_tf32=True: best of 10 / mean of 40 back to back"}


def ref_shaped(b200knn, K, dev, mode):
    """The call as the reference makes it (SURVEY.md §3.1): B = 64 queries per validation_step
    (scripts/WM811k_benchmark.py:71).  (a) the north-star bank, k=200; (b) the reference's own full
    bank size N=37,348 with its k=5 (:49; src/ssl_wafermap/models/knn.py:38).  us per call of
    b200knn.knn_predict (CUDA-graph replay + one status read) against the library bar."""
    import torch

    out = {}
    for name, n, k in (("N811457_k200", 811457, 200), ("N37348_k5", 37348, 5)):
        bank_nd, labels, q = make_inputs(dev, n, 64, DIM, seed=37)
        bank = bank_nd.t().contiguous()
        del bank_nd
        b200knn.set_default_mode(mode)
        ours = time_calls(lambda: b200knn.knn_predict(q, bank, labels, N_CLASSES, k, KNN_T), 100, 5)
        K.GRAPHS["enabled"] = False
        eager = time_calls(lambda: b200knn.knn_predict(q, bank, labels, N_CLASSES, k, KNN_T), 30, 3)
        K.GRAPHS["enabled"] = True
        b200knn.set_default_mode("exact")
        want = b200knn.knn_predict(q, bank, labels, N_CLASSES, k, KNN_T)
        b200knn.set_default_mode(mode)
        got = b200knn.knn_predict(q, bank, labels, N_CLASSES, k, KNN_T)
        entry = {"B": 64, "N": n, "k": k, "us_per_call": ours * 1e3, "us_per_call_without_graph": eager * 1e3,
                 "equals_exact_mode": bool(torch.equal(got, want)), "mode": mode}
        cand_bytes = n * DIM * 2  # fp16 candidate bank streamed once per call
        entry["hbm_floor_us"] = cand_bytes / (peaks()["hbm"] * 1e9) * 1e6
        entry["note"] = ("bank streamed once per call: HBM floor as stated" if cand_bytes > L2_BYTES else
                         "the prepared bank (%.0f MB) stays in L2: launch latency bound" % (cand_bytes / 1e6))
        for st in library_settings():
            with st:
                ms = time_calls(lambda: library_knn_predict(q, bank, labels, N_CLASSES, k, KNN_T), 50, 5)
            entry[f"library_{st.name}_us_per_call"] = ms * 1e3
        out[name] = entry
        del bank, labels, q
        K.bank_cache.clear()
        K.clear_call_graphs()
        torch.cuda.empty_cache()
    return out


def main():
    global DIM, KNN_K, N_BANK, N_CLASSES
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours")
    ap.add_argument("--mode", default=os.environ.get("B200KNN_BENCH_MODE", "fp32"))
    ap.add_argument("--config", default="north", choices=["north", "ref"],
                    help="north: BASELINE.json's metric config; ref: the reference-shaped call (N=37,348, B=64, k=5)")
    ap.add_argument("--queries", type=int, default=None, help="queries per step (default 151,552 = 8 waves)")
    ap.add_argument("--bank", type=int, default=None)
    ap.add_argument("--data", default="clustered", choices=["clustered", "gauss", "relu", "absgauss"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-library", action="store_true", help="skip the library bar / ref-shaped / side objects")
    ap.add_argument("--dim", type=int, default=DIM, help="vector dimension (default 512; 768 = config c5)")
    ap.add_argument("--k", type=int, default=None)
    ap.add_argument("--classes", type=int, default=N_CLASSES, help="9 = WM-811K priors; 38 = MixedWM38 (config c3)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the class ranking the last timed step returned to DIR/pred_labels.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs applies to --impl ours")
    if args.config == "ref":  # scripts/WM811k_benchmark.py:49,71; knn.py:38; train_data rows (notebook 1.0:1721)
        N_BANK, KNN_K = 37348, 5
        args.queries = args.queries or 64
    DIM, N_CLASSES = args.dim, args.classes
    N_BANK = args.bank or N_BANK
    KNN_K = args.k or KNN_K
    args.queries = args.queries or 8 * WAVE
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    import b200knn
    from b200knn import _lib
    from b200knn import knn as K

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    Q, N, mode = args.queries, N_BANK, args.mode
    b200knn.set_default_mode(mode)
    rescored = mode in K.RESCORED_MODES

    lo, hi = b200knn.shard_bounds(N, world, rank)
    bank_nd, labels, q = make_inputs(dev, N, Q, DIM, seed=811, row_range=(lo, hi) if world > 1 else None,
                                     kind=args.data)
    if world > 1:
        shard = bank_nd.t().contiguous()  # this rank's (D, rows) slice, reference layout
        del bank_nd
        sb = b200knn.ShardedBank(shard, labels, N, mode=mode)
        bank = shard
        n_local = hi - lo

        def predict(qd):
            return sb.knn_predict(qd, N_CLASSES, KNN_K, KNN_T)
    else:
        bank = bank_nd.t().contiguous()  # (D,N) contiguous as knn.py:80 builds it
        del bank_nd
        n_local = N

        def predict(qd):
            return b200knn.knn_predict(qd, bank, labels, N_CLASSES, KNN_K, KNN_T)

    # bank preparation (cached per bank tensor; once per validation epoch in the reference) — timed apart
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    pbank = None
    if mode != "exact":
        pbank = K.bank_cache.get(bank, K.RESCORED_MODES[mode]["cand"] if rescored else mode)
        if rescored:
            pbank.rescore_rows()
            pbank.max_norm()
    e1.record()
    torch.cuda.synchronize()
    prepare_ms = e0.elapsed_time(e1)

    q_host = q.cpu().pin_memory()
    top1_host = torch.empty(Q, dtype=torch.int64).pin_memory()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        barrier()
        s, e = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s.record()
        for _ in range(steps):
            fn()
        e.record()
        barrier()
        ms = torch.tensor([s.elapsed_time(e)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item())

    last = {}

    def step_resident():
        K.query_cache.clear()  # a new batch every step in real use: re-prepare (cast) the queries
        last["pred"] = predict(q)
        return last["pred"]

    # e2e: every step uploads its own batch from pinned host memory and reads its predictions
    # back.  The upload of step i+1 is enqueued on a copy stream before step i's compute, so
    # it overlaps the kernels (double-buffered device staging); knn_predict itself synchronises
    # once per call (status word), and the D2H of the result closes the step.
    copy_stream = torch.cuda.Stream(device=dev)
    staging = [torch.empty_like(q), torch.empty_like(q)]
    uploaded = [torch.cuda.Event(), torch.cuda.Event()]
    consumed = [torch.cuda.Event(), torch.cuda.Event()]
    e2e_state = {"i": 0, "primed": False}

    # N > 1: every rank uploads only its 1/N slice of the batch over its own PCIe link and the
    # full batch is assembled with an all-gather over NVLink (every rank needs all queries)
    q_per = (Q + world - 1) // world
    q_lo, q_hi = min(Q, rank * q_per), min(Q, (rank + 1) * q_per)
    if world > 1:
        slice_host = torch.zeros((q_per, DIM), dtype=q.dtype).pin_memory()
        slice_host[: q_hi - q_lo] = q_host[q_lo:q_hi]
        slice_dev = [torch.empty((q_per, DIM), dtype=q.dtype, device=dev) for _ in range(2)]
        gathered = [torch.empty((q_per * world, DIM), dtype=q.dtype, device=dev) for _ in range(2)]
        staging = [g[:Q] for g in gathered]

    def upload(slot):
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(consumed[slot])
            if world > 1:
                slice_dev[slot].copy_(slice_host, non_blocking=True)
                dist.all_gather_into_tensor(gathered[slot], slice_dev[slot])
            else:
                staging[slot].copy_(q_host, non_blocking=True)
            uploaded[slot].record(copy_stream)

    def step_e2e():
        i = e2e_state["i"]
        slot = i & 1
        if not e2e_state["primed"]:
            consumed[0].record()
            consumed[1].record()
            upload(slot)
            e2e_state["primed"] = True
        upload(slot ^ 1)  # next step's batch, overlapped with this step's kernels
        cur = torch.cuda.current_stream()
        cur.wait_event(uploaded[slot])
        K.query_cache.clear()
        pred = predict(staging[slot])
        consumed[slot].record(cur)
        top1_host.copy_(pred[:, 0], non_blocking=True)
        cur.synchronize()
        e2e_state["i"] = i + 1

    for _ in range(args.warmup):
        step_resident()
    K.profile_events = {}
    _lib.launch_counter["kernels"] = 0
    with ClockSampler(local) as clocks:
        total_ms = timed(step_resident, args.steps)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, last["pred"])
    n_abi_kernels = _lib.launch_counter["kernels"]
    events = K.profile_events
    K.profile_events = None
    topk_ms = sum(a.elapsed_time(b) for a, b in events.get("topk", [])) / max(1, args.steps)
    rescore_ms = sum(a.elapsed_time(b) for a, b in events.get("rescore", [])) / max(1, args.steps)
    rescore_stats, prepass_stats = dict(K.last_rescore_stats), dict(K.last_prepass_stats)
    uncertified = rescore_stats["uncertified"] if world == 1 else getattr(sb, "last_uncertified", 0)
    for _ in range(max(1, args.warmup // 2)):
        step_e2e()
    e2e_ms = timed(step_e2e, args.steps)

    clock_summary = clocks.summary()
    if world > 1:  # one sampler per rank (its own GPU): report every rank's median SM clock
        allc = [None] * world
        dist.all_gather_object(allc, clock_summary)
        clock_summary = dict(allc[0], per_rank_sm_mhz=[c.get("sm_mhz") for c in allc],
                             reasons=sorted({r for c in allc for r in c.get("reasons", [])}))

    # result quality, outside the timed regions, at EVERY world size: this mode's neighbours and
    # predictions for a sample of the batch against the exact mode (sequential-fma fp32 on CUDA
    # cores, bit-checked against the oracle by tests/; sharded the same way when N > 1): recall@k,
    # and bitwise key equality — the fp32-matching modes must be bitwise equal
    quality = None
    if mode != "exact":
        nq = min(Q, 256)
        qs = q[:nq].contiguous()
        if world > 1:
            exact_sb = b200knn.ShardedBank(shard, labels, N, mode="exact")
            ek = exact_sb.topk_keys(qs, KNN_K)
            tk = sb.topk_keys(qs, KNN_K)
            pe = exact_sb.knn_predict(qs, N_CLASSES, KNN_K, KNN_T)
            pm = sb.knn_predict(qs, N_CLASSES, KNN_K, KNN_T)
        else:
            ek = b200knn.topk_keys(qs, bank, KNN_K, mode="exact")
            tk = b200knn.topk_keys(qs, bank, KNN_K, mode=mode)
            b200knn.set_default_mode("exact")
            pe = b200knn.knn_predict(qs, bank, labels, N_CLASSES, KNN_K, KNN_T)
            b200knn.set_default_mode(mode)
            pm = b200knn.knn_predict(qs, bank, labels, N_CLASSES, KNN_K, KNN_T)
        ei = b200knn.decode_keys(ek)[1].cpu().numpy()
        ti = b200knn.decode_keys(tk)[1].cpu().numpy()
        recall = sum(len(set(a.tolist()) & set(b.tolist())) for a, b in zip(ei, ti)) / float(nq * KNN_K)
        quality = {"sample_queries": nq, "recall_at_k": recall,
                   "keys_bitwise_equal_exact_mode": bool(torch.equal(ek, tk)),
                   "top1_agreement_with_exact_mode": float((pe[:, 0] == pm[:, 0]).float().mean().item()),
                   "class_ranking_equal_exact_mode": bool(torch.equal(pe, pm)),
                   "against": "exact mode, sharded the same way" if world > 1 else "exact mode"}

    phases = None
    if world > 1:  # where a sharded step spends its time (one extra untimed step, rank 0's view)
        sb.phase_log = []
        step_resident()
        torch.cuda.synchronize()
        log, sb.phase_log = sb.phase_log, None
        phases = {}
        for i in range(1, len(log)):  # same-named phases (cascade levels) are summed
            if log[i][0] != "start":
                phases[log[i][0]] = round(phases.get(log[i][0], 0.0) + log[i - 1][1].elapsed_time(log[i][1]), 3)

    side = {}
    if world == 1 and not args.no_library and rank == 0:
        # ---- the fast approximate mode on the same workload
        if mode != "bf16":
            b200knn.set_default_mode("bf16")
            for _ in range(2):
                step_resident()
            n_b = max(2, min(5, args.steps))
            b_ms = timed(step_resident, n_b) / n_b
            nq = min(Q, 256)
            ek = b200knn.topk_keys(q[:nq].contiguous(), bank, KNN_K, mode="exact")
            bk = b200knn.topk_keys(q[:nq].contiguous(), bank, KNN_K, mode="bf16")
            ei, bi = b200knn.decode_keys(ek)[1].cpu().numpy(), b200knn.decode_keys(bk)[1].cpu().numpy()
            side["bf16_mode"] = {"mode": "bf16", "value": Q / (b_ms * 1e-3), "unit": "queries/s", "ms_per_step": b_ms,
                                 "steps": n_b, "recall_at_k": sum(len(set(a.tolist()) & set(b.tolist()))
                                                                  for a, b in zip(ei, bi)) / float(nq * KNN_K),
                                 "note": "raw bf16 tensor-core similarities, no re-scoring: not bit-exact"}
            b200knn.set_default_mode(mode)
            K.bank_cache.clear()
            torch.cuda.empty_cache()
        side["tf32_peak_measured"] = tf32_peak()
        side["gpu_library_baseline"] = library_baseline(q, bank, labels)

    if rank == 0:
        pk = peaks()
        ms_per_step = total_ms / args.steps
        value = Q / (ms_per_step * 1e-3)
        flops = 2.0 * Q * n_local * DIM  # algorithmic: 2*N*D per query (SURVEY.md §8d), this rank's rows
        whole_call = topk_ms <= 0.0  # captured (CUDA-graph) calls: no per-kernel events, time the whole call
        if whole_call:
            topk_ms = ms_per_step
        achieved = flops / (topk_ms * 1e-3) / 1e12
        cand_mode = K.RESCORED_MODES[mode]["cand"] if rescored else mode
        margin = K.RESCORED_MODES[mode]["margin"] if rescored else 0
        k_plan = KNN_K + margin
        plan = b200knn.plan_info(Q, n_local, DIM, k_plan, cand_mode) if mode != "exact" else \
            b200knn.plan_info(Q, n_local, DIM, KNN_K, "exact")
        mmas = {"bf16": 1, "f16": 1, "f16x2": 2, "bf16x3": 3, "tf32x3": 3}.get(cand_mode, 0)
        kern_name = {"bf16": "tc_topk_kernel<BF16,256,cta_group::2>", "f16": "tc_topk_kernel<F16,256,cta_group::2>",
                     "f16x2": "tc_topk_kernel<F16X2,256,cta_group::2>", "bf16x3": "tc_topk_kernel<BF16X3,128>",
                     "tf32x3": "tc_topk_kernel<TF32X3,128>", "exact": "exact_topk_kernel"}[cand_mode]
        if cand_mode == "exact":
            fp32_peak = 148 * 128 * 2 * 1.965e9 / 1e12
            roof = {"bound": "fp32-cuda-core", "achieved": achieved, "peak": fp32_peak, "unit": "TFLOP/s",
                    "frac": achieved / fp32_peak, "traffic": None, "kernel": kern_name,
                    "peak_source": "nominal 148 SM x 128 FMA/clk x 1.965 GHz", "kernel_ms": topk_ms}
        else:
            peak = pk["bf16"] / 2 if cand_mode == "tf32x3" else pk["bf16"]
            roof = {"bound": "tensor", "achieved": achieved, "peak": peak, "unit": "TFLOP/s", "frac": achieved / peak,
                    "traffic": ncu_traffic(mode, Q, N, world),
                    "kernel": f"{kern_name} candidate pass ({mmas} MMA per k-step; sum of the similarity + top-k "
                              f"launches of a step, incl. the small second-level pass)",
                    "peak_source": f"{pk['src']} bf16 sustained (MEASURED_PEAKS.json; fp16 runs at the bf16 rate"
                                   + (", tf32 at half of it)" if cand_mode == "tf32x3" else ")"),
                    "kernel_ms": topk_ms,
                    "useful_flops": "2*Q*N_local*D (algorithmic; executed = useful x MMAs per k-step)",
                    # the whole step against the same peak: what a user gets per useful flop
                    "step_frac": flops / (ms_per_step * 1e-3) / 1e12 / peak}
            if mmas > 1:
                roof["executed_frac"] = mmas * achieved / peak
            if whole_call:
                hbm_floor_ms = n_local * K.padded_dim(DIM) * elem_bytes(cand_mode) / (pk["hbm"] * 1e9) * 1e3
                roof["kernel"] = ("whole captured call (CUDA graph of ~12 kernels, B <= 512): launch-latency bound, "
                                  "not tensor bound; kernel_ms is the call")
                roof["latency_bound"] = {"us_per_call": ms_per_step * 1e3, "hbm_floor_us": hbm_floor_ms * 1e3,
                                         "note": "floor = candidate bank streamed once; a bank that fits L2 has no HBM floor"}
        if rescored and rescore_ms > 0:
            k_in = min(N, k_plan)
            gb = Q * k_in * K.padded_dim(DIM) * 4.0 / world / 1e9  # candidate rows gathered by this rank
            roof["rescore"] = {"bound": "hbm", "kernel": "rescore_dot_kernel + rescore_select_kernel (exact re-scoring gather)",
                               "achieved": gb / (rescore_ms * 1e-3), "peak": pk["hbm"], "unit": "GB/s",
                               "frac": gb / (rescore_ms * 1e-3) / pk["hbm"], "kernel_ms": rescore_ms,
                               "bytes": "Q*k_in*D_pad*4 / n_gpus (algorithmic: one fp32 row per candidate)"}
        # kernels launched through the C ABI inside the timed region (counted by the loader
        # proxy) + the split merges b200knn_topk* adds internally when its plan splits the bank
        splits_extra = args.steps if plan["splits"] > 1 else 0
        if K.prepass_stride(N, k_plan, Q) and mode != "exact":
            sp = b200knn.plan_info(Q, max(1, n_local // K.prepass_stride(N, k_plan, Q)), DIM, K.PREPASS["r"], cand_mode)
            splits_extra += args.steps if sp["splits"] > 1 else 0
        gpu_launches = n_abi_kernels + splits_extra
        elem = elem_bytes(cand_mode)
        bank_mb = n_local * K.padded_dim(DIM) * elem / 1e6
        step_mb = (Q * DIM * 4 + Q * k_plan * 8 + (Q * min(N, k_plan) * K.padded_dim(DIM) * 4 / world if rescored else 0)) / 1e6
        l2_note = (f"candidate bank {bank_mb:.0f} MB per rank "
                   + ("exceeds" if bank_mb * 1e6 > L2_BYTES else "fits")
                   + f" the 126 MB L2; every step additionally streams {step_mb:.0f} MB of queries, keys and "
                     "re-scoring rows (> L2), so no iteration starts with its inputs cached")
        line = {
            "metric": metric_name(), "value": value, "unit": "queries/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": {"bf16": "bf16", "tf32x3": "tf32x3", "bf16x3": "bf16x3", "f16x2": "f16x2", "f16": "f16", "exact": "f32",
                      "fp32": "f16+f32", "fp32_f16": "f16+f32", "fp32_f16x2": "f16x2+f32", "fp32_bf16x3": "bf16x3+f32",
                      "fp32_tf32": "tf32x3+f32", "fp32_bf16": "bf16+f32"}[mode], "data": "synthetic",
            "config": {"workload": f"knn_predict N={N} D={DIM} k={KNN_K} t={KNN_T} C={N_CLASSES}; "
                                   f"Q={Q} queries per step ({args.data} synthetic embeddings, WM-811K class priors)",
                       "mode": mode + (" (bit-exact: tensor-core candidates + exact sequential-fma re-scoring + "
                                       "per-row certificate)" if rescored else ""),
                       "bank_sharding": f"row-sharded over {world} GPU(s)" if world > 1 else "none",
                       "l2": l2_note, "plan": plan, "bank_prepare_ms_excluded": prepare_ms},
            "roofline": roof,
            "e2e": {"value": Q / (e2e_ms / args.steps * 1e-3), "unit": "queries/s",
                    "h2d_bytes_per_step": Q * DIM * 4, "d2h_bytes_per_step": Q * 8 * world,
                    "note": "whole-job bytes; the D2H is pred_labels[:, 0] (Q int64), the column the reference "
                            "consumes on the device (knn.py:99), not the full (Q, C) ranking; N>1: each rank uploads "
                            "1/N of the batch, an NVLink all-gather assembles it",
                    "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": gpu_launches,
            "clocks": clock_summary,
        }
        if quality is not None:
            line["quality"] = quality
        if phases is not None:
            line["config"]["phases_ms"] = phases
            line["config"]["exchange"] = (
                "candidate keys: stored by the top-k kernel into the query owner's buffer over NVLink peer memory; "
                "fp32: owner merges, stores each candidate into the inbox of the shard owning its bank row "
                "(route_scatter), that shard re-scores and stores the exact keys back (rescore_scatter); "
                "4 symmetric-memory barriers, NCCL only for the sampled thresholds and the final (Q,C+1) all-gather"
                if b200knn.ShardedBank.fused_exchange else "NCCL all_to_all_single")
        if rescored:
            line["config"]["uncertified_rows_last_step"] = uncertified
            line["config"]["cascade_last_step"] = rescore_stats.get("levels") if world == 1 else None
        line["config"]["prepass"] = {"stride": K.prepass_stride(N, k_plan, Q), "r": K.PREPASS["r"],
                                     "repaired_rows_last_step": prepass_stats["repaired"]}
        line.update(side)
        del side
        if world == 1 and not args.no_library and args.config == "north":
            # free the big bank first: the variants below build their own
            del bank, labels, q, staging
            pbank = None
            K.bank_cache.clear()
            torch.cuda.empty_cache()
            line["ref_shaped_call"] = ref_shaped(b200knn, K, dev, mode)
            if rescored and (N, DIM, KNN_K) == (811457, 512, 200):
                line["data_variants"] = data_variants(b200knn, K, dev, mode, exclude=args.data)
        if world == 1 and not args.no_cpu_baseline:
            rate, times, threads = cpu_reference_rate(64 if args.config == "ref" else 1024, 12)
            line["cpu_baseline"] = {"value": rate, "unit": "queries/s", "cores": threads, "kind": "port",
                                    "cpu": cpu_name(),
                                    "sample": f"12 calls of B={64 if args.config == 'ref' else 1024} queries against the "
                                              f"full {N_BANK}x{DIM} bank (oracle R32 = lightly knn_predict restated, "
                                              f"torch CPU fp32, {sum(times):.1f} s of CPU work)"}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def data_variants(b200knn, K, dev, mode, exclude):
    """The bit-exact mode on the other embedding distributions at the north-star size (2 waves of
    queries, 3 steps each): throughput, rows each cascade level left uncertified, and bitwise
    equality with the exact mode on a 256-query sample.  `relu` / `absgauss` are non-negative rows
    like the reference's post-ReLU features (knn.py:322): similarities bunched, same-sign products."""
    import torch

    out = {}
    Qv = 2 * WAVE
    for kind in ("gauss", "relu", "absgauss", "clustered"):
        if kind == exclude:
            continue
        bank_nd, labels, q = make_inputs(dev, N_BANK, Qv, DIM, seed=811, kind=kind)
        bank = bank_nd.t().contiguous()
        del bank_nd
        b200knn.set_default_mode(mode)

        def step():
            K.query_cache.clear()
            return b200knn.knn_predict(q, bank, labels, N_CLASSES, KNN_K, KNN_T)

        ms = time_calls(step, 3, 2)
        st = dict(K.last_rescore_stats)
        ek = b200knn.topk_keys(q[:256].contiguous(), bank, KNN_K, mode="exact")
        fk = b200knn.topk_keys(q[:256].contiguous(), bank, KNN_K, mode=mode)
        out[kind] = {"value": Qv / (ms * 1e-3), "unit": "queries/s", "Q": Qv, "ms_per_step": ms,
                     "cascade_last_step": st.get("levels"),
                     "keys_bitwise_equal_exact_mode": bool(torch.equal(ek, fk))}
        del bank, labels, q
        K.bank_cache.clear()
        torch.cuda.empty_cache()
    return out


if __name__ == "__main__":
    main()
