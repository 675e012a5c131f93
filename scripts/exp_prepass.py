"""Experiment (not a test): where does the sampling pre-pass spend its time?
(a) strided sample (production), (b) the same number of contiguous rows, (c) contiguous rows with
an admission threshold already in place (no list traffic), (d) k=200 main pass for scale."""
import os
import sys

ROOT = os.path.normpath(os.path.join(os.path.dirname(os.path.abspath(__file__)), ".."))
sys.path.insert(0, os.path.join(ROOT, "self-supervised-wafermaps_b200"))
import torch  # noqa: E402

import b200knn  # noqa: E402
from b200knn import knn as K  # noqa: E402

dev = torch.device("cuda:0")
Q, N, D = 75776, 811457, 512
g = torch.Generator(device=dev).manual_seed(1)
bank = torch.nn.functional.normalize(torch.randn(N, D, generator=g, device=dev), dim=1)
q = torch.nn.functional.normalize(torch.randn(Q, D, generator=g, device=dev), dim=1)
pb = b200knn.prepare_rows(bank.t(), "bf16", vectors_are_columns=True)
pq = b200knn.prepare_rows(q, "bf16", vectors_are_columns=False)


def timed(label, fn, reps=3):
    ts = []
    for _ in range(reps + 1):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        out = fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    print(f"{label:60s} {min(ts[1:]):8.3f} ms", flush=True)
    return out


for s, r in ((62, 16),):
    n_visit = (N + s - 1) // s
    keys = timed(f"(a) strided sample  s={s} n_visit={n_visit} k={r}",
                 lambda: K._search("bf16", pq, pb, Q, n_visit, D, r, stride=s))
    timed(f"(b) contiguous rows          n_visit={n_visit} k={r}",
          lambda: K._search("bf16", pq, pb, Q, n_visit, D, r))
    timed(f"(a') strided sample, register top-16 variant",
          lambda: K._search("bf16", pq, pb, Q, n_visit, D, r, stride=s, sample=True))
    tau = K.kth_sim(keys)
    timed(f"(c) contiguous rows, tau0 = own {r}-th best (few appends)",
          lambda: K._search("bf16", pq, pb, Q, n_visit, D, r, tau0=tau))
    timed(f"(c') strided rows, tau0 = own {r}-th best (few appends)",
          lambda: K._search("bf16", pq, pb, Q, n_visit, D, r, stride=s, tau0=tau))
keys = K._search("bf16", pq, pb, Q, (N + 61) // 62, D, 16, stride=62)
tau = K.kth_sim(keys)
timed("(d) main pass k=200 with prepass tau", lambda: K._search("bf16", pq, pb, Q, N, D, 200, tau0=tau))
timed("(d') main pass k=200 without tau", lambda: K._search("bf16", pq, pb, Q, N, D, 200), reps=1)
