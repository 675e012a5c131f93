"""GPU, >= 2 devices: the bank-row-sharded mode over NCCL + NVLink peer memory must reproduce the
single-GPU result BIT FOR BIT on every rank (SURVEY.md §8e invariant) — exact, fp32 (bit-exact,
fused route_scatter / rescore_scatter exchange and the NCCL fallback) and bf16 (fused
b200knn_topk_opt's peer exchange and NCCL all-to-all), including a batch large enough for the fused exchange,
forced second-level rows and the host-driven fallback.  Skipped on a single-GPU box."""
import os
import socket

import pytest
import torch

pytestmark = pytest.mark.gpu


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def run_cases(rank, dev, log=None):
    """The comparisons (every rank of an initialised NCCL group calls this); returns the failures."""
    import b200knn
    from b200knn import knn as K

    failures = []
    cases = [(200000, 512, 300, 200, 9, "gauss"), (30000, 512, 130, 20, 38, "gauss"), (50001, 384, 65, 5, 9, "gauss"),
             (120001, 512, 19001, 200, 9, "relu")]  # the last one: fused exchange, non-negative rows
    for (N, D, B, k, C, kind) in cases:
        g = torch.Generator(device=dev).manual_seed(811)  # same seed on every rank -> replicated inputs
        x = torch.randn(N, D, generator=g, device=dev)
        y = torch.randn(B, D, generator=g, device=dev)
        if kind == "relu":
            x, y = x.clamp_min(0) + 0.05, y.clamp_min(0) + 0.05
        bank = torch.nn.functional.normalize(x, dim=1).t().contiguous()
        q = torch.nn.functional.normalize(y, dim=1)
        lab = torch.randint(0, C, (N,), generator=g, device=dev)
        for mode in ("exact", "fp32", "bf16"):
            single = b200knn.topk_keys(q, bank, k, mode=mode)
            sb = b200knn.ShardedBank.from_full(bank, lab, mode=mode)
            sharded = sb.topk_keys(q, k)
            b200knn.set_default_mode(mode)
            p1 = b200knn.knn_predict(q, bank, lab, C, k, 0.1)
            p2 = sb.knn_predict(q, C, k, 0.1)                        # fused exchange where it applies
            p3 = sb.knn_predict(q, C, k, 0.1, exchange="allgather")  # the literal all-gather of keys
            b200knn.ShardedBank.fused_exchange = False                 # NCCL all-to-alls instead of P2P stores
            p4 = sb.knn_predict(q, C, k, 0.1)
            b200knn.ShardedBank.fused_exchange = True
            p5 = sb.knn_predict(q, C, k, 0.1)                        # buffers reused across calls
            b200knn.ShardedBank.fused_threshold = True                 # threshold exchange over peer memory too
            p6 = sb.knn_predict(q, C, k, 0.1)
            b200knn.ShardedBank.fused_threshold = False
            ok = bool(torch.equal(single, sharded)) and all(bool(torch.equal(p1, p)) for p in (p2, p3, p4, p5, p6))
            if log is not None:
                log(f"rank {rank} N={N} D={D} B={B} k={k} {kind} mode={mode}: sharded==single {ok}")
            if not ok:
                failures.append((N, D, B, k, mode))
        # second level on the device: make the first level's certificate unattainable for this call,
        # every row then goes through compact_rows -> per-shard exact keys -> all-gather -> merge
        b200knn.set_default_mode("fp32")
        sb = b200knn.ShardedBank.from_full(bank, lab, mode="fp32")
        n_sub = min(200, B)
        sub = q[:n_sub].contiguous()
        want = b200knn.knn_predict(sub, bank, lab, C, k, 0.1)
        old = K.LEVELS["fp32_f16"]["op_coef"]
        K.LEVELS["fp32_f16"]["op_coef"] = 10.0
        try:
            got = sb.knn_predict(sub, C, k, 0.1)
            n_open = sb.last_uncertified
            got2 = sb.knn_predict(sub, C, k, 0.1)
        finally:
            K.LEVELS["fp32_f16"]["op_coef"] = old
        ok = bool(torch.equal(got, want)) and bool(torch.equal(got2, want)) and n_open == n_sub
        if log is not None:
            log(f"rank {rank} N={N} D={D} B={n_sub} k={k} {kind} fp32 second level on {n_open} rows: sharded==single {ok}")
        if not ok:
            failures.append((N, D, B, k, "fp32-second-level", n_open))
    b200knn.set_default_mode("exact")
    return failures


def _worker(rank, world, port, out_dir):
    import torch.distributed as dist

    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        failures = run_cases(rank, dev)
        flag = torch.tensor([len(failures)], device=dev)
        dist.all_reduce(flag)
        with open(os.path.join(out_dir, f"rank{rank}.txt"), "w") as f:
            f.write(repr(failures))
        assert int(flag.item()) == 0, failures
    finally:
        dist.destroy_process_group()


def test_sharded_equals_single_bitwise_on_gpus(tmp_path):
    world = min(2, torch.cuda.device_count())
    if world < 2:
        pytest.skip("needs at least 2 GPUs")
    import torch.multiprocessing as mp

    mp.spawn(_worker, args=(world, _free_port(), str(tmp_path)), nprocs=world, join=True)
    for r in range(world):
        assert open(tmp_path / f"rank{r}.txt").read() == "[]"
