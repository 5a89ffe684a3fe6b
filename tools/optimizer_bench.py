#!/usr/bin/env python
"""Step time of sgd, momentum and RMSProp on the GPU path, alternated in one process.

The timed loop is bench.py's: inputs rotate through a device pool larger than the 126 MB L2, warm-up, CUDA events around K
steps, the maximum over ranks.  One engine per update rule shares the backend; the rules take turns for `--rounds` rounds
of K steps, so the three see the same machine state.  One JSON line per (model, rule) with the card's name and power limit;
at N >= 2 also the early-bucket phase stamps of the last step (start, arrived, reduced, pushed, landed, applied; us).

    python tools/optimizer_bench.py --model lenet --batch_size 256 --gpus 1
    python tools/optimizer_bench.py --model mlp3 --mlp_hidden 4096 --batch_size 8192 --gpus 1
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)


def card(index: int):
    import torch
    name = torch.cuda.get_device_name(index)
    try:
        q = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=power.limit", "--format=csv,noheader,nounits"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        power = float(q)
    except (OSError, ValueError, subprocess.SubprocessError):
        power = None
    return name, power


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--model", default="lenet")
    ap.add_argument("--mlp_hidden", type=int, default=4096)
    ap.add_argument("--batch_size", type=int, default=256)
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=50)
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--rules", default="sgd,momentum,rmsprop")
    args = ap.parse_args()
    if args.gpus > 1 and "RANK" not in os.environ:
        from distributedmnist_b200.parallel.launcher import run_replicas
        sys.exit(max(run_replicas([os.path.abspath(__file__)] + sys.argv[1:], args.gpus)))

    import torch
    import torch.distributed as dist

    from distributedmnist_b200.engine_cuda import CudaLeNetEngine, CudaMlpEngine
    from distributedmnist_b200.optim import UpdateRule
    from distributedmnist_b200.parallel.aggregators import SyncReplicasOptimizer
    from distributedmnist_b200.parallel.context import init_context, shutdown_context
    from distributedmnist_b200.parallel.fused import FusedBackend
    from distributedmnist_b200.schedule import LearningRateSchedule

    ctx = init_context(None, want_gpu=True)
    if not ctx.on_gpu:
        print(json.dumps({"error": "no CUDA device"}))
        sys.exit(1)
    n, rank, B = ctx.world_size, ctx.rank, args.batch_size
    backend = FusedBackend(ctx)
    rules = [UpdateRule(r) for r in args.rules.split(",")]
    engines = {}
    for rule in rules:
        eng = CudaLeNetEngine(B, backend, rank=rank) if args.model == "lenet" else \
            CudaMlpEngine(args.model, B, backend, hidden=args.mlp_hidden, rank=rank)
        eng.attach_optimizer(SyncReplicasOptimizer(backend, LearningRateSchedule(0.01, 1000, 0.95), n, n, update_rule=rule))
        engines[rule.name] = eng
    g = torch.Generator().manual_seed(1234 + rank)
    first = engines[rules[0].name]
    pool_n = int(160e6 / (B * 784 * 4)) + 1
    d_pool = torch.empty(pool_n, first._in_bytes, dtype=torch.uint8, device=ctx.device)
    for i in range(pool_n):
        d_pool[i].copy_(first.pack_batch(torch.rand(B, 28, 28, generator=g) - 0.5, torch.randint(0, 10, (B,), generator=g),
                                         pin=False))

    def barrier():
        torch.cuda.synchronize()
        backend.barrier()

    for eng in engines.values():
        for i in range(args.warmup):
            eng.step_packed(d_pool[i % pool_n])
        barrier()
    times = {r.name: [] for r in rules}
    phases = {}
    for rnd in range(args.rounds):
        for rule in rules:
            eng = engines[rule.name]
            barrier()
            backend.device_barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(args.steps):
                eng.step_packed(d_pool[(rnd * args.steps + i) % pool_n])
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=ctx.device)
            if n > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            times[rule.name].append(float(ms.item()) * 1e3 / args.steps)
            if n > 1 and eng._bucket_v2:
                phases[rule.name] = [round(x / 1e3, 2) for x in backend.read_phases_early()]
    backend.check_error()
    if rank == 0:
        name, power = card(ctx.device.index or 0)
        for rule in rules:
            t = times[rule.name]
            out = {"model": args.model, "hidden": args.mlp_hidden if args.model != "lenet" else None, "batch": B, "gpus": n,
                   "optimizer": rule.name, "us_per_step_median": round(statistics.median(t), 2),
                   "us_per_step_min": round(min(t), 2), "us_per_step_max": round(max(t), 2), "rounds": args.rounds,
                   "steps_per_round": args.steps, "bucketed": bool(engines[rule.name]._bucket_v2),
                   "card": name, "power_limit_w": power}
            if rule.name in phases:
                out["early_phases_us"] = phases[rule.name]
            print(json.dumps(out), flush=True)
    barrier()
    shutdown_context(ctx)


if __name__ == "__main__":
    main()
