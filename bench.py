#!/usr/bin/env python
"""Headline benchmark: MNIST images/sec of the synchronous-replica LeNet training step.

Metric / config (BASELINE.json): whole-box images/sec, device-timed, max over ranks;
LeNet-like convnet (reference src/mnist.py:76-147, 1,663,370 parameters), bf16 tensor-core
operands / fp32 accumulate + fp32 master weights, batch 256 per replica, plain SGD, K = N
sync replicas, synthetic 28x28 data, random-init weights.  Weak scaling (per-GPU batch fixed).

    python bench.py --gpus N --steps K --warmup W          # our engine (N>1: under torchrun, or self-spawned)
    python bench.py --impl reference ...                   # the unmodified reference (unavailable here: TF1/py2)
    python bench.py --impl torch_ddp ...                   # baseline/: torch + cuDNN/cuBLAS + NCCL (for BASELINE.md)
    python bench.py ... --dump-outputs DIR                 # also save the last timed step's results as DIR/*.npy

One JSON line on stdout from rank 0.  Two measurements per run:
  * ``value``  -- K steps replayed from the CUDA graph with inputs already on the device, rotating through a
                  device-resident input pool larger than L2 (so every step reads cold inputs); CUDA events;
  * ``e2e``    -- K steps through the public API (``engine.load_batch`` from pinned host memory ->
                  ``engine.train_step`` -> device->host read of the loss) -- H2D and D2H inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "MNIST images/sec (whole box, device-timed, max over ranks)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=300)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "torch_ddp"])
    ap.add_argument("--batch", type=int, default=256, help="per-replica batch (BASELINE.json: 256)")
    ap.add_argument("--k", type=int, default=-1, help="replicas_to_aggregate (-1 = all)")
    ap.add_argument("--model", default="lenet", choices=["lenet", "mlp2", "mlp3"],
                    help="lenet = the headline config; mlp3 at --batch 8192 = BASELINE.json large-message config")
    ap.add_argument("--hidden", type=int, default=4096, help="MLP hidden width")
    ap.add_argument("--no-graph", action="store_true")
    ap.add_argument("--graphed", action="store_true", help="--impl torch_ddp: capture the whole baseline step (incl. the NCCL "
                                                           "all-reduce) in a CUDA graph")
    ap.add_argument("--straggler", default="", help="rank:prob:usec device-side delay injection")
    ap.add_argument("--kernel-times", action="store_true", help="also print per-kernel device times (stderr)")
    ap.add_argument("--trace", default="", help="after the timed runs: CUPTI timeline (torch.profiler) of a few graph-replayed "
                                                "steps -> <path>.json (chrome trace) + <path>.txt (one step, kernel start/end)")
    ap.add_argument("--dump-outputs", default="", metavar="DIR",
                    help="after the timed steps: rank 0's results of the last timed step -> DIR/loss_acc.npy (loss, "
                         "accuracy) and DIR/params.npy (the updated fp32 weights; a fixed, seeded sample of %d of them "
                         "when the model is larger), to compare two builds output for output; the weight gradients sum "
                         "with fp32 atomics, so two runs agree closely, not bit for bit" % DUMP_MAX_PARAMS)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_MAX_PARAMS = 8 << 20            # 32 MB of fp32 weights at most in a --dump-outputs directory


def dump_outputs(out_dir: str, params, loss_acc) -> None:
    """Write what a caller of the training step gets back: its (loss, accuracy) and the weights it left behind."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    flat = params.detach().float().cpu().reshape(-1)
    if flat.numel() > DUMP_MAX_PARAMS:
        idx = torch.randperm(flat.numel(), generator=torch.Generator().manual_seed(0))[:DUMP_MAX_PARAMS].sort().values
        flat = flat[idx]
    np.save(os.path.join(out_dir, "params.npy"), flat.numpy().astype(np.float32))
    np.save(os.path.join(out_dir, "loss_acc.npy"), np.asarray(loss_acc, dtype=np.float32).reshape(2))


# ----------------------------------------------------------------------------------------------------
# clocks / throttle reasons sampled DURING the timed region
# ----------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = [(0x8, "hw_slowdown"), (0x40, "hw_thermal_slowdown"), (0x20, "sw_thermal_slowdown"),
               (0x4, "sw_power_cap"), (0x80, "hw_power_brake_slowdown"), (0x2, "applications_clocks_setting")]

    def __init__(self, index: int, period_s: float = 0.004):
        self.index, self.period = index, period_s
        self.sm, self.reasons, self.sm_max = [], set(), None
        self._stop = threading.Event()
        self._t = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:  # noqa: BLE001
            self.nv = None

    def _loop(self):
        while not self._stop.is_set():
            try:
                self.sm.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS:
                    if r & bit:
                        self.reasons.add(name)
            except Exception:  # noqa: BLE001
                pass
            self._stop.wait(self.period)

    def start(self):
        if self.nv is not None:
            self._t = threading.Thread(target=self._loop, daemon=True)
            self._t.start()

    def stop(self):
        self._stop.set()
        if self._t is not None:
            self._t.join()
        return {"sm_mhz": statistics.median(self.sm) if self.sm else None, "sm_max_mhz": self.sm_max,
                "reasons": sorted(self.reasons), "samples": len(self.sm)}


# ----------------------------------------------------------------------------------------------------
def run_reference(args):
    # The reference is Python-2 / TensorFlow<=1.0 / Twisted code with no setup.py; `pip install --no-index
    # --target baseline/_ref /root/reference` fails ("Neither 'setup.py' nor 'pyproject.toml' found") and
    # neither tensorflow nor twisted exists offline (DESIGN.md "Reference arm").
    print(json.dumps({"impl": "reference",
                      "unavailable": "reference is py2/TF<=1.0/Twisted with no setup.py; pip --no-index install fails "
                                     "and tensorflow/twisted are absent offline"}))
    return 0


def write_timeline(path: str, step_fn, barrier, rank: int, steps: int = 6) -> None:
    """Kernel timeline of graph-replayed steps (shows which kernels really overlap).  Never a bench value."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    barrier()
    with profile(activities=[ProfilerActivity.CUDA, ProfilerActivity.CPU]) as prof:
        for i in range(steps):
            step_fn(i)
        torch.cuda.synchronize()
    barrier()
    if rank != 0:
        return
    os.makedirs(os.path.dirname(os.path.abspath(path)) or ".", exist_ok=True)
    prof.export_chrome_trace(path + ".json")
    ev = [e for e in json.load(open(path + ".json"))["traceEvents"]
          if e.get("ph") == "X" and e.get("cat") in ("kernel", "gpu_memcpy", "gpu_memset")]
    ev.sort(key=lambda e: e["ts"])
    # one step = from a conv1_fwd kernel to the next; print the second-to-last complete one
    starts = [i for i, e in enumerate(ev) if "conv1_fwd" in e["name"] or "f32_to_bf16" in e["name"]]
    with open(path + ".txt", "w") as f:
        if len(starts) >= 3:
            a, b = starts[-3], starts[-2]
            t0 = ev[a]["ts"]
            f.write("# one graph-replayed step: kernel, stream, start_us, end_us, dur_us (relative to the step's first kernel)\n")
            for e in ev[a:b]:
                f.write("%-44s s=%-4s %8.2f %8.2f %7.2f\n" % (e["name"].split("(")[0][-44:], e.get("args", {}).get("stream", "?"),
                                                             e["ts"] - t0, e["ts"] + e["dur"] - t0, e["dur"]))
            f.write("# step period = %.2f us\n" % (ev[b]["ts"] - t0))
        else:
            f.write("# no step boundary found; %d device events\n" % len(ev))


def maybe_self_spawn(args) -> bool:
    """`python bench.py --gpus N` without torchrun: spawn the N ranks ourselves."""
    if args.gpus > 1 and "RANK" not in os.environ:
        from distributedmnist_b200.parallel.launcher import run_replicas
        codes = run_replicas([os.path.abspath(__file__)] + sys.argv[1:], args.gpus)
        sys.exit(max(codes))
    return False


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)
    maybe_self_spawn(args)

    import torch
    import torch.distributed as dist

    from distributedmnist_b200.flags import FLAGS
    from distributedmnist_b200.parallel.context import init_context, shutdown_context

    if args.impl == "torch_ddp":
        from baseline.torch_ddp import run_baseline
        return run_baseline(args)

    from distributedmnist_b200.engine_cuda import CudaLeNetEngine, CudaMlpEngine
    from distributedmnist_b200.parallel.aggregators import SyncReplicasOptimizer, parse_straggler_spec
    from distributedmnist_b200.parallel.fused import FusedBackend
    from distributedmnist_b200.schedule import LearningRateSchedule, decay_steps_for

    ctx = init_context(FLAGS, want_gpu=True)
    if not ctx.on_gpu:
        print(json.dumps({"metric": METRIC, "value": None, "error": "no CUDA device"}))
        return 1
    n, rank, B = ctx.world_size, ctx.rank, args.batch
    k = n if args.k < 0 else args.k
    # backup-worker runs: a short watchdog so a starved replica can cost seconds, never minutes
    backend = FusedBackend(ctx) if k == n else FusedBackend(ctx, timeout_ms=5000.0)
    if args.model == "lenet":
        engine = CudaLeNetEngine(B, backend, seed=66478, rank=rank, use_graph=not args.no_graph)
    else:
        engine = CudaMlpEngine(args.model, B, backend, hidden=args.hidden, seed=66478, rank=rank,
                               use_graph=not args.no_graph)
    sched = LearningRateSchedule(0.01, decay_steps_for(60000, B, 2.0, k), 0.999)
    opt = SyncReplicasOptimizer(backend, sched, replicas_to_aggregate=k, total_num_replicas=n,
                                straggler=parse_straggler_spec(args.straggler))
    engine.attach_optimizer(opt)

    # ---- synthetic data ------------------------------------------------------------------------------------
    # host pool (pinned) for the e2e path; device pool > L2 (126 MB) for the device-timed path
    # every batch is one packed buffer (images then labels, the device slot's layout): a step's input is ONE copy
    g = torch.Generator().manual_seed(1234 + rank)
    pool_n = int(160e6 / (B * 784 * 4)) + 1
    n_host = 32 if B <= 1024 else 4
    h_pool = [engine.pack_batch(torch.rand(B, 28, 28, generator=g) - 0.5, torch.randint(0, 10, (B,), generator=g))
              for _ in range(n_host)]                                             # page-locked host memory
    d_pool = torch.empty(pool_n, h_pool[0].numel(), dtype=torch.uint8, device=ctx.device)
    for i in range(pool_n):
        d_pool[i].copy_(h_pool[i % n_host])
    # drawn from the seeded generator too, not torch's process-wide one: identical inputs from run to run
    d_pool[:, :B * 784 * 4].view(torch.float32).view(pool_n, -1).add_(   # distinct images per pool entry
        ((torch.rand(pool_n, 1, generator=g) - 0.5) * 0.1).to(ctx.device))

    def barrier():
        torch.cuda.synchronize()
        if n > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def device_step(i: int):
        # inputs come from the device pool (cold in L2) through the same public call as the e2e path: the copy into the
        # slot buffer runs on the engine's copy stream and overlaps the previous step
        engine.step_packed(d_pool[i % pool_n])

    def e2e_step(i: int):
        # pinned host -> device (one DMA on the copy stream) + the step graph (which copies (loss, acc) to pinned host memory)
        # through the engine's public one-call step; returns (completion event, host loss buffer, seq): read one step later
        return engine.step_packed(h_pool[i % n_host])

    def run_global_steps(step_fn, steps: int) -> int:
        """K < N (backup workers, reference SyncReplicasOptimizer): replicas are NOT in lock step -- a delayed replica's
        gradient is dropped and it fast-forwards -- so a fixed number of LOCAL iterations per replica would leave the
        slowest one alone at the end, waiting for arrivals that never come.  Everyone instead free-runs until the GLOBAL
        step has advanced by ``steps`` (the device epoch is polled every 8 iterations; before every launch once the target is
        near or once this replica has been seen fast-forwarding -- so nobody launches a step at or beyond the target).  Returns the number of images whose
        gradients were accepted across all replicas."""
        ep = torch.tensor([backend.device_epoch], device=ctx.device, dtype=torch.int64)
        if n > 1:
            dist.broadcast(ep, src=0)                        # the chief's view defines the window for everybody
        target = int(ep.item()) + steps
        acc0 = backend._read_u32("accepted_steps")
        it, since, careful, known = 0, 0, False, backend.device_epoch
        t_abort = time.monotonic() + float(os.environ.get("DMNIST_BENCH_ABORT_S", "120"))
        while True:
            if time.monotonic() > t_abort:
                # host-side wall-clock abort: a K < N window can never hold a GPU lease hostage (round 1, call 36)
                print("bench: K<N window aborted after the wall-clock limit at global step %d (target %d)" % (known, target),
                      file=sys.stderr)
                backend.debug_dump(sys.stderr)
                os._exit(3)
            if careful or since >= 8 or known + since >= target - 16:
                now = backend.device_epoch                   # synchronises this replica's stream
                if now - known > since:
                    careful = True       # fast-forwarded past steps it did not take part in: a straggler checks before EVERY launch
                known, since = now, 0
            if known >= target:
                break
            step_fn(it)
            it += 1
            since += 1
        torch.cuda.synchronize()
        accepted = torch.tensor([backend._read_u32("accepted_steps") - acc0], device=ctx.device, dtype=torch.int64)
        if n > 1:
            dist.all_reduce(accepted)
        return int(accepted.item()) * B

    # ---- warm-up (captures the graphs) ------------------------------------------------------------------------
    # at least 30 untimed steps: the first two capture the step graphs, the next ones bring the host-side launch path, the
    # copy engine and the L2-resident working set (weights, activations) to steady state; the count is reported as `warmup`
    n_warm = max(args.warmup, 30)
    if k == n:
        for i in range(n_warm):
            device_step(i)
    else:
        # backup workers: replicas are not in lock step, so also the warm-up is a window of GLOBAL steps -- a fixed number of
        # local iterations would leave the delayed replica alone at the end, waiting for arrivals that never come
        for i in range(2):
            device_step(i)                   # both slot graphs get captured (every replica still launches: no starvation yet)
        barrier()
        run_global_steps(device_step, n_warm)
    barrier()

    # ---- device-timed K steps ------------------------------------------------------------------------------------
    # (NVML queries take a driver lock that kernel launches also need: one sampling thread per BOX, on rank 0's GPU -- eight of
    #  them polling every 4 ms showed up as launch jitter, i.e. as arrival skew in the aggregation kernel)
    sampler = ClockSampler(ctx.device.index or 0)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    if rank == 0:
        sampler.start()
    barrier()
    backend.device_barrier()          # the replicas' streams enter the timed region within a flag hop of each other
    e0.record()
    if k == n:
        for i in range(args.steps):
            device_step(i)
        images_dev = n * B * args.steps
    else:
        images_dev = run_global_steps(device_step, args.steps)
    e1.record()
    barrier()
    clocks = sampler.stop()
    ms = torch.tensor([e0.elapsed_time(e1)], device=ctx.device)
    if n > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_total = float(ms.item())
    launches = engine.launches_per_step * args.steps

    # ---- end-to-end K steps (public API: pinned H2D every step, loss D2H every step) --------------------------------
    if k == n:
        for i in range(3):
            e2e_step(i)[0].synchronize()
    else:
        run_global_steps(lambda i: e2e_step(i)[0].synchronize(), 3)
    barrier()
    backend.device_barrier()
    e0.record()
    pending = None
    last_loss = 0.0
    last_loss_acc = None                                          # host buffer with the last timed step's (loss, accuracy)
    if k == n:
        for i in range(args.steps):
            ev = e2e_step(i)
            if pending is not None:
                pending[0].synchronize()
                last_loss = float(pending[1][0])                  # the step's result is consumed on the host
            pending = ev
        pending[0].synchronize()
        last_loss = float(pending[1][0])
        last_loss_acc = pending[1]
        images_e2e = n * B * args.steps
    else:
        def e2e_consume(i):
            nonlocal last_loss, last_loss_acc
            ev = e2e_step(i)
            ev[0].synchronize()
            last_loss = float(ev[1][0])
            last_loss_acc = ev[1]
        images_e2e = run_global_steps(e2e_consume, args.steps)
    e1.record()
    barrier()
    ms2 = torch.tensor([e0.elapsed_time(e1)], device=ctx.device)
    if n > 1:
        dist.all_reduce(ms2, op=dist.ReduceOp.MAX)
    ms2_total = float(ms2.item())
    backend.check_error()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, engine.params, last_loss_acc)
    info = engine.step_info()
    if args.kernel_times:
        kt = engine.time_kernels(20)
        if rank == 0:
            print("KERNEL_TIMES_US " + json.dumps({k: round(v, 2) for k, v in kt.items()}) + " sum=%.1f" % sum(kt.values()),
                  file=sys.stderr)

    if args.trace:
        write_timeline(args.trace, device_step, barrier, rank)

    # per-rank %globaltimer phases of the LAST step's aggregation kernels: who waited for whom (the rank with the shortest
    # arrival wait is the one everybody else waited for)
    my_ph = {"late": backend.read_phases(), "early": backend.read_phases_early() if getattr(engine, "_bucketed", False) else None}
    all_ph = backend.all_gather_object(my_ph)
    if rank == 0:
        value = images_dev / (ms_total / 1e3)
        e2e_value = images_e2e / (ms2_total / 1e3)
        out = {
            "metric": METRIC, "value": value, "unit": "images/s", "n_gpus": n, "steps": args.steps,
            "warmup": n_warm, "ms_per_step": ms_total / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "impl": "ours",
            "config": {"model": ("LeNet-like MNIST convnet (1,663,370 params, reference src/mnist.py)" if args.model == "lenet"
                                 else "%s hidden=%d (%d params)" % (args.model, args.hidden, engine.spec.num_trainable)),
                       "global_batch": n * B, "batch_per_replica": B, "seq_len": None,
                       "parallelism": "dp%d (sync replicas, K=%d of %d, fused NVLink allreduce+SGD kernel, %s)"
                                      % (n, k, n, "NVLS multimem.ld_reduce/st" if backend.nvls_active else
                                         ("P2P ld/st" if n > 1 else "single replica")),
                       "optimizer": "SGD, staircase exp-decay LR evaluated on device",
                       "l2": "inputs rotate through a %d MB device pool (> 126 MB L2)" % int(d_pool.numel() / 1e6),
                       "cuda_graph": not args.no_graph},
            "clocks": {"sm_mhz": clocks["sm_mhz"], "sm_max_mhz": clocks["sm_max_mhz"], "reasons": clocks["reasons"],
                       "samples": clocks["samples"]},
            "e2e": {"value": e2e_value, "unit": "images/s", "ms_per_step": ms2_total / args.steps,
                    "h2d_bytes_per_step": engine.h2d_bytes_per_step(),
                    # (loss, accuracy) copied by a graph branch + the 8 status words the closing kernel stores into host memory
                    "d2h_bytes_per_step": 8 + 32,
                    "last_loss": last_loss},
            "backup_workers": (None if k == n else
                               {"k": k, "n": n, "window_global_steps": args.steps, "accepted_images_device_phase": images_dev,
                                "note": "replicas free-run until the global step advanced by `steps`; value = accepted images / time"}),
            "gpu_launches": launches, "gpu_launches_per_step": engine.launches_per_step,
            "final_global_step": info.global_step,
            "sync_phases_ns": dict(zip(["start", "decided", "reduced", "pushed", "landed", "end"], backend.read_phases())),
            "sync_early_phases_ns": (dict(zip(["start", "arrived", "reduced_cta0", "all_pushed", "all_landed", "applied_cta0"],
                                              backend.read_phases_early()))
                                     if getattr(engine, "_bucketed", False) else None),
            "sync_phases_all_ranks_ns": [p["late"] for p in all_ph],
            "sync_early_phases_all_ranks_ns": [p["early"] for p in all_ph],
            "aggregation": ("bucketed v2: bf16-wire fc1 bucket under the backward pass + pushed late bucket (csrc/fused_bucket.cu)"
                            if getattr(engine, "_bucket_v2", False) else
                            ("bucketed v1 (fp32 two-shot early + one-shot late)" if getattr(engine, "_bucketed", False)
                             else "single fused kernel")),
        }
        print(json.dumps(out))
    sys.stdout.flush()
    backend.close()
    shutdown_context(ctx)
    return 0


if __name__ == "__main__":
    sys.exit(main())
