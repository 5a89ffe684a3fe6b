"""Helper process for tests/test_optimizers_gpu.py (two or more GPUs): a stateful update rule through the multi-replica
aggregation kernels, driven directly.

argv: <out json with RANK placeholder> <momentum|rmsprop> <bucket|kofn_delayed|interval>.  DMNIST_NVLS selects multimem (1)
or peer loads / stores (0).  Every rank writes a fingerprint of its weights AND state after every step; `ok` says whether
the rank's own checks (the float64 rule, tests/_optim_ref.py) held."""
import hashlib
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))

import numpy as np  # noqa: E402
import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

from distributedmnist_b200.optim import UpdateRule  # noqa: E402
from distributedmnist_b200.parallel.context import init_context, shutdown_context  # noqa: E402
from distributedmnist_b200.parallel.fused import FusedBackend  # noqa: E402
from _optim_ref import RefState  # noqa: E402

U = 2.0 ** -23


def fp(*ts):
    h = hashlib.sha1()
    for t in ts:
        h.update(t.detach().cpu().numpy().tobytes())
    return h.hexdigest()


def gathered(t, n):
    out = [torch.empty_like(t) for _ in range(n)]
    dist.all_gather(out, t)
    return out


def main():
    out_json = sys.argv[1].replace("RANK", os.environ.get("RANK", "0"))
    name, case = sys.argv[2], sys.argv[3]
    ctx = init_context(None, want_gpu=True)
    n, r = ctx.world_size, ctx.rank
    be = FusedBackend(ctx, timeout_ms=10000.0)
    rule = UpdateRule(name)
    res = {"fingerprints": [], "masks": [], "ok": True, "dropped": 0, "worst": 0.0}
    if case == "bucket":
        numel, e0, e1 = 1665024, 52160, 52160 + 1605632          # the LeNet arena: fc1 weights = early bucket
    else:
        numel, e0, e1 = 1 << 20, 0, 0
    params, grads = be.allocate(numel), be.allocate(numel)
    be.attach_shadow(params)
    slots = rule.allocate_slots(be.allocate, numel)
    gen = torch.Generator(device="cpu").manual_seed(4321)
    w0 = torch.randn(numel, generator=gen) * 0.1
    params.copy_(w0.to(ctx.device))
    be.refresh_shadow(params)
    ref = RefState(name, w0.numpy())
    torch.cuda.synchronize()
    be.barrier()

    def record(mask=None):
        torch.cuda.synchronize()
        be.barrier()
        res["fingerprints"].append(fp(params, *slots))
        if mask is not None:
            res["masks"].append(int(mask))

    def check(what):
        try:
            res["worst"] = max(res["worst"], ref.check(params.cpu().numpy(), [s.cpu().numpy() for s in slots], what=what))
        except AssertionError as e:
            print("rank %d: %s" % (r, e), flush=True)
            res["ok"] = False

    if case == "bucket":
        n_late = numel - (e1 - e0)
        g16 = be.allocate_buffer((e1 - e0) * 2)
        inbox = be.allocate_buffer(2 * n * n_late * 8)
        g16v = g16.view(torch.bfloat16, 0, e1 - e0)
        late = torch.cat([torch.arange(0, e0), torch.arange(e1, numel)])
        for step in range(5):
            gg = torch.Generator(device="cpu").manual_seed(1000 * step + r)
            g = torch.randn(numel, generator=gg) * 0.01
            grads.copy_(g.to(ctx.device))
            g16v.copy_(g[e0:e1].to(torch.bfloat16).to(ctx.device))
            all_g = [x.cpu().double() for x in gathered(grads, n)]
            # NCCL oracle of the early bucket's bf16 sum (fp32 accumulation, rounded to bf16 once), taken as exact
            nccl = g16v.float().clone()
            dist.all_reduce(nccl)
            torch.cuda.synchronize()
            be.barrier()
            be.enqueue_bucket_v2(params, grads, g16, inbox, 1, e0, e1, 0.1, 0.7, 2, rule=rule, slots=slots)
            be.enqueue_bucket_v2(params, grads, g16, inbox, 2, e0, e1, 0.1, 0.7, 2, rule=rule, slots=slots)
            torch.cuda.synchronize()
            be.check_error()
            gsum = torch.zeros(numel, dtype=torch.float64)
            gsum[e0:e1] = g16v.cpu().double()                  # the reduced bf16 sum the kernel applied
            esum = torch.zeros(numel, dtype=torch.float64)
            esum[e0:e1] = (nccl.cpu().double() - gsum[e0:e1]).abs()   # distance to the NCCL sum: within bf16 rounding
            if be.late_bf16 and be.late_ll:
                parts = [x[late].float().to(torch.bfloat16).double() for x in all_g]
            else:
                parts = [x[late] for x in all_g]
            gsum[late] = sum(parts)
            esum[late] = n * U * sum(p.abs() for p in parts)
            if not bool((esum[e0:e1] <= 2 ** -7 * gsum[e0:e1].abs() + 1e-6).all()):
                print("rank %d: early bucket sum differs from NCCL" % r, flush=True)
                res["ok"] = False
            ref.step(gsum.numpy(), n, 0.1 * 0.7 ** (step // 2), e_gsum=(n * U * sum(x.abs() for x in all_g)).numpy())
            check("bucket step %d" % step)
            record((1 << n) - 1)
    elif case == "kofn_delayed":
        k = n - 1
        for step in range(6):
            gg = torch.Generator(device="cpu").manual_seed(1000 * step + r)
            grads.copy_(torch.randn(numel, generator=gg).to(ctx.device))
            all_g = [x.cpu().double() for x in gathered(grads, n)]
            torch.cuda.synchronize()
            be.barrier()
            info = be.sync_step(params, grads, 0.05, step, k, delay_s=0.02 if r == n - 1 else 0.0, rule=rule, slots=slots)
            # the delayed rank fast-forwards: once every rank is here, all pushes (weights and state) have landed everywhere
            torch.cuda.synchronize()
            be.barrier()
            mask = torch.tensor([info.mask if r == 0 else 0], device=ctx.device)
            dist.broadcast(mask, 0)
            mask = int(mask.item())
            members = [q for q in range(n) if (mask >> q) & 1]
            ref.step(sum(all_g[q] for q in members).numpy(), len(members), 0.05,
                     e_gsum=(n * U * sum(all_g[q].abs() for q in members)).numpy())
            check("kofn step %d" % step)
            res["dropped"] += 0 if info.accepted else 1
            record(mask)
    else:                                                     # interval: ticks committed by whichever replica is first
        acc = be.allocate(numel)
        be.interval_arm(0.2)
        for it in range(12):
            be.enqueue_interval_begin(params)
            gg = torch.Generator(device="cpu").manual_seed(1000 * it + r)
            grads.copy_(torch.randn(numel, generator=gg).to(ctx.device))
            be.enqueue_interval_end(params, grads, acc, 0.05, rule=rule, slots=slots)
            torch.cuda.synchronize()
            be.check_error()
            time.sleep(0.1)
        torch.cuda.synchronize()
        be.barrier()
        be.enqueue_interval_begin(params)                     # adopt the last commit
        record()
        st = be.read_status()
        res["steps"] = st["epoch"]
        if st["epoch"] < 2:
            print("rank %d: only %d ticks committed" % (r, st["epoch"]), flush=True)
            res["ok"] = False
        if rule.num_slots and torch.equal(slots[0], torch.full_like(slots[0], rule.slot_inits[0])):
            res["ok"] = False
    be.check_error()
    with open(out_json, "w") as f:
        json.dump(res, f)
    be.close()
    shutdown_context(ctx)


if __name__ == "__main__":
    main()
