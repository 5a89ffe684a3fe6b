"""Momentum and RMSProp in the sm_100a aggregation kernels: every kernel that owns an update, against the float64 TF
formulas with a derived fp32 bound (tests/_optim_ref.py), through the engines, across replicas, and from the entry point."""
import os

import numpy as np
import pytest
import torch

from distributedmnist_b200.parallel.launcher import run_replicas

from _optim_ref import RefState

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
STATEFUL = ["momentum", "rmsprop"]


def _backend():
    from distributedmnist_b200.parallel.context import ReplicaContext
    from distributedmnist_b200.parallel.fused import FusedBackend
    torch.cuda.set_device(0)
    return FusedBackend(ReplicaContext(0, 1, 0, torch.device("cuda", 0), "none"))


def _lr(lr0, rate, steps, k):
    return lr0 * rate ** (k // steps)


def _bf16(t):
    return t.to(torch.bfloat16).to(torch.float32)


# ---- 1. one rank, kernels driven directly -------------------------------------------------------------------------------
@pytest.mark.parametrize("name", STATEFUL)
def test_single_kernel_matches_float64_rule(name):
    from distributedmnist_b200.optim import UpdateRule
    be = _backend()
    rule = UpdateRule(name)
    n = 1 << 18
    params, grads = be.allocate(n), be.allocate(n)
    be.attach_shadow(params)
    slots = rule.allocate_slots(be.allocate, n)
    gen = torch.Generator().manual_seed(11)
    w0 = torch.randn(n, generator=gen)
    params.copy_(w0)
    ref = RefState(name, w0.numpy())
    lr0, rate, dsteps = 0.2, 0.5, 2
    for k in range(6):
        g = torch.randn(n, generator=gen) * torch.exp(torch.randn(n, generator=gen))
        grads.copy_(g)
        be.enqueue(params, grads, 1, lr0=lr0, decay_rate=rate, decay_steps=dsteps, rule=rule, slots=slots)
        torch.cuda.synchronize()
        be.check_error()
        ref.step(g.numpy(), 1, _lr(lr0, rate, dsteps, k), e_gsum=4 * 2.0 ** -23 * np.abs(g.numpy()))  # (__powf rate)
        ref.check(params.cpu().numpy(), [s.cpu().numpy() for s in slots], what="%s step %d" % (name, k))
        assert torch.equal(be.shadow, params.to(torch.bfloat16))           # shadow refreshed from the new weights
    assert be.device_epoch == 6


@pytest.mark.parametrize("name", STATEFUL)
@pytest.mark.parametrize("late_ll", [True, False], ids=["late_ll", "late_fp32"])
def test_bucket_v2_kernels_match_float64_rule(name, late_ll):
    """Phase 1 (early bucket, bf16 sum from g16) + phase 2 (late bucket: LL lines carry bf16, or fp32 data) on the LeNet
    arena split, one replica."""
    from distributedmnist_b200.optim import UpdateRule
    be = _backend()
    be.late_ll = late_ll
    rule = UpdateRule(name)
    numel, e0, e1 = 1665024, 52160, 52160 + 1605632
    params, grads = be.allocate(numel), be.allocate(numel)
    be.attach_shadow(params)
    slots = rule.allocate_slots(be.allocate, numel)
    g16 = be.allocate_buffer((e1 - e0) * 2)
    g16v = g16.view(torch.bfloat16, 0, e1 - e0)
    gen = torch.Generator().manual_seed(12)
    w0 = torch.randn(numel, generator=gen) * 0.1
    params.copy_(w0)
    be.refresh_shadow(params)
    ref = RefState(name, w0.numpy())
    late = torch.cat([torch.arange(0, e0), torch.arange(e1, numel)])
    lr0, rate, dsteps = 0.1, 0.7, 2
    for k in range(6):
        g = torch.randn(numel, generator=gen) * 0.01
        grads.copy_(g)
        g16v.copy_(g[e0:e1].to(torch.bfloat16))
        be.enqueue_bucket_v2(params, grads, g16, None, 1, e0, e1, lr0, rate, dsteps, rule=rule, slots=slots)
        be.enqueue_bucket_v2(params, grads, g16, None, 2, e0, e1, lr0, rate, dsteps, rule=rule, slots=slots)
        torch.cuda.synchronize()
        be.check_error()
        applied = g.clone()
        applied[e0:e1] = _bf16(g[e0:e1])                   # the early bucket sums bf16 gradients
        if late_ll:
            applied[late] = _bf16(g[late])                 # ... and the LL lines carry bf16 too
        ref.step(applied.numpy(), 1, _lr(lr0, rate, dsteps, k), e_gsum=4 * 2.0 ** -23 * np.abs(applied.numpy()))
        ref.check(params.cpu().numpy(), [s.cpu().numpy() for s in slots], what="%s step %d" % (name, k))
        assert torch.equal(be.shadow, params.to(torch.bfloat16))
    assert be.device_epoch == 6


# ---- 2. one GPU, through the engines ----------------------------------------------------------------------------------
@pytest.mark.parametrize("name", STATEFUL)
@pytest.mark.parametrize("model", ["lenet", "mlp3"])
def test_engine_step_applies_the_rule(model, name):
    """Every training step moves the weights by exactly the rule's step, from the state the kernels keep: lr_k * a_k
    (momentum) or mom_k (RMSProp), to fp32 rounding.  mlp3 at hidden 1024 sends its 3.3 MB late bucket through
    bucket_late_kernel, LeNet's through bucket_late_ll_kernel; the early bucket runs bucket_early_kernel."""
    from distributedmnist_b200.engine_cuda import CudaLeNetEngine, CudaMlpEngine
    from distributedmnist_b200.optim import UpdateRule
    from distributedmnist_b200.parallel.aggregators import SyncReplicasOptimizer
    from distributedmnist_b200.schedule import LearningRateSchedule
    be = _backend()
    B = 128
    eng = CudaLeNetEngine(B, be) if model == "lenet" else CudaMlpEngine("mlp3", B, be, hidden=1024)
    sched = LearningRateSchedule(0.05, 2, 0.5)
    rule = UpdateRule(name)
    opt = SyncReplicasOptimizer(be, sched, 1, 1, update_rule=rule)
    eng.attach_optimizer(opt)
    assert eng._bucket_v2 and len(eng.slots) == rule.num_slots
    valid = eng.spec.valid_mask().to(eng.params.device)
    gen = torch.Generator().manual_seed(13)
    u = 2.0 ** -23
    for k in range(5):
        x = torch.rand(B, 28, 28, generator=gen) - 0.5
        y = torch.randint(0, 10, (B,), generator=gen)
        w_prev = eng.params.clone()
        eng.load_batch(x.reshape(eng.images[0].shape).numpy(), y.numpy())
        eng.train_step()
        torch.cuda.synchronize()
        be.check_error()
        w = eng.params
        step = (w_prev - w)[valid].double()
        if name == "momentum":
            want = (sched(k) * eng.slots[0])[valid].double()
            tol = 4 * u * (w_prev.abs() + w.abs())[valid].double() + 8 * u * want.abs()
        else:
            want = eng.slots[1][valid].double()
            tol = 4 * u * (w_prev.abs() + w.abs())[valid].double()
        err = (step - want).abs()
        assert bool((err <= tol + 1e-30).all()), "%s %s step %d: max err/tol %.3f" % (model, name, k,
                                                                                   float((err / (tol + 1e-30)).max()))
        assert not torch.equal(eng.slots[0][valid], torch.full_like(eng.slots[0][valid], rule.slot_inits[0]))
        assert torch.equal(be.shadow, w.to(torch.bfloat16))


# ---- 3. multi-GPU ---------------------------------------------------------------------------------------------------------
def _gpus():
    return torch.cuda.device_count()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
@pytest.mark.parametrize("nvls", ["0", "1"])
@pytest.mark.parametrize("case", ["bucket", "kofn_delayed", "interval"])
@pytest.mark.parametrize("name", STATEFUL)
def test_replicas_hold_identical_weights_and_state(tmp_path, name, case, nvls):
    n = _gpus()
    out = str(tmp_path / "out")
    codes = run_replicas([os.path.join(HERE, "_optimizer_worker.py"), str(tmp_path / "res_RANK.json"), name, case], n,
                         timeout=300, out_dir=out, env={"DMNIST_NVLS": nvls})
    logs = "\n".join(open(os.path.join(out, f)).read()[-3000:] for f in sorted(os.listdir(out)))
    assert codes == [0] * n, logs
    import json
    res = [json.load(open(tmp_path / ("res_%d.json" % r))) for r in range(n)]
    for r in res[1:]:
        assert r["fingerprints"] == res[0]["fingerprints"], "replicas diverged"
    assert all(r["ok"] for r in res), logs
    if case == "kofn_delayed":
        assert all(m & (1 << (n - 1)) == 0 for m in res[0]["masks"])       # the delayed rank is never in the mask
        assert res[-1]["dropped"] > 0


# ---- 4. entry point, two ranks ----------------------------------------------------------------------------------------
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs at least two GPUs")
def test_entry_point_checkpoints_and_resumes_momentum(tmp_path):
    from distributedmnist_b200.checkpoint import Saver
    tdir = tmp_path / "train"
    argv = [os.path.join(ROOT, "src", "mnist_distributed_train.py"), "--optimizer=momentum", "--num_replicas_to_aggregate=1",
            "--inject_straggler=1:1.0:1000", "--model=lenet", "--batch_size=64", "--train_dir=%s" % tdir,
            "--save_interval_secs=1000"]
    for steps in (20, 40):
        codes = run_replicas(argv + ["--max_steps=%d" % steps], 2, timeout=300, out_dir=str(tmp_path / ("out%d" % steps)))
        assert codes == [0, 0]
        state, step = Saver.restore(Saver.latest(str(tdir)))
        assert {"Variable/Momentum"} | {"Variable_%d/Momentum" % i for i in range(1, 8)} <= set(state)
        assert step > steps
        if steps == 20:
            first = step
    assert step > first
    logs = "".join(open(os.path.join(tmp_path, "out40", f)).read() for f in os.listdir(tmp_path / "out40"))
    assert "Restored momentum optimizer slots" in logs
