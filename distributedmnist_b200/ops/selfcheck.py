"""Numerics self-checks of the sm_100a LeNet kernels against plain PyTorch fp32 references.

Each check returns ``(name, error, tolerance)``; ``tests/test_lenet_kernels_gpu.py``
asserts on them and ``tools/gpu_diag_lenet.py`` prints them all (one GPU call gives the
full picture when bringing a kernel up).
"""
from __future__ import annotations

import ctypes
from typing import List, Tuple

import torch
import torch.nn.functional as F

from ..models import dropout_keep_mask, dropout_seed_mix, get_model, lenet_forward, loss_and_accuracy
from ..parallel.context import ReplicaContext
from ..parallel.fused import FusedBackend
from .lib import check, load, ptr, stream_ptr

Result = Tuple[str, float, float]


def _bf(t: torch.Tensor) -> torch.Tensor:
    return t.to(torch.bfloat16)


def _nchw(t: torch.Tensor) -> torch.Tensor:
    return t.float().permute(0, 3, 1, 2).contiguous()


def _nhwc(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 2, 3, 1).contiguous()


def _decode_pool(code: torch.Tensor):
    return (code & 3).long(), ((code >> 2) & 1).bool()


def check_conv1_fwd(B: int = 8, seed: int = 0, tc: bool = False) -> List[Result]:
    lib, dev = load(), "cuda"
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = (torch.rand(B, 28, 28, generator=g) - 0.5).to(dev)
    w = (torch.randn(5, 5, 1, 32, generator=g) * 0.1).to(dev)
    b = (torch.randn(32, generator=g) * 0.1).to(dev)
    out = torch.zeros(B, 14, 14, 32, dtype=torch.bfloat16, device=dev)
    code = torch.zeros(B, 14, 14, 32, dtype=torch.uint8, device=dev)
    junk = torch.ones(100, device=dev)
    fn = lib.dm_conv1_fwd_tc if tc else lib.dm_conv1_fwd
    check(fn(ptr(x), ptr(w), ptr(b), ptr(out), ptr(code), B, ptr(junk), 100, ctypes.c_void_p(0), 0,
             ctypes.c_void_p(0), 0, stream_ptr()), "conv1_fwd")
    if tc:   # the tensor-core path rounds its operands to bf16: compare against the same rounding
        x, w = x.to(torch.bfloat16).float(), w.to(torch.bfloat16).float()
    conv = F.conv2d(x[:, None], w.permute(3, 2, 0, 1), b, padding=2)
    ref = _nhwc(F.max_pool2d(F.relu(conv), 2, 2))
    err = (out.float() - ref).abs().max().item()
    # argmax code: the selected position must hold the window maximum
    idx, act = _decode_pool(code)
    win = _nhwc(conv).reshape(B, 14, 2, 14, 2, 32).permute(0, 1, 3, 5, 2, 4).reshape(B, 14, 14, 32, 4)
    sel = torch.gather(win, 4, idx[..., None])[..., 0]
    err_idx = (sel - win.max(dim=4).values).abs().max().item()
    bad_act = ((sel > 1e-4) & ~act) | ((sel < -1e-4) & act)
    tag = "conv1_fwd_tc" if tc else "conv1_fwd"
    return [(tag + ".out", err, 0.02), (tag + ".argmax", err_idx, 1e-4 if tc else 1e-5),
            (tag + ".relu_flag", bad_act.float().sum().item(), 0.5), (tag + ".zeroing", junk.abs().max().item(), 1e-12)]


def check_conv1_fwd_tc(B: int = 8, seed: int = 0) -> List[Result]:
    return check_conv1_fwd(B, seed, tc=True)


def check_conv1_wgrad(B: int = 8, seed: int = 7, tc: bool = True) -> List[Result]:
    """conv1 weight/bias gradient fused with the maxpool1/ReLU1 backward (SIMT and tcgen05 versions)."""
    lib, dev = load(), "cuda"
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = (torch.rand(B, 28, 28, generator=g) - 0.5).to(dev)
    dpool = _bf(torch.randn(B, 14, 14, 32, generator=g) * 0.1).to(dev)
    code = (torch.randint(0, 4, (B, 14, 14, 32), generator=g) | (torch.randint(0, 2, (B, 14, 14, 32), generator=g) << 2)) \
        .to(torch.uint8).to(dev)
    gw = torch.zeros(25, 32, device=dev)
    gb = torch.zeros(32, device=dev)
    fn = lib.dm_conv1_wgrad_tc if tc else lib.dm_conv1_wgrad
    check(fn(ptr(x), ptr(dpool), ptr(code), ptr(gw), ptr(gb), B, stream_ptr()), "conv1_wgrad")
    idx, act = _decode_pool(code)
    masked = dpool.float() * act
    dy = torch.zeros(B, 14, 2, 14, 2, 32, device=dev)
    for q in range(4):
        dy[:, :, q >> 1, :, q & 1, :] = masked * (idx == q)
    dy = dy.reshape(B, 28, 28, 32)
    xr = x.to(torch.bfloat16).float() if tc else x
    ref = torch.nn.grad.conv2d_weight(xr[:, None], (32, 1, 5, 5), _nchw(dy), padding=2)    # [32,1,5,5]
    ref = ref[:, 0].permute(1, 2, 0).reshape(25, 32)
    tag = "conv1_wgrad_tc" if tc else "conv1_wgrad"
    return [(tag + ".g_w(rel)", (gw - ref).abs().max().item() / ref.abs().max().item(), 2e-3),
            (tag + ".g_b(rel)", (gb - masked.sum((0, 1, 2))).abs().max().item() / masked.sum((0, 1, 2)).abs().max().item(), 2e-3)]


def check_conv1_wgrad_simt(B: int = 8, seed: int = 7) -> List[Result]:
    return check_conv1_wgrad(B, seed, tc=False)


def check_conv2_fwd(B: int = 8, seed: int = 1) -> List[Result]:
    lib, dev = load(), "cuda"
    g = torch.Generator(device="cpu").manual_seed(seed)
    a1 = _bf(torch.rand(B, 14, 14, 32, generator=g)).to(dev)
    w = _bf(torch.randn(5, 5, 32, 64, generator=g) * 0.05).to(dev)
    b = (torch.randn(64, generator=g) * 0.1).to(dev)
    out = torch.zeros(B, 7, 7, 64, dtype=torch.bfloat16, device=dev)
    code = torch.zeros(B, 7, 7, 64, dtype=torch.uint8, device=dev)
    check(lib.dm_conv2_fwd(ptr(a1), ptr(w), ptr(b), ptr(out), ptr(code), B, stream_ptr()), "conv2_fwd")
    conv = F.conv2d(_nchw(a1), w.float().permute(3, 2, 0, 1), b, padding=2)
    ref = _nhwc(F.max_pool2d(F.relu(conv), 2, 2))
    err = (out.float() - ref).abs().max().item()
    idx, act = _decode_pool(code)
    win = _nhwc(conv).reshape(B, 7, 2, 7, 2, 64).permute(0, 1, 3, 5, 2, 4).reshape(B, 7, 7, 64, 4)
    sel = torch.gather(win, 4, idx[..., None])[..., 0]
    err_idx = (sel - win.max(dim=4).values).abs().max().item()
    bad_act = ((sel > 1e-3) & ~act) | ((sel < -1e-3) & act)
    return [("conv2_fwd.out", err, 0.05), ("conv2_fwd.argmax", err_idx, 2e-3),
            ("conv2_fwd.relu_flag", bad_act.float().sum().item(), 0.5)]


def check_conv2_dgrad(B: int = 8, seed: int = 2) -> List[Result]:
    lib, dev = load(), "cuda"
    g = torch.Generator(device="cpu").manual_seed(seed)
    dy = _bf(torch.randn(B, 14, 14, 64, generator=g) * 0.1).to(dev)
    w = _bf(torch.randn(5, 5, 32, 64, generator=g) * 0.05).to(dev)
    dx = torch.zeros(B, 14, 14, 32, dtype=torch.bfloat16, device=dev)
    check(lib.dm_conv2_dgrad(ptr(dy), ptr(w), ptr(dx), B, stream_ptr()), "conv2_dgrad")
    ref = _nhwc(torch.nn.grad.conv2d_input((B, 32, 14, 14), w.float().permute(3, 2, 0, 1), _nchw(dy), padding=2))
    return [("conv2_dgrad", (dx.float() - ref).abs().max().item(), 0.03)]


def check_conv2_wgrad(B: int = 8, seed: int = 3) -> List[Result]:
    lib, dev = load(), "cuda"
    g = torch.Generator(device="cpu").manual_seed(seed)
    a1 = _bf(torch.rand(B, 14, 14, 32, generator=g)).to(dev)
    dy = _bf(torch.randn(B, 14, 14, 64, generator=g) * 0.1).to(dev)
    gw = torch.zeros(5, 5, 32, 64, dtype=torch.float32, device=dev)
    check(lib.dm_conv2_wgrad(ptr(a1), ptr(dy), ptr(gw), B, stream_ptr()), "conv2_wgrad")
    ref = torch.nn.grad.conv2d_weight(_nchw(a1), (64, 32, 5, 5), _nchw(dy), padding=2).permute(2, 3, 1, 0)
    scale = ref.abs().max().item()
    return [("conv2_wgrad(rel)", (gw - ref).abs().max().item() / scale, 2e-3)]


def check_fc2_loss(B: int = 64, seed: int = 4) -> List[Result]:
    lib, dev = load(), "cuda"
    g = torch.Generator(device="cpu").manual_seed(seed)
    h_pre = torch.randn(B, 512, generator=g).to(dev)
    b1 = (torch.randn(512, generator=g) * 0.1).to(dev)
    w2 = (torch.randn(512, 10, generator=g) * 0.1).to(dev)
    b2 = (torch.randn(10, generator=g) * 0.1).to(dev)
    labels = torch.randint(0, 10, (B,), generator=g).to(dev)
    mix = dropout_seed_mix(123, 7, 2)
    step = torch.tensor([7], dtype=torch.int32, device=dev)
    mix0 = dropout_seed_mix(123, 0, 2)
    dh = torch.zeros(B, 512, dtype=torch.bfloat16, device=dev)
    gw2, gb2, gb1 = (torch.zeros(512, 10, device=dev), torch.zeros(10, device=dev), torch.zeros(512, device=dev))
    la = torch.zeros(2, device=dev)
    logits = torch.zeros(B, 10, device=dev)
    # the kernel consumes split-K partial sums: hand it three partials that add up to h_pre
    parts = torch.stack([h_pre * 0.5, h_pre * 0.25, h_pre * 0.25]).contiguous()
    h_act = torch.zeros(B, 512, device=dev)
    dl = torch.zeros(B, 12, device=dev)
    check(lib.dm_fc2_fwd_bwd(ptr(parts), ctypes.c_longlong(parts.stride(0)), 3, ptr(b1), ptr(w2), ptr(b2), ptr(labels),
                             ptr(dh), ptr(h_act), ptr(dl), ptr(la), ptr(logits), B, 1, ctypes.c_uint(mix0), ptr(step),
                             ctypes.c_float(0.5), stream_ptr()), "fc2_fwd_bwd")
    gw2.fill_(7.0), gb2.fill_(7.0), gb1.fill_(7.0)          # plain stores: stale contents must not matter
    check(lib.dm_fc2_wgrad(ptr(h_act), ptr(dl), ptr(dh), ptr(gw2), ptr(gb2), ptr(gb1), B, stream_ptr()), "fc2_wgrad")
    # reference
    hpre = (h_pre + b1).requires_grad_(True)
    keep = dropout_keep_mask(mix, B, 512, 0.5, device=dev)
    h = F.relu(hpre) * keep * 2.0
    w2r, b2r = w2.clone().requires_grad_(True), b2.clone().requires_grad_(True)
    lg = h @ w2r + b2r
    loss, acc = loss_and_accuracy(lg, labels)
    loss.backward()
    return [("fc2.logits", (logits - lg).abs().max().item(), 1e-3),
            ("fc2.loss", abs(la[0].item() - loss.item()), 1e-4), ("fc2.acc", abs(la[1].item() - acc.item()), 1e-6),
            ("fc2.dh", (dh.float() - hpre.grad).abs().max().item(), 2e-4 + 0.01 * hpre.grad.abs().max().item()),
            ("fc2.g_w2", (gw2 - w2r.grad).abs().max().item(), 1e-4), ("fc2.g_b2", (gb2 - b2r.grad).abs().max().item(), 1e-5),
            ("fc2.g_b1", (gb1 - hpre.grad.sum(0)).abs().max().item(), 1e-3)]


def check_fc1_dgrad_unpool(B: int = 200, seed: int = 6) -> List[Result]:
    """fc1 dgrad GEMM with the maxpool2/ReLU2 backward + conv2 bias gradient fused into its epilogue."""
    lib, dev = load(), "cuda"
    g = torch.Generator(device="cpu").manual_seed(seed)
    dh = _bf(torch.randn(B, 512, generator=g) * 0.1).to(dev)
    w1 = _bf(torch.randn(3136, 512, generator=g) * 0.05).to(dev)
    code = (torch.randint(0, 4, (B, 3136), generator=g) | (torch.randint(0, 2, (B, 3136), generator=g) << 2)).to(torch.uint8).to(dev)
    dy = torch.full((B, 14, 14, 64), 7.0, dtype=torch.bfloat16, device=dev)      # every element must be overwritten
    gb = torch.zeros(64, device=dev)
    check(lib.dm_fc1_dgrad_unpool(ptr(dh), ptr(w1), ptr(code), ptr(dy), ptr(gb), B, stream_ptr()), "fc1_dgrad_unpool")
    dx = dh.float() @ w1.float().t()                                              # [B,3136] = [B,7,7,64]
    idx, act = _decode_pool(code)
    masked = (dx * act).reshape(B, 7, 7, 64)
    ref = torch.zeros(B, 7, 2, 7, 2, 64, device=dev)
    idx = idx.reshape(B, 7, 7, 64)
    for q in range(4):
        ref[:, :, q >> 1, :, q & 1, :] = masked * (idx == q)
    ref = ref.reshape(B, 14, 14, 64)
    scale = dx.abs().max().item()
    return [("fc1_dgrad_unpool.dy(rel)", (dy.float() - ref).abs().max().item() / scale, 0.01),
            ("fc1_dgrad_unpool.g_bias(rel)", (gb - masked.sum((0, 1, 2))).abs().max().item() / masked.sum((0, 1, 2)).abs().max().item(), 2e-3)]


def _engine(B: int, seed: int = 5):
    from ..engine_cuda import CudaLeNetEngine
    ctx = ReplicaContext(0, 1, 0, torch.device("cuda", 0), "none")
    be = FusedBackend(ctx)
    return CudaLeNetEngine(B, be, seed=seed, rank=0, use_graph=False), be


# Per-tensor L2 bound of (gradients of the bf16-operand tensor-core step) vs (gradients of a PLAIN fp32 model, TF32 off).
# This is not a kernel-accuracy figure -- against the bf16-emulating reference every tensor agrees to <= 0.44 % (above) -- but
# the distance between bf16 and fp32 *training arithmetic*: activations rounded to bf16 flip ReLU / max-pool decisions, and the
# flips accumulate towards the input.  Measured on B200 (B = 64, seed 5; profiles/r2/): conv1_w 9.6 %, conv1_b 4.0 %,
# conv2_w 4.9 %, conv2_b 3.8 %, fc1_w 3.5 %, fc1_b 3.5 %, fc2_w 0.47 %, fc2_b 0.36 %.  Bounds = ~3x those: a wrong tap, a
# transposed tile or a dropped bias shows up as O(1).
FP32_GRAD_TOLS = {"conv1_weights": 0.30, "conv1_biases": 0.15, "conv2_weights": 0.15, "conv2_biases": 0.15,
                  "fc1_weights": 0.12, "fc1_biases": 0.12, "fc2_weights": 0.03, "fc2_biases": 0.03}


def check_end_to_end(B: int = 64, seed: int = 5) -> List[Result]:
    """Whole forward+backward through the CUDA engine vs torch autograd on the bf16-emulating reference."""
    eng, be = _engine(B, seed)
    spec, _ = get_model("lenet")
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = (torch.rand(B, 28, 28, 1, generator=g) - 0.5)
    y = torch.randint(0, 10, (B,), generator=g)
    eng.load_batch(x.numpy(), y.numpy())
    eng.forward_backward(0)
    torch.cuda.synchronize()
    loss, acc = eng.loss_acc()
    # reference on the same weights
    flat = eng.params.detach().clone().requires_grad_(True)
    mask = dropout_keep_mask(dropout_seed_mix(seed, 0, 0), B, 512, 0.5, device="cuda")
    logits = lenet_forward(spec.views(flat), x.cuda(), train=True, keep_mask=mask, emulate_bf16=True,
                           conv1_bf16=eng._conv1_tc)
    rloss, racc = loss_and_accuracy(logits, y.cuda())
    rloss.backward()
    out: List[Result] = [("e2e.loss", abs(loss - rloss.item()), 0.02 * max(1.0, abs(rloss.item()))),
                         ("e2e.acc", abs(acc - racc.item()), 2.0 / B + 1e-6)]
    gv, rv = spec.views(eng.grads), spec.views(flat.grad)
    for name in rv:
        scale = rv[name].abs().max().item() + 1e-8
        # measured on B200: <= 0.0044 for every tensor (profiles/r2); a wrong tap / transposed tile shows up as O(1)
        out.append(("e2e.grad.%s(rel)" % name, (gv[name] - rv[name]).abs().max().item() / scale, 0.02))
    # the same gradients against a PLAIN fp32 reference (no bf16 emulation anywhere): the remaining difference is the bf16
    # rounding of the tensor-core operands, bounded per tensor in the L2 norm
    flat32 = eng.params.detach().clone().requires_grad_(True)
    tf32_conv, tf32_mm = torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32
    torch.backends.cudnn.allow_tf32 = torch.backends.cuda.matmul.allow_tf32 = False      # a real fp32 reference
    try:
        logits32 = lenet_forward(spec.views(flat32), x.cuda(), train=True, keep_mask=mask, emulate_bf16=False, conv1_bf16=False)
        rloss32, _ = loss_and_accuracy(logits32, y.cuda())
        rloss32.backward()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32 = tf32_conv, tf32_mm
    r32 = spec.views(flat32.grad)
    for name in r32:
        num = (gv[name].double() - r32[name].double()).norm().item()
        den = r32[name].double().norm().item() + 1e-12
        out.append(("e2e.grad_vs_fp32.%s(L2 rel)" % name, num / den, FP32_GRAD_TOLS.get(name, 0.3)))
    out.append(("e2e.loss_vs_fp32", abs(loss - rloss32.item()), 0.02 * max(1.0, abs(rloss32.item()))))
    # padding of the gradient arena must stay zero (the fused kernel reduces the whole arena)
    out.append(("e2e.grad.padding", eng.grads[~spec.valid_mask().cuda()].abs().max().item(), 1e-12))
    return out


def check_bucketed_step_matches_single_kernel(B: int = 64, steps: int = 6, seed: int = 31, model: str = "lenet",
                                              hidden: int = 256) -> List[Result]:
    """One replica, whole graph-replayed training steps: bucketed aggregation (csrc/fused_bucket.cu: fc1 gradient as bf16,
    applied by the early kernel under the backward pass; small bucket by the late kernel) vs the single fused kernel."""
    import os
    from ..parallel.aggregators import SyncReplicasOptimizer
    from ..schedule import LearningRateSchedule
    g = torch.Generator(device="cpu").manual_seed(seed)
    xs = torch.rand(steps, B, 28, 28, generator=g) - 0.5
    ys = torch.randint(0, 10, (steps, B), generator=g)
    runs = {}
    old = os.environ.get("DMNIST_BUCKET")
    try:
        for mode in ("2", "0"):
            os.environ["DMNIST_BUCKET"] = mode
            if model == "lenet":
                eng, be = _engine(B, seed)
            else:
                from ..engine_cuda import CudaMlpEngine
                be = FusedBackend(ReplicaContext(0, 1, 0, torch.device("cuda", 0), "none"))
                eng = CudaMlpEngine(model, B, be, hidden=hidden, seed=seed, use_graph=True)
            eng.use_graph = True
            # lr 0.01: on random labels at lr 0.05 a 1e-6 relative change of the gradients (fp32 atomics summing in another
            # order) already moves the sixth loss by up to ~0.018, so the 0.02 loss bound below would sit inside that noise
            eng.attach_optimizer(SyncReplicasOptimizer(be, LearningRateSchedule(0.01, 2, 0.5), 1, 1))
            losses = []
            p_init = eng.params.clone()
            for s in range(steps):
                eng.load_batch(xs[s], ys[s])
                eng.train_step()
                losses.append(eng.loss_acc()[0])
                if s == 0:
                    torch.cuda.synchronize()
                    p_first = eng.params.clone()
            torch.cuda.synchronize()
            be.check_error()
            runs[mode] = (eng.params.clone(), eng.shadow.float().clone(), losses, eng.step_info().global_step,
                          bool(eng._bucket_v2), p_first, p_init)
    finally:
        if old is None:
            os.environ.pop("DMNIST_BUCKET", None)
        else:
            os.environ["DMNIST_BUCKET"] = old
    (p2, s2, l2, st2, v2, f2, i2), (p0, _s0, l0, st0, v0, f0, i0) = runs["2"], runs["0"]
    pmax = p0.abs().max().item()
    # after ONE step both paths applied the same gradient to the same weights, except that fc1's gradient went through bf16:
    # |difference| <= 2^-8 * |update| elementwise (+ fp32 atomics noise); later steps amplify it through ReLU / max-pool /
    # dropout decisions, so the final comparison is loose
    upd = (f0 - i0).abs()
    first_excess = ((f2 - f0).abs() - (upd * 2.0 ** -8 + 1e-6 * pmax)).max().item()
    tag = "bucket_v2" if model == "lenet" else "bucket_v2.%s" % model
    return [(tag + ".enabled", 0.0 if (v2 and not v0) else 1.0, 0.5),
            (tag + ".steps", abs(st2 - steps) + abs(st0 - steps), 0.5),
            (tag + ".first_step_excess", max(first_excess, 0.0) / pmax, 1e-6),
            (tag + ".first_update(rel, info)", upd.max().item() / pmax, 1e9),
            (tag + ".params_vs_single(rel)", (p2 - p0).abs().max().item() / pmax, 0.05),
            (tag + ".shadow(rel)", (s2 - p2).abs().max().item() / pmax, 0.01),
            (tag + ".loss", max(abs(a - b) for a, b in zip(l2, l0)), 0.02)]


def check_bucketed_mlp_step_matches_single_kernel() -> List[Result]:
    return (check_bucketed_step_matches_single_kernel(B=128, steps=4, seed=41, model="mlp3", hidden=256)
            + check_bucketed_step_matches_single_kernel(B=96, steps=3, seed=42, model="mlp2", hidden=128))


def check_training_reduces_loss(B: int = 128, steps: int = 40) -> List[Result]:
    from ..data import make_synthetic_mnist
    from ..parallel.aggregators import SyncReplicasOptimizer
    from ..schedule import LearningRateSchedule
    eng, be = _engine(B, 11)
    eng.use_graph = True
    opt = SyncReplicasOptimizer(be, LearningRateSchedule(0.05, 1000, 1.0), 1, 1)
    eng.attach_optimizer(opt)
    trx, try_, _, _ = make_synthetic_mnist(B * 8, 16, seed=3)
    losses = []
    for s in range(steps):
        i = (s % 8) * B
        eng.load_batch(trx[i:i + B], try_[i:i + B])
        eng.train_step()
        losses.append(eng.loss_acc()[0])
    info = eng.step_info()
    first, last = sum(losses[:5]) / 5, sum(losses[-5:]) / 5
    return [("train.loss_ratio(last/first)", last / first, 0.7), ("train.steps_missing", abs(info.global_step - steps), 0.5),
            ("train.nan", float(any(l != l for l in losses)), 0.5)]


def check_mlp_end_to_end(model: str = "mlp3", B: int = 256, hidden: int = 256, seed: int = 21) -> List[Result]:
    """CudaMlpEngine forward+backward vs torch autograd on the bf16-emulating reference."""
    from ..engine_cuda import CudaMlpEngine
    from ..models import mlp_forward
    ctx = ReplicaContext(0, 1, 0, torch.device("cuda", 0), "none")
    eng = CudaMlpEngine(model, B, FusedBackend(ctx), hidden=hidden, seed=seed, use_graph=False)
    g = torch.Generator(device="cpu").manual_seed(seed)
    x = (torch.rand(B, 28, 28, 1, generator=g) - 0.5)
    y = torch.randint(0, 10, (B,), generator=g)
    eng.load_batch(x.numpy(), y.numpy())
    eng.forward_backward(0)
    torch.cuda.synchronize()
    loss, acc = eng.loss_acc()
    flat = eng.params.detach().clone().requires_grad_(True)
    logits = mlp_forward(eng.spec.views(flat), x.cuda(), emulate_bf16=True)
    rloss, racc = loss_and_accuracy(logits, y.cuda())
    rloss.backward()
    out: List[Result] = [("%s.loss" % model, abs(loss - rloss.item()), 0.02 * max(1.0, abs(rloss.item()))),
                         ("%s.acc" % model, abs(acc - racc.item()), 2.0 / B + 1e-6)]
    gv, rv = eng.spec.views(eng.grads), eng.spec.views(flat.grad)
    for name in rv:
        scale = rv[name].abs().max().item() + 1e-8
        out.append(("%s.grad.%s(rel)" % (model, name), (gv[name] - rv[name]).abs().max().item() / scale, 0.06))
    out.append(("%s.grad.padding" % model, eng.grads[~eng.spec.valid_mask().cuda()].abs().max().item(), 1e-12))
    el, ea = eng.evaluate(x.numpy(), y.numpy())
    out.append(("%s.eval_loss" % model, abs(el - rloss.item()), 0.02 * max(1.0, abs(rloss.item()))))
    return out


def check_mlp2_end_to_end() -> List[Result]:
    return check_mlp_end_to_end("mlp2", B=96, hidden=128, seed=22)


ALL_CHECKS = [check_conv1_fwd, check_conv1_fwd_tc, check_conv1_wgrad, check_conv1_wgrad_simt, check_conv2_fwd, check_conv2_dgrad, check_conv2_wgrad, check_fc2_loss, check_fc1_dgrad_unpool,
              check_end_to_end, check_bucketed_step_matches_single_kernel, check_bucketed_mlp_step_matches_single_kernel,
              check_training_reduces_loss, check_mlp_end_to_end, check_mlp2_end_to_end]
