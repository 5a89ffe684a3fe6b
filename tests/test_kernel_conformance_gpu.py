"""Single-GPU kernels against float64 references at the batch sizes training and evaluation run.

Every check hands the kernel's exact operands to a float64 computation (tests/_fp64_ref.py) and judges the output by
the derived rounding bound, so a dropped tap, a wrong tile or a misplaced bias fails even where an fp32 comparison with
an absolute tolerance would not.  Batches 1000 and 1024 are the evaluator's and the 8-GPU configs' sizes: there the
persistent tensor-core kernels walk ~14 tiles per CTA, and with ``dm_set_max_ctas(8)`` the ones that honour it walk
tens of tiles per CTA even at small batches.  Outputs are surrounded by sentinels: what the code documents as fully
written must hold no sentinel afterwards, and rows beyond the batch must stay untouched.

The worst err / bound measured on a B200 is recorded beside each check.
"""
import ctypes

import numpy as np
import pytest
import torch

import _fp64_ref as R

pytestmark = pytest.mark.gpu

BATCHES = [1, 3, 37, 256, 1000, 1024]
NAN = float("nan")
SENT = 0xAB                      # uint8 sentinel: not a valid pooling code (codes are 0..7)


def _lib():
    from distributedmnist_b200.ops.lib import load
    return load()


def _check(rc, what):
    from distributedmnist_b200.ops.lib import check
    check(rc, what)


def _p(t):
    from distributedmnist_b200.ops.lib import ptr
    return ptr(t)


def _sp():
    from distributedmnist_b200.ops.lib import stream_ptr
    return stream_ptr()


def _gen(seed):
    return torch.Generator(device="cuda").manual_seed(seed)


@pytest.fixture
def max_ctas():
    """dm_set_max_ctas is process-global: whatever a test sets is put back to the full 148 SMs."""
    lib = _lib()
    try:
        yield lib.dm_set_max_ctas
    finally:
        lib.dm_set_max_ctas(148)


def _pool_ok(res, tag):
    # the pooled output within its bound; no argmax / ReLU decision contradicting the reference beyond the bound;
    # decisions the bound cannot settle (near-ties) are rare.  conv2's bound (800 terms) is ~1e-3 of values of order 1,
    # so on a B200 about 0.7 % of its windows hold an unresolvable near-tie and 0.3 % a near-zero ReLU input (random
    # inputs and the trained-weights evaluation alike); conv1 has almost none
    assert res["ratio"] <= 1.0, (tag, res)
    assert res["bad_idx"] == 0 and res["bad_act"] == 0, (tag, res)
    assert res["amb_idx"] <= 8 + 0.02 * res["count"] and res["amb_act"] <= 8 + 0.01 * res["count"], (tag, res)


# ---------------------------------------------------------------------------------------------------------------------
# LeNet kernels
# ---------------------------------------------------------------------------------------------------------------------
def run_conv1_fwd(B, tc, seed=0):
    lib = _lib()
    g = _gen(seed)
    x = torch.rand(B, 28, 28, generator=g, device="cuda") - 0.5
    w = torch.randn(25, 32, generator=g, device="cuda") * 0.1
    b = torch.randn(32, generator=g, device="cuda") * 0.1
    out = torch.full((B + 2, 14, 14, 32), NAN, dtype=torch.bfloat16, device="cuda")
    code = torch.full((B + 2, 14, 14, 32), SENT, dtype=torch.uint8, device="cuda")
    junk = torch.ones(1000, device="cuda")
    fn = lib.dm_conv1_fwd_tc if tc else lib.dm_conv1_fwd
    _check(fn(_p(x), _p(w), _p(b), _p(out), _p(code), B, _p(junk), 1000, ctypes.c_void_p(0), 0, ctypes.c_void_p(0), 0,
              _sp()), "conv1_fwd")
    torch.cuda.synchronize()
    if tc:      # the tensor-core path reads bf16 operands
        x, w = x.to(torch.bfloat16), w.to(torch.bfloat16)
    conv, S = R.conv_fwd(x[..., None], w.view(5, 5, 1, 32))
    res = R.check_pool_relu(conv, S, b, 25, out[:B], code[:B])
    assert not torch.isnan(out[:B].float()).any() and bool((code[:B] <= 7).all()), "a1/code1 not fully written"
    assert torch.isnan(out[B:].float()).all() and bool((code[B:] == SENT).all()), "rows beyond the batch written"
    assert float(junk.abs().max()) == 0.0, "zero range not cleared"
    return res


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("tc", [False, True], ids=["simt", "tc"])
def test_conv1_fwd(B, tc):
    # measured worst err/bound on a B200 (1000 W): 0.998 for both kernels (a bf16 output: its rounding alone reaches the
    # bound for values exactly halfway between two bf16 numbers); no argmax / ReLU decision contradicted
    res = run_conv1_fwd(B, tc, seed=B)
    print("RATIO conv1_fwd tc=%d B=%d" % (tc, B), res)
    _pool_ok(res, "conv1_fwd tc=%d B=%d" % (tc, B))


def _codes(shape, g):
    idx = torch.randint(0, 4, shape, generator=g, device="cuda")
    act = torch.randint(0, 2, shape, generator=g, device="cuda")
    return (idx | (act << 2)).to(torch.uint8)


def run_conv1_wgrad(B, tc, seed=0):
    lib = _lib()
    g = _gen(seed)
    x = torch.rand(B, 28, 28, generator=g, device="cuda") - 0.5
    dpool = (torch.randn(B, 14, 14, 32, generator=g, device="cuda") * 0.1).to(torch.bfloat16)
    code = _codes((B, 14, 14, 32), g)
    gw = torch.zeros(25, 32, device="cuda")
    gb = torch.zeros(32, device="cuda")
    fn = lib.dm_conv1_wgrad_tc if tc else lib.dm_conv1_wgrad
    _check(fn(_p(x), _p(dpool), _p(code), _p(gw), _p(gb), B, _sp()), "conv1_wgrad")
    torch.cuda.synchronize()
    xr = x.to(torch.bfloat16) if tc else x
    dy = R.unpool(dpool.double(), code)
    ref, S = R.conv_wgrad(xr[..., None], dy)
    n = B * 196 + 600                    # pixels + per-CTA partials
    r_w = R.worst_ratio(gw, ref.view(25, 32), R.acc_bound(S.view(25, 32), n))
    r_b = R.worst_ratio(gb, dy.sum((0, 1, 2)), R.acc_bound(dy.abs().sum((0, 1, 2)), n))
    return max(r_w, r_b)


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("tc", [False, True], ids=["simt", "tc"])
def test_conv1_wgrad(B, tc):
    # measured worst err/bound on a B200 (1000 W): SIMT 5.0e-4, tcgen05 4.6e-4
    r = run_conv1_wgrad(B, tc, seed=100 + B)
    print("RATIO conv1_wgrad tc=%d B=%d" % (tc, B), r)
    assert r <= 1.0, (B, tc, r)


def run_conv2_fwd(B, seed=0):
    lib = _lib()
    g = _gen(seed)
    a1 = torch.rand(B, 14, 14, 32, generator=g, device="cuda").to(torch.bfloat16)
    w = (torch.randn(5, 5, 32, 64, generator=g, device="cuda") * 0.05).to(torch.bfloat16)
    b = torch.randn(64, generator=g, device="cuda") * 0.1
    out = torch.full((B + 2, 7, 7, 64), NAN, dtype=torch.bfloat16, device="cuda")
    code = torch.full((B + 2, 7, 7, 64), SENT, dtype=torch.uint8, device="cuda")
    _check(lib.dm_conv2_fwd(_p(a1), _p(w), _p(b), _p(out), _p(code), B, _sp()), "conv2_fwd")
    torch.cuda.synchronize()
    conv, S = R.conv_fwd(a1, w)
    res = R.check_pool_relu(conv, S, b, 800, out[:B], code[:B])
    assert not torch.isnan(out[:B].float()).any() and bool((code[:B] <= 7).all()), "a2/code2 not fully written"
    assert torch.isnan(out[B:].float()).all() and bool((code[B:] == SENT).all()), "rows beyond the batch written"
    return res


@pytest.mark.parametrize("B", BATCHES)
def test_conv2_fwd(B):
    # measured worst err/bound on a B200 (1000 W): 0.80 (a bf16 output); no argmax / ReLU decision contradicted;
    # near-ties 0.72 % of windows, near-zero ReLU inputs 0.34 %
    res = run_conv2_fwd(B, seed=200 + B)
    print("RATIO conv2_fwd B=%d" % B, res)
    _pool_ok(res, "conv2_fwd B=%d" % B)


def run_conv2_dgrad(B, seed=0):
    lib = _lib()
    g = _gen(seed)
    dy = (torch.randn(B, 14, 14, 64, generator=g, device="cuda") * 0.1).to(torch.bfloat16)
    w = (torch.randn(5, 5, 32, 64, generator=g, device="cuda") * 0.05).to(torch.bfloat16)
    dx = torch.full((B + 2, 14, 14, 32), NAN, dtype=torch.bfloat16, device="cuda")
    _check(lib.dm_conv2_dgrad(_p(dy), _p(w), _p(dx), B, _sp()), "conv2_dgrad")
    torch.cuda.synchronize()
    assert not torch.isnan(dx[:B].float()).any(), "dx1 not fully written"
    assert torch.isnan(dx[B:].float()).all(), "rows beyond the batch written"
    ref, S = R.conv_dgrad(dy, w)
    return R.worst_ratio(dx[:B], ref, R.bf16_out_bound(ref, R.acc_bound(S, 1600)))


def run_conv2_wgrad(B, seed=0):
    lib = _lib()
    g = _gen(seed)
    a1 = torch.rand(B, 14, 14, 32, generator=g, device="cuda").to(torch.bfloat16)
    dy = (torch.randn(B, 14, 14, 64, generator=g, device="cuda") * 0.1).to(torch.bfloat16)
    gw = torch.zeros(5, 5, 32, 64, device="cuda")
    _check(lib.dm_conv2_wgrad(_p(a1), _p(dy), _p(gw), B, _sp()), "conv2_wgrad")
    torch.cuda.synchronize()
    ref, S = R.conv_wgrad(a1, dy)
    return R.worst_ratio(gw, ref, R.acc_bound(S, B * 196 + 148))


@pytest.mark.parametrize("B", BATCHES)
def test_conv2_dgrad_wgrad(B):
    # measured worst err/bound on a B200 (1000 W): dgrad 0.81 (bf16 output), wgrad 2.3e-3
    r_d, r_w = run_conv2_dgrad(B, seed=300 + B), run_conv2_wgrad(B, seed=400 + B)
    print("RATIO conv2 dgrad/wgrad B=%d" % B, r_d, r_w)
    assert r_d <= 1.0 and r_w <= 1.0, (B, r_d, r_w)


@pytest.mark.parametrize("B", [3, 37, 256])
def test_deep_persistent_loops_with_8_ctas(B, max_ctas):
    """dm_set_max_ctas(8): conv2 dgrad / wgrad and the tcgen05 conv1 wgrad walk tens of tiles per CTA, so the mbarrier
    phases and the TMEM double buffer wrap many times.  Measured worst err/bound on a B200 (1000 W): conv2 dgrad 0.77
    (bf16 output), conv2 wgrad 2.6e-3, conv1 wgrad 2.8e-4."""
    assert max_ctas(8) == 8
    r = [run_conv2_dgrad(B, seed=500 + B), run_conv2_wgrad(B, seed=600 + B), run_conv1_wgrad(B, True, seed=700 + B)]
    print("RATIO 8 CTAs B=%d" % B, r)
    assert max(r) <= 1.0, (B, r)


def run_fc1_dgrad_unpool(B, fused, seed=0):
    lib = _lib()
    g = _gen(seed)
    dh = (torch.randn(B, 512, generator=g, device="cuda") * 0.1).to(torch.bfloat16)
    w1 = (torch.randn(3136, 512, generator=g, device="cuda") * 0.05).to(torch.bfloat16)
    code = _codes((B, 3136), g)
    dy = torch.full((B + 2, 14, 14, 64), NAN, dtype=torch.bfloat16, device="cuda")
    gb = torch.zeros(64, device="cuda")
    dxfc_ref, S = dh.double() @ w1.double().t(), dh.double().abs() @ w1.double().abs().t()
    if fused:
        _check(lib.dm_fc1_dgrad_unpool(_p(dh), _p(w1), _p(code), _p(dy), _p(gb), B, _sp()), "fc1_dgrad_unpool")
        e = R.acc_bound(S, 512)
        vb = R.bf16_out_bound(dxfc_ref, e)
        gsum_ref = dxfc_ref
    else:
        # the unfused path: the bf16 dgrad output is given; the unpool kernel only scatters it and sums the bias gradient
        dxfc = dxfc_ref.to(torch.bfloat16)
        _check(lib.dm_unpool2(_p(dxfc), _p(code), _p(dy), _p(gb), B, _sp()), "unpool2")
        dxfc_ref, e = dxfc.double(), torch.zeros_like(S)
        vb = e
        gsum_ref = dxfc_ref
    torch.cuda.synchronize()
    assert not torch.isnan(dy[:B].float()).any(), "dy2 not fully written (zeros included)"
    assert torch.isnan(dy[B:].float()).all(), "rows beyond the batch written"
    ref = R.unpool(dxfc_ref.view(B, 7, 7, 64), code.view(B, 7, 7, 64))
    bound = R.unpool(vb.view(B, 7, 7, 64), code.view(B, 7, 7, 64))       # zero (exact) where nothing is scattered
    r_dy = R.worst_ratio(dy[:B], ref, bound)
    act = ((code >> 2) & 1).bool()
    gref = torch.where(act, gsum_ref, 0.0).view(B, 49, 64).sum((0, 1))
    gS = torch.where(act, S if fused else gsum_ref.abs(), 0.0).view(B, 49, 64).sum((0, 1))
    r_gb = R.worst_ratio(gb, gref, R.acc_bound(gS, (512 if fused else 0) + B * 49 + 600))
    return r_dy, r_gb


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("fused", [True, False], ids=["fused_epilogue", "unpool2"])
def test_fc1_dgrad_unpool_and_unpool2(B, fused):
    # measured worst err/bound on a B200 (1000 W): fused dy2 0.92 (bf16 output), bias gradient 1.2e-4; unpool2 exact
    # scatter, bias gradient 1.1e-4
    r = run_fc1_dgrad_unpool(B, fused, seed=800 + B)
    print("RATIO fc1_dgrad_unpool fused=%d B=%d" % (fused, B), r)
    assert max(r) <= 1.0, (B, fused, r)


def _xent_checks(logits, labels, la, B, tag):
    """Loss / accuracy accumulators against the float64 loss of the kernel's own logits."""
    row, row_bound, p, p_bound, hits = R.xent_ref(logits, labels)
    lb = float(row_bound.mean() + (R.gamma(B + 2) + 3 * R.U) * row.abs().mean())
    assert abs(float(la[0]) - float(row.mean())) <= lb, (tag, float(la[0]), float(row.mean()), lb)
    assert round(float(la[1]) * B) == hits, (tag, float(la[1]) * B, hits)
    return row, p, p_bound


def run_fc2(B, train, keep, seed=0, zero_w=False):
    from distributedmnist_b200.models import dropout_keep_mask, dropout_seed_mix
    lib = _lib()
    g = _gen(seed)
    splits = 7
    parts = torch.randn(splits, B, 512, generator=g, device="cuda") * 0.3
    b1 = torch.randn(512, generator=g, device="cuda") * 0.1
    w2 = torch.randn(512, 10, generator=g, device="cuda") * 0.1
    b2 = torch.randn(10, generator=g, device="cuda") * 0.1
    if zero_w:                                 # every logit equal: the tie goes to class 0
        w2.zero_(), b2.fill_(0.25)
    labels = torch.randint(0, 10, (B,), generator=g, device="cuda")
    seed_, step, rank = 1234, 5, 3
    step_t = torch.tensor([step], dtype=torch.int32, device="cuda")
    dh = torch.full((B + 1, 512), NAN, dtype=torch.bfloat16, device="cuda")
    h_act = torch.full((B + 1, 512), NAN, device="cuda")
    dl = torch.full((B + 1, 12), NAN, device="cuda")
    la = torch.zeros(2, device="cuda")
    logits = torch.full((B + 1, 10), NAN, device="cuda")
    _check(lib.dm_fc2_fwd_bwd(_p(parts), ctypes.c_longlong(parts.stride(0)), splits, _p(b1), _p(w2), _p(b2), _p(labels),
                              _p(dh), _p(h_act), _p(dl), _p(la), _p(logits), B, int(train),
                              ctypes.c_uint(dropout_seed_mix(seed_, 0, rank)), _p(step_t), ctypes.c_float(keep), _sp()),
           "fc2_fwd_bwd")
    torch.cuda.synchronize()
    tag = "fc2 B=%d train=%d keep=%g" % (B, train, keep)
    assert not torch.isnan(logits[:B]).any() and torch.isnan(logits[B:]).all(), tag
    # stage 1: hp = b1 + sum of the split-K partials, ReLU, dropout (train), 1/keep
    hp = b1.double() + parts.double().sum(0)
    e_hp = R.acc_bound(b1.double().abs() + parts.double().abs().sum(0), 8 + 1)
    mask = dropout_keep_mask(dropout_seed_mix(seed_, step, rank), B, 512, keep, device="cuda") if train \
        else torch.ones(B, 512, dtype=torch.bool, device="cuda")
    kp = keep if train else 1.0
    h_ref = torch.where(mask, hp.clamp_min(0), 0.0) / kp
    e_h = (e_hp / kp) * (1 + 2 * R.U) + 2 * R.U * h_ref.abs()
    amb = hp.abs() <= e_hp
    e_h = torch.where(amb, 2 * e_h + hp.abs() / kp, e_h)        # a ReLU decision the bound cannot settle: either way
    out = {}
    if train:
        assert not torch.isnan(h_act[:B]).any() and torch.isnan(h_act[B:]).all(), tag
        out["h"] = R.worst_ratio(h_act[:B], h_ref, e_h)
        # the dropout mask itself: wherever ReLU is clearly on, h != 0 exactly where the mask keeps
        on = hp > e_hp
        assert bool(((h_act[:B] != 0) == mask)[on].all()), tag + ": dropout mask differs from dropout_keep_mask"
        h_used, e_used = h_act[:B].double(), torch.zeros_like(e_h)     # judge fc2 on the kernel's own activations
    else:
        assert torch.isnan(h_act).all() and torch.isnan(dl).all() and torch.isnan(dh.float()).all(), \
            tag + ": eval wrote a training output"
        h_used, e_used = h_ref, e_h
    # stage 2: logits
    ref = h_used @ w2.double() + b2.double()
    S = (h_used.abs() + e_used) @ w2.double().abs() + b2.double().abs()
    out["logits"] = R.worst_ratio(logits[:B], ref, R.acc_bound(S, 513) + e_used @ w2.double().abs())
    # stage 3: loss / accuracy from the kernel's logits
    row, p, p_bound = _xent_checks(logits[:B], labels, la, B, tag)
    if zero_w:
        assert round(float(la[1]) * B) == int((labels == 0).sum()), tag + ": tie not resolved to class 0"
    if train:
        # stage 4: dlogits, then dh from the kernel's own dlogits
        assert not torch.isnan(dl[:B]).any() and torch.isnan(dl[B:]).all(), tag
        assert float(dl[:B, 10:].abs().max()) == 0.0, tag + ": dlogits padding columns not zero"
        onehot = torch.nn.functional.one_hot(labels, 10).double()
        dl_ref = (p - onehot) / B
        out["dl"] = R.worst_ratio(dl[:B, :10], dl_ref, p_bound / B + 3 * R.U * dl_ref.abs())
        dlk = dl[:B, :10].double()
        dref = torch.where(h_act[:B] != 0, (dlk @ w2.double().t()) / keep, 0.0)
        dS = (dlk.abs() @ w2.double().abs().t()) / keep
        assert not torch.isnan(dh[:B].float()).any() and torch.isnan(dh[B:].float()).all(), tag
        out["dh"] = R.worst_ratio(dh[:B], dref, R.bf16_out_bound(dref, R.acc_bound(dS, 12)))
    return out, (h_act, dl, dh, labels)


@pytest.mark.parametrize("B", BATCHES)
@pytest.mark.parametrize("train", [1, 0], ids=["train", "eval"])
@pytest.mark.parametrize("keep", [0.5, 0.75, 1.0])
def test_fc2_fwd_bwd(B, train, keep):
    # measured worst err/bound on a B200 (1000 W): h 0.20, logits 1.1e-3, dlogits 0.36, dh 1.00 (bf16 output: the
    # rounding of values exactly halfway between two bf16 numbers)
    out, _ = run_fc2(B, train, keep, seed=900 + B)
    print("RATIO fc2 B=%d train=%d keep=%g" % (B, train, keep), out)
    assert max(out.values()) <= 1.0, (B, train, keep, out)


def test_fc2_fwd_bwd_tie_goes_to_class_zero():
    run_fc2(37, 0, 0.5, seed=1, zero_w=True)
    run_fc2(37, 1, 0.5, seed=1, zero_w=True)


@pytest.mark.parametrize("B", BATCHES)
def test_fc2_wgrad(B):
    """From the fc2_fwd_bwd outputs of the same batch.  Measured worst err/bound on a B200 (1000 W): g_w2 0.17,
    g_b2 0.12, g_b1 2.6e-4."""
    lib = _lib()
    _, (h_act, dl, dh, _) = run_fc2(B, 1, 0.5, seed=950 + B)
    gw2 = torch.full((512, 10), 7.0, device="cuda")             # plain stores: stale contents must not matter
    gb2 = torch.full((10,), 7.0, device="cuda")
    gb1 = torch.full((512,), 7.0, device="cuda")
    _check(lib.dm_fc2_wgrad(_p(h_act), _p(dl), _p(dh), _p(gw2), _p(gb2), _p(gb1), B, _sp()), "fc2_wgrad")
    torch.cuda.synchronize()
    h, d, dh64 = h_act[:B].double(), dl[:B, :10].double(), dh[:B].double()
    n = B + 2
    r = [R.worst_ratio(gw2, h.t() @ d, R.acc_bound(h.abs().t() @ d.abs(), n)),
         R.worst_ratio(gb2, d.sum(0), R.acc_bound(d.abs().sum(0), n)),
         R.worst_ratio(gb1, dh64.sum(0), R.acc_bound(dh64.abs().sum(0), n))]
    print("RATIO fc2_wgrad B=%d" % B, r)
    assert max(r) <= 1.0, (B, r)


# ---------------------------------------------------------------------------------------------------------------------
# MLP SIMT kernels
# ---------------------------------------------------------------------------------------------------------------------
def run_dense10(B, H, train, seed=0, w_scale=0.05, zero_w=False):
    lib = _lib()
    g = _gen(seed)
    h = torch.randn(B, H, generator=g, device="cuda").clamp_min(0).to(torch.bfloat16)
    w = torch.randn(H, 10, generator=g, device="cuda") * w_scale
    b = torch.randn(10, generator=g, device="cuda") * 0.1
    if zero_w:
        w.zero_(), b.fill_(-0.5)
    labels = torch.randint(0, 10, (B,), generator=g, device="cuda")
    dh = torch.full((B + 1, H), NAN, dtype=torch.bfloat16, device="cuda")
    dl_pad = torch.full((B + 1, 64), NAN, dtype=torch.bfloat16, device="cuda")
    gb0 = torch.randn(10, generator=g, device="cuda")
    gb = gb0.clone()
    la = torch.zeros(2, device="cuda")
    logits = torch.full((B, 10), NAN, device="cuda")
    _check(lib.dm_dense10_xent(_p(h), _p(w), _p(b), _p(labels), _p(dh), _p(dl_pad), _p(gb), _p(la), _p(logits), B, H,
                               int(train), _sp()), "dense10_xent")
    torch.cuda.synchronize()
    tag = "dense10 B=%d H=%d train=%d" % (B, H, train)
    assert not torch.isnan(logits).any(), tag
    ref = h.double() @ w.double() + b.double()
    S = h.double().abs() @ w.double().abs() + b.double().abs()
    out = {"logits": R.worst_ratio(logits, ref, R.acc_bound(S, H + 1))}
    row, p, p_bound = _xent_checks(logits, labels, la, B, tag)
    assert torch.isfinite(row).all() and bool(torch.isfinite(la).all()), tag
    if zero_w:
        assert round(float(la[1]) * B) == int((labels == 0).sum()), tag + ": tie not resolved to class 0"
    if not train:
        assert torch.isnan(dh.float()).all() and torch.isnan(dl_pad.float()).all(), tag + ": eval wrote dh / dl"
        assert torch.equal(gb, gb0), tag + ": eval touched g_b"
        return out
    onehot = torch.nn.functional.one_hot(labels, 10).double()
    dl_ref = (p - onehot) / B
    dl_err = p_bound / B + 3 * R.U * dl_ref.abs()
    assert not torch.isnan(dl_pad[:B, :16].float()).any(), tag
    assert float(dl_pad[:B, 10:16].float().abs().max()) == 0.0, tag + ": dl_pad columns 10-15 not zero"
    assert torch.isnan(dl_pad[:B, 16:].float()).all() and torch.isnan(dl_pad[B:].float()).all(), tag + ": dl_pad guard"
    out["dl_pad"] = R.worst_ratio(dl_pad[:B, :10], dl_ref, R.bf16_out_bound(dl_ref, dl_err))
    wa = w.double().abs()
    dref = torch.where(h.double() > 0, dl_ref @ w.double().t(), 0.0)
    e = R.acc_bound(dl_ref.abs() @ wa.t() + dl_err @ wa.t(), 10) + dl_err @ wa.t()
    assert not torch.isnan(dh[:B].float()).any() and torch.isnan(dh[B:].float()).all(), tag
    out["dh"] = R.worst_ratio(dh[:B], dref, torch.where(h.double() > 0, R.bf16_out_bound(dref, e), 0.0))
    gref = gb0.double() + dl_ref.sum(0)
    out["g_b"] = R.worst_ratio(gb, gref, R.acc_bound(gb0.double().abs() + dl_ref.abs().sum(0), B + 160)
                               + dl_err.sum(0))
    return out


MLP_SHAPES = [(1, 64), (7, 128), (96, 128), (256, 256), (8192, 1024), (8192, 4096)]


@pytest.mark.parametrize("B,H", MLP_SHAPES)
@pytest.mark.parametrize("train", [1, 0], ids=["train", "eval"])
def test_dense10_xent(B, H, train):
    # measured worst err/bound on a B200 (1000 W): logits 6.7e-3, g_b 5.5e-3, dl_pad and dh 1.00 (bf16 outputs: the
    # rounding of values exactly halfway between two bf16 numbers)
    out = run_dense10(B, H, train, seed=B + H)
    print("RATIO dense10 B=%d H=%d train=%d" % (B, H, train), out)
    assert max(out.values()) <= 1.0, (B, H, train, out)


def test_dense10_xent_edges():
    """Zero weights + equal biases: the tie goes to class 0 (as in fc2_fwd_bwd).  Logits of ~1e4: the loss stays
    finite and matches the float64 log-sum-exp of the kernel's logits."""
    run_dense10(96, 128, 0, seed=5, zero_w=True)
    run_dense10(96, 128, 1, seed=5, zero_w=True)
    out = run_dense10(64, 256, 1, seed=6, w_scale=300.0)
    assert max(out.values()) <= 1.0, out


@pytest.mark.parametrize("B", [1, 255, 257, 8192, 20000])
@pytest.mark.parametrize("H", [2, 64, 130, 1024])
def test_relu_bwd_colsum(B, H):
    """h null (bias gradient only), separate output, in place.  At B = 20000 the 64-slab cap gives 313 rows per CTA.
    Measured worst err/bound of the bias gradient on a B200 (1000 W): 6.2e-3; dpre is exact."""
    lib = _lib()
    g = _gen(B * 7 + H)
    dh = (torch.randn(B, H, generator=g, device="cuda") * 0.1).to(torch.bfloat16)
    h = torch.randn(B, H, generator=g, device="cuda").clamp_min(0).to(torch.bfloat16)
    gb0 = torch.randn(H, generator=g, device="cuda")
    worst = 0.0
    for mode in ("no_mask", "separate", "in_place"):
        gb = gb0.clone()
        d_in = dh.clone()
        if mode == "no_mask":
            _check(lib.dm_relu_bwd_colsum(_p(d_in), ctypes.c_void_p(0), ctypes.c_void_p(0), _p(gb), B, H, _sp()), mode)
            dref = dh.double()
        elif mode == "separate":
            dpre = torch.full((B + 1, H), NAN, dtype=torch.bfloat16, device="cuda")
            _check(lib.dm_relu_bwd_colsum(_p(d_in), _p(h), _p(dpre), _p(gb), B, H, _sp()), mode)
            dref = torch.where(h.double() > 0, dh.double(), 0.0)
            torch.cuda.synchronize()
            assert torch.equal(dpre[:B].double(), dref), (B, H, mode)
            assert torch.isnan(dpre[B:].float()).all(), (B, H, mode)
        else:
            _check(lib.dm_relu_bwd_colsum(_p(d_in), _p(h), _p(d_in), _p(gb), B, H, _sp()), mode)
            dref = torch.where(h.double() > 0, dh.double(), 0.0)
            torch.cuda.synchronize()
            assert torch.equal(d_in.double(), dref), (B, H, mode)
        torch.cuda.synchronize()
        if mode == "no_mask":
            assert torch.equal(d_in, dh), "h == null must not write"
        r = R.worst_ratio(gb, gb0.double() + dref.sum(0), R.acc_bound(gb0.double().abs() + dref.abs().sum(0), B + 80))
        assert r <= 1.0, (B, H, mode, r)
        worst = max(worst, r)
    print("RATIO relu_bwd_colsum B=%d H=%d" % (B, H), worst)


def test_relu_bwd_colsum_odd_width_is_refused():
    lib = _lib()
    t = torch.zeros(4, 3, dtype=torch.bfloat16, device="cuda")
    gb = torch.zeros(3, device="cuda")
    assert lib.dm_relu_bwd_colsum(_p(t), ctypes.c_void_p(0), ctypes.c_void_p(0), _p(gb), 4, 3, _sp()) == -1


def test_f32_to_bf16_bit_exact():
    """The input conversion and the bf16 weight shadow: bit-identical to torch's round-to-nearest-even conversion."""
    lib = _lib()
    g = _gen(11)
    rnd = torch.randn(148 * 512 * 4 * 2, generator=g, device="cuda") * torch.exp2(
        torch.randint(-60, 60, (148 * 512 * 4 * 2,), generator=g, device="cuda").float())
    bits = torch.randint(0, 1 << 16, (4096,), generator=g, device="cuda", dtype=torch.int32)
    def f32(lo):
        v = (bits.long() << 16) | lo
        return torch.where(v >= 1 << 31, v - (1 << 32), v).to(torch.int32).view(torch.float32)
    ties = f32(0x8000)                                          # exactly halfway between two bf16 values (odd and even)
    near = f32(0x7FFF)
    special = torch.tensor([0.0, -0.0, float("inf"), float("-inf"), 1e-40, -1e-40, 1.4e-45, 1.1754942e-38,
                            3.3961e38, -3.3961e38, 3.3895e38, 65504.0, 1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8],
                           device="cuda")
    x = torch.cat([rnd, ties, near, special, torch.full((6,), NAN, device="cuda")])
    x = x[: x.numel() // 4 * 4].contiguous()
    dst = torch.zeros(x.numel() + 8, dtype=torch.bfloat16, device="cuda")
    dst[x.numel():] = 7.0
    _check(lib.dm_f32_to_bf16(_p(x), _p(dst), ctypes.c_longlong(x.numel()), _sp()), "f32_to_bf16")
    torch.cuda.synchronize()
    ref = x.to(torch.bfloat16)
    got = dst[: x.numel()]
    nan = torch.isnan(x)
    assert bool(torch.isnan(got[nan].float()).all()), "NaN must stay NaN"
    gb, rb = got[~nan].view(torch.int16), ref[~nan].view(torch.int16)
    bad = (gb != rb).nonzero()
    assert bad.numel() == 0, "first mismatches: %s" % [(float(x[~nan][i]), int(gb[i]), int(rb[i])) for i in bad[:5, 0]]
    assert bool((dst[x.numel():] == 7.0).all()), "wrote past the end"
    assert lib.dm_f32_to_bf16(_p(x), _p(dst), ctypes.c_longlong(6), _sp()) == -1


# ---------------------------------------------------------------------------------------------------------------------
# inference path at the engine level
# ---------------------------------------------------------------------------------------------------------------------
def _backend():
    from distributedmnist_b200.parallel.context import ReplicaContext
    from distributedmnist_b200.parallel.fused import FusedBackend
    return FusedBackend(ReplicaContext(0, 1, 0, torch.device("cuda", 0), "none"))


def _trained_params(make, steps, B, data):
    """A few hundred SGD steps of the CUDA engine on the synthetic set: weights that look trained."""
    from distributedmnist_b200.parallel.aggregators import SyncReplicasOptimizer
    from distributedmnist_b200.schedule import LearningRateSchedule
    be = _backend()
    eng = make(B, be)
    eng.attach_optimizer(SyncReplicasOptimizer(be, LearningRateSchedule(0.05, 1000, 1.0), 1, 1))
    trx, try_ = data
    nb = len(trx) // B
    for s in range(steps):
        i = (s % nb) * B
        eng.load_batch(trx[i:i + B], try_[i:i + B])
        eng.train_step()
    torch.cuda.synchronize()
    be.check_error()
    return eng.params.detach().clone()


@pytest.fixture(scope="module")
def synthetic():
    from distributedmnist_b200.data import make_synthetic_mnist
    trx, try_, tex, tey = make_synthetic_mnist(256 * 8, 2001, seed=17)
    return (trx.reshape(-1, 28, 28).astype(np.float32), try_), (tex.reshape(-1, 28, 28).astype(np.float32), tey)


def _reduction_checks(n, per_chunk):
    """evaluate() = mean over chunks of the kernel's per-row loss (float64, within the fp32 atomics bound) and the exact
    number of rows whose kernel-logit argmax matches the label."""
    loss_rows = torch.cat([c[0] for c in per_chunk])
    hits = sum(c[1] for c in per_chunk)
    lb = float(sum(c[2] for c in per_chunk)) / n + (R.gamma(1002) + 4 * R.U) * float(loss_rows.abs().mean())
    return loss_rows, hits, lb


def _lenet_ref64(eng, x):
    p, bf = eng.p, torch.bfloat16
    xr, w1 = (x.to(bf), p["conv1_weights"].to(bf)) if eng._conv1_tc else (x, p["conv1_weights"])
    c1 = R.conv_fwd(xr[..., None], w1)[0] + p["conv1_biases"].double()
    a1 = R.windows(c1).max(dim=4).values.clamp_min(0).to(bf)
    c2 = R.conv_fwd(a1, p["conv2_weights"].to(bf))[0] + p["conv2_biases"].double()
    a2 = R.windows(c2).max(dim=4).values.clamp_min(0).to(bf).double().reshape(x.shape[0], 3136)
    h = (a2 @ p["fc1_weights"].to(bf).double() + p["fc1_biases"].double()).clamp_min(0)
    return h @ p["fc2_weights"].double() + p["fc2_biases"].double()


def test_lenet_inference_path(synthetic):
    from distributedmnist_b200.engine_cuda import CudaLeNetEngine
    (trx, try_), (tex, tey) = synthetic
    params = _trained_params(lambda B, be: CudaLeNetEngine(B, be, seed=3, use_graph=True), 300, 256, (trx, try_))
    eng = CudaLeNetEngine(1000, _backend(), seed=3, use_graph=False)     # as make_cuda_eval_engine builds it
    eng.params.copy_(params)
    eng.params_updated()
    p, pb = eng.p, eng.pb
    worst = {}
    for n in (2001, 1500):                                     # final batches of one and of 500 images
        x = torch.from_numpy(tex[:n]).cuda()
        y = torch.from_numpy(tey[:n]).cuda()
        per_chunk = []
        for s in range(0, n, 1000):
            m = min(1000, n - s)
            xs, ys = x[s:s + m].contiguous(), y[s:s + m].contiguous()
            logits = eng.forward_logits(xs, ys, train=False)
            torch.cuda.synchronize()
            la = eng.d_loss_acc.clone()
            tag = "lenet eval n=%d chunk=%d m=%d" % (n, s, m)
            # stage by stage, each on the kernel's own previous output
            xr, w1 = (xs.to(torch.bfloat16), p["conv1_weights"].to(torch.bfloat16)) if eng._conv1_tc \
                else (xs, p["conv1_weights"])
            conv, S = R.conv_fwd(xr[..., None], w1)
            _pool_ok(R.check_pool_relu(conv, S, p["conv1_biases"], 25, eng.a1[:m], eng.code1[:m]), tag + " conv1")
            conv, S = R.conv_fwd(eng.a1[:m], pb["conv2_weights"])
            res = R.check_pool_relu(conv, S, p["conv2_biases"], 800, eng.a2[:m].view(m, 7, 7, 64),
                                    eng.code2[:m].view(m, 7, 7, 64))
            _pool_ok(res, tag + " conv2")
            a2, w1f = eng.a2[:m].double(), pb["fc1_weights"].double()
            for z in range(7):                                  # 49 k-blocks of 64: seven per split
                k0, k1 = 448 * z, 448 * (z + 1)
                r = R.worst_ratio(eng.h_part[z, :m], a2[:, k0:k1] @ w1f[k0:k1],
                                  R.acc_bound(a2[:, k0:k1].abs() @ w1f[k0:k1].abs(), 448))
                assert r <= 1.0, (tag, "fc1 split", z, r)
            hp = p["fc1_biases"].double() + eng.h_part[:, :m].double().sum(0)
            e_hp = R.acc_bound(p["fc1_biases"].double().abs() + eng.h_part[:, :m].double().abs().sum(0), 9)
            h = hp.clamp_min(0)
            e_h = torch.where(hp.abs() <= e_hp, 2 * e_hp, e_hp)
            w2 = p["fc2_weights"].double()
            ref = h @ w2 + p["fc2_biases"].double()
            bound = R.acc_bound((h + e_h) @ w2.abs() + p["fc2_biases"].double().abs(), 513) + e_h @ w2.abs()
            worst[tag] = R.worst_ratio(logits, ref, bound)
            assert worst[tag] <= 1.0, (tag, worst[tag])
            row, row_bound, _, _, hits = R.xent_ref(logits, ys)
            _xent_checks(logits, ys, la, m, tag)
            per_chunk.append((row, hits, float(row_bound.sum())))
        loss_rows, hits, lb = _reduction_checks(n, per_chunk)
        el, ea = eng.evaluate(tex[:n], tey[:n])
        assert abs(el - float(loss_rows.mean())) <= lb, (n, el, float(loss_rows.mean()), lb)
        assert round(ea * n) == hits, (n, ea * n, hits)
        # the whole chain in float64 with the kernels' bf16 rounding points (a1, a2, bf16 weights; fc1's activations
        # stay fp32 as in the kernels): decisions near ties may go either way, so this is a stated tolerance, not the bound
        ref_logits = _lenet_ref64(eng, x)
        rl = torch.nn.functional.cross_entropy(ref_logits, y)
        ra = (ref_logits.argmax(1) == y).double().mean()
        assert abs(el - float(rl)) <= 2e-3 * max(1.0, float(rl)), (n, el, float(rl))
        chunk_logits = torch.cat([eng.forward_logits(x[s:s + 1000].contiguous(), y[s:s + 1000].contiguous(), False)
                                  for s in range(0, n, 1000)])
        dev = float((chunk_logits.double() - ref_logits).abs().max())
        assert dev <= 0.05, (n, dev)
        close = int((R.margin_top2(ref_logits) <= 2 * dev).sum())
        assert abs(round(ea * n) - round(float(ra) * n)) <= close, (n, ea, float(ra), close)
        assert ea > 0.9, (n, ea)
    print("lenet inference worst err/bound:", max(worst.values()))


def test_mlp_inference_path(synthetic):
    from distributedmnist_b200.engine_cuda import CudaMlpEngine
    (trx, try_), (tex, tey) = synthetic
    H = 256
    params = _trained_params(lambda B, be: CudaMlpEngine("mlp3", B, be, hidden=H, seed=4, use_graph=True), 300, 256,
                             (trx.reshape(-1, 784), try_))
    eng = CudaMlpEngine("mlp3", 1000, _backend(), hidden=H, seed=4, use_graph=False)
    eng.params.copy_(params)
    eng.params_updated()
    p, pb = eng.p, eng.pb
    n = 1037
    x = torch.from_numpy(tex[:n].reshape(n, 784)).cuda()
    y = torch.from_numpy(tey[:n]).cuda()
    per_chunk = []
    worst = 0.0
    for s in range(0, n, 1000):
        m = min(1000, n - s)
        xs, ys = x[s:s + m].contiguous(), y[s:s + m].contiguous()
        logits = torch.zeros(m, 10, device="cuda")
        eng.d_loss_acc.zero_()
        eng._forward(xs, ys, m, False, logits_out=logits)
        torch.cuda.synchronize()
        la = eng.d_loss_acc.clone()
        tag = "mlp3 eval chunk=%d m=%d" % (s, m)
        assert torch.equal(eng.x16[:m].view(torch.int16), xs.to(torch.bfloat16).view(torch.int16)), tag
        src = eng.x16[:m].double()
        for i in range(1, eng.n_layers):
            W, b = pb["fc%d_weights" % i].double(), p["fc%d_biases" % i].double()
            ref = (src @ W + b).clamp_min(0)
            e = R.acc_bound(src.abs() @ W.abs() + b.abs(), src.shape[1] + 1)
            r = R.worst_ratio(eng.h[i - 1][:m], ref, R.bf16_out_bound(ref, e))
            assert r <= 1.0, (tag, i, r)
            worst = max(worst, r)
            src = eng.h[i - 1][:m].double()
        L = eng.n_layers
        W, b = p["fc%d_weights" % L].double(), p["fc%d_biases" % L].double()
        r = R.worst_ratio(logits, src @ W + b, R.acc_bound(src.abs() @ W.abs() + b.abs(), H + 1))
        assert r <= 1.0, (tag, "logits", r)
        worst = max(worst, r)
        row, row_bound, _, _, hits = R.xent_ref(logits, ys)
        _xent_checks(logits, ys, la, m, tag)
        per_chunk.append((row, hits, float(row_bound.sum())))
    loss_rows, hits, lb = _reduction_checks(n, per_chunk)
    el, ea = eng.evaluate(tex[:n].reshape(n, 784), tey[:n])
    assert abs(el - float(loss_rows.mean())) <= lb, (el, float(loss_rows.mean()), lb)
    assert round(ea * n) == hits, (ea * n, hits)
    assert ea > 0.9, ea
    print("mlp3 inference worst err/bound:", worst)
