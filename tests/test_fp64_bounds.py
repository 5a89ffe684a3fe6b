"""The float64 error bound of tests/_fp64_ref.py, checked on the CPU.

A bound is only useful if it holds for every correct summation order and fails for a wrong kernel.  Here bf16 x bf16
dot products are accumulated in fp32 (numpy) in several orders, including a truncating accumulator, and must stay
within the bound; then the faults a tensor-core kernel typically has (a dropped k-block, a dropped filter tap, the
neighbouring column's bias, a transposed sub-tile) must each exceed it.
"""
import numpy as np
import pytest
import torch

import _fp64_ref as R


def _bf16(rng, shape, scale=1.0, offset=0.0):
    x = torch.from_numpy(rng.standard_normal(shape) * scale + offset).float()
    return x.to(torch.bfloat16).float().numpy()


def _trunc32(x: np.ndarray) -> np.ndarray:
    """float64 -> fp32 rounded toward zero."""
    f = x.astype(np.float32)
    over = np.abs(f.astype(np.float64)) > np.abs(x)
    return np.where(over, np.nextafter(f, np.float32(0)), f).astype(np.float32)


def _dot_orders(a: np.ndarray, b: np.ndarray) -> dict:
    """out[M,N] = a[M,K] @ b[K,N] with exact products and fp32 accumulation in several orders."""
    M, K = a.shape
    prods = (a[:, :, None].astype(np.float32) * b[None, :, :].astype(np.float32))        # exact: 8 x 8 significant bits
    out = {}
    acc = np.zeros((M, b.shape[1]), np.float32)
    for k in range(K):
        acc = acc + prods[:, k]
    out["sequential"] = acc
    acc = np.zeros_like(acc)
    for k in reversed(range(K)):
        acc = acc + prods[:, k]
    out["reversed"] = acc
    p = prods
    while p.shape[1] > 1:                                         # pairwise tree
        if p.shape[1] % 2:
            p = np.concatenate([p, np.zeros_like(p[:, :1])], axis=1)
        p = p[:, 0::2] + p[:, 1::2]
    out["pairwise"] = p[:, 0]
    acc = np.zeros_like(acc)                                      # k-blocks of 64 summed apart, then added (split-K)
    for k0 in range(0, K, 64):
        blk = np.zeros_like(acc)
        for k in range(k0, min(K, k0 + 64)):
            blk = blk + prods[:, k]
        acc = acc + blk
    out["split_k"] = acc
    acc = np.zeros_like(acc)                                      # an accumulator that truncates every addition
    for k in range(K):
        acc = _trunc32(acc.astype(np.float64) + prods[:, k].astype(np.float64))
    out["truncating"] = acc
    return out


def _ref(a, b):
    A, Bm = torch.from_numpy(a).double(), torch.from_numpy(b).double()
    return A @ Bm, A.abs() @ Bm.abs()


@pytest.mark.parametrize("K", [1, 37, 64, 512, 3136])
def test_correct_summation_orders_stay_within_bound(K):
    rng = np.random.default_rng(K)
    a = _bf16(rng, (16, K), 0.5)
    b = _bf16(rng, (K, 12), 0.5, 0.1)                             # nonzero mean: partial cancellation and growth
    ref, S = _ref(a, b)
    bound = R.acc_bound(S, K)
    for name, out in _dot_orders(a, b).items():
        r = R.worst_ratio(torch.from_numpy(out), ref, bound)
        assert r <= 1.0, (name, K, r)
        # and once rounded to bf16 like the kernels' bf16 stores
        o16 = torch.from_numpy(out).to(torch.bfloat16)
        r16 = R.worst_ratio(o16, ref, R.bf16_out_bound(ref, bound))
        assert r16 <= 1.0, (name, K, r16)


def test_mutations_exceed_bound():
    rng = np.random.default_rng(7)
    K = 512
    a = _bf16(rng, (64, K), 0.5)
    b = _bf16(rng, (K, 64), 0.5)
    ref, S = _ref(a, b)
    bound = R.acc_bound(S, K)
    good = _dot_orders(a, b)["sequential"].astype(np.float64)
    assert R.worst_ratio(torch.from_numpy(good), ref, bound) <= 1.0
    # one k-block of 64 missing
    a_drop = a.copy()
    a_drop[:, 128:192] = 0
    assert R.worst_ratio(torch.from_numpy(a_drop.astype(np.float64) @ b), ref, bound) > 1.0
    # the neighbouring column's bias
    bias = _bf16(rng, (64,), 0.1)
    ref_b, Sb = ref + torch.from_numpy(bias).double(), S + torch.from_numpy(np.abs(bias)).double()
    wrong = good + np.roll(bias, -1)[None, :]
    assert R.worst_ratio(torch.from_numpy(wrong), ref_b, R.acc_bound(Sb, K + 1)) > 1.0
    # a transposed 32 x 32 sub-tile
    t = good.copy()
    t[:32, :32] = t[:32, :32].T.copy()
    assert R.worst_ratio(torch.from_numpy(t), ref, bound) > 1.0


def test_dropped_conv2_tap_channel_exceeds_bound():
    """conv2-shaped sums (800 terms): zeroing one (tap, input-channel) weight row must exceed the bound somewhere."""
    g = torch.Generator().manual_seed(1)
    a1 = torch.rand(2, 14, 14, 32, generator=g).to(torch.bfloat16)
    w = (torch.randn(5, 5, 32, 64, generator=g) * 0.05).to(torch.bfloat16)
    ref, S = R.conv_fwd(a1, w)
    bound = R.acc_bound(S, 800)
    fp32 = R.conv_fwd(a1.float(), w.float())[0]                       # correct result, summed in some other order
    assert R.worst_ratio(fp32.float(), ref, bound) <= 1.0
    for tap, ci in [(0, 0), (12, 5), (24, 31)]:
        wm = w.clone()
        wm[tap // 5, tap % 5, ci, :] = 0
        assert R.worst_ratio(R.conv_fwd(a1, wm)[0].float(), ref, bound) > 1.0, (tap, ci)


def test_pool_relu_checker_flags_a_wrong_argmax():
    g = torch.Generator().manual_seed(3)
    a1 = torch.rand(2, 14, 14, 32, generator=g).to(torch.bfloat16)
    w = (torch.randn(5, 5, 32, 64, generator=g) * 0.05).to(torch.bfloat16)
    bias = torch.randn(64, generator=g) * 0.1
    conv, S = R.conv_fwd(a1, w)
    win = R.windows(conv.float())
    mx, idx = win.max(dim=4)
    pre = mx + bias
    out = pre.clamp_min(0).to(torch.bfloat16)
    code = (idx | ((pre > 0).long() << 2)).to(torch.uint8)
    res = R.check_pool_relu(conv, S, bias, 800, out, code)
    assert res["ratio"] <= 1.0 and res["bad_idx"] == 0 and res["bad_act"] == 0, res
    wrong = code.clone()
    wrong[0, 0, 0, :] = (wrong[0, 0, 0, :] & 4) | ((wrong[0, 0, 0, :] & 3) ^ 1)
    assert R.check_pool_relu(conv, S, bias, 800, out, wrong)["bad_idx"] > 0
    assert R.check_pool_relu(conv, S, bias, 800, out, code ^ 4)["bad_act"] > 0


def test_bf16_half_ulp():
    x = torch.tensor([1.0, 1.5, 2.0 - 2 ** -10, 2.0, 3.0, 0.0], dtype=torch.float64)
    assert R.bf16_half_ulp(x).tolist() == [2 ** -8, 2 ** -8, 2 ** -8, 2 ** -7, 2 ** -7, 0.0]
