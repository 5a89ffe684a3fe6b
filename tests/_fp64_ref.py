"""Float64 references of the kernels' operations and the rounding-error bounds the kernels are judged by.

Method: the reference is given the kernel's exact operands (bf16 where the kernel reads bf16, fp32 where it reads
fp32) and computes in float64, so the only difference left is the kernel's own rounding.  Every dot product of n
terms summed in fp32 (any order, any split into partials or atomics) stays within

    |out - ref| <= gamma_n * sum|a||b|,        gamma_n = n*u / (1 - n*u)

and a result stored as bf16 adds half a bf16 ulp of the value it rounds, |ref| + gamma_n * sum|a||b| at most.
Max-pool and ReLU never increase the infinity-norm error, so the bound of a pooled output is the window maximum of
the per-element bounds.

u = 2^-23 (one fp32 ulp, not half of one) leaves room for an accumulator that truncates instead of rounding: how
precisely the tcgen05 tensor core accumulates has not been documented.  Products of two bf16 values are exact in
fp32, so for the tensor-core kernels the bound covers accumulation only; for the SIMT kernels the fused multiply-add
rounds once per term, which the same gamma_n covers.  Measured worst err / bound values are recorded beside each
check in the tests.

The module only needs torch, so the CPU test of the bound itself runs without a GPU.
"""
from __future__ import annotations

from typing import Tuple

import torch
import torch.nn.functional as F

U = 2.0 ** -23          # unit of the fp32 accumulation model (allows truncation)
U_BF16 = 2.0 ** -8      # bf16 unit roundoff (round to nearest even, 8 significant bits)


def gamma(n: int, u: float = U) -> float:
    nu = n * u
    assert nu < 0.5, "gamma_%d undefined for u=%g" % (n, u)
    return nu / (1.0 - nu)


def bf16_half_ulp(x: torch.Tensor) -> torch.Tensor:
    """Half a bf16 ulp at |x| (x >= 0, float64): for x in [2^(e-1), 2^e) the bf16 spacing is 2^(e-8)."""
    _, e = torch.frexp(x)
    h = torch.ldexp(torch.ones_like(x), e - 9)
    return torch.where(x > 0, h, torch.zeros_like(x))


def acc_bound(S: torch.Tensor, n: int, u: float = U) -> torch.Tensor:
    """Bound of an fp32 sum of n terms whose absolute values add up to S."""
    return gamma(n, u) * S


def bf16_out_bound(ref: torch.Tensor, e: torch.Tensor) -> torch.Tensor:
    """Bound of a value within e of ref, then rounded to bf16."""
    return e + bf16_half_ulp(ref.abs() + e)


def worst_ratio(out: torch.Tensor, ref: torch.Tensor, bound: torch.Tensor) -> float:
    """max |out - ref| / bound (float64); an element with bound 0 must match exactly (else inf); NaN out is inf."""
    err = (out.double() - ref.double()).abs()
    r = torch.where(bound > 0, err / bound.clamp_min(1e-300), torch.where(err > 0, torch.inf, 0.0))
    r = torch.where(torch.isnan(err), torch.inf, r)
    return float(r.max()) if r.numel() else 0.0


# ---------------------------------------------------------------------------------------------------------------------
# convolutions (NHWC activations, HWIO weights, 5x5 SAME), float64 on whatever device the operands live on
# ---------------------------------------------------------------------------------------------------------------------
def _nchw(t: torch.Tensor) -> torch.Tensor:
    return t.double().permute(0, 3, 1, 2)


def _nhwc(t: torch.Tensor) -> torch.Tensor:
    return t.permute(0, 2, 3, 1).contiguous()


def conv_fwd(x: torch.Tensor, w: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """x [B,H,W,Ci], w [5,5,Ci,Co] -> (sum x*w, sum |x||w|), both [B,H,W,Co] float64, no bias."""
    wt = w.double().permute(3, 2, 0, 1)
    xn = _nchw(x)
    return (_nhwc(F.conv2d(xn, wt, padding=2)), _nhwc(F.conv2d(xn.abs(), wt.abs(), padding=2)))


def conv_dgrad(dy: torch.Tensor, w: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """dy [B,H,W,Co], w [5,5,Ci,Co] -> d input [B,H,W,Ci] and its sum of |terms|."""
    B, H, W, _ = dy.shape
    wt = w.double().permute(3, 2, 0, 1)
    shape = (B, w.shape[2], H, W)
    dn = _nchw(dy)
    return (_nhwc(torch.nn.grad.conv2d_input(shape, wt, dn, padding=2)),
            _nhwc(torch.nn.grad.conv2d_input(shape, wt.abs(), dn.abs(), padding=2)))


def conv_wgrad(x: torch.Tensor, dy: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
    """x [B,H,W,Ci], dy [B,H,W,Co] -> HWIO weight gradient [5,5,Ci,Co] and its sum of |terms|."""
    ci, co = x.shape[3], dy.shape[3]
    xn, dn = _nchw(x), _nchw(dy)
    g = torch.nn.grad.conv2d_weight(xn, (co, ci, 5, 5), dn, padding=2).permute(2, 3, 1, 0)
    s = torch.nn.grad.conv2d_weight(xn.abs(), (co, ci, 5, 5), dn.abs(), padding=2).permute(2, 3, 1, 0)
    return g.contiguous(), s.contiguous()


def windows(t: torch.Tensor) -> torch.Tensor:
    """[B,2h,2w,C] -> [B,h,w,C,4] with window position q = dy*2 + dx (the kernels' argmax code)."""
    B, H, W, C = t.shape
    return t.reshape(B, H // 2, 2, W // 2, 2, C).permute(0, 1, 3, 5, 2, 4).reshape(B, H // 2, W // 2, C, 4)


def check_pool_relu(conv: torch.Tensor, S: torch.Tensor, bias: torch.Tensor, n: int, out: torch.Tensor,
                    code: torch.Tensor) -> dict:
    """Judge a fused  conv + bias -> ReLU -> 2x2 max-pool -> bf16  output and its pooling code.

    conv / S: float64 pre-bias sums and sums of |terms| ([B,2h,2w,C]); n: terms per sum (bias excluded).
    Returns worst err/bound of the output, the number of argmax / ReLU-flag decisions that contradict the reference
    beyond the bound, the number of decisions the bound cannot settle, and the element count."""
    e_pre = acc_bound(S, n)                                     # pre-bias accumulator
    cw, ew = windows(conv), windows(e_pre)
    b = bias.double().view(1, 1, 1, -1)
    mx, amax = cw.max(dim=4)
    E = ew.max(dim=4).values + gamma(n + 1) * (windows(S).max(dim=4).values + b.abs())   # + the bias add
    r = mx + b
    ref = r.clamp_min(0.0)
    ratio = worst_ratio(out, ref, bf16_out_bound(ref, E))
    idx, act = (code & 3).long(), ((code >> 2) & 1).bool()
    # argmax: the chosen window value must be within the two errors of the maximum
    sel = torch.gather(cw, 4, idx[..., None])[..., 0]
    esel = torch.gather(ew, 4, idx[..., None])[..., 0]
    emax = torch.gather(ew, 4, amax[..., None])[..., 0]
    bad_idx = int((sel < mx - (esel + emax)).sum())
    # near-ties the bound cannot order (exact sums, e.g. all-zero patches, have a bound of 0 and are not counted: any
    # tied choice is then exactly the maximum)
    top2 = cw.topk(2, dim=4).values
    emx = ew.max(dim=4).values
    amb_idx = int(((top2[..., 0] - top2[..., 1] <= 2 * emx) & (emx > 0)).sum())
    # ReLU flag: decided by the sign of max + bias wherever |max + bias| exceeds the bound; and the stored output is
    # nonzero exactly where the flag is set (a positive fp32 value never rounds to bf16 zero here)
    bad_act = int(((r > E) & ~act).sum() + ((r < -E) & act).sum() + ((out.float() > 0) != act).sum())
    amb_act = int(((r.abs() <= E) & (E > 0)).sum())
    return dict(ratio=ratio, bad_idx=bad_idx, amb_idx=amb_idx, bad_act=bad_act, amb_act=amb_act, count=out.numel())


def unpool(g: torch.Tensor, code: torch.Tensor) -> torch.Tensor:
    """Pooled gradient [B,h,w,C] -> dense [B,2h,2w,C]: each value at its window's argmax, where ReLU was active."""
    B, h, w, C = g.shape
    idx, act = (code & 3).long(), ((code >> 2) & 1).bool()
    gm = torch.where(act, g, torch.zeros_like(g))
    out = torch.zeros(B, h, 2, w, 2, C, dtype=g.dtype, device=g.device)
    for q in range(4):
        out[:, :, q >> 1, :, q & 1, :] = torch.where(idx == q, gm, torch.zeros_like(gm))
    return out.reshape(B, 2 * h, 2 * w, C)


# ---------------------------------------------------------------------------------------------------------------------
# softmax cross entropy with the kernels' fast-math exp / log
# ---------------------------------------------------------------------------------------------------------------------
def expf_rel(x: torch.Tensor) -> torch.Tensor:
    """Relative error bound of __expf(x) (CUDA programming guide: 2 + floor(|1.173 x|) ulp; fast-math exp2 path)."""
    return (2.0 + torch.floor((1.173 * x).abs())) * U


def xent_ref(logits: torch.Tensor, labels: torch.Tensor):
    """From the kernel's own fp32 logits [B,10]: float64 per-row loss, its error bound, softmax p, bound of p, hits.

    Per row the kernel computes m = max, e_c = __expf(l_c - m), s = sum e_c, loss = __logf(s) - (l_label - m),
    p_c = e_c / s.  __logf: 2^-21.41 absolute on [0.5, 2], 3 ulp elsewhere (s is in [1, 10])."""
    L = logits.double()
    m = L.max(dim=1, keepdim=True).values
    x = L - m
    e = x.exp()
    s = e.sum(dim=1, keepdim=True)
    lab = labels.long().view(-1, 1)
    row = (s.log() - torch.gather(x, 1, lab))[:, 0]
    re = expf_rel(x)                                            # exp
    ftz = 2.0 ** -126                                           # fast-math exp flushes results below FLT_MIN to zero
    rs = ((e * (re + 2 * U)).sum(dim=1, keepdim=True) + 10 * ftz) / s + gamma(10)   # relative error of s
    lse = s.log()
    log_err = torch.where(s <= 2, torch.full_like(s, 2.0 ** -21.41), 3 * U * lse.abs()) + rs * (1 + U)
    row_bound = (log_err + 4 * U * (lse.abs() + torch.gather(x, 1, lab).abs()))[:, 0]
    p = e / s
    p_bound = p * (re + rs + 3 * U) + ftz / s
    hits = int((logits.argmax(dim=1) == labels.long()).sum())   # torch argmax returns the first maximal index
    return row, row_bound, p, p_bound, hits


def margin_top2(logits: torch.Tensor) -> torch.Tensor:
    t = logits.double().topk(2, dim=1).values
    return t[:, 0] - t[:, 1]
