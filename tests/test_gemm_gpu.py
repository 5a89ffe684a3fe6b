"""tcgen05 GEMM vs a plain PyTorch fp32 reference of the same op (SURVEY §4 item 2)."""
import pytest
import torch

pytestmark = pytest.mark.gpu


def _ref(a, b, a_major, b_major):
    A = a.float().t() if a_major == "mn" else a.float()
    Bm = b.float() if b_major == "mn" else b.float().t()
    return A @ Bm


CASES = [
    # (M, N, K) incl. partial tiles and K not a multiple of 64
    (128, 128, 64), (256, 512, 3136), (256, 3136, 512), (3136, 512, 256), (200, 72, 784), (128, 64, 100 * 8),
]


@pytest.mark.parametrize("a_major", ["k", "mn"])
@pytest.mark.parametrize("b_major", ["k", "mn"])
@pytest.mark.parametrize("bn", [64, 128])
def test_gemm_all_majors(a_major, b_major, bn):
    from distributedmnist_b200.ops.gemm import gemm_bf16
    torch.manual_seed(0)
    for (M, N, K) in CASES:
        a = (torch.randn((K, M) if a_major == "mn" else (M, K), device="cuda") * 0.5).to(torch.bfloat16)
        b = (torch.randn((K, N) if b_major == "mn" else (N, K), device="cuda") * 0.5).to(torch.bfloat16)
        out = gemm_bf16(a, b, a_major, b_major, bn=bn)
        ref = _ref(a, b, a_major, b_major)
        err = (out - ref).abs().max().item()
        tol = 2e-3 * (K ** 0.5) + 1e-3
        assert err < tol, "M=%d N=%d K=%d majors=%s/%s bn=%d: max err %g (tol %g)" % (M, N, K, a_major, b_major, bn, err, tol)


def test_gemm_split_k_atomic_and_bf16_out():
    from distributedmnist_b200.ops.gemm import gemm_bf16
    torch.manual_seed(1)
    a = (torch.randn(256, 3136, device="cuda") * 0.3).to(torch.bfloat16)
    w = (torch.randn(3136, 512, device="cuda") * 0.1).to(torch.bfloat16)
    ref = a.float() @ w.float()
    out = gemm_bf16(a, w, "k", "mn", splits=16)
    assert (out - ref).abs().max().item() < 0.05
    out16 = gemm_bf16(a, w, "k", "mn", out_dtype=torch.bfloat16)
    assert (out16.float() - ref).abs().max().item() < 0.25


# ---------------------------------------------------------------------------------------------------------------------
# Every epilogue x tile width x operand major against a float64 reference with the derived bound (tests/_fp64_ref.py),
# at the call sites' shapes, with NaN guard bands around the output.
# ---------------------------------------------------------------------------------------------------------------------
import ctypes                                                   # noqa: E402

import _fp64_ref as R                                           # noqa: E402

EPIS = [0, 1, 2, 3]
BNS = [64, 128, 256]


def _operands(M, N, K, a_mn, b_mn, g, lda=None, ldb=None):
    """bf16 operands in the requested majors, leading dimensions padded to a multiple of 8 (TMA stride rule); the
    padding holds garbage that must never be read.  Returns the storage tensors and float64 logical A [M,K], B [K,N]."""
    pad8 = lambda v: (v + 7) // 8 * 8                          # noqa: E731
    ra, ca = (K, M) if a_mn else (M, K)
    rb, cb = (K, N) if b_mn else (N, K)
    lda, ldb = lda or pad8(ca), ldb or pad8(cb)
    a = (torch.randn(ra, lda, generator=g, device="cuda") * 0.5).to(torch.bfloat16)
    b = (torch.randn(rb, ldb, generator=g, device="cuda") * 0.5 + 0.05).to(torch.bfloat16)
    A = a[:, :ca].double()
    Bm = b[:, :cb].double()
    A = A.t() if a_mn else A
    Bm = Bm if b_mn else Bm.t()
    return a, b, lda, ldb, A, Bm


def _run_case(M, N, K, a_mn, b_mn, epi, bn, splits=1, partials=False, ldo=None, seed=0, sample_rows=None):
    from distributedmnist_b200.ops.gemm import gemm_bf16_raw
    g = torch.Generator(device="cuda").manual_seed(seed)
    a, b, lda, ldb, A, Bm = _operands(M, N, K, a_mn, b_mn, g)
    ldo = ldo or (N + 8)                                        # padding columns beyond N: a guard band
    rows = M + 3                                                # rows beyond M: a guard band
    f32 = epi in (0, 1)
    dt = torch.float32 if f32 else torch.bfloat16
    nz = splits if partials else 1
    out = torch.full((nz, rows, ldo), float("nan"), dtype=dt, device="cuda")
    init = None
    if epi == 1:                                                # atomics add onto what is there: start from a known value
        init = torch.randn(M, N, generator=g, device="cuda")
        out[0, :M, :N] = init
    bias = None
    if epi == 3:                                                # nonzero, mostly negative: ReLU clips a real share
        bias = torch.randn(N, generator=g, device="cuda") * 0.5 - 0.3
    gemm_bf16_raw(a, b, out, M, N, K, lda, ldb, ldo, a_mn, b_mn, epi, splits=splits, bn=bn,
                  split_stride=rows * ldo if partials else 0, bias=bias)
    torch.cuda.synchronize()
    tag = "M=%d N=%d K=%d a_mn=%d b_mn=%d epi=%d bn=%d splits=%d partials=%d ldo=%d" % (
        M, N, K, a_mn, b_mn, epi, bn, splits, partials, ldo)
    # guard bands: everything in the M x N extent written, nothing else touched
    assert not torch.isnan(out[:, :M, :N].float()).any(), "unwritten output element: " + tag
    assert torch.isnan(out[:, :M, N:].float()).all() and torch.isnan(out[:, M:].float()).all(), "guard band written: " + tag
    sel = slice(None) if sample_rows is None else sample_rows
    Ar = A[sel]
    worst = 0.0
    if partials:
        nkb = (K + 63) // 64
        for z in range(splits):                                 # split z owns k-blocks [nkb*z/splits, nkb*(z+1)/splits)
            k0, k1 = 64 * (nkb * z // splits), min(K, 64 * (nkb * (z + 1) // splits))
            ref = Ar[:, k0:k1] @ Bm[k0:k1]
            S = Ar[:, k0:k1].abs() @ Bm[k0:k1].abs()
            worst = max(worst, R.worst_ratio(out[z, :M, :N][sel], ref, R.acc_bound(S, max(k1 - k0, 1))))
        return worst, tag
    ref, S = Ar @ Bm, Ar.abs() @ Bm.abs()
    n = K + (splits if epi == 1 else 0)
    if epi == 1:
        ref, S, n = ref + init.double()[sel], S + init.double().abs()[sel], n + 1
    if epi == 3:
        ref, S, n = (ref + bias.double()).clamp_min(0), S + bias.double().abs(), n + 1
    e = R.acc_bound(S, max(n, 1))
    bound = e if f32 else R.bf16_out_bound(ref, e)
    return R.worst_ratio(out[0, :M, :N][sel], ref, bound), tag


EDGE_SHAPES = [(128, 128, 64), (200, 72, 784), (37, 130, 40), (129, 257, 1), (1, 96, 200), (130, 10, 96)]


@pytest.mark.parametrize("epi", EPIS)
@pytest.mark.parametrize("bn", BNS)
def test_gemm_epilogue_tile_major_matrix(epi, bn):
    """Edge shapes (K < 64, K = 1, M = 1, N = 10, partial tiles) in every operand major.
    Measured worst err / bound on a B200 (1000 W): fp32 stores 0.04, fp32 atomics 0.10, bf16 stores 1.00 (the rounding
    of values exactly halfway between two bf16 numbers)."""
    if bn == 256 and epi == 1:
        pytest.skip("128 x 256 tiles have no atomic epilogue (dm_gemm_bf16 returns -1)")
    worst = []
    for i, (M, N, K) in enumerate(EDGE_SHAPES):
        for a_mn in (False, True):
            for b_mn in (False, True):
                r, tag = _run_case(M, N, K, a_mn, b_mn, epi, bn, splits=3 if epi == 1 else 1, seed=i)
                print("RATIO", tag, r)
                assert r <= 1.0, "err/bound %.3g: %s" % (r, tag)
                worst.append(r)
    print("gemm matrix epi=%d bn=%d worst err/bound %.3g" % (epi, bn, max(worst)))


def test_gemm_bn256_atomic_is_refused():
    from distributedmnist_b200.ops.lib import load, ptr, stream_ptr
    a = torch.zeros(128, 64, dtype=torch.bfloat16, device="cuda")
    out = torch.zeros(128, 256, device="cuda")
    rc = load().dm_gemm_bf16(ptr(a), ptr(a), ptr(out), 128, 256, 64, 64, 64, 256, 0, 0, 1, 1, 256,
                             ctypes.c_longlong(0), ptr(None), stream_ptr())
    assert rc == -1


def test_gemm_unpadded_leading_dimension_is_refused():
    """TMA needs 16-byte global strides: an lda / ldb that is not a multiple of 8 elements returns -3."""
    from distributedmnist_b200.ops.lib import load, ptr, stream_ptr
    a = torch.zeros(64, 100, dtype=torch.bfloat16, device="cuda")
    b = torch.zeros(100, 64, dtype=torch.bfloat16, device="cuda")
    out = torch.full((64, 64), float("nan"), device="cuda")
    lib = load()
    for lda, ldb in [(100, 64), (104, 60), (97, 64)]:
        rc = lib.dm_gemm_bf16(ptr(a), ptr(b), ptr(out), 64, 64, 97, lda, ldb, 64, 0, 1, 0, 1, 128,
                              ctypes.c_longlong(0), ptr(None), stream_ptr())
        assert rc == -3, (lda, ldb, rc)
    torch.cuda.synchronize()
    assert torch.isnan(out).all()


@pytest.mark.parametrize("B", [1, 37, 256, 1000, 1024])
def test_gemm_lenet_fc1_call_sites(B):
    """fc1 forward (7 split-K partials), dgrad (bf16 out) and wgrad (K = batch, fp32 and bf16) as the engine calls them.
    Measured worst err / bound on a B200 (1000 W): fp32 stores 0.04, fp32 atomics 0.10, bf16 stores 1.00 (the rounding
    of values exactly halfway between two bf16 numbers)."""
    cases = [
        dict(M=B, N=512, K=3136, a_mn=False, b_mn=True, epi=0, bn=64, splits=7, partials=True),    # fc1 fwd
        dict(M=B, N=3136, K=512, a_mn=False, b_mn=False, epi=2, bn=64),                          # fc1 dgrad (unfused)
        dict(M=3136, N=512, K=B, a_mn=True, b_mn=True, epi=0, bn=128),                           # fc1 wgrad
        dict(M=3136, N=512, K=B, a_mn=True, b_mn=True, epi=2, bn=128),                           # fc1 wgrad, bf16 wire
    ]
    for c in cases:
        r, tag = _run_case(seed=B, **c)
        print("RATIO", tag, r)
        assert r <= 1.0, "err/bound %.3g: %s" % (r, tag)


def test_gemm_split_k_partials_with_more_splits_than_k_blocks():
    """Splits beyond the k-block count: CTAs that own no k-block must still store zero partial tiles."""
    for (M, N, K, splits) in [(200, 512, 100, 7), (37, 64, 64, 5), (128, 130, 300, 8)]:
        for bn in BNS:
            r, tag = _run_case(M, N, K, False, True, 0, bn, splits=splits, partials=True, seed=splits)
            print("RATIO", tag, r)
            assert r <= 1.0, "err/bound %.3g: %s" % (r, tag)


def test_gemm_split_k_atomics_more_splits_than_k_blocks():
    for bn in (64, 128):
        r, tag = _run_case(256, 512, 130, False, True, 1, bn, splits=16, seed=3)
        print("RATIO", tag, r)
        assert r <= 1.0, "err/bound %.3g: %s" % (r, tag)


@pytest.mark.parametrize("B,H", [(96, 128), (256, 256), (8192, 1024), (8192, 4096)])
def test_gemm_mlp_call_sites(B, H):
    """The MLP layers as CudaMlpEngine calls them: bias+ReLU forward, dgrad to bf16, wgrad with K = batch, and the
    output layer's weight gradient (N = 10, ldo = 10: the scalar-store tail).  Rows are sampled for the float64
    reference at batch 8192.  Measured worst err / bound on a B200 (1000 W): fp32 stores 0.04, fp32 atomics 0.10,
    bf16 stores 1.00 (the rounding of values exactly halfway between two bf16 numbers)."""
    bn = 256 if H % 256 == 0 else 128
    rows = None
    if B > 2048:
        rows = torch.cat([torch.arange(0, 160), torch.arange(B // 2 - 64, B // 2 + 64), torch.arange(B - 160, B)]).cuda()
    wrows = torch.cat([torch.arange(0, 130), torch.arange(H - 130, H)]).cuda() if H > 1024 else None
    cases = [
        (dict(M=B, N=H, K=784, a_mn=False, b_mn=True, epi=3, bn=bn), rows),            # layer 1 forward
        (dict(M=B, N=H, K=H, a_mn=False, b_mn=True, epi=3, bn=bn), rows),              # hidden forward
        (dict(M=B, N=H, K=H, a_mn=False, b_mn=False, epi=2, bn=bn), rows),             # dgrad
        (dict(M=H, N=H, K=B, a_mn=True, b_mn=True, epi=0, bn=bn), wrows),              # hidden wgrad
        (dict(M=784, N=H, K=B, a_mn=True, b_mn=True, epi=0, bn=bn), None),             # layer 1 wgrad
        (dict(M=H, N=10, K=B, a_mn=True, b_mn=True, epi=0, bn=64, ldo=10), wrows),     # output-layer wgrad
    ]
    for c, sel in cases:
        r, tag = _run_case(seed=H, sample_rows=sel, **c)
        print("RATIO", tag, r)
        assert r <= 1.0, "err/bound %.3g: %s" % (r, tag)
