"""tcgen05 plumbing self-test on real hardware (descriptors / swizzle / TMEM mapping)."""
import pytest
import torch

from samble_b200 import _lib as L

pytestmark = pytest.mark.gpu


def _tf32_trunc(t):
    return (t.view(torch.int32) & ~0x1FFF).view(torch.float32)


@pytest.mark.parametrize("K", [32, 64, 128])
def test_tc_gemm_selftest(K):
    g = torch.Generator().manual_seed(K)
    A = torch.randn(128, K, generator=g).cuda()
    B = torch.randn(128, K, generator=g).cuda()
    D = torch.zeros(128, 128, device="cuda")
    L.check(L.lib().samble_selftest_tc_gemm(L.ptr(A), L.ptr(B), K, L.ptr(D), None, None, L.stream()), "selftest")
    torch.cuda.synchronize()
    exact = A.double() @ B.double().t()
    trunc = _tf32_trunc(A).double() @ _tf32_trunc(B).double().t()
    err_exact = (D.double() - exact).abs().max().item()
    err_trunc = (D.double() - trunc).abs().max().item()
    print(f"K={K}: max|D-fp64| = {err_exact:.3e}, max|D-tf32trunc| = {err_trunc:.3e}")
    assert err_exact < 0.05 * (K ** 0.5), "tcgen05 result is not the GEMM: descriptor/swizzle/TMEM mapping is wrong"


@pytest.mark.parametrize("K", [32, 128, 256])
def test_tc_gemm_selftest_a_in_tmem(K):
    """tcgen05.mma reading A from tensor memory (parked with tcgen05.st): the operand path of csrc/mlp2.cu."""
    g = torch.Generator().manual_seed(K)
    A, B = torch.randn(128, K, generator=g).cuda(), torch.randn(128, K, generator=g).cuda()
    D = torch.zeros(128, 128, device="cuda")
    L.check(L.lib().samble_selftest_tc_gemm_ts(L.ptr(A), L.ptr(B), K, L.ptr(D), 0, 1, None, L.stream()), "selftest ts")
    torch.cuda.synchronize()
    ref = _tf32_trunc(A).double() @ _tf32_trunc(B).double().t()
    err = (D.double() - ref).abs().max().item()
    print(f"K={K}: max|D-tf32trunc| = {err:.3e}")
    assert err < 2e-3


def test_tc_gemm_selftest_nonswizzled_extra_k_step():
    """the compact SWIZZLE_NONE [128 x 32 B] slice that carries |b|^2 through the kNN GEMM."""
    g = torch.Generator().manual_seed(1)
    A, B = torch.randn(128, 64, generator=g).cuda(), torch.randn(128, 64, generator=g).cuda()
    Ax, Bx = torch.randn(128, 8, generator=g).cuda(), torch.randn(128, 8, generator=g).cuda()
    D = torch.zeros(128, 128, device="cuda")
    L.check(L.lib().samble_selftest_tc_gemm(L.ptr(A), L.ptr(B), 64, L.ptr(D), L.ptr(Ax), L.ptr(Bx), L.stream()), "selftest")
    torch.cuda.synchronize()
    ref = _tf32_trunc(A).double() @ _tf32_trunc(B).double().t() + _tf32_trunc(Ax).double() @ _tf32_trunc(Bx).double().t()
    err = (D.double() - ref).abs().max().item()
    print(f"ext: max|D-tf32trunc| = {err:.3e}")
    assert err < 1e-3


LIN_CASES = [  # (B, P, K, Nout, x_layout, out_layout, scale, shift, lrelu, residual, res_first)
    (2, 300, 128, 384, "rows", "rows", False, None, False, False, False),
    (2, 2048, 128, 512, "rows", "rows", True, "shared", True, False, False),
    (3, 257, 512, 128, "rows", "bcn", True, "shared", False, True, True),
    (2, 1000, 128, 1024, "bcn", "bcn", True, "cloud", True, False, False),
    (1, 130, 64, 128, "bcn", "rows", False, "shared", False, True, False),
    (2, 64, 1024, 256, "bcn", "bcn", True, "shared", True, False, False),
    (1, 77, 256, 50, "bcn", "bcn", False, None, False, False, False),
    (2, 96, 6, 64, "rows", "rows", False, "shared", False, False, False),
    (1, 128, 100, 200, "rows", "rows", True, None, True, True, False),
    (2, 515, 512, 128, "rows", "bcn", True, "shared", False, "rows", True),      # the N2P feed-forward tail
]


@pytest.mark.parametrize("case", LIN_CASES, ids=[f"B{c[0]}_P{c[1]}_K{c[2]}_N{c[3]}_{c[4]}_{c[5]}" for c in LIN_CASES])
def test_linear_3xtf32_matches_fp64(case):
    from samble_b200 import ops

    B, P, K, Nout, xl, ol, use_scale, shift_kind, lrelu, use_res, res_first = case
    g = torch.Generator().manual_seed(B * 1000 + P + K)
    x_rows = torch.randn(B, P, K, generator=g) * 2
    w = torch.randn(Nout, K, generator=g) / K ** 0.5
    scale = torch.rand(Nout, generator=g) + 0.5 if use_scale else None
    shift = None if shift_kind is None else (torch.randn(Nout, generator=g) if shift_kind == "shared" else torch.randn(B, Nout, generator=g))
    res_rows = torch.randn(B, P, Nout, generator=g) if use_res else None
    ref = x_rows.double() @ w.double().t()
    if use_res and res_first:
        ref = ref + res_rows.double()
    if scale is not None:
        ref = ref * scale.double()
    if shift is not None:
        ref = ref + (shift.double() if shift.dim() == 1 else shift.double().unsqueeze(1))
    if lrelu:
        ref = torch.where(ref > 0, ref, 0.2 * ref)
    if use_res and not res_first:
        ref = ref + res_rows.double()
    x = x_rows.cuda() if xl == "rows" else x_rows.transpose(1, 2).contiguous().cuda()
    rl = use_res if isinstance(use_res, str) else ol
    res = None if res_rows is None else (res_rows.cuda() if rl == "rows" else res_rows.transpose(1, 2).contiguous().cuda())
    y = ops.linear(x, w.cuda(), x_layout=xl, out_layout=ol, scale=None if scale is None else scale.cuda(),
                   shift=None if shift is None else shift.cuda(), lrelu=lrelu, residual=res, residual_first=res_first,
                   residual_layout=rl)
    torch.cuda.synchronize()
    y_rows = y if ol == "rows" else y.transpose(1, 2)
    assert tuple(y_rows.shape) == (B, P, Nout)
    err = (y_rows.double().cpu() - ref).abs().max().item()
    fp32 = (x_rows @ w.t()).double()                    # what a plain fp32 GEMM on the CPU gives, for scale
    print(f"max err vs fp64 {err:.2e}; an fp32 CPU GEMM is off by {(fp32 - x_rows.double() @ w.double().t()).abs().max().item():.2e}")
    assert err < 2e-5 * max(1.0, ref.abs().max().item())


SWAP_CASES = [(2, 2048, 128, 1024, False, None, True), (3, 384, 128, 512, True, "cloud", True), (2, 512, 512, 128, True, "shared", False),
              (16, 128, 64, 200, True, "shared", True)]


@pytest.mark.parametrize("case", SWAP_CASES, ids=[f"B{c[0]}_P{c[1]}_K{c[2]}_N{c[3]}" for c in SWAP_CASES])
def test_linear_pool_swapped_orientation_matches_row_per_thread(case):
    """samble_linear_pool on clouds of whole 128-row tiles runs linear_tma in the swapped orientation (weight tile as the A
    operand, the reduction over the points down each thread's own accumulator columns): same products in the same order as the
    row-per-thread butterfly kernel (samble_set_linear_debug(128)), so the maxima are identical; the means differ by the
    summation order only."""
    from samble_b200 import ops

    B, P, K, Nout, use_scale, shift_kind, lrelu = case
    g = torch.Generator().manual_seed(P + K + Nout)
    x = (torch.randn(B, P, K, generator=g) * 2).cuda()
    w = (torch.randn(Nout, K, generator=g) / K ** 0.5).cuda()
    scale = (torch.rand(Nout, generator=g) + 0.5).cuda() if use_scale else None
    shift = None if shift_kind is None else (torch.randn(Nout, generator=g) if shift_kind == "shared" else torch.randn(B, Nout, generator=g)).cuda()
    mx, mean = ops.linear_pool(x, w, scale=scale, shift=shift, lrelu=lrelu)
    L.lib().samble_set_linear_debug(128)
    try:
        mx0, mean0 = ops.linear_pool(x, w, scale=scale, shift=shift, lrelu=lrelu)
    finally:
        L.lib().samble_set_linear_debug(0)
    torch.cuda.synchronize()
    assert torch.equal(mx, mx0)
    assert (mean - mean0).abs().max().item() <= 1e-5 * max(1.0, mean0.abs().max().item())


POOL_CASES = [(2, 256, 128, 1024, True, "shared", True), (3, 96, 64, 200, False, None, False), (1, 2048, 128, 1024, True, "cloud", True),
              (4, 32, 36, 50, True, "shared", True), (2, 512, 512, 128, False, "shared", True)]


@pytest.mark.parametrize("case", POOL_CASES, ids=[f"B{c[0]}_P{c[1]}_K{c[2]}_N{c[3]}" for c in POOL_CASES])
def test_linear_pool_matches_fp64(case):
    """samble_linear_pool: max / mean over each cloud's points of the fused layer, activation never stored."""
    from samble_b200 import ops

    B, P, K, Nout, use_scale, shift_kind, lrelu = case
    g = torch.Generator().manual_seed(B * 77 + P + K)
    x = torch.randn(B, P, K, generator=g) * 2
    w = torch.randn(Nout, K, generator=g) / K ** 0.5
    scale = torch.rand(Nout, generator=g) + 0.5 if use_scale else None
    shift = None if shift_kind is None else (torch.randn(Nout, generator=g) if shift_kind == "shared" else torch.randn(B, Nout, generator=g))
    ref = x.double() @ w.double().t()
    if scale is not None:
        ref = ref * scale.double()
    if shift is not None:
        ref = ref + (shift.double() if shift.dim() == 1 else shift.double().unsqueeze(1))
    if lrelu:
        ref = torch.where(ref > 0, ref, 0.2 * ref)
    mx, mean = ops.linear_pool(x.cuda(), w.cuda(), scale=None if scale is None else scale.cuda(),
                               shift=None if shift is None else shift.cuda(), lrelu=lrelu)
    torch.cuda.synchronize()
    tol = 2e-5 * max(1.0, ref.abs().max().item())
    assert (mx.double().cpu() - ref.max(dim=1)[0]).abs().max().item() < tol
    assert (mean.double().cpu() - ref.mean(dim=1)).abs().max().item() < tol
    only_max, none = ops.linear_pool(x.cuda(), w.cuda(), scale=None if scale is None else scale.cuda(),
                                     shift=None if shift is None else shift.cuda(), lrelu=lrelu, want_mean=False)
    assert none is None and torch.equal(only_max, mx)
    # deterministic: fixed reduction order, no atomics
    mx2, mean2 = ops.linear_pool(x.cuda(), w.cuda(), scale=None if scale is None else scale.cuda(),
                                 shift=None if shift is None else shift.cuda(), lrelu=lrelu)
    assert torch.equal(mx, mx2) and torch.equal(mean, mean2)


@pytest.mark.parametrize("case", [(2, 256, 128, 640), (3, 128, 64, 100), (2, 512, 1024, 128), (2, 256, 4096, 128), (1, 128, 4100, 64)],
                         ids=lambda c: f"B{c[0]}_R{c[1]}_K{c[2]}_N{c[3]}")
def test_cloud_matmul_matches_fp64(case):
    """samble_cloud_matmul: per-cloud weights, and the softmax-row epilogue with known row statistics.  K = 4096 is the
    longest contraction it takes (DownSampleToken's attention rows x V at N = 4096 keys, with the token share as the
    residual); one key more is refused."""
    from samble_b200 import ops

    B, R, K, Nout = case
    g = torch.Generator().manual_seed(B + R + K)
    x = torch.randn(B, R, K, generator=g)
    w = torch.randn(B, Nout, K, generator=g) / K ** 0.5
    if K > 4096:
        with pytest.raises(ValueError, match="too large"):
            ops.cloud_matmul(x.cuda(), w.cuda())
        return
    ref = torch.matmul(x.double(), w.double().transpose(1, 2))
    y = ops.cloud_matmul(x.cuda(), w.cuda())
    assert (y.double().cpu() - ref).abs().max().item() < 2e-5 * max(1.0, ref.abs().max().item())
    res = torch.randn(B, R, Nout, generator=g)
    y_res = ops.cloud_matmul(x.cuda(), w.cuda(), residual=res.cuda())
    assert (y_res.double().cpu() - ref - res.double()).abs().max().item() < 2e-5 * max(1.0, (ref + res.double()).abs().max().item())
    div = 3.0
    logits = ref / div
    rmax = logits.max(dim=-1)[0]
    rsum = torch.exp(logits - rmax.unsqueeze(-1)).sum(-1)
    p = ops.cloud_matmul(x.cuda(), w.cuda(), row_max=rmax.float().cuda(), row_sum=rsum.float().cuda(), logit_div=div)
    pref = torch.softmax(logits, dim=-1)
    assert (p.double().cpu() - pref).abs().max().item() < 2e-6
    assert (p.double().cpu().sum(-1) - 1).abs().max().item() < 1e-5


# ---------------------------------------------------------------- exact-product GEMM (csrc/xgemm.cu)

XG_SHAPES = [  # (Ba, Ra, Bb, Rb, C, scale of A, scale of B)
    (2, 300, 2, 200, 128, 1.0, 1.0),
    (3, 128, 1, 384, 128, 40.0, 0.09),        # shared B (a weight matrix), magnitudes far from 1
    (1, 1000, 1, 70, 64, 1e-3, 1e3),
    (2, 257, 2, 129, 20, 1.0, 1.0),           # channel count padded to 64, ragged tiles
    (4, 2048, 4, 2048, 128, 3.0, 1.0),        # DownSampleToken q k^T at N=2048: a CTA walks several row tiles
]


@pytest.mark.parametrize("shape", XG_SHAPES, ids=lambda s: f"A{s[0]}x{s[1]}_B{s[2]}x{s[3]}_C{s[4]}")
def test_xgemm_is_exact_and_order_independent(shape):
    """The tensor-core accumulation of the digit products is EXACT: bit-identical to the int32 restatement, and
    within the digit truncation bound of the fp64 product."""
    from samble_b200 import ops

    Ba, Ra, Bb, Rb, C, sa, sb = shape
    g = torch.Generator().manual_seed(Ra + Rb)
    A = (torch.randn(Ba, Ra, C, generator=g) * sa).cuda()
    Bm = (torch.randn(Bb, Rb, C, generator=g) * sb).cuda()
    A[0, 0] = 0                                                 # a zero row; one cloud much smaller than the others
    if Ba > 1:
        A[-1] *= 1e-2
    ad, bd = ops.digits(A), ops.digits(Bm)
    out = ops.xgemm(ad, bd)
    ref = ops.xgemm(ad, bd, reference=True)
    torch.cuda.synchronize()
    assert torch.equal(out, ref), f"max |tc - int32| = {(out - ref).abs().max().item():.3e}"
    exact = A.double() @ (Bm.double().transpose(1, 2) if Bb > 1 else Bm[0].double().t())
    # digit pairs of weight < 2^-24 are dropped (<= ~K 2^-29 maxA maxB with the power-of-two ceilings), then three fused
    # roundings of a partial sum no larger than the result: C is the fp64 product to within ~2 ulp
    amax = A.abs().amax(dim=(1, 2)).double().clamp_min(1e-30)
    bmax = Bm.abs().amax(dim=(1, 2)).double()
    bound = (C * 2.0 ** -26 * amax * (bmax if Bb > 1 else bmax[0])).view(Ba, 1, 1) + 2.0 ** -22 * exact.abs()
    err = (out.double() - exact).abs()
    assert bool((err <= bound + 1e-30).all()), float((err / bound).max())
    rel = err.max().item() / exact.abs().max().item()
    print(f"xgemm {shape}: max err / max|C| = {rel:.2e}")


def test_xgemm_amax_feeds_the_next_slicing():
    from samble_b200 import ops

    g = torch.Generator().manual_seed(5)
    x = torch.randn(3, 640, 128, generator=g).cuda()
    w = (torch.randn(384, 128, generator=g) / 11.3).cuda()
    out, amax = ops.xgemm(ops.digits(x), ops.weight_digits(w), amax_group=128)
    want = out.view(3, 640, 3, 128).abs().amax(dim=(1, 3))                     # (B, 3 groups)
    assert torch.equal(amax.view(torch.float32), want)
    q, k = out[..., :128], out[..., 128:256]
    qd, kd = ops.digits(q, amax, 0), ops.digits(k, amax, 1)
    qd2, kd2 = ops.digits(q.contiguous()), ops.digits(k.contiguous())          # own reduction pass
    assert torch.equal(qd.planes, qd2.planes) and torch.equal(kd.planes, kd2.planes) and torch.equal(qd.scale, qd2.scale)
    # the digits reconstruct the value to 2^-32 of the cloud's power-of-two ceiling (exactly, for all but tiny elements)
    pl = qd.planes.view(torch.bfloat16).view(4, 3, 640, 128).double()
    rec = (pl[0] + pl[1] / 2 ** 8 + pl[2] / 2 ** 16 + pl[3] / 2 ** 24) * qd.scale.double().view(3, 1, 1)
    ceil2 = torch.exp2(torch.floor(torch.log2(want[:, 0].double())) + 1).view(3, 1, 1)
    assert float(((rec - q.double()).abs() / ceil2).max()) <= 2.0 ** -32
    assert float((rec == q.double()).double().mean()) > 0.95


ROW_STATS_CASES = [(2, 2048, 4, 4.0, 128), (1, 1000, 6, 8.0, 128), (2, 512, 4, 1.0, 128), (2, 1000, 8, 4.0, 64)]


@pytest.mark.parametrize("B,N,nb,sharp,D", ROW_STATS_CASES,
                         ids=["-".join(map(str, c[:4])) + ("" if c[4] == 128 else f"-D{c[4]}") for c in ROW_STATS_CASES])
def test_ds_row_stats_exact_vs_fp64(B, N, nb, sharp, D):
    """logsumexp of q [k | k_tok]^T / sqrt(D) from the exact GEMM: error of one fp32 rounding of the logit, not of a
    tensor-core accumulation chain."""
    import math

    from samble_b200 import ops

    g = torch.Generator().manual_seed(N + nb)
    q = (torch.randn(B, N, D, generator=g) * sharp).cuda()
    k = torch.randn(B, N, D, generator=g).cuda()
    k_tok = torch.randn(nb, D, generator=g).cuda()
    rowmax, rowsum, tok = ops.ds_row_stats_exact(ops.digits(q), ops.digits(k), q, k_tok)
    logits = torch.cat([q.double() @ k.double().transpose(1, 2), q.double() @ k_tok.double().t()], -1) / math.sqrt(D)
    lse = rowmax.double() + torch.log(rowsum.double())
    err = (lse - torch.logsumexp(logits, -1)).abs().max().item()
    ulp = 2.0 ** -23 * float(logits.abs().max())
    print(f"LSE error {err:.2e} (one ulp of the largest logit: {ulp:.2e})")
    assert err <= 2 * ulp + 5e-7
    torch.testing.assert_close(tok.double(), logits[..., N:], atol=1e-4, rtol=1e-5)
