"""The native backward kernels (csrc/backward.cu) one op at a time, off the shipped shapes, against fp64 on the CPU.

Every reference is the literal statement of the operation in fp64, fed the indices the native call used, so a failure
points at one kernel:
  - ops.n2p_attend forward and backward (n2p_attend_bwd_kernel) against autograd of the reference's gathered-difference
    form (samble_b200.testing.n2p_attend_literal), at every lanes-per-head value the kernel takes, K up to 32, N not a
    multiple of 8, with kNN, repeated, hub, self-only and all-points neighbour sets, and ordinary, saturated and uniform
    softmaxes.
  - index_points / group / gather_by_idx backward (index_points_bwd_kernel, gather_by_idx_bwd_kernel) with small-integer
    upstream gradients: the fp32 atomic sums are then exact in any order, so the gradient must equal fp64 bit for bit.
  - the kNN distance gradient at coincident and duplicated points, k = 1 and Nq != Nr.
Also the layout contract of the ops that consume neighbour indices (strided views in, the contiguous call's bits out)
and the widths the Neighbor2Point kernels refuse.
"""
import pytest
import torch

from samble_b200 import _lib as L
from samble_b200 import blocks, ops
from samble_b200.config import Cfg, _attention
from samble_b200.testing import n2p_attend_literal, synthetic_features
from tests.test_gpu_backward import _group_ref, _knn_ref_dist

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

# Per point row r of a gradient (or output) g against its fp64 reference:
#     max_r |g - g_ref|  <=  N2P_TOL * max(max_r |g_ref|, 1e-3 * max_all |g_ref|)  +  ROUNDING * max_r A
# A is the fp64 sum of the absolute values of the terms the kernel adds up for that element (each softmax weight
# counted with the fp32 rounding of its logit).  The second term is fp32 rounding where the terms cancel: a saturated
# softmax (dq, dk ~ e^-60 of their natural size) or self-only rows (exactly 0 in the reference).  A dropped, doubled or
# misplaced term is an error of the order of A itself.
# Measured over all N2P_CASES on an NVIDIA B200 (1000 W power limit), both kernel selections:
#   worst |g - g_ref| per row <= 3.8 * 2^-24 * A (C=128 H=32 K=32 repeat/uniform, dv), so ROUNDING = 16 ulps of A;
#   worst |g - g_ref| / max(|g_ref|_row, 1e-3 |g_ref|_all) = 3.8e-6 where the terms do not cancel (C=128 H=2 K=2 kNN,
#   uniform), so N2P_TOL = 2e-5.  (Where they do, it is up to 8.2e-4 in the saturated cases and unbounded in the
#   self-only ones, whose reference is 0; those rows are within the rounding term.)
#   The largest share of the whole bound any tensor used was 0.046 with ROUNDING = 64 ulps.
N2P_TOL = 2e-5
ROUNDING = 16 * 2.0 ** -24


def cu(t):
    return t.to(DEV)


def _id(v):
    return str(v).replace("torch.", "") if isinstance(v, torch.dtype) else ("hub" if v is True else "spread" if v is False else None)


def _rowwise(g, ref, A):
    """Per-row errors of g against ref: (share of the bound above used, worst |g - ref| / max(|ref|_row, 1e-3 |ref|_all),
    worst |g - ref| / A_row in units of 2^-24), each the max over the rows."""
    g, ref, A = g.detach().cpu().double(), ref.detach().cpu().double(), A.double()
    C = g.shape[-1]
    err = (g - ref).abs().reshape(-1, C).amax(1)
    scale = torch.clamp(ref.abs().reshape(-1, C).amax(1), min=1e-3 * float(ref.abs().max()))
    a = A.reshape(-1, C).amax(1)
    bound = N2P_TOL * scale + ROUNDING * a

    def worst(den):
        r = torch.where(err > 0, err / den, torch.zeros_like(err))   # (0 / 0: an exact zero where the reference is 0)
        return float(r.max())
    return worst(bound), worst(scale), worst(a * 2.0 ** -24)


def _n2p_term_scales(qkv, idx, heads, probe):
    """fp64 magnitudes A of the terms the native kernels sum, per element: (out (B,N,C), grad (B,N,3C)).
      forward   out_i = sum_j p_ij v_j - v_i
      backward  ds_ij = p_ij (dp_ij - sum_j' p_ij' dp_ij') / sqrt(d),  dp_ij = g_i . v_j
                dq_i = sum_j ds_ij k_j,  dk_j += ds_ij q_i,  dv_j += p_ij g_i,  dv_i -= g_i
    plus the terms of the reference's own form that cancel in exact arithmetic (sum_j ds_ij (k_i | q_i), with
    k_ij = k_j - k_i), each p_ij weighted by (1 + L_ij), L_ij = sum_c |q_ic k_jc| / sqrt(d): the fp32 logit error is
    ~eps L_ij."""
    B, N, C3 = qkv.shape
    C, K = C3 // 3, idx.shape[-1]
    D = C // heads
    x = qkv.double()
    q, k, v = (x[..., i * C:(i + 1) * C] for i in range(3))
    flat = idx.long().reshape(B, -1, 1).expand(-1, -1, C)
    kj = torch.gather(k, 1, flat).view(B, N, K, heads, D)
    vj = torch.gather(v, 1, flat).view(B, N, K, heads, D)
    qh, gh = q.reshape(B, N, heads, D), probe.double().reshape(B, N, heads, D)
    p = torch.softmax(torch.einsum("bnhd,bnkhd->bnhk", qh, kj - k.view(B, N, 1, heads, D)) / D ** 0.5, -1)
    L = torch.einsum("bnhd,bnkhd->bnhk", qh.abs(), kj.abs()) / D ** 0.5
    pw = p * (1 + L)
    a_out = torch.einsum("bnhk,bnkhd->bnhd", pw, vj.abs()).reshape(B, N, C) + v.abs()
    dp = torch.einsum("bnhd,bnkhd->bnhk", gh.abs(), vj.abs())
    w = pw * (dp + (p * dp).sum(-1, keepdim=True)) / D ** 0.5                          # |ds_ij|, with its rounding
    a_q = torch.einsum("bnhk,bnkhd->bnhd", w, kj.abs()).reshape(B, N, C) + w.sum(-1).repeat_interleave(D, -1) * k.abs()

    def scatter(t):                                                                   # (B,N,K,C) -> rows j
        return torch.zeros(B, N, C, dtype=torch.float64).scatter_add_(1, flat, t.reshape(B, N * K, C))

    a_k = scatter(torch.einsum("bnhk,bnhd->bnkhd", w, qh.abs())) + w.sum(-1).repeat_interleave(D, -1) * q.abs()
    a_v = scatter(torch.einsum("bnhk,bnhd->bnkhd", pw, gh.abs())) + probe.double().abs()
    return a_out, torch.cat([a_q, a_k, a_v], -1)


# ---------------------------------------------------------------- a. ops.n2p_attend, forward and backward

# (C, heads) covers lanes per head lph = C / heads / 4 = 32, 16, 8, 4, 2, 1, and C < 128 with idle lanes (64/1, 96/3,
# 48/3, 48/12, 4/1).  Pairwise over K in {1, 2, 7, 31, 32}, N in {9, 300, 1027} (the last CTA is partial), B up to 3,
# int32 / int64, the index patterns and the logit regimes.
N2P_CASES = [  # C, heads, K, N, B, idx dtype, pattern, regime
    (128, 1, 32, 1027, 2, torch.int32, "knn", "ordinary"),
    (128, 2, 31, 300, 3, torch.int64, "repeat", "saturated"),
    (128, 4, 32, 300, 2, torch.int32, "hub", "ordinary"),
    (128, 4, 7, 1027, 1, torch.int64, "knn", "uniform"),
    (128, 4, 31, 31, 2, torch.int64, "all", "saturated"),
    (128, 8, 2, 9, 3, torch.int32, "repeat", "ordinary"),
    (128, 8, 31, 31, 1, torch.int32, "all", "ordinary"),
    (128, 16, 7, 300, 1, torch.int64, "hub", "saturated"),
    (128, 16, 1, 9, 2, torch.int32, "hub", "ordinary"),
    (128, 32, 1, 1027, 2, torch.int32, "knn", "ordinary"),
    (128, 32, 32, 300, 3, torch.int64, "repeat", "uniform"),
    (128, 1, 1, 300, 3, torch.int64, "self", "saturated"),
    (128, 2, 2, 1027, 1, torch.int32, "knn", "uniform"),
    (64, 1, 32, 9, 2, torch.int64, "repeat", "saturated"),
    (64, 1, 7, 300, 1, torch.int32, "self", "uniform"),
    (96, 3, 31, 31, 1, torch.int32, "all", "ordinary"),
    (96, 3, 32, 1027, 2, torch.int64, "knn", "saturated"),
    (48, 3, 2, 1027, 3, torch.int64, "hub", "uniform"),
    (48, 12, 32, 300, 2, torch.int32, "self", "ordinary"),
    (48, 12, 31, 9, 2, torch.int64, "repeat", "uniform"),
    (4, 1, 7, 9, 3, torch.int32, "knn", "saturated"),
    (4, 1, 31, 1027, 1, torch.int64, "hub", "ordinary"),
    (4, 1, 2, 300, 2, torch.int64, "self", "ordinary"),
]


def _n2p_inputs(C, K, N, B, pattern, regime, seed):
    g = torch.Generator().manual_seed(seed)
    qkv = torch.randn(B, N, 3 * C, generator=g)
    qkv[..., :C] *= {"ordinary": 1.0, "saturated": 200.0, "uniform": 0.0}[regime]     # logits up to ~1e3: exp overflows
    if pattern == "knn":           # the training path's own neighbour sets (Neighbor2PointAttention's differentiable branch)
        idx = ops.knn_indices(cu(synthetic_features(B, 8, N, seed)), K, ordered=False).cpu()
    elif pattern == "self":        # every entry of row i is i
        idx = torch.arange(N).view(1, N, 1).expand(B, N, K)
    elif pattern == "all":         # K = N: every row lists every point, in its own order
        assert K == N
        idx = torch.argsort(torch.rand(B, N, N, generator=g), dim=-1)
    else:
        idx = torch.randint(0, N, (B, N, K), generator=g)
        if pattern == "repeat":    # the second half of every row repeats the first
            idx[..., K // 2:] = idx[..., :K - K // 2]
        else:                      # hub: half of all rows list point 0
            idx[:, ::2, 0] = 0
    probe = torch.randn(B, N, C, generator=g)
    return qkv, idx.contiguous(), probe


@pytest.mark.parametrize("C,H,K,N,B,dt,pattern,regime", N2P_CASES,
                         ids=[f"C{c[0]}_H{c[1]}_K{c[2]}_N{c[3]}_B{c[4]}_{str(c[5])[-5:]}_{c[6]}_{c[7]}" for c in N2P_CASES])
def test_n2p_attend_vs_fp64(C, H, K, N, B, dt, pattern, regime):
    """The grad path's forward equals the fused no-grad forward bit for bit under both kernel selections (the eight-lane
    kernel runs for C = 128 / 4 heads in mode 0); the output and dq, dk, dv match fp64 autograd of the literal form row by
    row.  K = 1 gives dq = dk = 0 exactly; self-only rows give output 0 (exactly for K <= 2: the kernels form
    sum_j p_j v_j / sum_j p_j - v_i, which rounds for longer sums)."""
    qkv, idx, probe = _n2p_inputs(C, K, N, B, pattern, regime, seed=C * 7 + K * 3 + N)
    r = qkv.double().requires_grad_(True)
    ref = n2p_attend_literal(r, idx, H)
    (g_ref,) = torch.autograd.grad(ref, r, probe.double())
    a_out, a_g = _n2p_term_scales(qkv, idx, H, probe)
    worst = {}
    for mode in (0, 1):
        L.lib().samble_set_n2p_mode(mode)
        try:
            with torch.no_grad():
                fused = ops.n2p_attend(cu(qkv), cu(idx).to(dt), H)
            rc = cu(qkv).requires_grad_(True)
            out = ops.n2p_attend(rc, cu(idx).to(dt), H)
            (g,) = torch.autograd.grad(out, rc, cu(probe))
        finally:
            L.lib().samble_set_n2p_mode(0)
        assert torch.equal(out.detach(), fused), mode
        worst[f"out{mode}"] = _rowwise(out, ref, a_out)
        for i, name in enumerate("qkv"):
            sl = slice(i * C, (i + 1) * C)
            worst[f"d{name}{mode}"] = _rowwise(g[..., sl], g_ref[..., sl], a_g[..., sl])
        if K == 1:
            assert int(torch.count_nonzero(g[..., :2 * C])) == 0, "K = 1: dq and dk must be exactly 0"
        if pattern == "self" and K <= 2:
            assert int(torch.count_nonzero(out)) == 0
        assert bool(torch.isfinite(g).all())
    print(f"n2p C={C} H={H} K={K} N={N} {pattern}/{regime} -- tensor: share of bound, rel. to |ref|, ulps of A:",
          ", ".join(f"{k} {v[0]:.3f} {v[1]:.1e} {v[2]:.2f}" for k, v in worst.items()))
    bad = {k: v for k, v in worst.items() if not v[0] <= 1.0}
    assert not bad, bad


# ---------------------------------------------------------------- b. gather / group / gather_by_idx backward, exact

def _int_probe(shape, seed):
    """Upstream gradient of small integers (|g| <= 16): with fewer than 2^20 contributions per element every partial
    sum is an integer below 2^24, so fp32 atomics in any order give the exact sum."""
    return torch.randint(-16, 17, shape, generator=torch.Generator().manual_seed(seed)).float()


def _indices(B, R, N, hub, seed):
    if hub:                                                   # every row points at one point
        return torch.full((B, R), N // 3, dtype=torch.int64)
    return torch.randint(0, N, (B, R), generator=torch.Generator().manual_seed(seed))


# R*C = 2048*32*16 = 1,048,576 per cloud is above the 148*16*256 = 606,208 threads the backward grid launches, so every
# thread takes at least two grid-stride steps.
GATHER_CASES = [  # B, N, M, K, C, idx dtype, hub
    (3, 2048, 2048, 32, 16, torch.int32, False),
    (3, 2048, 2048, 32, 16, torch.int64, True),
    (3, 300, 200, 7, 1, torch.int64, False),
    (3, 300, 200, 7, 3, torch.int32, True),
    (3, 257, 129, 5, 5, torch.int64, False),
    (2, 513, 100, 9, 130, torch.int32, False),
]


@pytest.mark.parametrize("B,N,M,K,C,dt,hub", GATHER_CASES, ids=_id)
def test_index_points_backward_is_exact(B, N, M, K, C, dt, hub):
    p = synthetic_features(B, N, C, N + C)
    idx = _indices(B, M * K, N, hub, seed=M + K).view(B, M, K)
    probe = _int_probe((B, M, K, C), seed=C)
    pr = p.double().requires_grad_(True)
    ref = torch.gather(pr, 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, M, K, C)
    (g_ref,) = torch.autograd.grad(ref, pr, probe.double())
    pc = cu(p).requires_grad_(True)
    out = ops.index_points(pc, cu(idx).to(dt))
    assert torch.equal(out.detach().cpu(), ref.detach().float())
    (g,) = torch.autograd.grad(out, pc, cu(probe))
    assert torch.equal(g.cpu(), g_ref.float())


GROUP_CASES = [  # B, N, K, C, idx dtype, hub
    (3, 2048, 32, 16, torch.int64, False),
    (3, 300, 7, 1, torch.int32, True),
    (3, 129, 9, 5, torch.int64, False),
    (2, 200, 20, 130, torch.int32, False),
    (3, 100, 4, 3, torch.int32, False),
]


@pytest.mark.parametrize("group_type", ["neighbor", "diff", "center_neighbor", "center_diff"])
@pytest.mark.parametrize("B,N,K,C,dt,hub", GROUP_CASES, ids=_id)
def test_group_backward_is_exact(B, N, K, C, dt, hub, group_type):
    x = synthetic_features(B, C, N, N + K)
    idx = _indices(B, N * K, N, hub, seed=N * K).view(B, N, K)
    xr = x.double().requires_grad_(True)
    ref = _group_ref(xr, idx, group_type)
    probe = _int_probe(tuple(ref.shape), seed=K + C)
    (g_ref,) = torch.autograd.grad(ref, xr, probe.double())
    xc = cu(x).requires_grad_(True)
    out = ops._group_from_idx(xc, cu(idx).to(dt), group_type)
    assert torch.equal(out.detach().cpu(), ref.detach().float())
    (g,) = torch.autograd.grad(out, xc, cu(probe))
    assert torch.equal(g.cpu(), g_ref.float())


GATHER_BY_IDX_CASES = [  # B, C, N, M, idx dtype, hub   (M > N: indices repeat)
    (3, 130, 50, 700, torch.int32, False),
    (3, 1, 300, 1000, torch.int64, False),
    (3, 5, 7, 2000, torch.int32, False),
    (3, 16, 1000, 40000, torch.int64, False),        # C*M = 640,000 per cloud: two grid-stride steps
    (3, 3, 10, 5000, torch.int64, True),
]


@pytest.mark.parametrize("B,C,N,M,dt,hub", GATHER_BY_IDX_CASES, ids=_id)
def test_gather_by_idx_backward_is_exact(B, C, N, M, dt, hub):
    x = synthetic_features(B, C, N, C + N)
    idx = _indices(B, M, N, hub, seed=M).view(B, 1, M)
    xr = x.double().requires_grad_(True)
    ref = torch.gather(xr, 2, idx.expand(-1, C, -1))
    probe = _int_probe((B, C, M), seed=N)
    (g_ref,) = torch.autograd.grad(ref, xr, probe.double())
    xc = cu(x).requires_grad_(True)
    out = ops.gather_by_idx(xc, cu(idx).to(dt))
    assert torch.equal(out.detach().cpu(), ref.detach().float())
    (g,) = torch.autograd.grad(out, xc, cu(probe))
    assert torch.equal(g.cpu(), g_ref.float())


# ---------------------------------------------------------------- c. kNN distance gradient edges

# per row, |g - g_ref| / max(|g_ref|_row, 1e-3 |g_ref|_all); worst measured on an NVIDIA B200 (1000 W): 3.1e-6
KNN_TOL = 1e-5
KNN_CASES = [  # C, k, Nq, Nr, query points repeated in the reference set, duplicated reference points
    (3, 1, 300, 160, "some", False),
    (3, 8, 257, 513, "some", True),
    (16, 32, 100, 700, "none", True),
    (3, 1, 500, 500, "all", False),
]


@pytest.mark.parametrize("C,k,Nq,Nr,coincident,duplicated", KNN_CASES)
def test_knn_distance_gradient_edges(C, k, Nq, Nr, coincident, duplicated):
    """Gradients of ops.knn's distances w.r.t. both point sets against fp64 autograd of the reference's cdist form
    (_knn_ref_dist) on the native indices, per row.  A pair of coincident points has subgradient 0: the native gradient
    must come out finite and take nothing from those pairs, so the reference's probe is zeroed there (and only there)."""
    B = 2
    g = torch.Generator().manual_seed(C + k + Nq)
    a = torch.randn(B, Nq, C, generator=g)
    b = a.clone() if coincident == "all" else torch.randn(B, Nr, C, generator=g)
    if coincident == "some":
        b[:, :min(Nq, Nr) // 2] = a[:, :min(Nq, Nr) // 2]
    if duplicated:
        b[:, -40:-20] = b[:, -20:]
    ac, bc = cu(a).requires_grad_(True), cu(b).requires_grad_(True)
    neg, idx = ops.knn(ac, bc, k)
    probe = torch.randn(B, Nq, k, generator=g)
    ga, gb = torch.autograd.grad(-neg, (ac, bc), cu(probe))
    assert bool(torch.isfinite(ga).all()) and bool(torch.isfinite(gb).all())
    idx = idx.cpu()
    same = (a.unsqueeze(2) == torch.gather(b, 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, Nq, k, C)).all(-1)
    assert bool(same.any()) == (coincident != "none")
    ar, br = a.double().requires_grad_(True), b.double().requires_grad_(True)
    ga_ref, gb_ref = torch.autograd.grad(_knn_ref_dist(ar, br, idx), (ar, br), probe.double() * ~same)
    if coincident == "all":                 # k = 1 and every query is its own nearest point: no gradient at all
        assert int(torch.count_nonzero(ga)) == 0 and int(torch.count_nonzero(gb)) == 0
        return
    worst = []
    for x, r in ((ga, ga_ref), (gb, gb_ref)):
        x, r = x.cpu().double(), r.double()
        err = (x - r).abs().amax(-1)
        scale = r.abs().amax(-1).clamp(min=1e-3 * float(r.abs().max()))
        worst.append(float((err / scale).max()))
    print(f"knn C={C} k={k} Nq={Nq} Nr={Nr}: worst per-row relative error (a, b) {worst[0]:.2e} {worst[1]:.2e}")
    assert max(worst) <= KNN_TOL, worst


# ---------------------------------------------------------------- d. layout contract of the index-consuming ops

def _idx_views(idx32):
    """(B,N,32) search -> [(name, idx (B,N,16) non-contiguous view, the same indices contiguous)]."""
    sl = idx32[..., :16]
    perm = sl.transpose(1, 2).contiguous().transpose(1, 2)             # strides (16N, 1, N)
    assert not sl.is_contiguous() and not perm.is_contiguous()
    return [("slice", sl), ("permuted", perm), ("int64 slice", idx32.long()[..., :16])]


def _row_views(t, seed):
    """t (B,N,W) -> [(name, the same values as a view the kernels address differently)]."""
    B, N, W = t.shape
    wide = torch.full((B, N, W + 12), float("nan"), device=t.device)
    wide[..., 4:4 + W] = t                                             # column slice of a wider row buffer, aligned
    odd = torch.full((B, N, W + 13), float("nan"), device=t.device)
    odd[..., 1:1 + W] = t                                              # misaligned rows, odd pitch
    strided = torch.full((B, N, 2 * W), float("nan"), device=t.device)
    strided[..., ::2] = t                                              # inner stride 2
    nbw = t.transpose(0, 1).contiguous().transpose(0, 1)               # batch pitch W != N * row pitch
    return [("column slice", wide[..., 4:4 + W]), ("misaligned", odd[..., 1:1 + W]), ("inner stride 2", strided[..., ::2]),
            ("batch-inner", nbw)]


@pytest.mark.parametrize("C,H", [(128, 4), (64, 2)])
def test_n2p_attend_layouts(C, H):
    """ops.n2p_attend with and without grad: non-contiguous indices and strided qkv give the contiguous call's bits."""
    B, N = 2, 300
    g = torch.Generator().manual_seed(C)
    qkv = cu(torch.randn(B, N, 3 * C, generator=g))
    idx32 = ops.knn_indices(cu(synthetic_features(B, 8, N, 1)), 32, ordered=False)
    for grad in (False, True):
        def call(t, i):
            with torch.set_grad_enabled(grad):                   # (detach keeps the view's strides and makes it a leaf)
                return ops.n2p_attend(t.detach().requires_grad_(grad), i, H).detach()
        for name, idx in _idx_views(idx32):
            want = call(qkv, idx.contiguous())
            assert torch.equal(call(qkv, idx), want), (grad, name)
            for rname, view in _row_views(qkv, 0):
                assert torch.equal(call(view, idx), want), (grad, name, rname)
        with pytest.raises(TypeError, match="qkv must be float32"):
            call(qkv.double(), idx32)
        with pytest.raises(TypeError, match="int32 or int64"):
            call(qkv, idx32.float())
        with pytest.raises(TypeError, match="int32 or int64"):
            call(qkv, idx32.to(torch.int16))


def test_n2p_attend_grad_path_refuses_float_indices():
    """autograd.N2PAttend itself (not only the ops wrapper) refuses an index dtype the kernels cannot read."""
    from samble_b200 import autograd as AG
    qkv = cu(torch.randn(1, 64, 3 * 32)).requires_grad_(True)
    idx = ops.knn_indices(cu(synthetic_features(1, 8, 64, 2)), 8)
    with pytest.raises(TypeError, match="int32 or int64"):
        AG.N2PAttend.apply(qkv, idx.float(), 1)
    with pytest.raises(TypeError, match="int32 or int64"):
        AG.IndexPoints.apply(cu(torch.randn(1, 64, 4)).requires_grad_(True), idx.to(torch.uint8))


@pytest.mark.parametrize("mode", [0, 1])
@pytest.mark.parametrize("C1,C2,K", [(64, 128, 16), (48, 64, 16)])
def test_edge_mlp_max_layouts(C1, C2, K, mode):
    """ops.edge_mlp_max (tensor-core and FFMA kernels): non-contiguous indices and strided pr give the contiguous call's
    bits."""
    B, N = 2, 300
    g = torch.Generator().manual_seed(C1 + C2)
    pr = cu(torch.randn(B, N, 2 * C1, generator=g))
    w2, b2 = cu(torch.randn(C2, C1, generator=g) / C1 ** 0.5), cu(torch.randn(C2, generator=g))
    idx32 = ops.knn_indices(cu(synthetic_features(B, 8, N, 3)), 32, ordered=False)
    L.lib().samble_set_edge_mode(mode)
    try:
        with torch.no_grad():
            for name, idx in _idx_views(idx32):
                idx = idx[..., :K]
                want = ops.edge_mlp_max(pr, idx.contiguous(), w2, b2)
                assert torch.equal(ops.edge_mlp_max(pr, idx, w2, b2), want), name
                for rname, view in _row_views(pr, 0):
                    assert torch.equal(ops.edge_mlp_max(view, idx, w2, b2), want), (name, rname)
            with pytest.raises(TypeError, match="pr must be float32"):
                ops.edge_mlp_max(pr.double(), idx32, w2, b2)
            with pytest.raises(TypeError, match="int32 or int64"):
                ops.edge_mlp_max(pr, idx32.to(torch.int16), w2, b2)
            with pytest.raises(RuntimeError, match="neighbour indices must be"):
                ops.edge_mlp_max(pr, idx32[:, :-1], w2, b2)
    finally:
        L.lib().samble_set_edge_mode(0)


def test_ds_edge_score_layouts():
    """ops.ds_edge_score: non-contiguous indices, q / k as column slices of one row buffer (as DownSampleToken passes
    them) or other strided views, and strided row statistics give the contiguous call's bits."""
    B, N, D = 2, 384, 64
    g = torch.Generator().manual_seed(D)
    q, k = torch.randn(B, N, D, generator=g), torch.randn(B, N, D, generator=g)
    logits = q.double() @ k.double().transpose(1, 2) / D ** 0.5
    m = logits.max(-1)[0]
    s = torch.exp(logits - m.unsqueeze(-1)).sum(-1)
    q, k, m, s = cu(q), cu(k), cu(m.float()), cu(s.float())
    idx32 = ops.knn_indices(cu(synthetic_features(B, 8, N, 4)), 32, ordered=False)
    ms = torch.stack([m, s], -1)                                       # (B,N,2): rowmax / rowsum with stride 2
    with torch.no_grad():
        for name, idx in _idx_views(idx32):
            want = ops.ds_edge_score(q, k, m, s, idx.contiguous())
            assert torch.equal(ops.ds_edge_score(q, k, m, s, idx), want), name
            assert torch.equal(ops.ds_edge_score(q, k, ms[..., 0], ms[..., 1], idx), want), name
            for (rname, qv), (_, kv) in zip(_row_views(q, 0), _row_views(k, 1)):
                assert torch.equal(ops.ds_edge_score(qv, kv, m, s, idx), want), (name, rname)
        with pytest.raises(TypeError, match="q must be float32"):
            ops.ds_edge_score(q.half(), k, m, s, idx32)
        with pytest.raises(TypeError, match="int32 or int64"):
            ops.ds_edge_score(q, k, m, s, idx32.float())


# ---------------------------------------------------------------- e. widths the Neighbor2Point kernels refuse

@pytest.mark.parametrize("train", [False, True], ids=["eval", "train"])
@pytest.mark.parametrize("C,H,match", [(256, 4, r"C=256 must be a multiple of 4, <= 128"),
                                       (96, 2, r"\(C/heads\)/4 = 12 must be a power of two")], ids=["C256", "C96_H2"])
def test_n2p_attention_refuses_widths_its_kernels_cannot_take(C, H, match, train):
    """The attention kernels take C <= 128 with a power-of-two number of float4 lanes per head.  A block outside that
    raises the kernel's own message in both modes; there is no other implementation to fall back to."""
    att = blocks.Neighbor2PointAttention(Cfg(_attention(1, C=C, K=16, heads=H)), 0).to(DEV).train(train)
    x = cu(synthetic_features(2, C, 128, C))
    with torch.set_grad_enabled(train), pytest.raises(ValueError, match=match):
        att(x)
