"""The ordered backward scatters (csrc/backward_ordered.cu) that the differentiable path takes under
torch.use_deterministic_algorithms(True).

Order contract: for cloud b, edge e has target idx[b, e]; every gradient element is the fp32 left fold of its terms over
the target's edges in ascending e, each product and sum rounded on its own.  numpy's np.add.at on float32 folds in index
order, so the contract is checked bit for bit against it, on values (+-2^k, k in [-20, 20]) where another order gives
other bits -- which each such test asserts of its own data.

  1. ops.reverse_index against numpy's stable argsort.
  2. ops.scatter_rows_ordered against the host fold, unweighted and per-head weighted, row- and channel-major.
  3. The public ops with the flag on: the scatter part against the host fold, the gradient against fp64.
  4. Neighbor2Point: the edge pass against fp64, dk / dv against the host fold of the exported p and ds.
  5. Invariance: a cloud's gradient alone, inside a batch, run twice, on a side stream: the same bits.
  6. Selection: the flag alone picks the kernels (the library's launch profiler).
  7. Whole models, in a subprocess with torch.use_deterministic_algorithms(True) (errors, not warnings): two seeded
     training steps from the same state, with different stream use and allocator history, give the same bits.
  8. Whole models against the oracle's autograd with the flag on.
"""
import contextlib
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

from oracle import harness
from samble_b200 import _lib as L
from samble_b200 import autograd as AG
from samble_b200 import ops
from samble_b200.testing import n2p_attend_literal, synthetic_clouds, synthetic_features
from tests.test_gpu_backward import _group_ref, _knn_ref_dist, _prepared, rel
from tests.test_gpu_backward_kernels import N2P_CASES, _n2p_inputs, _n2p_term_scales, _rowwise

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@contextlib.contextmanager
def deterministic(warn_only=True):
    prev = (torch.are_deterministic_algorithms_enabled(), torch.is_deterministic_algorithms_warn_only_enabled())
    torch.use_deterministic_algorithms(True, warn_only=warn_only)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev[0], warn_only=prev[1])


def cu(t):
    return t.to(DEV)


def pow2(shape, seed):
    """+-2^k, k uniform in [-20, 20]: sums of such values round differently in different orders."""
    g = np.random.default_rng(seed)
    return (g.choice([-1.0, 1.0], size=shape) * np.exp2(g.integers(-20, 21, size=shape))).astype(np.float32)


def host_fold(terms, tgt, N, reverse=False):
    """terms (R,C) float32, tgt (R,) -> (N,C): np.add.at folds in index order (reverse: descending order instead)."""
    out = np.zeros((N, terms.shape[1]), np.float32)
    ok = (tgt >= 0) & (tgt < N)
    t, x = tgt[ok], terms[ok]
    if reverse:
        t, x = t[::-1], x[::-1]
    np.add.at(out, t, x)
    return out


def assert_order_matters(terms, tgt, N):
    assert not np.array_equal(host_fold(terms, tgt, N), host_fold(terms, tgt, N, reverse=True)), \
        "the data does not tell the summation orders apart"


# ---------------------------------------------------------------- 1. reverse index


def _targets(pattern, B, R, N, seed):
    g = np.random.default_rng(seed)
    if pattern == "random":
        return g.integers(0, N, size=(B, R))
    if pattern == "knn":                                  # R = N * K kNN lists of the cloud itself
        K = R // N
        idx = ops.knn_indices(cu(synthetic_features(B, 8, N, seed)), K, ordered=False)
        return idx.reshape(B, -1).cpu().numpy().astype(np.int64)
    if pattern == "hub":                                  # every edge on one point
        return np.full((B, R), N // 2, dtype=np.int64)
    if pattern == "sparse":                               # most targets have no edge
        return g.integers(0, max(1, N // 10), size=(B, R)) * 7 % N
    if pattern == "out_of_range":                         # a third of the entries outside [0, N)
        t = g.integers(0, N, size=(B, R))
        bad = g.random((B, R)) < 0.33
        t[bad] = g.choice([-1, -5, N, N + 3, 2 ** 20], size=int(bad.sum()))
        return t
    raise ValueError(pattern)


REV_CASES = [  # pattern, B, R, N
    ("random", 3, 1001, 300),
    ("random", 1, 65536 + 7, 2048),
    ("knn", 2, 300 * 17, 300),
    ("hub", 3, 4099, 50),
    ("hub", 1, 5, 1),
    ("sparse", 2, 777, 4096),
    ("out_of_range", 3, 2049, 257),
    ("random", 2, 31, 100),
]


@pytest.mark.parametrize("dt", [torch.int32, torch.int64], ids=["int32", "int64"])
@pytest.mark.parametrize("pattern,B,R,N", REV_CASES)
def test_reverse_index_is_a_stable_sort(pattern, B, R, N, dt):
    t = _targets(pattern, B, R, N, seed=R + N)
    if dt == torch.int32:
        t = np.where(t > 2 ** 30, -7, t)
    offsets, edges = ops.reverse_index(cu(torch.from_numpy(t).to(dt)), N)
    offsets, edges = offsets.cpu().numpy(), edges.cpu().numpy()
    for b in range(B):
        ok = np.nonzero((t[b] >= 0) & (t[b] < N))[0]
        want = ok[np.argsort(t[b][ok], kind="stable")]
        cnt = np.bincount(t[b][ok], minlength=N)
        assert np.array_equal(offsets[b], np.concatenate([[0], np.cumsum(cnt)])), b
        assert np.array_equal(edges[b, :len(ok)], want), b
        assert (edges[b, len(ok):] == -1).all(), b


# ---------------------------------------------------------------- 2. ordered scatter against the host fold


SCATTER_CASES = [  # B, N, R, C, heads (0: no weight), src_div, channel-major, sub, pattern
    (3, 300, 1001, 64, 0, 1, False, False, "random"),
    (2, 257, 2049, 3, 0, 1, True, False, "out_of_range"),
    (2, 300, 300 * 17, 128, 4, 17, False, True, "knn"),
    (3, 50, 4099, 40, 8, 1, True, False, "hub"),
    (1, 2048, 2048 * 32, 130, 0, 32, False, False, "random"),
    (2, 100, 700, 96, 3, 7, False, True, "sparse"),
]


@pytest.mark.parametrize("B,N,R,C,heads,src_div,cm,with_sub,pattern", SCATTER_CASES)
def test_scatter_rows_ordered_matches_the_host_fold(B, N, R, C, heads, src_div, cm, with_sub, pattern):
    seed = B + N + R + C
    t = _targets(pattern, B, R, N, seed)
    S = -(-R // src_div)
    x = pow2((B, S, C), seed)
    w = pow2((B, R, heads), seed + 1) if heads else None
    sub = pow2((B, N, C), seed + 2) if with_sub else None
    offsets, edges = ops.reverse_index(cu(torch.from_numpy(t)), N)
    xt = cu(torch.from_numpy(x))
    xt = xt.transpose(1, 2).contiguous() if cm else xt                      # (B,C,S) channel-major storage
    out = ops.scatter_rows_ordered(xt, offsets, edges, channel_major=cm,
                                   weight=None if w is None else cu(torch.from_numpy(w)), src_div=src_div,
                                   sub=None if sub is None else cu(torch.from_numpy(sub)))
    out = (out.transpose(1, 2) if cm else out).cpu().numpy()
    differs = False
    for b in range(B):
        rows = x[b][np.arange(R) // src_div]                                 # (R,C)
        if w is not None:
            rows = w[b][:, np.arange(C) // (C // heads)] * rows             # float32 products, rounded once
        want = host_fold(rows, t[b], N)
        if sub is not None:
            want = want - sub[b]
        assert np.array_equal(out[b], want), b
        differs |= not np.array_equal(host_fold(rows, t[b], N), host_fold(rows, t[b], N, reverse=True))
    assert differs, "the data does not tell the summation orders apart"


def test_scatter_rows_ordered_writes_into_a_column_slice():
    """out= a column slice of a wider buffer: every element of the slice is written, nothing outside it."""
    B, N, R, C = 2, 129, 900, 24
    t = cu(torch.from_numpy(_targets("random", B, R, N, 3)))
    x = cu(torch.from_numpy(pow2((B, R, C), 4)))
    offsets, edges = ops.reverse_index(t, N)
    want = ops.scatter_rows_ordered(x, offsets, edges)
    wide = torch.full((B, N, 3 * C), float("nan"), device=DEV)
    AG.scatter_rows_ordered(x, offsets, edges, out=wide[..., C:2 * C])
    assert torch.equal(wide[..., C:2 * C], want)
    assert bool(wide[..., :C].isnan().all()) and bool(wide[..., 2 * C:].isnan().all())


# ---------------------------------------------------------------- 3. the public ops with the flag on


def _fold_rows(g_rows, idx, N):
    """g_rows (B,R,C) float32 tensor, idx (B,R) -> (B,N,C) host fold."""
    g, i = g_rows.cpu().numpy(), idx.cpu().numpy()
    return torch.from_numpy(np.stack([host_fold(g[b], i[b], N) for b in range(g.shape[0])]))


@pytest.mark.parametrize("dt", [torch.int32, torch.int64], ids=["int32", "int64"])
def test_index_points_ordered(dt):
    B, N, C, M, K = 3, 300, 24, 200, 7
    p = synthetic_features(B, N, C, 1)
    idx = torch.randint(0, N, (B, M, K), generator=torch.Generator().manual_seed(2))
    probe = torch.from_numpy(pow2((B, M, K, C), 3))
    pc = cu(p).requires_grad_(True)
    with deterministic():
        out = ops.index_points(pc, cu(idx).to(dt))
        (g,) = torch.autograd.grad(out, pc, cu(probe))
    want = _fold_rows(probe.view(B, -1, C), idx.view(B, -1), N)
    assert torch.equal(g.cpu(), want)
    assert_order_matters(probe[0].reshape(-1, C).numpy(), idx[0].reshape(-1).numpy(), N)
    pr = p.double().requires_grad_(True)
    ref = torch.gather(pr, 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, M, K, C)
    (g_ref,) = torch.autograd.grad(ref, pr, probe.double())
    assert rel(g, g_ref) <= 1e-6


@pytest.mark.parametrize("group_type", ["neighbor", "diff", "center_neighbor", "center_diff"])
@pytest.mark.parametrize("C", [3, 64])
def test_group_ordered(group_type, C):
    """The scatter part is the host fold; the ATen reductions the Group backward applies around it are repeated here on
    the GPU from the folded value, and the result must be the native gradient bit for bit."""
    B, N, K = 2, 256, 32
    x = synthetic_features(B, C, N, 5)
    xc = cu(x).requires_grad_(True)
    with deterministic():
        out, idx = ops.group(xc, K, group_type)
        xr = x.double().requires_grad_(True)
        ref = _group_ref(xr, idx.cpu(), group_type)
        probe = torch.from_numpy(pow2(tuple(ref.shape), C + K)).float()
        (g,) = torch.autograd.grad(out, xc, cu(probe))
        gp = cu(probe)
        g_center = None
        if group_type.startswith("center"):
            g_center, gp = gp[:, :C].sum(dim=-1), gp[:, C:]
        g_rows = gp.permute(0, 2, 3, 1).contiguous()                        # (B,N,K,C)
        want = cu(_fold_rows(g_rows.view(B, N * K, C), idx.view(B, -1), N))
        if group_type in ("diff", "center_diff"):
            want = want - g_rows.sum(dim=2)
        want = want.transpose(1, 2)
        if g_center is not None:
            want = want + g_center
    assert torch.equal(g, want)
    (g_ref,) = torch.autograd.grad(ref, xr, probe.double())
    assert rel(g, g_ref) <= 1e-5


@pytest.mark.parametrize("dt", [torch.int32, torch.int64], ids=["int32", "int64"])
def test_gather_by_idx_ordered(dt):
    B, C, N, M = 3, 128, 512, 1500                                             # M > N: indices repeat
    x = synthetic_features(B, C, N, 7)
    idx = torch.randint(0, N, (B, 1, M), generator=torch.Generator().manual_seed(8))
    probe = torch.from_numpy(pow2((B, C, M), 9))
    xc = cu(x).requires_grad_(True)
    with deterministic():
        out = ops.gather_by_idx(xc, cu(idx).to(dt))
        (g,) = torch.autograd.grad(out, xc, cu(probe))
    want = _fold_rows(probe.transpose(1, 2), idx.view(B, M), N).transpose(1, 2)
    assert torch.equal(g.cpu(), want)
    assert_order_matters(probe[0].t().numpy(), idx[0, 0].numpy(), N)
    xr = x.double().requires_grad_(True)
    (g_ref,) = torch.autograd.grad(torch.gather(xr, 2, idx.expand(-1, C, -1)), xr, probe.double())
    assert rel(g, g_ref) <= 1e-6


@pytest.mark.parametrize("C,k,same", [(3, 3, False), (3, 32, True), (64, 16, False)])
def test_knn_distance_gradient_ordered(C, k, same):
    B, Nq = 2, 300
    Nr = 300 if same else 160
    a = synthetic_features(B, Nq, C, 11)
    b = a.clone() if same else a[:, torch.randperm(Nq, generator=torch.Generator().manual_seed(1))[:Nr]].clone()
    ac, bc = cu(a).requires_grad_(True), cu(b).requires_grad_(True)
    probe = torch.randn(B, Nq, k, generator=torch.Generator().manual_seed(2))
    with deterministic():
        neg, idx = ops.knn(ac, bc, k)
        ar, br = a.double().requires_grad_(True), b.double().requires_grad_(True)
        d_ref = _knn_ref_dist(ar, br, idx.cpu())
        probe = probe * (d_ref.detach() > 1e-3)
        ga, gb = torch.autograd.grad(-neg, (ac, bc), cu(probe))
        # the scatter part: PairDistance's backward on the normalised sets, its terms formed here by the same ATen statements
        an, bn = (cu(torch.randn(B, n, C, generator=torch.Generator().manual_seed(n))).requires_grad_(True) for n in (Nq, Nr))
        d = (an.detach().unsqueeze(2) - torch.gather(bn.detach(), 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, Nq, k, C)).norm(dim=-1)
        (gbn,) = torch.autograd.grad(AG.PairDistance.apply(an, bn, idx, d), bn, cu(probe))
        diff = an.detach().unsqueeze(2) - AG.IndexPoints.apply(bn.detach(), idx)
        dist = diff.norm(dim=-1)
        t = (cu(probe) / dist).masked_fill(dist == 0, 0.0).unsqueeze(-1) * diff
    assert torch.equal(gbn.cpu(), _fold_rows((-t).reshape(B, Nq * k, C), idx.reshape(B, -1), Nr))
    ga_ref, gb_ref = torch.autograd.grad((d_ref * probe.double()).sum(), (ar, br))
    assert rel(ga, ga_ref) <= 1e-4 and rel(gb, gb_ref) <= 1e-4


# ---------------------------------------------------------------- 4. Neighbor2Point


def _n2p_edges_fp64(qkv, idx, heads, probe):
    """fp64 p_ij and ds_ij (B,N,K,heads) and the magnitudes A of their fp32 rounding (p (1 + L) and |ds| with its
    rounding, as _n2p_term_scales counts them)."""
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
    dp = torch.einsum("bnhd,bnkhd->bnhk", gh, vj)
    ds = p * (dp - (p * dp).sum(-1, keepdim=True)) / D ** 0.5
    Lg = torch.einsum("bnhd,bnkhd->bnhk", qh.abs(), kj.abs()) / D ** 0.5
    pw = p * (1 + Lg)
    dpa = torch.einsum("bnhd,bnkhd->bnhk", gh.abs(), vj.abs())
    a_ds = pw * (dpa + (p * dpa).sum(-1, keepdim=True)) / D ** 0.5
    perm = (0, 1, 3, 2)
    return p.permute(perm), ds.permute(perm), pw.permute(perm), a_ds.permute(perm)


@pytest.mark.parametrize("C,H,K,N,B,dt,pattern,regime", N2P_CASES,
                         ids=[f"C{c[0]}_H{c[1]}_K{c[2]}_N{c[3]}_B{c[4]}_{str(c[5])[-5:]}_{c[6]}_{c[7]}" for c in N2P_CASES])
def test_n2p_ordered_backward(C, H, K, N, B, dt, pattern, regime):
    qkv, idx, probe = _n2p_inputs(C, K, N, B, pattern, regime, seed=C * 7 + K * 3 + N)
    r = qkv.double().requires_grad_(True)
    (g_ref,) = torch.autograd.grad(n2p_attend_literal(r, idx, H), r, probe.double())
    _, a_g = _n2p_term_scales(qkv, idx, H, probe)
    p64, ds64, a_p, a_ds = _n2p_edges_fp64(qkv, idx, H, probe)
    qc, ic, gc = cu(qkv), cu(idx).to(dt), cu(probe)
    gq, p, ds = ops.n2p_attend_backward_edges(qc, ic, H, gc)
    worst = {"dq(edge)": _rowwise(gq, g_ref[..., :C], a_g[..., :C]),
             "p": _rowwise(p.reshape(B, N, -1), p64.reshape(B, N, -1), a_p.reshape(B, N, -1)),
             "ds": _rowwise(ds.reshape(B, N, -1), ds64.reshape(B, N, -1), a_ds.reshape(B, N, -1))}
    rc = qc.clone().requires_grad_(True)
    with deterministic():
        (g,) = torch.autograd.grad(ops.n2p_attend(rc, ic, H), rc, gc)
    assert torch.equal(g[..., :C], gq)
    # dk / dv: the host fold of the exported terms
    q32, g32, P, DS = qkv[..., :C].numpy(), probe.numpy(), p.cpu().numpy(), ds.cpu().numpy()
    t = idx.reshape(B, -1).numpy()
    hc = np.arange(C) // (C // H)
    src = np.arange(N * K) // K
    for b in range(B):
        dk = host_fold(DS[b].reshape(N * K, H)[:, hc] * q32[b][src], t[b], N)
        dv = host_fold(P[b].reshape(N * K, H)[:, hc] * g32[b][src], t[b], N) - g32[b]
        assert np.array_equal(g[b, :, C:2 * C].cpu().numpy(), dk), b
        assert np.array_equal(g[b, :, 2 * C:].cpu().numpy(), dv), b
    for i, name in enumerate("qkv"):
        sl = slice(i * C, (i + 1) * C)
        worst[f"d{name}"] = _rowwise(g[..., sl], g_ref[..., sl], a_g[..., sl])
    assert bool(torch.isfinite(g).all())
    print(f"ordered n2p C={C} H={H} K={K} N={N} {pattern}/{regime} -- tensor: share of bound, rel. to |ref|, ulps of A:",
          ", ".join(f"{k} {v[0]:.3f} {v[1]:.1e} {v[2]:.2f}" for k, v in worst.items()))
    bad = {k: v for k, v in worst.items() if not v[0] <= 1.0}
    assert not bad, bad


def test_n2p_ordered_order_matters():
    """On +-2^k data the dv fold in descending order gives other bits: the bitwise checks above pin the order."""
    B, N, K, C = 1, 300, 32, 128
    idx = _targets("knn", B, N * K, N, 1)[0]
    terms = pow2((N * K, C), 2)
    assert_order_matters(terms, idx, N)


# ---------------------------------------------------------------- 5. invariance


def _grads(kind, x, idx, probe):
    """Gradient of one op w.r.t. its input, flag on."""
    xc = x.detach().clone().requires_grad_(True)
    with deterministic():
        if kind == "index_points":
            out = ops.index_points(xc, idx)
        elif kind == "gather_by_idx":
            out = ops.gather_by_idx(xc, idx)
        elif kind == "n2p":
            out = ops.n2p_attend(xc, idx, 4)
        elif kind.startswith("group_"):
            out = ops._group_from_idx(xc, idx, kind[6:])
        elif kind == "knn":
            out = -ops.knn(xc, idx, 16)[0]
        else:                                               # knn_pairs: the distance gradient on given normalised sets
            bn = idx.detach().clone().requires_grad_(True)
            nn_idx = ops.knn(xc.detach(), bn.detach(), 16)[1]
            d = (xc.detach().unsqueeze(2) - AG.IndexPoints.apply(bn.detach(), nn_idx)).norm(dim=-1)
            (g,) = torch.autograd.grad(AG.PairDistance.apply(xc, bn, nn_idx, d), bn, probe)
            return g
        (g,) = torch.autograd.grad(out, xc, probe)
    return g


def _invariance_inputs(kind, B, seed):
    gen = torch.Generator().manual_seed(seed)
    N = 1024
    if kind == "index_points":
        x, idx = torch.randn(B, N, 64, generator=gen), torch.randint(0, N, (B, N, 32), generator=gen)
        probe = torch.randn(B, N, 32, 64, generator=gen)
    elif kind == "gather_by_idx":
        x, idx = torch.randn(B, 128, N, generator=gen), torch.randint(0, N, (B, 1, 1024), generator=gen)
        probe = torch.randn(B, 128, 1024, generator=gen)
    elif kind == "n2p":
        x = torch.randn(B, N, 384, generator=gen)
        idx = torch.randint(0, N, (B, N, 32), generator=gen)
        probe = torch.randn(B, N, 128, generator=gen)
    elif kind.startswith("group_"):
        x, idx = torch.randn(B, 64, N, generator=gen), torch.randint(0, N, (B, N, 32), generator=gen)
        ref = _group_ref(x[:1].double(), idx[:1], kind[6:])
        probe = torch.randn(B, *ref.shape[1:], generator=gen)
    else:                                                   # knn / knn_pairs: idx is the reference set
        x, idx = torch.randn(B, N, 3, generator=gen), torch.randn(B, 700, 3, generator=gen)
        probe = torch.randn(B, N, 16, generator=gen)
    return cu(x), cu(idx), cu(probe)


@pytest.mark.parametrize("kind", ["index_points", "gather_by_idx", "n2p", "group_neighbor", "group_diff", "group_center_neighbor",
                                  "group_center_diff", "knn", "knn_pairs"])
def test_ordered_gradients_are_invariant(kind):
    """Each cloud's gradient is the same bits alone and inside a batch of 3, run twice, and run on a side stream.

    ops.knn's gradient is only checked run to run and across streams: before the selected pairs it runs through the
    per-cloud normalisation of utils/ops.py:23-29 (mean and std over the points), ATen reductions whose strategy follows
    the tensor's shape, so one cloud alone and the same cloud in a batch round differently there in either mode.  The
    part of it that is native, PairDistance's scatter onto the reference set, is checked alone and in a batch as
    knn_pairs."""
    x, idx, probe = _invariance_inputs(kind, 3, seed=17)
    batch = _grads(kind, x, idx, probe)
    assert torch.equal(_grads(kind, x, idx, probe), batch)
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        on_side = _grads(kind, x, idx, probe)
    torch.cuda.current_stream().wait_stream(side)
    assert torch.equal(on_side, batch)
    for b in range(3 if kind != "knn" else 0):
        alone = _grads(kind, x[b:b + 1].contiguous(), idx[b:b + 1].contiguous(), probe[b:b + 1].contiguous())
        assert torch.equal(alone, batch[b:b + 1]), b


# ---------------------------------------------------------------- 6. selection


ATOMIC = {"index_points_bwd_kernel", "gather_by_idx_bwd_kernel", "n2p_attend_bwd_kernel"}
ORDERED = {"reverse_index_kernel", "scatter_rows_ordered_kernel", "n2p_attend_bwd_edges_kernel"}


def _backward_launches(flag):
    """Names of the kernels the three backward passes launch.  The autograd engine runs CUDA backward passes on a worker
    thread of its own and the launch profiler records per thread, so it is switched on and read by hooks that run there:
    one on the op's output (before the op's backward) and one on its input (after it)."""
    x, idx, probe = _invariance_inputs("index_points", 2, 1)
    xg, ig, pg = _invariance_inputs("gather_by_idx", 2, 2)
    xn, inn, pn = _invariance_inputs("n2p", 2, 3)
    names = set()

    def start(g):
        L.profile_report()                                  # (drop anything recorded before)
        L.profile(True)
        return g

    def stop(g):
        torch.cuda.synchronize()
        names.update(L.profile_report())
        L.profile(False)
        return g

    ctx = deterministic() if flag else contextlib.nullcontext()
    with ctx:
        for fn, inp, pr in ((lambda t: ops.index_points(t, idx), x, probe), (lambda t: ops.gather_by_idx(t, ig), xg, pg),
                            (lambda t: ops.n2p_attend(t, inn, 4), xn, pn)):
            inp = inp.detach().requires_grad_(True)
            inp.register_hook(stop)
            out = fn(inp)
            out.register_hook(start)
            out.backward(pr)
    return names


def test_the_flag_selects_the_kernels():
    off = _backward_launches(False)
    assert ATOMIC <= off and not (off & ORDERED), off
    on = _backward_launches(True)
    assert ORDERED <= on and not (on & ATOMIC), on


# ---------------------------------------------------------------- 7. whole models, reproducible


_STEP = r"""
import sys
sys.path.insert(0, ROOT)
import torch
import torch.nn.functional as F
torch.use_deterministic_algorithms(True)
from samble_b200 import blocks, models, ops
from samble_b200.config import cls_config, seg_config
from samble_b200.testing import fill_state_dict_, synthetic_clouds

DEV = "cuda:0"


def step(which, second):
    ops.CONCURRENT_BRANCHES = not second
    junk = [torch.empty(n, device=DEV) for n in (12345, 987653, 77)] if second else []   # another allocator history
    B, N = (4, 1024) if which == "seg" else (8, 1024)
    cfg = (seg_config if which == "seg" else cls_config)(M=(512, 256))
    m = (models.ShapeNetModel if which == "seg" else models.ModelNetModel)(cfg)
    m.load_state_dict(fill_state_dict_(m.state_dict(), seed=3, sharpen=2.0))
    m = m.to(DEV).train()
    sampled = []
    for mod in m.modules():
        if isinstance(mod, blocks.DownSampleToken):
            mod.register_forward_hook(lambda mod, inp, out: sampled.append(out[0][1].detach().cpu()))
    xc, catc = synthetic_clouds(B, N, 20)
    torch.manual_seed(7)
    with torch.no_grad():                                   # first boundary estimate; the step below then runs the EMA
        m(xc.to(DEV), catc.to(DEV)) if which == "seg" else m(xc.to(DEV))
    x, cat = synthetic_clouds(B, N, 21)
    x = x.to(DEV).requires_grad_(True)
    labels = torch.randint(0, 50 if which == "seg" else 40, (B, N) if which == "seg" else (B,),
                           generator=torch.Generator().manual_seed(5)).to(DEV)
    opt = torch.optim.SGD(m.parameters(), lr=0.05, momentum=0.9)
    torch.manual_seed(11)                                   # (dropout)
    out = m(x, cat.to(DEV)) if which == "seg" else m(x)
    loss = F.cross_entropy(out.transpose(1, 2).reshape(-1, 50), labels.reshape(-1)) if which == "seg" else F.cross_entropy(out, labels)
    opt.zero_grad()
    loss.backward()
    opt.step()
    torch.cuda.synchronize()
    del junk
    res = {"loss": loss.detach().cpu(), "input grad": x.grad.cpu()}
    res.update({"grad " + n: p.grad.cpu() for n, p in m.named_parameters() if p.grad is not None})
    res.update({"state " + n: t.detach().cpu() for n, t in m.state_dict().items()})
    for i, mod in enumerate(mm for mm in m.modules() if isinstance(mm, blocks.DownSampleToken)):
        for j, t in enumerate(mod.bin_boundaries):
            res[f"boundaries {i}.{j}"] = t.detach().cpu()
    for i, t in enumerate(sampled):
        res[f"sampled {i}"] = t
    return res


bad = []
for which in ("seg", "cls"):
    a, b = step(which, False), step(which, True)
    assert a.keys() == b.keys()
    assert any(k.startswith("grad ") for k in a) and any(k.startswith("sampled") for k in a)
    bad += [f"{which}: {k}" for k in a if not torch.equal(a[k], b[k])]
    print(which, len(a), "tensors compared")
print("MISMATCH", [k for k in bad if " state " not in k], "and", sum(" state " in k for k in bad), "state tensors")
sys.exit(1 if bad else 0)
"""


def test_whole_model_training_step_is_reproducible():
    env = dict(os.environ, CUBLAS_WORKSPACE_CONFIG=":4096:8")
    p = subprocess.run([sys.executable, "-c", f"ROOT = {ROOT!r}\n" + _STEP], env=env, cwd=ROOT, capture_output=True,
                       text=True, timeout=1200)
    print(p.stdout[-4000:], p.stderr[-4000:])
    assert p.returncode == 0, (p.stdout[-2000:], p.stderr[-4000:])


# ---------------------------------------------------------------- 8. whole models, accurate


@pytest.mark.parametrize("which", ["seg", "cls"])
def test_model_backward_vs_oracle_autograd_ordered(which):
    B, N, M = (8 if which == "cls" else 2), 256, (128, 64)
    m, sd, cfg = _prepared(which, B, N, M, seed=4, train=True)
    x, cat = synthetic_clouds(B, N, 6)
    with deterministic():
        rep = harness.gradient_parity(m, sd, cfg, x, cat, which=which)
    allp = list(rep["params"].items()) + [("<input>", rep["input"])]
    for n, e in sorted(allp, key=lambda kv: -kv[1]["rel"])[:4]:
        print(f"  {n}: rel {e['rel']:.2e} (reference fp32 autograd: {e['rel_oracle32']:.2e})")
    assert rep["logits_close_frac_fp64"] == 1.0
    harness.assert_gradient_report(rep, tol=1e-4)
