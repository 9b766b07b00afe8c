"""The differentiable path (SURVEY 8 row f1): torch.autograd.Functions whose forward AND backward run the sm_100a kernels.

The reference trains through ATen autograd of gather / softmax / cdist (train_shapenet.py:398-428): gradients reach the
STN through the xyz distances of the 3-NN interpolation (models/upsample.py:206-212 <- models/seg_model.py:187-192),
the q/k/v convolutions through the per-neighbourhood softmax (models/attention.py:207-250), and every feature through
the neighbour gathers (utils/ops.py:5-14).  The discrete decisions (neighbour indices, sampled indices) carry no
gradient in the reference either, so they come from the same forward-only kernels as in inference.

What is native here: the gathers and their scatter-add backward, the Neighbor2Point attention core and its backward
(nothing of size N*K*C is saved or formed in either direction: the forward saves the (B,N,3C) projections and the
indices, the backward recomputes the probabilities), and the distance gradient in at::_euclidean_dist_backward's form
evaluated only on the k selected pairs.  Dense layers (1x1 convolutions, BatchNorm with batch statistics) stay ATen.

The scatters of these backward passes add their terms with fp32 atomics (csrc/backward.cu), so the last bits of a
gradient change from run to run.  While torch.use_deterministic_algorithms(True) is in force -- the switch ATen's own
gather backward honours -- they take the ordered kernels of csrc/backward_ordered.cu instead: a reverse neighbour index
built once per backward call, then a fold of each target's terms in ascending edge order, bitwise reproducible.
"""
from __future__ import annotations

import torch
from torch.autograd import Function
from torch.autograd.function import once_differentiable

from . import _lib as L

Tensor = torch.Tensor


def wants_grad(*tensors) -> bool:
    return torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors)


def _bits(idx: Tensor) -> int:
    """Index width for the C ABI; any dtype other than int32 / int64 would be read as garbage, so it is refused."""
    if idx.dtype == torch.int64:
        return 64
    if idx.dtype == torch.int32:
        return 32
    raise TypeError(f"index tensor must be int32 or int64, got {idx.dtype}")


def deterministic() -> bool:
    """True while torch.use_deterministic_algorithms(True) is in force (with or without warn_only): the backward scatters
    then take the ordered kernels of csrc/backward_ordered.cu instead of the fp32 atomics of csrc/backward.cu."""
    return torch.are_deterministic_algorithms_enabled()


def reverse_index(idx: Tensor, N: int):
    """idx (B, ...) int32 / int64, flattened per cloud to (B,R) -> (offsets (B,N+1) int32, edges (B,R) int32): the edges of
    target j are edges[b, offsets[b,j]:offsets[b,j+1]] in ascending order; entries outside [0,N) are left out."""
    idx = idx.contiguous()
    B = idx.shape[0]
    R = idx[0].numel()
    dev = idx.device
    offsets = torch.empty(B, N + 1, dtype=torch.int32, device=dev)
    edges = torch.empty(B, R, dtype=torch.int32, device=dev)
    lib = L.lib()
    ws = L.workspace(lib.samble_reverse_index_workspace_bytes(B, N), dev)
    L.check(lib.samble_reverse_index(L.ptr(idx), _bits(idx), B, N, R, L.ptr(offsets), L.ptr(edges), L.ptr(ws), ws.numel(),
                                     L.stream()), "samble_reverse_index")
    return offsets, edges


def scatter_rows_ordered(x: Tensor, offsets: Tensor, edges: Tensor, *, channel_major: bool = False, weight: Tensor = None,
                         src_div: int = 1, sub: Tensor = None, out: Tensor = None) -> Tensor:
    """The ordered scatter: out[b, j, c] = fold over the edges e of target j (ascending) of weight[b, e, h(c)] * x[b, e // src_div, c]
    (weight None: x alone), minus sub[b, j, c] if given.  x (B,S,C) rows, or (B,C,S) when channel_major, any strides;
    weight (B,R,heads); sub (B,N,C) with unit channel stride; out (B,N,C) (or (B,C,N)) is written, allocated if None."""
    B, N = offsets.shape[0], offsets.shape[1] - 1
    R = edges.shape[1]
    if channel_major:
        C = x.shape[1]
        xs = (x.stride(0), x.stride(2), x.stride(1))
    else:
        C = x.shape[2]
        xs = (x.stride(0), x.stride(1), x.stride(2))
    if out is None:
        out = torch.empty((B, C, N) if channel_major else (B, N, C), dtype=torch.float32, device=x.device)
    os_ = (out.stride(0), out.stride(2), out.stride(1)) if channel_major else (out.stride(0), out.stride(1), out.stride(2))
    heads = 1
    if weight is not None:
        weight = weight.contiguous()
        heads = weight.shape[-1]
    if sub is not None and sub.stride(2) != 1:
        sub = sub.contiguous()
    sb = (sub.stride(0), sub.stride(1)) if sub is not None else (0, 0)
    L.check(L.lib().samble_scatter_rows_ordered(L.ptr(x), *xs, src_div, L.ptr(weight), heads, L.ptr(offsets), L.ptr(edges),
                                                L.ptr(sub), *sb, B, N, R, C, L.ptr(out), *os_, L.stream()),
            "samble_scatter_rows_ordered")
    return out


def _scatter_rows(grad_rows: Tensor, idx: Tensor, N: int) -> Tensor:
    """grad_rows (B,R,C) contiguous, idx (B,R) -> (B,N,C) with out[b, idx[b,r]] += grad_rows[b,r]."""
    B, R, C = grad_rows.shape
    if deterministic():
        offsets, edges = reverse_index(idx, N)
        return scatter_rows_ordered(grad_rows, offsets, edges)
    out = torch.zeros(B, N, C, dtype=torch.float32, device=grad_rows.device)
    L.check(L.lib().samble_index_points_backward(L.ptr(grad_rows), L.ptr(idx), _bits(idx), B, N, C, R, L.ptr(out), L.stream()),
            "samble_index_points_backward")
    return out


class IndexPoints(Function):
    """utils/ops.py:5-14: points (B,N,C), idx (B,M,K) -> (B,M,K,C); backward = row scatter-add."""

    @staticmethod
    def forward(ctx, points: Tensor, idx: Tensor) -> Tensor:
        points, idx = points.contiguous(), idx.contiguous()
        B, N, C = points.shape
        R = idx[0].numel()
        out = torch.empty(*idx.shape, C, dtype=torch.float32, device=points.device)
        L.check(L.lib().samble_index_points(L.ptr(points), L.ptr(idx), _bits(idx), B, N, C, R, L.ptr(out), L.stream()),
                "samble_index_points")
        ctx.save_for_backward(idx)
        ctx.n = N
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g: Tensor):
        (idx,) = ctx.saved_tensors
        B, C = g.shape[0], g.shape[-1]
        return _scatter_rows(g.contiguous().view(B, -1, C), idx.view(B, -1), ctx.n), None


class Group(Function):
    """utils/ops.py:47-65, 83-112 after the kNN: pcd (B,C,N), idx (B,N,K) -> (B,C,N,K) view / (B,2C,N,K)."""

    @staticmethod
    def forward(ctx, pcd: Tensor, idx: Tensor, gtype: int) -> Tensor:
        pcd, idx = pcd.contiguous(), idx.contiguous()
        B, C, N = pcd.shape
        K = idx.shape[-1]
        buf = torch.empty((B, N, K, C) if gtype < 2 else (B, 2 * C, N, K), dtype=torch.float32, device=pcd.device)
        L.check(L.lib().samble_group(L.ptr(pcd), L.ptr(idx), _bits(idx), B, C, N, K, gtype, L.ptr(buf), L.stream()), "samble_group")
        ctx.save_for_backward(idx)
        ctx.gtype, ctx.dims = gtype, (B, C, N, K)
        return buf.permute(0, 3, 1, 2) if gtype < 2 else buf

    @staticmethod
    @once_differentiable
    def backward(ctx, g: Tensor):
        (idx,) = ctx.saved_tensors
        B, C, N, K = ctx.dims
        t = ctx.gtype
        g_center = None
        if t >= 2:                                   # (B,2C,N,K): [centre repeated over K | neighbour or difference]
            g_center = g[:, :C].sum(dim=-1)                                   # (B,C,N)
            g = g[:, C:]
        g_rows = g.permute(0, 2, 3, 1).contiguous()                           # (B,N,K,C): free for the neighbor/diff view
        gp = _scatter_rows(g_rows.view(B, N * K, C), idx.view(B, N * K), N)   # (B,N,C)
        if t in (1, 3):                              # diff: every gathered row also subtracted the centre
            gp = gp - g_rows.sum(dim=2)
        gp = gp.transpose(1, 2)
        return (gp if g_center is None else gp + g_center), None, None


class GatherByIdx(Function):
    """utils/ops.py:136-145: pcd (B,C,N), idx (B,1,M) -> (B,C,M)."""

    @staticmethod
    def forward(ctx, pcd: Tensor, idx: Tensor) -> Tensor:
        pcd, idx = pcd.contiguous(), idx.contiguous()
        B, C, N = pcd.shape
        M = idx.shape[2]
        out = torch.empty(B, C, M, dtype=torch.float32, device=pcd.device)
        L.check(L.lib().samble_gather_by_idx(L.ptr(pcd), L.ptr(idx), _bits(idx), B, C, N, M, L.ptr(out), L.stream()),
                "samble_gather_by_idx")
        ctx.save_for_backward(idx)
        ctx.n = N
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g: Tensor):
        (idx,) = ctx.saved_tensors
        g = g.contiguous()
        B, C, M = g.shape
        if deterministic():
            offsets, edges = reverse_index(idx.view(B, M), ctx.n)
            return scatter_rows_ordered(g, offsets, edges, channel_major=True), None
        out = torch.zeros(B, C, ctx.n, dtype=torch.float32, device=g.device)
        L.check(L.lib().samble_gather_by_idx_backward(L.ptr(g), L.ptr(idx), _bits(idx), B, C, ctx.n, M, L.ptr(out), L.stream()),
                "samble_gather_by_idx_backward")
        return out, None


class N2PAttend(Function):
    """Core of models/attention.py:165-185, 207-250 on the hoisted projections: qkv (B,N,3C) = [q|k|v] of the points,
    idx (B,N,K) -> (B,N,C); csrc/attention.cu forward, csrc/backward.cu backward."""

    @staticmethod
    def forward(ctx, qkv: Tensor, idx: Tensor, heads: int) -> Tensor:
        qkv, idx = qkv.contiguous(), idx.contiguous()
        B, N, C3 = qkv.shape
        C, K = C3 // 3, idx.shape[-1]
        out = torch.empty(B, N, C, dtype=torch.float32, device=qkv.device)
        base = qkv.data_ptr()
        import ctypes as Ct

        q, k, v = (Ct.c_void_p(base + 4 * C * i) for i in range(3))
        L.check(L.lib().samble_n2p_attend(q, k, v, C3, L.ptr(idx), _bits(idx), B, N, C, K, heads, None, C, None, None,
                                          L.ptr(out), C, L.stream()), "samble_n2p_attend")
        ctx.save_for_backward(qkv, idx)
        ctx.heads = heads
        return out

    @staticmethod
    @once_differentiable
    def backward(ctx, g: Tensor):
        import ctypes as Ct

        qkv, idx = ctx.saved_tensors
        g = g.contiguous()
        B, N, C3 = qkv.shape
        C, K = C3 // 3, idx.shape[-1]
        if deterministic():
            return n2p_attend_backward_ordered(qkv, idx, ctx.heads, g), None, None
        gqkv = torch.zeros_like(qkv)
        q, k, v = (Ct.c_void_p(qkv.data_ptr() + 4 * C * i) for i in range(3))
        gq, gk, gv = (Ct.c_void_p(gqkv.data_ptr() + 4 * C * i) for i in range(3))
        L.check(L.lib().samble_n2p_attend_backward(q, k, v, C3, L.ptr(idx), _bits(idx), B, N, C, K, ctx.heads, L.ptr(g), C,
                                                   gq, gk, gv, C3, L.stream()), "samble_n2p_attend_backward")
        return gqkv, None, None


def n2p_attend_backward_edges(qkv: Tensor, idx: Tensor, heads: int, g: Tensor, grad_q: Tensor = None):
    """The per-edge pass of the ordered N2P backward: qkv (B,N,3C) contiguous, idx (B,N,K), g (B,N,C) contiguous ->
    (grad_q, p, ds): grad_q (B,N,C) (or written into the given (B,N,*) view with unit inner stride), p / ds (B,N,K,heads)."""
    import ctypes as Ct

    B, N, C3 = qkv.shape
    C, K = C3 // 3, idx.shape[-1]
    if grad_q is None:
        grad_q = torch.empty(B, N, C, dtype=torch.float32, device=qkv.device)
    p = torch.empty(B, N, K, heads, dtype=torch.float32, device=qkv.device)
    ds = torch.empty_like(p)
    q, k, v = (Ct.c_void_p(qkv.data_ptr() + 4 * C * i) for i in range(3))
    L.check(L.lib().samble_n2p_attend_backward_edges(q, k, v, C3, L.ptr(idx), _bits(idx), B, N, C, K, heads, L.ptr(g), C,
                                                     L.ptr(grad_q), grad_q.stride(1), L.ptr(p), L.ptr(ds), L.stream()),
            "samble_n2p_attend_backward_edges")
    return grad_q, p, ds


def n2p_attend_backward_ordered(qkv: Tensor, idx: Tensor, heads: int, g: Tensor) -> Tensor:
    """N2PAttend's gradient w.r.t. qkv without atomics: the edge pass, then dk_j = fold of ds_ij q_i and
    dv_j = (fold of p_ij g_i) - g_j over the edges i -> j in ascending i*K + slot."""
    B, N, C3 = qkv.shape
    C, K = C3 // 3, idx.shape[-1]
    gqkv = torch.empty_like(qkv)
    _, p, ds = n2p_attend_backward_edges(qkv, idx, heads, g, grad_q=gqkv[..., :C])
    offsets, edges = reverse_index(idx.view(B, N * K), N)
    scatter_rows_ordered(qkv[..., :C], offsets, edges, weight=ds.view(B, N * K, heads), src_div=K, out=gqkv[..., C:2 * C])
    scatter_rows_ordered(g, offsets, edges, weight=p.view(B, N * K, heads), src_div=K, sub=g, out=gqkv[..., 2 * C:])
    return gqkv


class PairDistance(Function):
    """Distances of the k selected pairs as a differentiable function of the (normalised) point sets.

    forward: the values the native kNN produced (the GEMM form of torch.cdist, utils/ops.py:35).
    backward: at::_euclidean_dist_backward's formula -- grad_a_i = sum_j (g_ij / d_ij)(a_i - b_j), zero where d == 0 --
    restricted to the selected pairs (the reference's topk passes no gradient to the others), with d_ij taken as
    |a_i - b_j| rather than the forward's GEMM-form value."""

    @staticmethod
    def forward(ctx, a_n: Tensor, b_n: Tensor, idx: Tensor, d: Tensor) -> Tensor:
        ctx.save_for_backward(a_n, b_n, idx, d)
        return d.clone()

    @staticmethod
    @once_differentiable
    def backward(ctx, g: Tensor):
        a_n, b_n, idx, d = ctx.saved_tensors
        B, Nq, k = idx.shape
        b_sel = IndexPoints.apply(b_n.detach(), idx)                                    # (B,Nq,k,C)
        diff = a_n.unsqueeze(2) - b_sel
        # the reference divides by ITS forward value, whose small entries are GEMM-form cancellation noise (1e-4 relative
        # at d ~ 1e-2, and 0 or ~1e-3 for coincident points); the norm of the difference itself is exact to fp32 rounding
        # and vanishes exactly where the points coincide, which is where the subgradient 0 belongs
        dist = diff.norm(dim=-1)
        ratio = (g / dist).masked_fill(dist == 0, 0.0)                                  # (B,Nq,k)
        t = ratio.unsqueeze(-1) * diff
        ga = t.sum(dim=2)
        gb = _scatter_rows((-t).contiguous().view(B, Nq * k, -1), idx.reshape(B, Nq * k), b_n.shape[1])
        return ga, gb, None, None


def knn_distance(a: Tensor, b: Tensor, idx: Tensor, d_native: Tensor) -> Tensor:
    """a (B,Nq,C), b (B,Nr,C) (autograd-tracked), idx (B,Nq,k), d_native >= 0 the kernel's distances -> the same values with
    the reference's gradient, through the per-cloud normalisation of utils/ops.py:23-29."""
    a_mean = torch.mean(a, dim=1, keepdim=True)
    a0, b0 = a - a_mean, b - a_mean
    a_std = torch.mean(torch.std(a0, dim=1, keepdim=True), dim=2, keepdim=True)
    return PairDistance.apply((a0 / a_std).contiguous(), (b0 / a_std).contiguous(), idx.contiguous(), d_native)
