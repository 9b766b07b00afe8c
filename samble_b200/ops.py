"""Drop-in for the reference's `utils/ops.py` hot-path functions, backed by the sm_100a kernels.

Same names, argument meaning, return layouts and error behaviour as reference
utils/ops.py:5-145, 174-236, 385-505, so the reference's own models can use this
module in place of `utils.ops` (see samble_b200.patch).  Every function runs through
the C ABI (include/samble_b200.h); nothing falls back to PyTorch or the CPU.

Functions with a leading underscore-free "fast" name (`knn_indices`, `n2p_attend`,
`ds_*`, `interpolate3`) are the fused entry points our own blocks use; they have no
reference counterpart because the reference materialises the intermediate instead.
"""
from __future__ import annotations

import ctypes as C
from typing import List, Optional, Tuple

import torch

from . import _lib as L
from . import autograd as AG

Tensor = torch.Tensor

_GROUP_TYPES = {"neighbor": 0, "diff": 1, "center_neighbor": 2, "center_diff": 3}


def _f32(t: Tensor, name: str) -> Tensor:
    if t.dtype != torch.float32:
        raise TypeError(f"{name} must be float32, got {t.dtype}")
    return t


_idx_bits = AG._bits


def _rows(t: Tensor, name: str) -> Tensor:
    """t (B,N,W) float32 as rows a kernel addresses with one row pitch t.stride(1): unit inner stride, a batch pitch of
    N rows, 16-byte aligned rows.  A contiguous tensor or an aligned column slice of a wider row-major buffer passes as it
    is; anything else is copied."""
    _f32(t, name)
    if (t.stride(2) != 1 or t.stride(0) != t.shape[1] * t.stride(1) or t.stride(1) % 4 != 0
            or t.data_ptr() % 16 != 0):
        t = t.clone(memory_format=torch.contiguous_format)       # (fresh storage: aligned even if t was contiguous)
    return t


def _neighbour_idx(idx: Tensor, B: int, N: int) -> Tensor:
    """idx (B,N,K) int32 / int64 as the contiguous array the kernels index."""
    _idx_bits(idx)
    if idx.dim() != 3 or tuple(idx.shape[:2]) != (B, N):
        raise RuntimeError(f"neighbour indices must be ({B},{N},K), got {tuple(idx.shape)}")
    return idx.contiguous()


# ------------------------------------------------------------------ kNN


def _knn_strided(a: Tensor, b: Tensor, k: int, layout: str, want_dist: bool, idx_dtype=torch.int64, ordered=True):
    """a, b: 3-D fp32 CUDA tensors in 'bnc' (B,N,C) or 'bcn' (B,C,N) layout, any strides."""
    dev = L.need_cuda(a, b)
    a, b = a.detach(), b.detach()            # discrete output + forward values; callers attach the distance gradient (autograd.py)
    _f32(a, "a"), _f32(b, "b")
    if layout == "bnc":
        (B, Nq, Cc), (Bb, Nr, Cb) = a.shape, b.shape
        sa, sb_ = (a.stride(0), a.stride(1), a.stride(2)), (b.stride(0), b.stride(1), b.stride(2))
    else:
        (B, Cc, Nq), (Bb, Cb, Nr) = a.shape, b.shape
        sa, sb_ = (a.stride(0), a.stride(2), a.stride(1)), (b.stride(0), b.stride(2), b.stride(1))
    if B != Bb or Cc != Cb:
        raise RuntimeError(f"knn: batch/channel mismatch {tuple(a.shape)} vs {tuple(b.shape)}")
    if k > Nr:   # torch.topk's own complaint (utils/ops.py:43)
        raise RuntimeError("selected index k out of range")
    lib = L.lib()
    idx = torch.empty(B, Nq, k, dtype=idx_dtype, device=dev)
    dist = torch.empty(B, Nq, k, dtype=torch.float32, device=dev) if want_dist else None
    nbytes = lib.samble_knn_workspace_bytes(B, Nq, Nr, Cc)
    ws = L.workspace(nbytes, dev)
    rc = lib.samble_knn(L.ptr(a), *sa, L.ptr(b), *sb_, B, Nq, Nr, Cc, k, L.ptr(idx), _idx_bits(idx), L.ptr(dist),
                        0 if ordered else 1, L.ptr(ws), ws.numel(), L.stream())
    L.check(rc, "samble_knn")
    return dist, idx


def knn(a: Tensor, b: Tensor, k: int) -> Tuple[Tensor, Tensor]:
    """utils/ops.py:17-44.  a (B,N,C), b (B,M,C) -> (negative distance (B,N,k), idx (B,N,k) int64).
    When a or b requires grad the distances carry the reference's gradient (autograd.knn_distance)."""
    neg, idx = _knn_strided(a, b, k, "bnc", True)
    if AG.wants_grad(a, b):
        neg = -AG.knn_distance(a, b, idx, -neg)
    return neg, idx


def knn_indices(pcd: Tensor, K: int, idx_dtype=torch.int32, ordered: bool = True) -> Tensor:
    """Self-kNN of a channel-major cloud (B,C,N) -> idx (B,N,K); the internal fast path
    (int32 indices, no distance output, no permute copy).  ordered=False (SAMBLE_KNN_ANY_ORDER): the same
    neighbour SET per row in arbitrary order, for consumers that reduce over the neighbours."""
    return _knn_strided(pcd, pcd, K, "bcn", False, idx_dtype, ordered)[1]


# ------------------------------------------------------------------ concurrent branches
#
# Inside a block the neighbour search and the dense projections depend on the same input and on nothing else, and
# neither fills the GPU alone (a 512-point layer launches 64 search CTAs on 148 SMs; the persistent GEMM kernels have
# tails).  `fork(fn)` runs fn on a per-device side stream and returns a join() that makes the current stream wait for
# it; under CUDA-graph capture the two become parallel branches of the graph.  Scratch space is per (device, stream)
# (_lib.workspace), so the branches never share a workspace.

CONCURRENT_BRANCHES = True
_SIDE_STREAMS: dict = {}


def fork(fn):
    """Run fn() on the side stream; returns join() -> fn's result, valid on the current stream afterwards."""
    if not CONCURRENT_BRANCHES or not torch.cuda.is_available():     # (no GPU: fn raises the library's own "CUDA only" error)
        out = fn()
        return lambda: out
    main = torch.cuda.current_stream()
    key = (main.device.index, main.cuda_stream)      # one side stream per calling stream (sub-batches may run side by side)
    side = _SIDE_STREAMS.get(key)
    if side is None:
        side = _SIDE_STREAMS[key] = torch.cuda.Stream(device=main.device)
    side.wait_stream(main)                       # everything fn reads has been produced on the current stream
    with torch.cuda.stream(side):
        out = fn()
    done = torch.cuda.Event()
    done.record(side)

    def join():
        main.wait_event(done)
        for t in (out if isinstance(out, (tuple, list)) else (out,)):
            if isinstance(t, torch.Tensor):
                t.record_stream(main)            # allocated on the side stream, consumed here
        return out

    return join


# ------------------------------------------------------------------ gathers


def index_points(points: Tensor, idx: Tensor) -> Tensor:
    """utils/ops.py:5-14.  points (B,N,C), idx (B,M,K) -> (B,M,K,C)."""
    dev = L.need_cuda(points, idx)
    if AG.wants_grad(points):
        return AG.IndexPoints.apply(_f32(points, "points"), idx)
    points = _f32(points, "points").contiguous()
    idx = idx.contiguous()
    B, N, Cc = points.shape
    R = idx[0].numel()
    out = torch.empty(*idx.shape, Cc, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_index_points(L.ptr(points), L.ptr(idx), _idx_bits(idx), B, N, Cc, R, L.ptr(out), L.stream()),
            "samble_index_points")
    return out


def _group_from_idx(pcd: Tensor, idx: Tensor, group_type: str) -> Tensor:
    B, Cc, N = pcd.shape
    K = idx.shape[-1]
    t = _GROUP_TYPES[group_type]
    if AG.wants_grad(pcd):
        return AG.Group.apply(pcd, idx, t)
    if t < 2:
        buf = torch.empty(B, N, K, Cc, dtype=torch.float32, device=pcd.device)
    else:
        buf = torch.empty(B, 2 * Cc, N, K, dtype=torch.float32, device=pcd.device)
    L.check(L.lib().samble_group(L.ptr(pcd), L.ptr(idx), _idx_bits(idx), B, Cc, N, K, t, L.ptr(buf), L.stream()),
            "samble_group")
    # neighbor/diff: the reference hands out this exact memory as a permuted view (utils/ops.py:57,60)
    return buf.permute(0, 3, 1, 2) if t < 2 else buf


def select_neighbors(pcd: Tensor, K: int, neighbor_type: str, normal_channel: bool = False):
    """utils/ops.py:47-65.  pcd (B,C,N) -> ((B,C,N,K) view of (B,N,K,C), idx (B,N,K) int64)."""
    if neighbor_type not in ("neighbor", "diff"):
        raise ValueError(f'neighbor_type should be "neighbor" or "diff", but got {neighbor_type}')
    L.need_cuda(pcd)
    pcd = _f32(pcd, "pcd").contiguous()
    key = pcd[:, :3, :] if (normal_channel and pcd.shape[1] == 6) else pcd
    _, idx = _knn_strided(key, key, K, "bcn", False)
    return _group_from_idx(pcd, idx, neighbor_type), idx


def group(pcd: Tensor, K: int, group_type: str, normal_channel: bool = False):
    """utils/ops.py:83-112."""
    if group_type not in _GROUP_TYPES:
        raise ValueError(
            f"group_type should be neighbor, diff, center_neighbor or center_diff, but got {group_type}")
    L.need_cuda(pcd)
    pcd = _f32(pcd, "pcd").contiguous()
    key = pcd[:, :3, :] if (normal_channel and pcd.shape[1] == 6) else pcd
    _, idx = _knn_strided(key, key, K, "bcn", False)
    return _group_from_idx(pcd, idx, group_type), idx


def select_neighbors_interpolate(unknown: Tensor, known: Tensor, known_feature: Tensor, K: int = 3):
    """utils/ops.py:68-80.  -> (neighbors (B,C,N,K) view, idx (B,N,K), distance (B,N,K) >= 0)."""
    L.need_cuda(unknown, known, known_feature)
    neg, idx = _knn_strided(unknown, known, K, "bcn", True)
    d = -1 * neg
    if AG.wants_grad(unknown, known):        # the distances feed the interpolation weights (models/upsample.py:206-209)
        d = AG.knn_distance(unknown.permute(0, 2, 1), known.permute(0, 2, 1), idx, d)
    nbr = index_points(known_feature.permute(0, 2, 1), idx)
    return nbr.permute(0, 3, 1, 2), idx, d


def neighbor_mask(pcd: Tensor, K: int) -> Tensor:
    """utils/ops.py:125-133.  dense 0/1 (B,N,N) float32."""
    dev = L.need_cuda(pcd)
    pcd = _f32(pcd, "pcd")
    idx = knn_indices(pcd, K)
    B, N, _ = idx.shape
    out = torch.empty(B, N, N, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_neighbor_mask(L.ptr(idx), 32, B, N, K, L.ptr(out), L.stream()), "samble_neighbor_mask")
    return out


def gather_by_idx(pcd: Tensor, idx: Tensor) -> Tensor:
    """utils/ops.py:136-145.  pcd (B,C,N), idx (B,1,M) -> (B,C,M)."""
    dev = L.need_cuda(pcd, idx)
    if idx.dim() != 3 or idx.shape[1] != 1:
        raise RuntimeError(f"gather_by_idx expects idx of shape (B,1,M), got {tuple(idx.shape)}")
    if AG.wants_grad(pcd):
        return AG.GatherByIdx.apply(_f32(pcd, "pcd"), idx)
    pcd = _f32(pcd, "pcd").contiguous()
    B, Cc, N = pcd.shape
    idx = idx.contiguous()
    M = idx.shape[2]
    out = torch.empty(B, Cc, M, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_gather_by_idx(L.ptr(pcd), L.ptr(idx), _idx_bits(idx), B, Cc, N, M, L.ptr(out), L.stream()),
            "samble_gather_by_idx")
    return out


# ------------------------------------------------------------------ fused block cores


_W_SPLIT: dict = {}      # id(base tensor) -> (weakref(base), version, {view key: (W padded, W_lo)})


def rows_of(x: Tensor) -> Tensor:
    """Point-major rows (B,N,C), contiguous, of a cloud given in the reference's (B,C,N) shape.  Block outputs are
    (B,C,N) VIEWS of point-major storage (stride(1) == 1), so between our own blocks this is free; a genuinely
    channel-major tensor is transposed once (samble_transpose)."""
    if x.dim() == 3 and x.stride(1) == 1 and x.stride(2) >= x.shape[1] and x.stride(0) == x.stride(2) * x.shape[2]:
        return x.transpose(1, 2)            # (B,N,C) rows, possibly a column slice of a wider buffer (row pitch = stride)
    return transpose12(x)


def transpose12(x: Tensor) -> Tensor:
    """x (B,R,C) -> contiguous (B,C,R) (samble_transpose); x.transpose(1,2).contiguous() without ATen's strided copy."""
    dev = L.need_cuda(x)
    x = _f32(x, "x")
    if x.dim() != 3:
        raise RuntimeError("transpose12: expected a 3-D tensor")
    B, R, Cc = x.shape
    if x.stride(2) != 1 or x.stride(1) < Cc:
        x = x.contiguous()
    out = torch.empty(B, Cc, R, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_transpose(L.ptr(x), x.stride(0), x.stride(1), B, R, Cc, L.ptr(out), L.stream()), "samble_transpose")
    return out


def _split_weight(weight: Tensor):
    """(W padded to a multiple of 4 columns, W_lo = W - tf32_trunc(W)).  Cached per LIVE base tensor (weak reference:
    an address recycled by the allocator for a new tensor never hits), its in-place version, and the view taken of it."""
    import weakref

    base = weight._base if weight._base is not None else weight
    vkey = (weight.data_ptr(), tuple(weight.shape), tuple(weight.stride()))
    ent = _W_SPLIT.get(id(base))
    if ent is not None and ent[0]() is base and ent[1] == base._version:
        hit = ent[2].get(vkey)
        if hit is not None:
            return hit
    else:
        ent = (weakref.ref(base, lambda _r, k=id(base): _W_SPLIT.pop(k, None)), base._version, {})
        _W_SPLIT[id(base)] = ent
    with torch.no_grad():
        w = _f32(weight, "weight").detach().flatten(1)
        Nout, K = w.shape
        K4 = (K + 3) // 4 * 4
        if K4 != K or w.stride(1) != 1 or w.stride(0) % 4 != 0 or w.data_ptr() % 16 != 0:
            wp = torch.zeros(Nout, K4, dtype=torch.float32, device=w.device)
            wp[:, :K] = w
            w = wp
        lo = torch.empty(w.shape[0], w.stride(0), dtype=torch.float32, device=w.device)[:, : w.shape[1]]
        if w.is_contiguous():
            L.check(L.lib().samble_split_tf32(L.ptr(w), L.ptr(lo), w.numel(), L.stream()), "samble_split_tf32")
        else:                       # strided view (e.g. a column slice of a bigger weight): split via torch bit ops
            lo.copy_(w - (w.view(torch.int32) & -8192).view(torch.float32))
    ent[2][vkey] = (w, lo)
    return w, lo


def linear(x: Tensor, weight: Tensor, *, x_layout: str = "rows", out_layout: str = "rows", scale: Optional[Tensor] = None,
           shift: Optional[Tensor] = None, lrelu: bool = False, residual: Optional[Tensor] = None,
           residual_first: bool = False, residual_layout: Optional[str] = None) -> Tensor:
    """Point-wise linear layer on the tensor cores, fp32-class accuracy (csrc/linear_tc.cu).

    x: 'rows' -> (..., K) with unit inner stride (leading dims flattened, one common row stride), or
       'bcn'  -> (B, K, P) contiguous channel-major cloud.
    weight: (Nout, K[,1[,1]]).  scale: (Nout,), shift: (Nout,) or per cloud (B, Nout).
    out_layout 'rows' -> (..., Nout) ; 'bcn' -> (B, Nout, P).  residual_layout defaults to out_layout.
    y = ((x W^T [+ residual if residual_first]) * scale + shift) -> LeakyReLU(0.2) if lrelu [-> + residual]."""
    dev = L.need_cuda(x, weight, scale, shift, residual)
    L.no_grad_check(x, weight)
    w, w_lo = _split_weight(weight)
    Nout, K = weight.shape[0], weight[0].numel()
    if x_layout == "bcn" and x.shape[1] >= 32:
        # measured: the row-major loader (cp.async, two stages ahead) is 2x faster than the channel-major one even
        # after paying for this transposing copy (tools/time_linear_calls.py)
        x, x_layout = rows_of(x), "rows"
    if x_layout == "bcn":
        x = _f32(x, "x").contiguous()
        B, Kx, P = x.shape
        M, ldx, lead = B * P, 0, None
    else:
        x = _f32(x, "x")
        if x.stride(-1) != 1:
            x = x.contiguous()
        lead, Kx = x.shape[:-1], x.shape[-1]
        x2 = x.reshape(-1, Kx) if x.dim() != 2 else x
        if x2.stride(1) != 1:
            x2 = x2.contiguous()
        if Kx % 4 != 0 or x2.stride(0) % 4 != 0 or x2.data_ptr() % 16 != 0:     # cp.async rows must be 16-byte chunks
            x2 = torch.nn.functional.pad(x2, (0, (-Kx) % 4)).contiguous()
        x, M, ldx = x2, x2.shape[0], x2.stride(0)
        B, P = (lead[0], M // lead[0]) if len(lead) >= 2 else (1, M)
    if Kx != K:
        raise RuntimeError(f"linear: x has {Kx} channels, weight expects {K}")
    if out_layout == "bcn":
        out = torch.empty(B, Nout, P, dtype=torch.float32, device=dev)
        ldo = 0
    else:
        out = torch.empty(*(lead if lead is not None else (B, P)), Nout, dtype=torch.float32, device=dev)
        ldo = Nout
    shift_ldb = 0
    if shift is not None:
        shift = _f32(shift, "shift").contiguous()
        if shift.dim() == 2:
            shift_ldb = Nout
    if scale is not None:
        scale = _f32(scale, "scale").contiguous()
    ldr = 0
    res_layout = residual_layout or out_layout
    if residual is not None:
        residual = _f32(residual, "residual")
        want = (B, Nout, P) if res_layout == "bcn" else (M, Nout)
        if (tuple(residual.shape) != want) if res_layout == "bcn" else (residual.numel() != M * Nout or residual.shape[-1] != Nout):
            raise RuntimeError(f"linear: residual shape {tuple(residual.shape)} does not match layout '{res_layout}' of a "
                               f"{M} x {Nout} result")
        if res_layout == "bcn":
            residual = residual.contiguous()
        else:
            if residual.stride(-1) != 1:
                residual = residual.contiguous()
            r2 = residual.reshape(-1, Nout)
            residual, ldr = r2, r2.stride(0)
    L.check(L.lib().samble_linear(L.ptr(x), ldx, 1 if x_layout == "bcn" else 0, L.ptr(w), L.ptr(w_lo), w.stride(0), L.ptr(scale), L.ptr(shift),
                                  shift_ldb, 1 if lrelu else 0, L.ptr(residual), ldr, 1 if res_layout == "bcn" else 0,
                                  1 if residual_first else 0, L.ptr(out), ldo,
                                  1 if out_layout == "bcn" else 0, M, K, Nout, P, L.stream()), "samble_linear")
    return out


def ds_select_rows(q: Tensor, rowmax: Tensor, rowsum: Tensor, tok_logits: Tensor, v_tok: Tensor, idx: Tensor):
    """For the selected points idx (B,M) int64: q_sel (B,M,D), m_sel, s_sel (B,M) and tok_mix (B,M,C) = the token
    columns' share softmax(row)[N:] @ v_tok of the block's output (samble_ds_select_rows)."""
    dev = L.need_cuda(q, rowmax, rowsum, tok_logits, v_tok, idx)
    B, N, D = q.shape
    M, nb, Cc = idx.shape[1], tok_logits.shape[-1], v_tok.shape[-1]
    v_tok, idx = _f32(v_tok, "v_tok").contiguous(), idx.contiguous()
    q_sel = torch.empty(B, M, D, dtype=torch.float32, device=dev)
    m_sel = torch.empty(B, M, dtype=torch.float32, device=dev)
    s_sel = torch.empty(B, M, dtype=torch.float32, device=dev)
    tok_mix = torch.empty(B, M, Cc, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_ds_select_rows(L.ptr(q), q.stride(1), L.ptr(rowmax), L.ptr(rowsum), L.ptr(tok_logits), L.ptr(v_tok),
                                          L.ptr(idx), B, N, M, D, nb, Cc, L.ptr(q_sel), L.ptr(m_sel), L.ptr(s_sel),
                                          L.ptr(tok_mix), L.stream()), "samble_ds_select_rows")
    return q_sel, m_sel, s_sel, tok_mix


def cloud_matmul(x: Tensor, w: Tensor, *, row_max: Optional[Tensor] = None, row_sum: Optional[Tensor] = None,
                 logit_div: float = 1.0, w_split=None, residual: Optional[Tensor] = None) -> Tensor:
    """Per-cloud products on the tensor cores (3xTF32, samble_cloud_matmul): x (B,R,K), w (B,Nout,K) -> (B,R,Nout) with
    out[b] = x[b] w[b]^T; R a multiple of 128.  With row_max/row_sum (B,R) the result is
    exp(out / logit_div - row_max) / row_sum, i.e. softmax rows whose statistics are already known."""
    dev = L.need_cuda(x, w, row_max, row_sum)
    L.no_grad_check(x, w)
    x, w = _f32(x, "x"), _f32(w, "w")
    B, R, K = x.shape
    Bw, Nout, Kw = w.shape
    if Bw != B or Kw != K:
        raise RuntimeError(f"cloud_matmul: x {tuple(x.shape)} vs w {tuple(w.shape)}")
    if K % 4 != 0:
        x = torch.nn.functional.pad(x, (0, (-K) % 4))
    x = x.contiguous()
    w, w_lo = w_split if w_split is not None else split_operand(w)     # a (B,K,Nout) view is transposed by one tiled kernel
    lib = L.lib()
    out = torch.empty(B, R, Nout, dtype=torch.float32, device=dev)
    if row_max is not None:
        row_max, row_sum = _f32(row_max, "row_max").contiguous(), _f32(row_sum, "row_sum").contiguous()
    if residual is not None:
        residual = _f32(residual, "residual").contiguous()
        if tuple(residual.shape) != (B, R, Nout):
            raise RuntimeError(f"cloud_matmul: residual {tuple(residual.shape)} != {(B, R, Nout)}")
    L.check(lib.samble_cloud_matmul(L.ptr(x), x.stride(1), L.ptr(w), L.ptr(w_lo), w.stride(1), B * R, K, Nout, R, L.ptr(row_max),
                                    L.ptr(row_sum), float(logit_div), L.ptr(residual), Nout, L.ptr(out), Nout, L.stream()),
            "samble_cloud_matmul")
    return out


# two-layer MLPs (N2P feed-forward, seg head conv2 -> conv3) as one kernel; False = the two `linear` launches (A/B measurements)
FUSED_MLP2 = True


def mlp2_eligible(K1: int, Hd: int, N2: int) -> bool:
    """shapes the fused two-layer kernel (csrc/mlp2.cu) takes; anything else stays two `linear` calls."""
    return K1 <= 128 and K1 % 4 == 0 and Hd >= 128 and Hd % 128 == 0 and N2 in (128, 256)


def mlp2(x: Tensor, w1: Tensor, w2: Tensor, *, scale1: Optional[Tensor] = None, shift1: Optional[Tensor] = None,
         lrelu1: bool = True, scale2: Optional[Tensor] = None, shift2: Optional[Tensor] = None, lrelu2: bool = False,
         residual: Optional[Tensor] = None, residual_first: bool = False) -> Tensor:
    """Two point-wise linear layers in one kernel, the hidden activation kept in tensor memory (csrc/mlp2.cu):
        h = lrelu?((x W1^T) * scale1 + shift1);  y = ((h W2^T [+ residual if residual_first]) * scale2 + shift2) -> lrelu? [-> + residual]
    x: (B, P, K1) rows (K1 <= 128); w1: (Hd, K1[,1]); w2: (N2, Hd[,1]) with N2 in {128, 256}; shifts (C,) or per cloud (B, C).
    models/attention.py:187-192 (feed-forward + bn2 of Neighbor2PointAttention), models/seg_model.py:205-214 (conv2 -> conv3)."""
    dev = L.need_cuda(x, w1, w2, scale1, shift1, scale2, shift2, residual)
    L.no_grad_check(x, w1, w2)
    w1s, w1lo = _split_weight(w1)
    w2s, w2lo = _split_weight(w2)
    Hd, K1 = w1.shape[0], w1[0].numel()
    N2 = w2.shape[0]
    if w2[0].numel() != Hd or not mlp2_eligible(K1, Hd, N2):
        raise RuntimeError(f"mlp2: unsupported widths {K1} -> {Hd} -> {N2} (K1 <= 128, Hd % 128 == 0, N2 in (128, 256))")
    x = _f32(x, "x")
    if x.dim() != 3 or x.shape[-1] != K1:
        raise RuntimeError(f"mlp2: x must be (B, P, {K1}) rows, got {tuple(x.shape)}")
    B, P, _ = x.shape
    x2 = x.reshape(B * P, K1)
    if x2.stride(1) != 1 or x2.stride(0) % 4 != 0 or x2.data_ptr() % 16 != 0:
        x2 = x2.contiguous()
    M = B * P

    def col(v, name, width):
        if v is None:
            return None, 0
        v = _f32(v, name).contiguous()
        if v.shape[-1] != width or v.dim() > 2 or (v.dim() == 2 and v.shape[0] != B):
            raise RuntimeError(f"mlp2: {name} must be ({width},) or ({B}, {width}), got {tuple(v.shape)}")
        if v.data_ptr() % 16 != 0:
            v = v.clone()
        return v, (width if v.dim() == 2 else 0)

    scale1, _ = col(scale1, "scale1", Hd)
    shift1, s1_ldb = col(shift1, "shift1", Hd)
    scale2, _ = col(scale2, "scale2", N2)
    shift2, s2_ldb = col(shift2, "shift2", N2)
    if (s1_ldb or s2_ldb) and P % 128 != 0:
        raise RuntimeError("mlp2: per-cloud shifts need clouds of a multiple of 128 points")
    ldr = 0
    if residual is not None:
        residual = _f32(residual, "residual")
        if residual.numel() != M * N2 or residual.shape[-1] != N2:
            raise RuntimeError(f"mlp2: residual shape {tuple(residual.shape)} does not match a {M} x {N2} result")
        if residual.stride(-1) != 1:
            residual = residual.contiguous()
        residual = residual.reshape(-1, N2)
        ldr = residual.stride(0)
    out = torch.empty(B, P, N2, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_mlp2(L.ptr(x2), x2.stride(0), M, K1, L.ptr(w1s), L.ptr(w1lo), w1s.stride(0), Hd, L.ptr(scale1), L.ptr(shift1),
                                s1_ldb, 1 if lrelu1 else 0, L.ptr(w2s), L.ptr(w2lo), w2s.stride(0), N2, L.ptr(scale2), L.ptr(shift2),
                                s2_ldb, 1 if lrelu2 else 0, L.ptr(residual), ldr, 1 if residual_first else 0, L.ptr(out), N2, P,
                                L.stream()), "samble_mlp2")
    return out


def linear_pool(x: Tensor, weight: Tensor, *, scale: Optional[Tensor] = None, shift: Optional[Tensor] = None,
                lrelu: bool = False, want_max: bool = True, want_mean: bool = True):
    """max / mean over the points of each cloud of  lrelu(x W^T * scale + shift)  without storing the activation
    (samble_linear_pool).  x: (B, P, K) row-major with P % 32 == 0.  Returns (max (B,Nout) | None, mean (B,Nout) | None)."""
    dev = L.need_cuda(x, weight, scale, shift)
    L.no_grad_check(x, weight)
    w, w_lo = _split_weight(weight)
    Nout, K = weight.shape[0], weight[0].numel()
    x = _f32(x, "x")
    B, P, Kx = x.shape
    if Kx != K:
        raise RuntimeError(f"linear_pool: x has {Kx} channels, weight expects {K}")
    x2 = x.reshape(B * P, Kx)
    if x2.stride(1) != 1 or Kx % 4 != 0 or x2.stride(0) % 4 != 0 or x2.data_ptr() % 16 != 0:
        x2 = torch.nn.functional.pad(x2, (0, (-Kx) % 4)).contiguous()
    shift_ldb = 0
    if shift is not None:
        shift = _f32(shift, "shift").contiguous()
        shift_ldb = Nout if shift.dim() == 2 else 0
    if scale is not None:
        scale = _f32(scale, "scale").contiguous()
    omax = torch.empty(B, Nout, dtype=torch.float32, device=dev) if want_max else None
    omean = torch.empty(B, Nout, dtype=torch.float32, device=dev) if want_mean else None
    lib = L.lib()
    ws = L.workspace(lib.samble_linear_pool_workspace_bytes(B * P, Nout), dev)
    L.check(lib.samble_linear_pool(L.ptr(x2), x2.stride(0), L.ptr(w), L.ptr(w_lo), w.stride(0), L.ptr(scale), L.ptr(shift),
                                   shift_ldb, 1 if lrelu else 0, B * P, K, Nout, P, L.ptr(omax), L.ptr(omean),
                                   L.ptr(ws), ws.numel(), L.stream()), "samble_linear_pool")
    return omax, omean


def edge_mlp_max(pr: Tensor, idx: Tensor, w2: Tensor, b2: Tensor, out_rows: Optional[Tensor] = None) -> Tensor:
    """Fused EdgeConv core (csrc/edgeconv.cu): pr (B,N,2*C1) = [P'|R'] point projections, idx (B,N,K),
    w2 (C2,C1), b2 (C2) -> (B,C2,N).  models/embedding.py:29-39 after folding eval-mode BatchNorm.
    The result is stored point-major -- in `out_rows` (B,N,C2), which may be a column slice of a wider row-major buffer, or
    in fresh storage -- and handed back in the reference's (B,C2,N) shape as a view of it (ops.rows_of is then free)."""
    dev = L.need_cuda(pr, idx, w2, b2, out_rows)
    pr = _rows(pr, "pr")
    B, N, two_c1 = pr.shape
    idx = _neighbour_idx(idx, B, N)
    C1, C2, K = two_c1 // 2, w2.shape[0], idx.shape[-1]
    w2, b2 = w2.contiguous(), b2.contiguous()
    if out_rows is None:
        out_rows = torch.empty(B, N, C2, dtype=torch.float32, device=dev)
    elif tuple(out_rows.shape) != (B, N, C2) or out_rows.stride(2) != 1 or out_rows.stride(0) != N * out_rows.stride(1):
        raise RuntimeError("edge_mlp_max: out_rows must be (B,N,C2) rows with unit inner stride and a common pitch")
    L.check(L.lib().samble_edge_mlp_max(L.ptr(pr), pr.stride(1), L.ptr(idx), _idx_bits(idx), L.ptr(w2), L.ptr(b2), B, N, K,
                                        C1, C2, L.ptr(out_rows), out_rows.stride(1), L.stream()), "samble_edge_mlp_max")
    return out_rows.transpose(1, 2)


def n2p_attend(qkv: Tensor, idx: Tensor, heads: int, residual: Optional[Tensor] = None,
               scale: Optional[Tensor] = None, shift: Optional[Tensor] = None) -> Tensor:
    """qkv (B,N,3C) point-major [q|k|v] projections of the points; idx (B,N,K) -> (B,N,C).
    Core of models/attention.py:165-185,207-250 with the k/v convolutions hoisted (attention.cu).
    With residual (B,N,C) / scale,shift (C,): returns (residual + attention) * scale + shift (folded bn1, :187)."""
    dev = L.need_cuda(qkv, idx, residual, scale, shift)
    _f32(qkv, "qkv")
    if AG.wants_grad(qkv, residual, scale, shift):
        y = AG.N2PAttend.apply(qkv, idx, heads)
        if residual is not None:
            y = y + residual
        return y * scale + shift if scale is not None else y
    qkv = _rows(qkv, "qkv")
    B, N, C3 = qkv.shape
    idx = _neighbour_idx(idx, B, N)
    Cc = C3 // 3
    K = idx.shape[-1]
    out = torch.empty(B, N, Cc, dtype=torch.float32, device=dev)
    q, k, v = qkv[..., :Cc], qkv[..., Cc:2 * Cc], qkv[..., 2 * Cc:]
    if residual is not None:
        residual = residual.contiguous()
    if scale is not None:
        scale, shift = scale.contiguous(), shift.contiguous()
    L.check(L.lib().samble_n2p_attend(L.ptr(q), L.ptr(k), L.ptr(v), qkv.stride(1), L.ptr(idx), _idx_bits(idx), B, N, Cc, K, heads,
                                      L.ptr(residual), Cc, L.ptr(scale), L.ptr(shift), L.ptr(out), Cc, L.stream()),
            "samble_n2p_attend")
    return out


def split_operand(w: Tensor):
    """(w contiguous, w_lo = w - trunc_tf32(w)) for an ACTIVATION used as the per-cloud weight of cloud_matmul /
    ds_row_stats (weights proper go through the cached _split_weight).  w: (B,R,K) rows, or its (B,K,R) transpose."""
    w = _f32(w, "w")
    if not w.is_contiguous():
        wt = w.transpose(1, 2)
        w = transpose12(wt) if (wt.stride(2) == 1 and wt.stride(1) >= wt.shape[2]) else w.contiguous()
    if w.shape[-1] % 4 != 0:
        w = torch.nn.functional.pad(w, (0, (-w.shape[-1]) % 4))
    w_lo = torch.empty_like(w)
    L.check(L.lib().samble_split_tf32(L.ptr(w), L.ptr(w_lo), w.numel(), L.stream()), "samble_split_tf32")
    return w, w_lo


# ------------------------------------------------------------------ exact-product tensor-core GEMM (csrc/xgemm.cu)


class Digits:
    """Three signed-8-bit digit planes (bf16 integers) of a (B,R,C) fp32 array + the per-cloud power-of-two scale."""

    __slots__ = ("planes", "scale", "B", "R", "C")

    def __init__(self, planes, scale, B, R, C):
        self.planes, self.scale, self.B, self.R, self.C = planes, scale, B, R, C


def digits(x: Tensor, amax: Optional[Tensor] = None, group: int = 0) -> Digits:
    """x (B,R,C) fp32 rows (unit inner stride, common row pitch; a column slice of a wider buffer is fine) -> Digits.
    amax (B,G) int32 = bit patterns of max|x| per cloud and column group (xgemm(..., amax_group=C)); `group` picks the
    column of amax that belongs to x.  Without amax a reduction pass finds the magnitudes."""
    dev = L.need_cuda(x, amax)
    x = _f32(x, "x")
    if x.dim() != 3:
        raise RuntimeError("digits: expected (B,R,C)")
    B, R, Cc = x.shape
    if x.stride(2) != 1 or x.stride(1) % 4 or x.stride(0) % 4 or x.data_ptr() % 16 or Cc % 4:
        x = torch.nn.functional.pad(x, (0, (-Cc) % 4)).contiguous()
    lib = L.lib()
    planes = torch.empty(lib.samble_digits_bytes(B, R, x.shape[2]), dtype=torch.uint8, device=dev)
    scale = torch.empty(B, dtype=torch.float32, device=dev)
    if amax is None:
        scratch = torch.empty(B, dtype=torch.int32, device=dev)
        a_ptr, a_stride = None, 0
    else:
        scratch = None
        a_ptr, a_stride = C.c_void_p(amax.data_ptr() + 4 * group), amax.shape[1]
    L.check(lib.samble_digits(L.ptr(x), x.stride(1), x.stride(0), B, R, x.shape[2], a_ptr, a_stride, L.ptr(planes), L.ptr(scale),
                              L.ptr(scratch), L.stream()), "samble_digits")
    return Digits(planes, scale, B, R, x.shape[2])


_W_DIGITS: dict = {}


def weight_digits(weight: Tensor) -> Digits:
    """digits() of a (Nout,K[,1[,1]]) weight as one 'cloud', cached per live tensor and in-place version."""
    import weakref

    key = id(weight)
    ent = _W_DIGITS.get(key)
    if ent is not None and ent[0]() is weight and ent[1] == weight._version:
        return ent[2]
    with torch.no_grad():
        d = digits(weight.detach().flatten(1).unsqueeze(0))
    _W_DIGITS[key] = (weakref.ref(weight, lambda _r, k=key: _W_DIGITS.pop(k, None)), weight._version, d)
    return d


def xgemm(a: Digits, b: Digits, amax_group: int = 0, reference: bool = False):
    """out (Ba,Ra,Rb) = A[b] B[b or 0]^T, exact accumulation (samble_xgemm).  amax_group > 0 also returns the int32 bit
    patterns of max|out| per cloud and group of `amax_group` output columns, which digits() of a column slice takes."""
    if a.C != b.C or (b.B != a.B and b.B != 1):
        raise RuntimeError(f"xgemm: A is ({a.B},{a.R},{a.C}), B is ({b.B},{b.R},{b.C})")
    dev = a.planes.device
    out = torch.empty(a.B, a.R, b.R, dtype=torch.float32, device=dev)
    amax = torch.empty(a.B, (b.R + amax_group - 1) // amax_group, dtype=torch.int32, device=dev) if amax_group else None
    L.check(L.lib().samble_xgemm(L.ptr(a.planes), L.ptr(a.scale), a.B, a.R, L.ptr(b.planes), L.ptr(b.scale), b.B, b.R, a.C,
                                 L.ptr(out), b.R, L.ptr(amax), amax_group, 1 if reference else 0, L.stream()), "samble_xgemm")
    return (out, amax) if amax_group else out


def ds_row_stats_exact(qd: Digits, kd: Digits, q: Tensor, k_tok: Tensor):
    """Row statistics of softmax(q [k | k_tok]^T / sqrt(D)) from the digit planes of q and k (point columns, exact
    accumulation) and the fp32 q rows (token columns): -> rowmax (B,N), rowsum (B,N), token_logits (B,N,nb)."""
    dev = L.need_cuda(q, k_tok)
    B, N, D = q.shape
    nb = k_tok.shape[0]
    k_tok = _f32(k_tok, "k_tok").contiguous()
    rowmax = torch.empty(B, N, dtype=torch.float32, device=dev)
    rowsum = torch.empty(B, N, dtype=torch.float32, device=dev)
    tok = torch.empty(B, N, nb, dtype=torch.float32, device=dev)
    lib = L.lib()
    ws = L.workspace(lib.samble_ds_row_stats_exact_workspace_bytes(B, N), dev)
    L.check(lib.samble_ds_row_stats_exact(L.ptr(qd.planes), L.ptr(qd.scale), L.ptr(kd.planes), L.ptr(kd.scale), L.ptr(q), q.stride(1),
                                          L.ptr(k_tok), B, N, D, nb, L.ptr(rowmax), L.ptr(rowsum), L.ptr(tok), L.ptr(ws), ws.numel(),
                                          L.stream()), "samble_ds_row_stats_exact")
    return rowmax, rowsum, tok


def ds_attend_rows(qd: Digits, kd: Digits, v: Tensor, idx: Tensor, rowmax: Tensor, rowsum: Tensor, tok_logits: Tensor,
                   v_tok: Tensor) -> Tensor:
    """The attention rows of the selected points times V, flash-style (samble_ds_attend_rows; models/downsample.py:242-252):
    qd/kd digit planes of q/k (B,N,D), v (B,N,C) fp32 rows (unit inner stride), idx (B,M) int64, row statistics (B,N),
    tok_logits (B,N,nb), v_tok (nb,C) -> (B,M,C)."""
    dev = L.need_cuda(v, idx, rowmax, rowsum, tok_logits, v_tok)
    B, N, Cc = v.shape
    M, nb, D = idx.shape[1], tok_logits.shape[-1], qd.C
    if v.stride(2) != 1 or v.stride(0) != N * v.stride(1):
        v = v.contiguous()
    idx, v_tok = idx.contiguous(), _f32(v_tok, "v_tok").contiguous()
    out = torch.empty(B, M, Cc, dtype=torch.float32, device=dev)
    lib = L.lib()
    ws = L.workspace(lib.samble_ds_attend_rows_workspace_bytes(B, N, Cc), dev)
    L.check(lib.samble_ds_attend_rows(L.ptr(qd.planes), L.ptr(qd.scale), L.ptr(kd.planes), L.ptr(kd.scale), L.ptr(v), v.stride(1),
                                      L.ptr(idx), L.ptr(rowmax), L.ptr(rowsum), L.ptr(tok_logits), L.ptr(v_tok), B, N, M, D, Cc, nb,
                                      L.ptr(out), L.ptr(ws), ws.numel(), L.stream()), "samble_ds_attend_rows")
    return out


# Two tensor-core kernels compute the row statistics: the row-statistics epilogue of linear_tma.cu (default:
# samble_ds_row_stats_fast; TMA-fed, shares k's tf32 split with cloud_matmul) and ds_rowstats_tc.cu (cp.async loaders).
# Tests flip this to cross-check one against the other.
_DS_FAST = True


def ds_row_stats(q: Tensor, k: Tensor, k_tok: Tensor, k_split=None):
    """q,k: (B,N,D) point-major views (last stride 1, row stride ld); k_tok (nb,D).
    -> rowmax (B,N), rowsum (B,N), token_logits (B,N,nb).  models/downsample.py:139-153.
    k_split = split_operand(k) lets the caller share k's tf32 split with cloud_matmul."""
    dev = L.need_cuda(q, k, k_tok)
    B, N, D = q.shape
    nb = k_tok.shape[0]
    k_tok = k_tok.contiguous()
    rowmax = torch.empty(B, N, dtype=torch.float32, device=dev)
    rowsum = torch.empty(B, N, dtype=torch.float32, device=dev)
    tok = torch.empty(B, N, nb, dtype=torch.float32, device=dev)
    if _DS_FAST and N % 128 == 0 and D % 4 == 0 and q.stride(2) == 1 and q.stride(0) == N * q.stride(1):
        kc, klo = k_split if k_split is not None else split_operand(k)
        lib = L.lib()
        ws = L.workspace(lib.samble_ds_row_stats_fast_workspace_bytes(B, N), dev)
        L.check(lib.samble_ds_row_stats_fast(L.ptr(q), q.stride(1), L.ptr(kc), L.ptr(klo), kc.stride(1), L.ptr(k_tok), B, N, D, nb,
                                             L.ptr(rowmax), L.ptr(rowsum), L.ptr(tok), L.ptr(ws), ws.numel(), L.stream()),
                "samble_ds_row_stats_fast")
        return rowmax, rowsum, tok
    L.check(L.lib().samble_ds_row_stats(L.ptr(q), q.stride(1), L.ptr(k), k.stride(1), L.ptr(k_tok), B, N, D, nb,
                                        L.ptr(rowmax), L.ptr(rowsum), L.ptr(tok), L.stream()), "samble_ds_row_stats")
    return rowmax, rowsum, tok


def ds_edge_score(q: Tensor, k: Tensor, rowmax: Tensor, rowsum: Tensor, idx: Tensor) -> Tensor:
    """sparse_col_sqr point score (B,N) from the kNN edges only.  models/downsample.py:300-344."""
    dev = L.need_cuda(q, k, rowmax, rowsum, idx)
    q, k = _rows(q, "q"), _rows(k, "k")
    B, N, D = q.shape
    idx = _neighbour_idx(idx, B, N)
    rowmax, rowsum = _f32(rowmax, "rowmax").contiguous(), _f32(rowsum, "rowsum").contiguous()
    K = idx.shape[-1]
    lib = L.lib()
    score = torch.empty(B, N, dtype=torch.float32, device=dev)
    ws = L.workspace(lib.samble_ds_edge_score_workspace_bytes(B, N), dev)
    L.check(lib.samble_ds_edge_score(L.ptr(q), q.stride(1), L.ptr(k), k.stride(1), L.ptr(rowmax), L.ptr(rowsum),
                                     L.ptr(idx), _idx_bits(idx), B, N, D, K, L.ptr(score), L.ptr(ws), ws.numel(),
                                     L.stream()), "samble_ds_edge_score")
    return score


def zscore(score: Tensor) -> Tensor:
    """(score - mean) / population std over the last dim (utils/ops.py:450-452)."""
    L.need_cuda(score)
    score = _f32(score, "score").contiguous()
    N = score.shape[-1]
    z = torch.empty_like(score)
    L.check(L.lib().samble_zscore(L.ptr(score), score.numel() // N, N, L.ptr(z), L.stream()), "samble_zscore")
    return z


def ds_sample(score: Tensor, token_logits: Tensor, cuts: Tensor, M: int, want_z: bool = False):
    """Fused bin stage (models/downsample.py:205-240): score (B,N), token_logits (B,N,nb), cuts (nb-1,)
    descending thresholds on the z-score -> dict(idx (B,M) int64, bin_id (B,N) uint8, counts, k, w_raw, z)."""
    dev = L.need_cuda(score, token_logits, cuts)
    B, N = score.shape
    nb = token_logits.shape[-1]
    cuts = _f32(cuts, "cuts").contiguous()
    if cuts.numel() != nb - 1:
        raise ValueError(f"ds_sample: expected {nb - 1} cuts, got {cuts.numel()}")
    out = dict(idx=torch.empty(B, M, dtype=torch.int64, device=dev),
               bin_id=torch.empty(B, N, dtype=torch.uint8, device=dev),
               counts=torch.empty(B, nb, dtype=torch.int32, device=dev),
               k=torch.empty(B, nb, dtype=torch.int32, device=dev),
               w_raw=torch.empty(B, nb, dtype=torch.float32, device=dev),
               z=torch.empty(B, N, dtype=torch.float32, device=dev) if want_z else None)
    L.check(L.lib().samble_ds_sample(L.ptr(score), L.ptr(token_logits), L.ptr(cuts), B, N, nb, M, L.ptr(out["idx"]),
                                     L.ptr(out["bin_id"]), L.ptr(out["counts"]), L.ptr(out["k"]), L.ptr(out["w_raw"]),
                                     L.ptr(out["z"]), L.stream()), "samble_ds_sample")
    return out


def interpolate3(xyz_up: Tensor, xyz_sel: Tensor, feat: Tensor, want_idx: bool = False):
    """Fused 3-NN inverse-distance interpolation (models/upsample.py:194-212): xyz_up (B,3,N),
    xyz_sel (B,3,M), feat (B,C,M) -> (B,C,N) [, idx (B,N,3) int64, dist (B,N,3)]."""
    dev = L.need_cuda(xyz_up, xyz_sel, feat)
    L.no_grad_check(xyz_up, xyz_sel, feat)
    xyz_up, xyz_sel, feat = (_f32(t, "input").contiguous() for t in (xyz_up, xyz_sel, feat))
    B, three, N = xyz_up.shape
    M, Cc = xyz_sel.shape[2], feat.shape[1]
    if three != 3 or xyz_sel.shape[1] != 3:
        raise ValueError("interpolate3: xyz tensors must be (B,3,N)")
    lib = L.lib()
    out = torch.empty(B, Cc, N, dtype=torch.float32, device=dev)
    idx = torch.empty(B, N, 3, dtype=torch.int64, device=dev) if want_idx else None
    dist = torch.empty(B, N, 3, dtype=torch.float32, device=dev) if want_idx else None
    ws = L.workspace(lib.samble_interpolate3_workspace_bytes(B, N, M), dev)
    L.check(lib.samble_interpolate3(L.ptr(xyz_up), L.ptr(xyz_sel), L.ptr(feat), B, N, M, Cc, L.ptr(out), L.ptr(idx),
                                    L.ptr(dist), L.ptr(ws), ws.numel(), L.stream()), "samble_interpolate3")
    return (out, idx, dist) if want_idx else out


def interpolate3_rows(xyz_up: Tensor, xyz_sel: Tensor, feat_rows: Tensor, out: Tensor) -> Tensor:
    """interpolate3 with point-major features: feat_rows (B,M,C) -> written into `out` (B,N,C), which may be a column
    slice of a wider row-major buffer (unit inner stride)."""
    dev = L.need_cuda(xyz_up, xyz_sel, feat_rows, out)
    L.no_grad_check(xyz_up, xyz_sel, feat_rows)
    xyz_up, xyz_sel = (_f32(t, "xyz").contiguous() for t in (xyz_up, xyz_sel))
    feat_rows = _f32(feat_rows, "feat")
    if feat_rows.stride(2) != 1:
        feat_rows = feat_rows.contiguous()
    B, three, N = xyz_up.shape
    M, Cc = xyz_sel.shape[2], feat_rows.shape[2]
    if three != 3 or xyz_sel.shape[1] != 3:
        raise ValueError("interpolate3: xyz tensors must be (B,3,N)")
    if tuple(out.shape) != (B, N, Cc) or out.stride(2) != 1 or out.stride(0) != N * out.stride(1) or \
            feat_rows.stride(0) != M * feat_rows.stride(1):
        raise RuntimeError("interpolate3_rows: out must be (B,N,C) rows with a common pitch")
    lib = L.lib()
    ws = L.workspace(lib.samble_interpolate3_workspace_bytes(B, N, M), dev)
    L.check(lib.samble_interpolate3_rows(L.ptr(xyz_up), L.ptr(xyz_sel), L.ptr(feat_rows), feat_rows.stride(1), B, N, M, Cc,
                                         L.ptr(out), out.stride(1), L.ptr(ws), ws.numel(), L.stream()), "samble_interpolate3_rows")
    return out


def interpolate3_search(xyz_up: Tensor, xyz_sel: Tensor):
    """3-NN of every up point among the selected points + normalised inverse-distance weights (models/upsample.py:194-209):
    xyz_up (B,3,N), xyz_sel (B,3,M) -> nn_idx (B,N,3) int32, nn_w (B,N,3).  Needs the coordinates only."""
    dev = L.need_cuda(xyz_up, xyz_sel)
    L.no_grad_check(xyz_up, xyz_sel)
    xyz_up, xyz_sel = (_f32(t, "xyz").contiguous() for t in (xyz_up, xyz_sel))
    B, three, N = xyz_up.shape
    M = xyz_sel.shape[2]
    if three != 3 or xyz_sel.shape[1] != 3:
        raise ValueError("interpolate3: xyz tensors must be (B,3,N)")
    nn_idx = torch.empty(B, N, 3, dtype=torch.int32, device=dev)
    nn_w = torch.empty(B, N, 3, dtype=torch.float32, device=dev)
    lib = L.lib()
    ws = L.workspace(lib.samble_interpolate3_workspace_bytes(B, N, M), dev)
    L.check(lib.samble_interpolate3_search(L.ptr(xyz_up), L.ptr(xyz_sel), B, N, M, L.ptr(nn_idx), L.ptr(nn_w), L.ptr(ws), ws.numel(),
                                           L.stream()), "samble_interpolate3_search")
    return nn_idx, nn_w


def interpolate3_gather_rows(nn_idx: Tensor, nn_w: Tensor, feat_rows: Tensor, out: Tensor) -> Tensor:
    """out[b,n,:] = sum_j nn_w[b,n,j] * feat_rows[b, nn_idx[b,n,j], :] (models/upsample.py:210-212); feat_rows (B,M,C), out
    (B,N,C) rows with unit inner stride (may be a column slice of a wider buffer)."""
    L.need_cuda(nn_idx, nn_w, feat_rows, out)
    L.no_grad_check(feat_rows)
    feat_rows = _f32(feat_rows, "feat")
    if feat_rows.stride(2) != 1:
        feat_rows = feat_rows.contiguous()
    B, N, _ = nn_idx.shape
    M, Cc = feat_rows.shape[1], feat_rows.shape[2]
    if tuple(out.shape) != (B, N, Cc) or out.stride(2) != 1 or out.stride(0) != N * out.stride(1) or \
            feat_rows.stride(0) != M * feat_rows.stride(1):
        raise RuntimeError("interpolate3_gather_rows: out must be (B,N,C) rows with a common pitch")
    L.check(L.lib().samble_interpolate3_gather_rows(L.ptr(nn_idx), L.ptr(nn_w), L.ptr(feat_rows), feat_rows.stride(1), B, N, M, Cc,
                                                    L.ptr(out), out.stride(1), L.stream()), "samble_interpolate3_gather_rows")
    return out


# ------------------------------------------------------------------ bins (reference signatures)


def _quantile_pick(ranked: Tensor, num_bins: int) -> Tensor:
    """cut[j-1] = ranked[int(j / num_bins * n)] (utils/ops.py:182-189), one native launch."""
    dev = L.need_cuda(ranked)
    cut = torch.empty(num_bins - 1, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_quantile_pick(L.ptr(ranked), ranked.numel(), num_bins, L.ptr(cut), L.stream()), "samble_quantile_pick")
    return cut


def _boundary_ema(cut_sum: Tensor, world: int, old_bin_boundaries, num_bins: int, momentum_update_factor: float):
    """rank average + EMA blend (or creation with the +-inf sentinels) of the [upper, lower] pair (utils/ops.py:198-233), one
    native launch."""
    dev = L.need_cuda(cut_sum)
    if old_bin_boundaries is not None:
        upper = old_bin_boundaries[0].detach().to(device=dev, dtype=torch.float32).contiguous()
        lower = old_bin_boundaries[1].detach().to(device=dev, dtype=torch.float32).contiguous()
    else:
        upper = torch.empty(1, 1, 1, num_bins, dtype=torch.float32, device=dev)
        lower = torch.empty(1, 1, 1, num_bins, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_boundary_ema(L.ptr(cut_sum), world, float(momentum_update_factor), 1 if old_bin_boundaries is not None else 0,
                                        num_bins, L.ptr(upper), L.ptr(lower), L.stream()), "samble_boundary_ema")
    return [upper, lower]


def update_sampling_score_bin_boundary(old_bin_boundaries, attention_point_score: Tensor, num_bins: int,
                                       momentum_update_factor: float):
    """utils/ops.py:174-236.  Batch quantiles of the z-scored point score -> [upper, lower] pair, rank-averaged when a
    process group exists (:191-199) and EMA-blended into the old pair.  One device sort (ATen's radix sort of B*N keys),
    then two native launches around ONE all_reduce of nb-1 floats (quantile pick; average + EMA + sentinels): a
    training-time, latency-bound step.  The collective plumbing is covered by a world_size-2 gloo test in which the two
    native steps are replaced by their oracle statements (tests/test_distributed_cpu.py)."""
    z = attention_point_score
    ranked, _ = torch.sort(z.detach().flatten(), dim=0, descending=True)
    cut = _quantile_pick(ranked, num_bins)
    world = 1
    if torch.distributed.is_available() and torch.distributed.is_initialized():
        torch.distributed.all_reduce(cut)
        world = torch.distributed.get_world_size()
    return _boundary_ema(cut, world, old_bin_boundaries, num_bins, momentum_update_factor)


def bin_partition(attention_point_score: Tensor, bin_boundaries, dynamic_boundaries_enable: bool,
                  momentum_update_factor: float, num_bins: int):
    """utils/ops.py:435-464.  score (B,H,N) -> ([upper, lower], mask (B,H,N,num_bins) bool)."""
    dev = L.need_cuda(attention_point_score)
    attention_point_score = attention_point_score.detach()      # a partition: no gradient in the reference either
    B, H, N = attention_point_score.shape
    if bin_boundaries is not None:
        bin_boundaries = [t.to(dev) for t in bin_boundaries]
    z = zscore(attention_point_score)
    if dynamic_boundaries_enable:
        bin_boundaries = update_sampling_score_bin_boundary(bin_boundaries, z.reshape(B, H, N, 1), num_bins,
                                                            momentum_update_factor)
    upper = bin_boundaries[0].reshape(-1).to(torch.float32).contiguous()
    lower = bin_boundaries[1].reshape(-1).to(torch.float32).contiguous()
    mask = torch.empty(B, H, N, num_bins, dtype=torch.uint8, device=dev)
    L.check(L.lib().samble_bin_mask(L.ptr(z), L.ptr(upper), L.ptr(lower), B * H, N, num_bins, L.ptr(mask), L.stream()),
            "samble_bin_mask")
    return bin_boundaries, mask.view(torch.bool)


def calculate_num_points_to_choose(bin_prob: Tensor, max_num_points: Tensor, total_points_to_choose: int) -> Tensor:
    """utils/ops.py:385-432.  (B,nb) fp32, (B,nb) int64, int -> (B,nb) int32."""
    dev = L.need_cuda(bin_prob, max_num_points)
    B, nb = bin_prob.shape
    bin_prob = _f32(bin_prob, "bin_prob").contiguous()
    cnt = max_num_points.to(torch.int64).contiguous()
    k = torch.empty(B, nb, dtype=torch.int32, device=dev)
    L.check(L.lib().samble_num_points_to_choose(L.ptr(bin_prob), L.ptr(cnt), B, nb, int(total_points_to_choose), L.ptr(k),
                                                L.stream()), "samble_num_points_to_choose")
    return k


def sampling_probabilities(attention_point_score: Tensor, bin_points_mask: Tensor, bin_sample_mode: str, boltzmann_t) -> Tensor:
    """utils/ops.py:507-592: the per-(cloud, bin) categorical distribution the 'uniform' / 'random' sampling modes draw
    from, (B*nb, N) on the device -- one native launch per batch (csrc/sampler.cu: z-score, tanh, exp, mask, per-bin
    normalisation in one CTA per cloud) instead of the reference's chain of element-wise ops over (B,N,nb)."""
    import numbers

    dev = L.need_cuda(attention_point_score, bin_points_mask)
    B, H, N, nb = bin_points_mask.shape
    if H != 1:
        raise ValueError("sampling_probabilities: one attention head expected (reference: 'has to be 1 head')")
    inv_t, t_div = 0.0, 0.0
    if bin_sample_mode == "uniform":
        mode = 0
    elif bin_sample_mode == "random":
        mode = 1
        if boltzmann_t in ("mode_1", "mode_3"):
            t_div = 100.0 if boltzmann_t == "mode_1" else 200.0
        elif boltzmann_t == "mode_2":
            inv_t = N / (100.0 * nb)
        elif boltzmann_t == "mode_4":
            inv_t = N / (200.0 * nb)
        elif isinstance(boltzmann_t, numbers.Number):
            inv_t = 1 / boltzmann_t
        else:
            raise NotImplementedError
    else:
        raise ValueError("Please check the setting of bin sample mode. It must be topk, multinomial or random!")
    score = _f32(attention_point_score.detach(), "score").reshape(B, N).contiguous()
    mask = bin_points_mask.reshape(B, N, nb).to(torch.uint8).contiguous()
    p = torch.empty(B * nb, N, dtype=torch.float32, device=dev)
    L.check(L.lib().samble_sampling_probabilities(L.ptr(score), L.ptr(mask), B, N, nb, mode, float(inv_t), float(t_div), L.ptr(p),
                                                  L.stream()), "samble_sampling_probabilities")
    return p


def generating_downsampled_index(M: int, attention_point_score: Tensor, bin_points_mask: Tensor, bin_sample_mode: str,
                                 boltzmann_t, k_point_to_choose: Tensor) -> Tensor:
    """utils/ops.py:467-619.  'topk' (:476-505) is the native per-bin top-k kernel.  'uniform' / 'random' (:507-613)
    draw M indices per (cloud, bin) without replacement with torch.multinomial -- the reference's own sampler, so
    the stream of random numbers is the device generator's -- and keep the first k of each bin, bins in order."""
    if bin_sample_mode in ("uniform", "random"):
        L.need_cuda(attention_point_score, bin_points_mask, k_point_to_choose)
        B, H, N, nb = bin_points_mask.shape
        p = sampling_probabilities(attention_point_score, bin_points_mask, bin_sample_mode, boltzmann_t)
        draws = torch.multinomial(p, M).reshape(B, nb, M)
        keep = torch.arange(M, device=draws.device).view(1, 1, M) < k_point_to_choose.view(B, nb, 1)
        return draws[keep].reshape(B, 1, M)            # row-major over (cloud, bin, draw): bins in order, sum_k = M
    if bin_sample_mode != "topk":
        raise ValueError("Please check the setting of bin sample mode. It must be topk, multinomial or random!")
    dev = L.need_cuda(attention_point_score, bin_points_mask, k_point_to_choose)
    B, H, N, nb = bin_points_mask.shape
    if H != 1:
        raise ValueError("generating_downsampled_index: one attention head expected (reference: 'has to be 1 head')")
    score = _f32(attention_point_score, "score").reshape(B, N).contiguous()
    mask = bin_points_mask.reshape(B, N, nb).to(torch.uint8).contiguous()
    k = k_point_to_choose.to(torch.int32).contiguous()
    idx = torch.empty(B, 1, M, dtype=torch.int64, device=dev)
    L.check(L.lib().samble_downsample_index_topk(L.ptr(score), L.ptr(mask), L.ptr(k), B, N, nb, M, L.ptr(idx), L.stream()),
            "samble_downsample_index_topk")
    return idx
