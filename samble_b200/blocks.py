"""The four hot-path blocks as nn.Modules, state_dict-compatible with the reference's.

Constructor signature `Cls(config_subtree, layer)`, forward signatures, parameter
names/shapes and the public attributes callers read (SURVEY 3.4-10, 8b) follow
  models/embedding.py:7-39     EdgeConv
  models/attention.py:130-250  Neighbor2PointAttention
  models/downsample.py:15-378  DownSampleToken
  models/upsample.py:136-213   UpSampleInterpolation
so a reference checkpoint loads with load_state_dict and the reference's model wiring
can construct these in place of its own (samble_b200.patch).

Forward passes run the sm_100a kernels through samble_b200.ops; plain library GEMMs
(1x1 convolutions on N points, BatchNorm) stay in PyTorch/cuBLAS.  There is no CPU path.
"""
from __future__ import annotations

import math

import torch
import torch.nn.functional as F
from torch import nn

from . import ops
from ._precision import fp32_forward

Tensor = torch.Tensor


def differentiable(mod: nn.Module, *tensors) -> bool:
    """True when a forward must take the differentiable path (samble_b200.autograd + ATen dense layers): BatchNorm needs
    batch statistics (train mode), or a gradient could be asked for (grad mode on and an input or a parameter of `mod`
    requires grad).  Otherwise the fused inference kernels run; they refuse tensors that require grad (_lib.no_grad_check)."""
    if mod.training:
        return True
    if not torch.is_grad_enabled():
        return False
    return any(t is not None and t.requires_grad for t in tensors) or any(p.requires_grad for p in mod.parameters())


def fold_bn(bn: nn.modules.batchnorm._BatchNorm):
    """eval-mode BatchNorm as y = a*x + b."""
    a = bn.weight / torch.sqrt(bn.running_var + bn.eps)
    return a, bn.bias - bn.running_mean * a


_BN_CACHE: "weakref.WeakKeyDictionary" = None


def folded(bn: nn.modules.batchnorm._BatchNorm):
    """fold_bn with a per-module cache keyed on the in-place version counters of its tensors."""
    global _BN_CACHE
    import weakref

    if _BN_CACHE is None:
        _BN_CACHE = weakref.WeakKeyDictionary()
    ts = (bn.weight, bn.bias, bn.running_mean, bn.running_var)
    key = tuple((t.data_ptr(), t._version) for t in ts)
    hit = _BN_CACHE.get(bn)
    if hit is None or hit[0] != key:
        with torch.no_grad():
            a, b = fold_bn(bn)
        hit = (key, (a.contiguous(), b.contiguous()))
        _BN_CACHE[bn] = hit
    return hit[1]


def cbl(seq: nn.Sequential, x: Tensor, x_layout: str = "bcn", out_layout: str = "bcn", shift_extra: Tensor = None) -> Tensor:
    """eval-mode nn.Sequential(Conv1d 1x1 (no bias), BatchNorm1d, LeakyReLU(0.2)) as ONE tensor-core GEMM with the
    BatchNorm folded into the epilogue (csrc/linear_tc.cu)."""
    a, b = folded(seq[1])
    return ops.linear(x, seq[0].weight, x_layout=x_layout, out_layout=out_layout, scale=a,
                      shift=b if shift_extra is None else shift_extra, lrelu=True)


def cbl_pool(seq: nn.Sequential, x: Tensor, x_layout: str = "bcn", want_max: bool = True, want_mean: bool = True):
    """(cbl(seq, x).max over points, .mean over points) with the activation never stored (ops.linear_pool).
    Falls back to the unfused form when a cloud is not a whole number of 32-point groups."""
    a, b = folded(seq[1])
    x_rows = ops.rows_of(x) if x_layout == "bcn" else x
    if x_rows.shape[1] % 32:
        y = ops.linear(x_rows, seq[0].weight, scale=a, shift=b, lrelu=True)
        return (y.max(dim=1)[0] if want_max else None), (y.mean(dim=1) if want_mean else None)
    return ops.linear_pool(x_rows, seq[0].weight, scale=a, shift=b, lrelu=True, want_max=want_max, want_mean=want_mean)


class _FoldCache:
    """Folded weights of an edge MLP, recomputed only when a parameter/buffer was modified in place
    (tensor._version) or moved."""

    def __init__(self):
        self.key, self.val = None, None

    def get(self, tensors, build):
        key = tuple((t.data_ptr(), t._version) for t in tensors)
        if key != self.key:
            with torch.no_grad():
                self.val = build()
            self.key = key
        return self.val


def edge_mlp_weights(conv1, bn1, conv2, bn2, group_type: str):
    """Fold conv1+BN1 into per-point projections and BN2 into conv2 (csrc/edgeconv.cu header)."""
    w1 = conv1.weight.flatten(1)                         # (C1, Cin_total)
    c1 = w1.shape[0]
    if group_type.startswith("center"):
        cin = w1.shape[1] // 2
        wa, wb = w1[:, :cin], w1[:, cin:]
        a_mat = wa - wb if group_type == "center_diff" else wa
        b_mat = wb
    else:
        a_mat = -w1 if group_type == "diff" else torch.zeros_like(w1)
        b_mat = w1
    a1, b1 = fold_bn(bn1)
    a2, b2 = fold_bn(bn2)
    w_pr = torch.cat([a1[:, None] * a_mat, a1[:, None] * b_mat], dim=0).contiguous()          # (2*C1, Cin)
    bias_pr = torch.cat([b1, torch.zeros_like(b1)]).contiguous()                               # shift rides on P
    w2 = (a2[:, None] * conv2.weight.flatten(1)).contiguous()                                  # (C2, C1)
    return w_pr, bias_pr, w2, b2.contiguous()


def fused_edge_mlp(x: Tensor, idx: Tensor, weights, out_rows: Tensor = None) -> Tensor:
    """x (B,Cin,N), idx (B,N,K) -> (B,C2,N): one library GEMM over the N points + the fused kernel."""
    w_pr, bias_pr, w2, b2 = weights
    pr = ops.linear(x, w_pr, x_layout="bcn", out_layout="rows", shift=bias_pr)                  # (B,N,2*C1)
    return ops.edge_mlp_max(pr, idx() if callable(idx) else idx, w2, b2, out_rows=out_rows)


class EdgeConv(nn.Module):
    """models/embedding.py:7-39: group -> (conv1x1+BN+LeakyReLU) x2 -> max over K.

    eval mode: fused (csrc/edgeconv.cu), nothing of size N*K touches HBM.  train mode (BatchNorm batch
    statistics cannot be folded): native group kernel + library convolutions, as the reference computes it."""

    def __init__(self, config_embedding, layer):
        super().__init__()
        self.K = config_embedding.K[layer]
        self.group_type = config_embedding.group_type[layer]
        self.normal_channel = config_embedding.normal_channel

        def cbl(cin, cout):
            return nn.Sequential(nn.Conv2d(cin, cout, kernel_size=1, bias=False), nn.BatchNorm2d(cout),
                                 nn.LeakyReLU(negative_slope=0.2))

        self.conv1 = cbl(config_embedding.conv1_in[layer], config_embedding.conv1_out[layer])
        self.conv2 = cbl(config_embedding.conv2_in[layer], config_embedding.conv2_out[layer])
        self._fold = _FoldCache()

    @fp32_forward
    def forward(self, x: Tensor, out_rows: Tensor = None) -> Tensor:
        """out_rows (optional, ours): a (B,N,C2) row-major slot -- e.g. this layer's columns of the concatenated embedding
        (seg_model.py:98-102) -- that the fused kernel fills in place; the result is returned as its (B,C2,N) view."""
        if self.group_type not in ("neighbor", "diff", "center_neighbor", "center_diff"):
            raise ValueError(
                f"group_type should be neighbor, diff, center_neighbor or center_diff, but got {self.group_type}")
        c2 = self.conv2[0].out_channels
        if differentiable(self, x) or self.K > 32 or c2 not in (32, 64, 128) or self.conv1[0].out_channels % 4:
            x, _ = ops.group(x, self.K, self.group_type, self.normal_channel)
            y = self.conv2(self.conv1(x)).max(dim=-1, keepdim=False)[0]
            if out_rows is not None:
                out_rows.copy_(y.transpose(1, 2))
            return y
        key = x[:, :3, :] if (self.normal_channel and x.shape[1] == 6) else x
        idx = ops.fork(lambda: ops.knn_indices(key, self.K, ordered=False))      # concurrent with the point projections
        params = [self.conv1[0].weight, self.conv2[0].weight, *self.conv1[1].parameters(), *self.conv1[1].buffers(),
                  *self.conv2[1].parameters(), *self.conv2[1].buffers()]
        weights = self._fold.get(params, lambda: edge_mlp_weights(self.conv1[0], self.conv1[1], self.conv2[0],
                                                                  self.conv2[1], self.group_type))
        return fused_edge_mlp(x, idx, weights, out_rows)


class Neighbor2PointAttention(nn.Module):
    """models/attention.py:130-250 (scalar_dot / asm 'dot' / group 'diff', the shipped setting).

    The reference convolves the gathered (B,C,N,K) differences with k_conv/v_conv; both are
    bias-free and linear, so the N points are projected ONCE ([q|k|v] in one GEMM) and the fused
    kernel gathers projected rows (csrc/attention.cu): 32x fewer projection FLOPs, no (B,C,N,K)."""

    def __init__(self, config_attention, layer):
        super().__init__()
        self.K = config_attention.K[layer]
        self.group_type = config_attention.group_type[layer]
        self.num_heads = config_attention.num_heads[layer]
        self.attention_mode = config_attention.attention_mode[layer]
        self.asm = config_attention.asm[layer]
        q_in, q_out = config_attention.q_in[layer], config_attention.q_out[layer]
        k_in, k_out = config_attention.k_in[layer], config_attention.k_out[layer]
        v_in, v_out = config_attention.v_in[layer], config_attention.v_out[layer]
        self.q_depth, self.k_depth, self.v_depth = (int(c / self.num_heads) for c in (q_out, k_out, v_out))
        self.q_conv = nn.Conv2d(q_in, q_out, 1, bias=False)
        self.k_conv = nn.Conv2d(k_in, k_out, 1, bias=False)
        self.v_conv = nn.Conv2d(v_in, v_out, 1, bias=False)
        self.softmax = nn.Softmax(dim=-1)
        self.ff = nn.Sequential(
            nn.Conv1d(config_attention.ff_conv1_channels_in[layer], config_attention.ff_conv1_channels_out[layer], 1, bias=False),
            nn.LeakyReLU(negative_slope=0.2),
            nn.Conv1d(config_attention.ff_conv2_channels_in[layer], config_attention.ff_conv2_channels_out[layer], 1, bias=False),
        )
        self.bn1 = nn.BatchNorm1d(v_out)
        self.bn2 = nn.BatchNorm1d(v_out)
        self._wqkv = _FoldCache()

    @fp32_forward
    def forward(self, x: Tensor) -> Tensor:
        if self.group_type != "diff" or self.attention_mode != "scalar_dot" or self.asm != "dot":
            raise NotImplementedError("native Neighbor2PointAttention covers group_type='diff', "
                                      "attention_mode='scalar_dot', asm='dot' (the shipped configs)")
        B, C, N = x.shape
        if differentiable(self, x):
            idx = ops.knn_indices(x, self.K, ordered=False)                                    # (B,N,K) int32
            # train mode / gradients: the same hoisted form, projections and BatchNorm (batch statistics) in ATen, the
            # attention core and its backward native (autograd.N2PAttend) -- still no (B,C,N,K) tensor in either direction
            w = torch.cat([self.q_conv.weight, self.k_conv.weight, self.v_conv.weight], dim=0).view(3 * C, C)
            qkv = torch.matmul(x.transpose(1, 2), w.t())                        # (B,N,3C) point-major
            y = ops.n2p_attend(qkv, idx, self.num_heads)                        # (B,N,C)
            x = self.bn1(x + y.transpose(1, 2))
            return self.bn2(x + self.ff(x))
        w = self._wqkv.get([self.q_conv.weight, self.k_conv.weight, self.v_conv.weight], lambda: torch.cat(
            [self.q_conv.weight, self.k_conv.weight, self.v_conv.weight], dim=0).view(3 * C, C).contiguous())
        # eval: everything point-major, projections / feed-forward on the tensor cores, BatchNorms folded into epilogues
        join_idx = ops.fork(lambda: ops.knn_indices(x, self.K, ordered=False))  # (B,N,K) int32, concurrent with the projection
        x_pm = ops.rows_of(x)                                                   # (B,N,C)
        qkv = ops.linear(x_pm, w)                                               # (B,N,3C)
        a1, b1 = folded(self.bn1)
        a2, b2 = folded(self.bn2)
        x1 = ops.n2p_attend(qkv, join_idx(), self.num_heads, residual=x_pm, scale=a1, shift=b1)     # bn1(x + attention)
        w1, w2 = self.ff[0].weight, self.ff[2].weight
        if ops.FUSED_MLP2 and ops.mlp2_eligible(w1.shape[1], w1.shape[0], w2.shape[0]):
            # feed-forward + residual + bn2 in one kernel, the (B,N,4C) hidden activation stays in tensor memory (csrc/mlp2.cu)
            y = ops.mlp2(x1, w1, w2, lrelu1=True, scale2=a2, shift2=b2, residual=x1, residual_first=True)
        else:
            h = ops.linear(x1, w1, lrelu=True)                                  # (B,N,4C)
            y = ops.linear(h, w2, scale=a2, shift=b2, residual=x1, residual_first=True)      # (B,N,C)
        return y.transpose(1, 2)          # the reference's (B,C,N) shape as a view of point-major storage (ops.rows_of)


# DownSampleToken's score-deciding contractions on the exact-product GEMM (csrc/xgemm.cu).  False = the 3xTF32 kernels
# of round 1 (kept for A/B measurements: tools/diag_parity.py).
DS_EXACT = True


class DownSampleToken(nn.Module):
    """models/downsample.py:15-378 for the shipped configuration: asm 'dot', one head, multi_token,
    idx_mode sparse_col_sqr, mean_relu, res off, sample_mode 'topk'.

    Pipeline (no N x N tensor is ever written):
      [q|k|v] projection -> feature kNN (knn.cu) -> row softmax statistics -> edge-only column score (downsample.cu)
      -> z-score / bins / k per bin / per-bin top-k (sampler.cu) -> attention rows of the M selected points x V.

    Two branches compute the projection, the row statistics and the selected rows (_forward_native):
      exact  (C <= 128, C % 32 == 0, D == C; DS_EXACT): exact-product GEMM for [q|k|v] and q k^T (xgemm.cu), the rows
             as one flash-style kernel over the N + nb keys (ds_attend.cu);
      3xTF32 (every other width, or DS_EXACT = False): tensor-core projection (linear_tc.cu), row statistics on the fast
             tensor-core kernel when N % 128 == 0 (else ds_rowstats_tc.cu / the FFMA kernel of downsample.cu), the
             selected rows gathered by ds_select_rows and multiplied by two per-cloud GEMMs (cloud_matmul) when
             M % 128 == 0 and N <= 4096, else by ATen matmuls on the (B,M,N) slab.
    """

    def __init__(self, config_ds, layer):
        super().__init__()
        self.M = config_ds.M[layer]
        self.K = config_ds.K
        self.asm = config_ds.asm[layer]
        self.res = config_ds.res.enable[layer]
        self.ff = config_ds.res.ff[layer]
        self.num_heads = config_ds.num_heads[layer]
        self.idx_mode = config_ds.idx_mode[layer]
        self.relu_mean_order = config_ds.bin.relu_mean_order[layer]
        self.num_bins = config_ds.bin.num_bins[layer]
        q_in, q_out = config_ds.q_in[layer], config_ds.q_out[layer]
        k_in, k_out = config_ds.k_in[layer], config_ds.k_out[layer]
        v_in, v_out = config_ds.v_in[layer], config_ds.v_out[layer]
        self.q_depth, self.k_depth, self.v_depth = (int(c / self.num_heads) for c in (q_out, k_out, v_out))
        self.q_conv = nn.Conv1d(q_in, q_out, 1, bias=False)
        self.k_conv = nn.Conv1d(k_in, k_out, 1, bias=False)
        self.v_conv = nn.Conv1d(v_in, v_out, 1, bias=False)
        self.token_mode = config_ds.bin.token_mode[layer]
        if self.token_mode != "multi_token":
            raise NotImplementedError("only token_mode 'multi_token' (the shipped setting) is built")
        self.bin_tokens = nn.Parameter(torch.normal(mean=0, std=1 / math.sqrt(q_in), size=(1, q_in, self.num_bins)))
        self.softmax = nn.Softmax(dim=-1)
        if self.res:
            raise NotImplementedError("DownSampleToken residual link is off in every shipped config (default.yaml:188-190)")
        self.scaling_factor = config_ds.bin.scaling_factor[layer]
        self.bin_sample_mode = config_ds.bin.sample_mode[layer]
        self.bin_norm_mode = config_ds.bin.norm_mode[layer]
        self.momentum_update_factor = config_ds.bin.momentum_update_factor[layer]
        self.dynamic_boundaries_enable = config_ds.bin.dynamic_boundaries_enable
        if self.dynamic_boundaries_enable:
            self.bin_boundaries = None
        else:
            cuts = [float(v) for v in config_ds.bin.bin_boundaries[layer]]     # not mutated (cf. downsample.py:98-99)
            self.bin_boundaries = [torch.tensor([float("inf")] + cuts).reshape(1, 1, 1, self.num_bins),
                                   torch.tensor(cuts + [float("-inf")]).reshape(1, 1, 1, self.num_bins)]
        self.boltzmann_enable = config_ds.boltzmann.enable[layer]
        self.boltzmann_T = config_ds.bin.boltzmann_T[layer]
        self.boltzmann_norm_mode = config_ds.boltzmann.norm_mode[layer]
        self.token_orthognonal_loss_factor = config_ds.bin.token_orthognonal_loss_factor
        self._wqkv = _FoldCache()

    # -- helpers -------------------------------------------------------------------------------
    def _cuts(self, device) -> Tensor:
        """the nb-1 finite thresholds of the [upper, lower] pair.  The native partition assigns a point to the FIRST bin whose
        interval holds its z-score, which equals the reference's mask (utils/ops.py:460-462) only for non-increasing cuts
        with lower[j] == upper[j+1]; that is checked once per boundary update outside graph capture (one host sync) and
        anything else is refused rather than partitioned differently."""
        upper = self.bin_boundaries[0]
        if upper.device != device:
            self.bin_boundaries = [t.to(device) for t in self.bin_boundaries]
            upper = self.bin_boundaries[0]
        cuts = upper.reshape(-1)[1:].to(torch.float32).contiguous()
        key = (upper.data_ptr(), upper._version, self.bin_boundaries[1].data_ptr(), self.bin_boundaries[1]._version)
        if key != getattr(self, "_cuts_checked", None) and not self.dynamic_boundaries_enable and not torch.cuda.is_current_stream_capturing():
            lower = self.bin_boundaries[1].reshape(-1)[:-1].to(device=device, dtype=torch.float32)
            ok = bool(((cuts[:-1] >= cuts[1:]).all() if cuts.numel() > 1 else torch.tensor(True)) & (lower == cuts).all())
            if not ok:
                raise ValueError("DownSampleToken: bin boundaries must be non-increasing with lower[j] == upper[j+1] "
                                 "(the [upper, lower] pair utils/ops.py:174-236 maintains)")
            self._cuts_checked = key
        return cuts

    @fp32_forward
    def forward(self, x: Tensor, x_xyz=None):
        if self.asm != "dot" or self.idx_mode != "sparse_col_sqr" or self.relu_mean_order != "mean_relu" or self.num_heads != 1:
            raise NotImplementedError("native DownSampleToken covers asm='dot', idx_mode='sparse_col_sqr', "
                                      "relu_mean_order='mean_relu', one head (the shipped configs)")
        if self.bin_sample_mode not in ("topk", "uniform", "random"):
            raise ValueError("Please check the setting of bin sample mode. It must be topk, multinomial or random!")
        if differentiable(self, x):
            # train mode / gradients.  The sampled indices are a discrete decision (no gradient in the reference either):
            # they come from the same native scoring + sampling kernels.  Gradients flow through the selected attention
            # rows times V (:242-252) and through the token logits (token-orthogonality loss, train_shapenet.py:401-413),
            # which are formed here in ATen on an (B,M,N+nb) slab -- not the reference's (B,N,N+nb).
            with torch.no_grad():
                _, index_down = self._forward_native(x.detach(), want_rows=False)
            x_ds, tok = self._selected_rows_autograd(x, index_down)
            self.attention_bins_beforesoftmax = tok
            return (x_ds, index_down), (None, None)
        x_ds, index_down = self._forward_native(x, want_rows=True)
        return (x_ds, index_down), (None, None)

    def _selected_rows_autograd(self, x: Tensor, index_down: Tensor):
        """x_ds (B,C,M) and the pre-softmax token logits (B,1,N,nb) as differentiable functions of x and the parameters."""
        B, C, N = x.shape
        nb, scale = self.num_bins, math.sqrt(self.q_depth)
        xt = torch.cat([x, self.bin_tokens.expand(B, -1, -1)], dim=2)          # (B,C,N+nb)  (:116-118)
        q, k, v = self.q_conv(x), self.k_conv(xt), self.v_conv(xt)             # (B,D,N), (B,D,N+nb) x2
        tok = torch.matmul(q.transpose(1, 2), k[:, :, N:]) / scale             # (B,N,nb)
        q_sel = ops.gather_by_idx(q, index_down)                               # (B,D,M), native gather + scatter-add backward
        att = torch.softmax(torch.matmul(q_sel.transpose(1, 2), k) / scale, dim=-1)          # (B,M,N+nb)
        x_ds = torch.matmul(att, v.transpose(1, 2)).transpose(1, 2)            # (B,C,M)
        return x_ds, tok.view(B, 1, N, nb)

    def _forward_native(self, x: Tensor, want_rows: bool):
        B, C, N = x.shape
        D, nb = self.q_depth, self.num_bins
        # projections of the points and of the nb bin tokens (shared by the whole batch, :116-118)
        w = self._wqkv.get([self.q_conv.weight, self.k_conv.weight, self.v_conv.weight], lambda: torch.cat(
            [self.q_conv.weight, self.k_conv.weight, self.v_conv.weight], dim=0).view(3 * C, C).contiguous())
        # The two contractions that decide the sampled indices run on the exact-product tensor-core GEMM (csrc/xgemm.cu):
        # fp32-class accuracy independent of accumulation order (the 3xTF32 kernels' logit error is exponentiated here).
        # The projection's per-cloud max|q|, |k|, |v| come out of the GEMM in groups of C columns, whole 32-column tiles.
        exact = DS_EXACT and C <= 128 and C % 32 == 0 and D == C
        join_idx = ops.fork(lambda: ops.knn_indices(x, self.K, ordered=False))                # neighbor_mask's kNN (:301), concurrent
        if exact:
            x_rows = ops.rows_of(x)                                            # (B,N,C)
            qkv, amax = ops.xgemm(ops.digits(x_rows), ops.weight_digits(w), amax_group=C)     # (B,N,3C) + max|q|,|k|,|v| per cloud
        else:
            qkv = ops.linear(x, w, x_layout="bcn")                             # (B,N,3C), 3xTF32
        q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
        tok = self.bin_tokens[0].t()                                           # (nb,C)
        k_tok = torch.matmul(tok, self.k_conv.weight.view(C, C).t()).contiguous()   # (nb,D)
        v_tok = torch.matmul(tok, self.v_conv.weight.view(C, C).t())

        k_split = None
        if exact:
            qd, kd = ops.digits(q, amax, 0), ops.digits(k, amax, 1)
            rowmax, rowsum, tok_logits = ops.ds_row_stats_exact(qd, kd, q, k_tok)
        else:
            k_split = ops.split_operand(k) if (self.M % 128 == 0 and N <= 4096) else None     # for the M selected rows
            rowmax, rowsum, tok_logits = ops.ds_row_stats(q, k, k_tok, k_split=k_split)
        score = ops.ds_edge_score(q, k, rowmax, rowsum, join_idx())            # (B,N)
        self.attention_point_score = score.view(B, 1, N)

        if self.dynamic_boundaries_enable:
            z = ops.zscore(score)
            self.bin_boundaries = ops.update_sampling_score_bin_boundary(
                self.bin_boundaries, z.view(B, 1, N, 1), nb, self.momentum_update_factor)
        s = ops.ds_sample(score, tok_logits, self._cuts(x.device), self.M)
        self.bin_points_mask = (s["bin_id"].view(B, 1, N, 1) == torch.arange(nb, device=x.device, dtype=torch.uint8))
        if self.bin_sample_mode != "topk":           # stochastic modes (ops.py:507-613): bins and k as above, indices drawn
            s["idx"] = ops.generating_downsampled_index(self.M, score.view(B, 1, N), self.bin_points_mask, self.bin_sample_mode,
                                                        self.boltzmann_T, s["k"]).view(B, self.M)
        index_down = s["idx"].view(B, 1, self.M)
        self.k_point_to_choose = s["k"]
        self.bin_weights_beforerelu = s["w_raw"]

        # attention rows of the selected points over all N+nb keys, times V (:242-252).  The softmax statistics of every
        # row are already known (pass 1), so one flash-style kernel forms S = Q_sel K^T in TMEM, turns it into
        # probabilities in registers and feeds them to the second MMA through shared memory (csrc/ds_attend.cu): no
        # (B,M,N) tensor exists.
        sel = s["idx"]
        scale = math.sqrt(D)
        self.idx = index_down
        self.attention_bins_beforesoftmax = tok_logits.view(B, 1, N, nb)
        if not want_rows:
            return None, index_down
        if exact:
            x_ds = ops.ds_attend_rows(qd, kd, v, sel, rowmax, rowsum, tok_logits, v_tok)          # (B,M,C)
        else:
            q_sel, m_sel, s_sel, tok_mix = ops.ds_select_rows(q, rowmax, rowsum, tok_logits, v_tok, sel)
            if self.M % 128 == 0 and N <= 4096:        # (samble_cloud_matmul contracts at most 4096 keys)
                att = ops.cloud_matmul(q_sel, k, row_max=m_sel, row_sum=s_sel, logit_div=scale, w_split=k_split)     # (B,M,N)
                x_ds = ops.cloud_matmul(att, v.transpose(1, 2), residual=tok_mix)                     # (B,M,C)
            else:
                att = torch.exp(torch.matmul(q_sel, k.transpose(1, 2)) / scale - m_sel.unsqueeze(-1)) / s_sel.unsqueeze(-1)
                x_ds = torch.matmul(att, v) + tok_mix
        return x_ds.transpose(1, 2), index_down

    # reference API kept for callers (downsample.py:346-378)
    def output_variable_calculatio(self):
        B, _, _, num_bins = self.bin_points_mask.shape
        index_batch, _, index_point, index_bin = torch.where(self.bin_points_mask)
        self.idx_chunks = [[index_point[(index_bin == i) & (index_batch == j)].reshape(1, -1) for j in range(B)]
                           for i in range(num_bins)]
        self.bin_prob = self.bin_weights_beforerelu

    def output_variables(self, *args):
        vals = tuple(getattr(self, key) for key in args)
        return vals[0] if len(vals) == 1 else (vals if vals else None)


class UpSampleInterpolation(nn.Module):
    """models/upsample.py:136-213: conv on the coarse features -> 3-NN inverse-distance interpolation
    (fused kernel, csrc/upsample.cu) -> concat skip -> conv."""

    def __init__(self, config_upsample, layer):
        super().__init__()
        q_in, v_out = config_upsample.q_in[layer], config_upsample.v_out[layer]
        self.distance_type = config_upsample.interpolation.distance_type[layer]
        self.K = config_upsample.interpolation.K[layer]

        def cbl(cin, cout):
            return nn.Sequential(nn.Conv1d(cin, cout, 1, bias=False), nn.BatchNorm1d(cout), nn.LeakyReLU(negative_slope=0.2))

        self.conv = cbl(q_in, v_out)
        self.res_conv = cbl(2 * v_out, v_out)

    @fp32_forward
    def forward(self, pcd_up, pcd_down, pcd_up_xyz):
        (points_select, idx_select, points_select_xyz), (points_drop, idx_drop) = pcd_down
        slow = differentiable(self, pcd_up, points_select, pcd_up_xyz, points_select_xyz)
        # the row kernels (csrc/upsample.cu) read and write 16-byte chunks: the feature width and the column offset of the
        # interpolated half in [pcd_up | interpolated] must be multiples of 4 floats
        rows = self.conv[0].out_channels % 4 == 0 and pcd_up.shape[1] % 4 == 0
        if not slow and self.distance_type == "xyz" and self.K == 3 and rows:
            # point-major throughout: [pcd_up | interpolated] is assembled as rows (the interpolation writes its half in
            # place), res_conv reads it as a GEMM operand, the result is handed on as a (B,C,N) view of rows
            B, C, N = pcd_up.shape
            search = ops.fork(lambda: ops.interpolate3_search(pcd_up_xyz, points_select_xyz))   # needs xyz only: parallel branch
            feat = cbl(self.conv, points_select, out_layout="rows")                        # (B,M,C')
            both = torch.empty(B, N, C + feat.shape[2], dtype=torch.float32, device=pcd_up.device)
            both[..., :C].copy_(ops.rows_of(pcd_up))
            nn_idx, nn_w = search()
            ops.interpolate3_gather_rows(nn_idx, nn_w, feat, both[..., C:])
            return cbl(self.res_conv, both, x_layout="rows", out_layout="rows").transpose(1, 2)
        interpolated = self.interpolate(pcd_up, points_select, pcd_up_xyz, points_select_xyz,
                                        distance_type=self.distance_type, K=self.K)
        x = torch.cat([pcd_up, interpolated], dim=1)
        return self.res_conv(x) if slow else cbl(self.res_conv, x)

    def interpolate(self, pcd_up, points_select, pcd_up_xyz, points_select_xyz, distance_type="feature", K=3):
        slow = differentiable(self, pcd_up, points_select, pcd_up_xyz, points_select_xyz)
        feat = self.conv(points_select) if slow else cbl(self.conv, points_select)
        if distance_type == "xyz" and K == 3 and not slow:
            return ops.interpolate3(pcd_up_xyz, points_select_xyz, feat)
        if distance_type == "feature":
            nbr, _, d = ops.select_neighbors_interpolate(pcd_up, points_select, feat, K=K)
        elif distance_type == "xyz":
            nbr, _, d = ops.select_neighbors_interpolate(pcd_up_xyz, points_select_xyz, feat, K=K)
        else:
            raise ValueError(f"upsample interpolation distance type can only be feature or xyz! Got: {distance_type}")
        w = 1.0 / (d + 1e-8)
        w = w / torch.sum(w, dim=-1, keepdim=True)
        return torch.sum(nbr * w.unsqueeze(dim=1), dim=-1)
