"""CPU oracle for the SAMBLE neighbourhood + sampling hot path.  TEST INFRASTRUCTURE ONLY.

Only tests/, __graft_entry__.smoke() and bench.py's cpu_baseline / --impl reference
legs may import this file.  The product (samble_b200/) never does: it fails loudly
when its CUDA library is missing.

What this is
------------
A functional (state_dict in, tensors out) fp32 restatement of the reference's
*algorithm* for the hot path, written against the same ATen primitives the
reference calls (torch.cdist / topk / gather / scatter_ / sort / softmax / conv),
so that on one machine it reproduces the reference bit for bit while sharing no
module structure with it.  Every function cites the reference lines it follows
(paths relative to the upstream repo root).

The arithmetic itself lives in a third-party dependency that is not under the
reference tree: PyTorch's ATen (reference README.md:29 pins pytorch==1.11.0; this
image has torch 2.11.0+cu128).  Parity is therefore anchored on the reference's
own call sites.

Pinning status
--------------
The reference ships NO tests, golden vectors or known-answer files (SURVEY 4), so
nothing upstream pins this oracle.  It is pinned instead against outputs of the
reference itself, run by tests/golden/make_golden.py (committed fixtures in
tests/golden/*.npz) and, when SAMBLE_REFERENCE names a checkout of the reference,
live in tests/test_oracle_vs_reference.py.
"""
from __future__ import annotations

import math
import numbers
from typing import Dict, List, Optional, Sequence, Tuple

import torch
import torch.nn.functional as F

Tensor = torch.Tensor
SD = Dict[str, Tensor]

# --------------------------------------------------------------------------
# L0 ops (utils/ops.py)
# --------------------------------------------------------------------------


class Forcing:
    """Teacher forcing for the parity tests (inactive unless installed with `forcing(...)`).

    The hot path contains two kinds of DISCRETE decisions -- neighbour sets (knn) and sampled
    point indices (DownSampleToken) -- whose fp32 near-ties no two implementations are obliged
    to break alike (SURVEY 7 hard part 1).  To compare everything downstream of such a decision
    within plain fp32 tolerance, the decision of the implementation under test is fed to the
    oracle: `knn_log` is a list of ((Nq, Nr, C, k), idx (B,Nq,k)[, dist (B,Nq,k)]) in call order (entries are
    consumed by signature), `ds_idx` a list with one (B,1,M) index tensor per DownSample layer.
    What the oracle itself would have decided is still computed and kept in `knn_seen`
    (raw inputs + its own indices) / the `record` dict, so the decisions are compared stage by
    stage on IDENTICAL inputs with the tie-aware comparators of samble_b200.testing."""

    def __init__(self, knn_log=None, ds_idx=None, keep_inputs: bool = True, lrelu_masks=None):
        self.knn_log = list(knn_log or [])
        self.ds_idx = list(ds_idx or [])
        self.keep_inputs = keep_inputs
        self.knn_seen: List[dict] = []
        self.lrelu_masks = None if lrelu_masks is None else list(lrelu_masks)     # (x > 0) per LeakyReLU call, call order
        self.lrelu_flips = 0                                                        # forced sides that differ from the oracle's own

    def take_lrelu(self, shape):
        for n, m in enumerate(self.lrelu_masks):
            if tuple(m.shape) == tuple(shape):
                return self.lrelu_masks.pop(n)
        return None

    def take_knn(self, sig):
        """-> (idx, dist or None) of the first unconsumed entry with this signature, or None.  An entry may carry the
        (positive) distances too: utils/ops.py:35's clamped GEMM-form distance of COINCIDENT points is pure fp32
        cancellation noise (0 or ~1e-3), and upsample.py:206 turns it into a weight 1/(d + 1e-8) -- a quantity no two
        fp32 implementations agree on, so it is forced like a decision and judged where it is computed."""
        for n, entry in enumerate(self.knn_log):
            if tuple(entry[0]) == tuple(sig):
                del self.knn_log[n]
                return entry[1], (entry[2] if len(entry) > 2 else None)
        return None


_FORCE: Optional[Forcing] = None


class forcing:
    """with forcing(Forcing(...)): ...   -- context manager installing the teacher-forcing state."""

    def __init__(self, f: Forcing):
        self.f = f

    def __enter__(self):
        global _FORCE
        self.prev, _FORCE = _FORCE, self.f
        return self.f

    def __exit__(self, *exc):
        global _FORCE
        _FORCE = self.prev


def knn(a: Tensor, b: Tensor, k: int) -> Tuple[Tensor, Tensor]:
    """utils/ops.py:17-44.  a (B,Nq,C), b (B,Nr,C) -> (-euclid (B,Nq,k), idx (B,Nq,k)).

    Both clouds are centred by a's per-channel mean over points and divided by ONE
    scalar per cloud: the mean over channels of a's per-channel unbiased std
    (:23-29).  Distances come from torch.cdist (:35) and the k largest of the
    negated matrix, sorted, are returned (:43).
    """
    mu = a.mean(dim=1, keepdim=True)
    a0, b0 = a - mu, b - mu
    sigma = a0.std(dim=1, keepdim=True).mean(dim=2, keepdim=True)
    neg = -torch.cdist(a0 / sigma, b0 / sigma)
    if _FORCE is None:
        return neg.topk(k=k, dim=-1)
    # teacher-forced (tests only): same distance matrix, the neighbour choice of the implementation under test
    own = neg.topk(k=k, dim=-1)
    sig = (a.shape[1], b.shape[1], a.shape[2], k)
    taken = _FORCE.take_knn(sig)
    forced, fdist = taken if taken is not None else (None, None)
    _FORCE.knn_seen.append(dict(sig=sig, idx=own[1], dist=own[0], forced=forced, a=a if _FORCE.keep_inputs else None,
                                b=b if _FORCE.keep_inputs else None))
    if forced is None:
        return own
    forced = forced.to(torch.int64)
    mine = neg.gather(2, forced)
    if fdist is None:
        return mine, forced
    # forced VALUES, own gradient (straight-through): under autograd (the f1 gradient tests) the distance keeps the
    # reference's graph through cdist and the normalisation; without autograd this is exactly -fdist
    return (mine + (-fdist - mine).detach() if mine.requires_grad else -fdist), forced


def index_points(points: Tensor, idx: Tensor) -> Tensor:
    """utils/ops.py:5-14.  points (B,N,C), idx (B,M,K) -> (B,M,K,C)."""
    B, C = points.shape[0], points.shape[-1]
    flat = idx.reshape(B, -1, 1).expand(-1, -1, C)
    return points.gather(1, flat).view(*idx.shape, C)


def select_neighbors(pcd: Tensor, K: int, neighbor_type: str, normal_channel: bool = False):
    """utils/ops.py:47-65.  pcd (B,C,N) -> ((B,C,N,K) permuted view, idx (B,N,K))."""
    pts = pcd.transpose(1, 2)
    key = pts[..., :3] if (normal_channel and pts.shape[-1] == 6) else pts
    _, idx = knn(key, key, K)
    nbr = index_points(pts, idx)
    if neighbor_type == "diff":
        nbr = nbr - pts.unsqueeze(2)
    elif neighbor_type != "neighbor":
        raise ValueError(f'neighbor_type should be "neighbor" or "diff", but got {neighbor_type}')
    return nbr.permute(0, 3, 1, 2), idx


def group(pcd: Tensor, K: int, group_type: str, normal_channel: bool = False):
    """utils/ops.py:83-112."""
    if group_type not in ("neighbor", "diff", "center_neighbor", "center_diff"):
        raise ValueError(
            f"group_type should be neighbor, diff, center_neighbor or center_diff, but got {group_type}")
    kind = "diff" if group_type.endswith("diff") else "neighbor"
    out, idx = select_neighbors(pcd, K, kind, normal_channel)
    if group_type.startswith("center"):
        out = torch.cat([pcd.unsqueeze(-1).repeat(1, 1, 1, K), out], dim=1)
    return out, idx


def neighbor_mask(pcd: Tensor, K: int) -> Tensor:
    """utils/ops.py:125-133.  dense 0/1 (B,N,N): row i marks the K nearest of point i."""
    pts = pcd.transpose(1, 2)
    _, idx = knn(pts, pts, K)
    B, N, _ = idx.shape
    return torch.zeros(B, N, N, dtype=torch.float32).scatter_(2, idx, 1.0)


def gather_by_idx(pcd: Tensor, idx: Tensor) -> Tensor:
    """utils/ops.py:136-145.  pcd (B,C,N), idx (B,1,M) -> (B,C,M)."""
    return pcd.gather(2, idx.expand(-1, pcd.shape[1], -1))


def select_neighbors_interpolate(unknown: Tensor, known: Tensor, known_feature: Tensor, K: int = 3):
    """utils/ops.py:68-80.  returns (nbr (B,C,N,K) view, idx (B,N,K), positive distance (B,N,K))."""
    neg, idx = knn(unknown.transpose(1, 2), known.transpose(1, 2), K)
    nbr = index_points(known_feature.transpose(1, 2), idx)
    return nbr.permute(0, 3, 1, 2), idx, -1 * neg


def update_sampling_score_bin_boundary(old, z: Tensor, num_bins: int, momentum: float,
                                       all_reduce=None):
    """utils/ops.py:174-236.  z is the (B,H,N,1) z-scored point score.

    Boundaries are the values found at ranks j/num_bins of ALL B*N scores sorted
    descending (:182-189), averaged over ranks when a process group exists
    (:191-199; `all_reduce` is a callable(t)->(t_sum, world) supplied by tests),
    then either blended into the previous pair with the EMA factor (:201-213) or
    used to create the [upper, lower] pair with +-inf sentinels (:214-233).
    """
    n = z.nelement()
    pos = (torch.arange(1, num_bins) / num_bins * n).int().long()
    ranked, _ = torch.sort(z.flatten(), dim=0, descending=True)
    cut = ranked[pos]
    if all_reduce is not None:
        total, world = all_reduce(cut)
        cut = total / world
    if old is not None:
        upper, lower = old[0].detach(), old[1].detach()
        cut = upper[0, 0, 0, 1:] * momentum + (1 - momentum) * cut
        upper[0, 0, 0, 1:] = cut
        lower[0, 0, 0, :-1] = cut
        return [upper, lower]
    upper = torch.cat([torch.tensor([float("inf")]), cut]).reshape(1, 1, 1, num_bins)
    lower = torch.cat([cut, torch.tensor([float("-inf")])]).reshape(1, 1, 1, num_bins)
    return [upper, lower]


def bin_partition(score: Tensor, boundaries, dynamic: bool, momentum: float, num_bins: int,
                  all_reduce=None):
    """utils/ops.py:435-464.  score (B,H,N) -> ([upper,lower], mask (B,H,N,nb) bool)."""
    B, H, N = score.shape
    z = (score - score.mean(dim=2, keepdim=True)) / score.std(dim=2, unbiased=False, keepdim=True)
    z = z.reshape(B, H, N, 1)
    if dynamic:
        boundaries = update_sampling_score_bin_boundary(boundaries, z, num_bins, momentum, all_reduce)
    mask = (z < boundaries[0]) & (z >= boundaries[1])
    return boundaries, mask


def calculate_num_points_to_choose(bin_prob: Tensor, max_num_points: Tensor, total: int) -> Tensor:
    """utils/ops.py:385-432.  water-filling of `total` points over bins, capped by bin size.

    p = w*cnt + 1e-10 (:396-397); up to nb rounds of {normalise p; spread what is
    left proportionally; clamp to the bin size; zero p of saturated bins}
    (:403-422) with a batch-wide early exit (:409); truncate to int (:424); give
    the remainder to the bin with the most room, first index on ties (:427-430).
    """
    B, nb = bin_prob.shape
    p = bin_prob * max_num_points
    p = p + 1e-10
    chosen = torch.zeros_like(p)
    for _ in range(nb):
        p = p / p.sum(dim=1, keepdim=True)
        left = total - chosen.sum(dim=1, keepdim=True)
        if bool((left == 0).all()):
            break
        chosen = chosen + p * left
        full = chosen >= max_num_points
        chosen = torch.where(full, max_num_points, chosen)
        p = p * torch.where(full, 0, 1)
    k = chosen.int()
    rows = torch.arange(B)
    k[rows, torch.argmax(max_num_points - k, dim=1)] += total - k.sum(dim=1)
    return k


def sampling_probabilities(score: Tensor, mask: Tensor, mode: str, boltzmann_t) -> Tensor:
    """utils/ops.py:507-592: per-(cloud, bin) categorical distribution over the N points, (B*nb, N).
    'uniform': the bin's membership mask (an empty bin -> all ones, :511-513).
    'random' : z-score -> tanh -> exp(score * 1/T) restricted to the bin and normalised; NaN -> 1e-8 (:515-590)."""
    B, _, N, nb = mask.shape
    if mode == "uniform":
        p = mask.float().squeeze(dim=1)
        p = p + (torch.sum(p, dim=1, keepdim=True) == 0)
    elif mode == "random":
        z = (score - torch.mean(score, dim=2, keepdim=True)) / torch.std(score, dim=2, unbiased=False, keepdim=True)
        z = torch.tanh(z)
        if boltzmann_t in ("mode_1", "mode_3"):
            inv_t = torch.sum(mask, dim=2, keepdim=True).float() / (100.0 if boltzmann_t == "mode_1" else 200.0)
        elif boltzmann_t == "mode_2":
            inv_t = N / (100.0 * nb)
        elif boltzmann_t == "mode_4":
            inv_t = N / (200.0 * nb)
        elif isinstance(boltzmann_t, numbers.Number):
            inv_t = 1 / boltzmann_t
        else:
            raise NotImplementedError
        p = torch.exp(z.unsqueeze(3) * inv_t) * mask
        p = p / torch.sum(p, dim=2, keepdim=True)
        p = p.squeeze(dim=1)
        p[torch.isnan(p)] = 1e-8
    else:
        raise ValueError("Please check the setting of bin sample mode. It must be topk, multinomial or random!")
    return p.permute(0, 2, 1).reshape(-1, N)


def generating_downsampled_index(M: int, score: Tensor, mask: Tensor, mode: str, boltzmann_t,
                                 k: Tensor, generator=None) -> Tensor:
    """utils/ops.py:467-619.  Returns (B,1,M) int64: bins in order; within a bin `topk` takes descending
    score+1e-8 (:476-505), `uniform`/`random` take the first k of M draws without replacement from
    sampling_probabilities (:594-612; torch.multinomial, so bit-equal to the reference only under the same
    CPU RNG state -- tests/test_oracle_vs_reference.py seeds both)."""
    B, _, N, nb = mask.shape
    if mode == "topk":
        masked = (score + 1e-8).unsqueeze(3) * mask
        order = torch.sort(masked, dim=2, descending=True)[1].squeeze(1)      # (B,N,nb)
        rows = [torch.cat([order[b, : int(k[b, j]), j] for j in range(nb)]) for b in range(B)]
        return torch.stack(rows).reshape(B, 1, M)
    p = sampling_probabilities(score, mask, mode, boltzmann_t)
    draws = torch.multinomial(p, M, generator=generator).reshape(B, nb, M)
    rows = [torch.cat([draws[b, j, : int(k[b, j])] for j in range(nb)]) for b in range(B)]
    return torch.stack(rows).reshape(B, 1, M)


# --------------------------------------------------------------------------
# L1 blocks (models/*.py), functional over a state_dict
# --------------------------------------------------------------------------


def _conv(sd: SD, name: str, x: Tensor) -> Tensor:
    """1x1 Conv1d/Conv2d without bias == the stored weight applied as a conv."""
    w = sd[name + ".weight"]
    return F.conv2d(x, w) if w.dim() == 4 else F.conv1d(x, w)


_BN_TRAINING = False


class bn_training:
    """with bn_training(True): BatchNorm normalises with the batch statistics (nn.BatchNorm in train mode, as under
    train_shapenet.py:398; running statistics are not updated here).  Default: eval mode."""

    def __init__(self, on: bool):
        self.on = bool(on)

    def __enter__(self):
        global _BN_TRAINING
        self.prev, _BN_TRAINING = _BN_TRAINING, self.on

    def __exit__(self, *exc):
        global _BN_TRAINING
        _BN_TRAINING = self.prev


def _bn(sd: SD, name: str, x: Tensor) -> Tensor:
    """BatchNorm: eval mode (running statistics) unless inside `bn_training(True)`."""
    if _BN_TRAINING:
        return F.batch_norm(x, None, None, sd[name + ".weight"], sd[name + ".bias"], True, 0.0, 1e-5)
    return F.batch_norm(x, sd[name + ".running_mean"], sd[name + ".running_var"],
                        sd[name + ".weight"], sd[name + ".bias"], False, 0.0, 1e-5)


def _lrelu(x: Tensor) -> Tensor:
    """LeakyReLU(0.2).  Under teacher forcing with recorded activation masks (gradient tests only) the side of the kink
    is the one the implementation under test took: a pre-activation within fp32 rounding of zero changes the output by
    ~1e-7 but the derivative by 0.8, i.e. it is one more discrete decision."""
    if _FORCE is not None and _FORCE.lrelu_masks is not None:
        m = _FORCE.take_lrelu(tuple(x.shape))
        if m is not None:
            _FORCE.lrelu_flips += int((m != (x > 0)).sum())
            return torch.where(m, x, x * 0.2)
    return F.leaky_relu(x, 0.2)


def _cbl(sd: SD, name: str, x: Tensor) -> Tensor:
    """nn.Sequential(conv, bn, LeakyReLU(0.2)) as used all over the reference."""
    return _lrelu(_bn(sd, name + ".1", _conv(sd, name + ".0", x)))


def edgeconv(sd: SD, pre: str, x: Tensor, K: int, group_type: str = "center_diff") -> Tensor:
    """models/embedding.py:29-39."""
    g, _ = group(x, K, group_type)
    return _cbl(sd, pre + "conv2", _cbl(sd, pre + "conv1", g)).max(dim=-1)[0]


def n2p_attention(sd: SD, pre: str, x: Tensor, K: int, heads: int = 4) -> Tensor:
    """models/attention.py:165-250, scalar_dot / asm 'dot' (the shipped setting)."""
    B, C, N = x.shape
    nb, _ = group(x, K, "diff")                                    # (B,C,N,K)
    D = C // heads

    def split(t):                                                  # (B,C,N,k)->(B,H,N,k,D)
        return t.view(B, heads, D, N, t.shape[-1]).permute(0, 1, 3, 4, 2)

    q = split(_conv(sd, pre + "q_conv", x.unsqueeze(-1)))          # (B,H,N,1,D)
    k = split(_conv(sd, pre + "k_conv", nb))                       # (B,H,N,K,D)
    v = split(_conv(sd, pre + "v_conv", nb))
    att = torch.softmax(q @ k.transpose(-1, -2) / math.sqrt(D), dim=-1)   # (B,H,N,1,K)
    y = (att @ v)[:, :, :, 0, :].permute(0, 2, 1, 3).reshape(B, N, C).permute(0, 2, 1)
    x = _bn(sd, pre + "bn1", x + y)
    ff = _conv(sd, pre + "ff.2", _lrelu(_conv(sd, pre + "ff.0", x)))
    return _bn(sd, pre + "bn2", x + ff)


class DSState:
    """Per-layer mutable state of DownSampleToken that lives outside the state_dict
    (bin boundaries; models/downsample.py:91-103, train_shapenet.py:666-672)."""

    def __init__(self, dynamic: bool = True, boundaries=None, momentum: float = 0.99):
        self.dynamic = dynamic
        self.boundaries = boundaries
        self.momentum = momentum


def downsample_token(sd: SD, pre: str, x: Tensor, M: int, K: int, num_bins: int, state: DSState,
                     sample_mode: str = "topk", all_reduce=None, force_idx: Optional[Tensor] = None) -> Dict[str, Tensor]:
    """models/downsample.py:112-262 with asm='dot', idx_mode='sparse_col_sqr',
    relu_mean_order='mean_relu', multi_token, one head, res off (shipped configs)."""
    B, C, N = x.shape
    tokens = sd[pre + "bin_tokens"].expand(B, -1, -1)
    xt = torch.cat([x, tokens], dim=2)                                       # :116-118
    q = _conv(sd, pre + "q_conv", x).unsqueeze(1).transpose(2, 3)            # (B,1,N,D)
    k = _conv(sd, pre + "k_conv", xt).unsqueeze(1)                           # (B,1,D,N+nb)
    v = _conv(sd, pre + "v_conv", xt).unsqueeze(1)
    logits = (q @ k) / math.sqrt(q.shape[-1])                                # :139-143
    amap = torch.softmax(logits, dim=-1)                                     # :145
    token_logits = logits[..., N:]                                           # :149 (pre-softmax)
    a_pts = amap[..., :N]
    # sparse column score (:300-344)
    m = neighbor_mask(x, K).unsqueeze(1)
    indeg = m.sum(dim=-2) + 1e-8
    score = (a_pts * m).sum(dim=-2) / indeg / indeg
    score[torch.isnan(score)] = 0
    # bins (:205-227)
    state.boundaries, mask = bin_partition(score, state.boundaries, state.dynamic, state.momentum,
                                           num_bins, all_reduce)
    w_raw = ((token_logits * mask).sum(dim=2) / (torch.count_nonzero(mask, dim=2) + 1e-8)).squeeze(1)
    counts = mask.squeeze(1).sum(dim=1)
    kpb = calculate_num_points_to_choose(F.relu(w_raw), counts, M)
    idx = own_idx = generating_downsampled_index(M, score, mask, sample_mode, None, kpb)
    if force_idx is not None:            # teacher-forced (tests only): gather the rows the implementation under test chose
        idx = force_idx.to(torch.int64).reshape(B, 1, M)
    a_down = amap.gather(2, idx.unsqueeze(3).expand(-1, -1, -1, amap.shape[-1]))   # :242-246
    x_ds = (a_down @ v.transpose(2, 3)).permute(0, 2, 1, 3).reshape(B, M, C).permute(0, 2, 1)
    return dict(x_ds=x_ds, idx=idx, own_idx=own_idx, score=score, mask=mask, k=kpb, bin_weights_beforerelu=w_raw,
                token_logits=token_logits, boundaries=state.boundaries, x_in=x)


def upsample_interpolation(sd: SD, pre: str, pcd_up: Tensor, selected: Tensor, xyz_up: Tensor,
                           xyz_sel: Tensor, K: int = 3) -> Tensor:
    """models/upsample.py:162-213 with distance_type='xyz'."""
    feat = _cbl(sd, pre + "conv", selected)
    nbr, _, d = select_neighbors_interpolate(xyz_up, xyz_sel, feat, K)
    w = 1.0 / (d + 1e-8)
    w = w / w.sum(dim=-1, keepdim=True)
    interp = (nbr * w.unsqueeze(1)).sum(dim=-1)
    return _cbl(sd, pre + "res_conv", torch.cat([pcd_up, interp], dim=1))


def stn(sd: SD, pre: str, x0: Tensor) -> Tensor:
    """models/embedding.py:78-97 (eval: dropout is identity).  Out of hot-path scope;
    restated only because the seg forward cannot run without it."""
    B = x0.shape[0]
    x = _cbl(sd, pre + "conv2", _cbl(sd, pre + "conv1", x0)).max(dim=-1)[0]
    x = _cbl(sd, pre + "conv3", x).max(dim=-1)[0]
    for name in ("linear1", "linear2"):
        x = _lrelu(_bn(sd, f"{pre}{name}.1", F.linear(x, sd[f"{pre}{name}.0.weight"])))
    return F.linear(x, sd[pre + "transform.weight"], sd[pre + "transform.bias"]).view(B, 3, 3)


# --------------------------------------------------------------------------
# L2 wiring (models/seg_model.py, models/cls_model.py)
# --------------------------------------------------------------------------


def _block_down(sd: SD, cfg, x: Tensor, states: Sequence[DSState], record: Optional[dict]):
    """shared front half: EdgeConv x2 -> N2P -> (DownSample -> N2P)*L.
    seg_model.py:96-117 / cls_model.py:102-136."""
    ds, emb, att = cfg.downsample, cfg.embedding, cfg.attention
    xyz = x[:, :3, :]
    feats = []
    for l in range(len(emb.K)):
        x = edgeconv(sd, f"block.embedding_list.{l}.", x, emb.K[l], emb.group_type[l])
        feats.append(x)
    x = n2p_attention(sd, "block.feature_learning_layer_list.0.", torch.cat(feats, dim=1),
                      att.K[0], att.num_heads[0])
    xs, xyzs, idxs = [x], [xyz], []
    for i in range(len(ds.M)):
        out = downsample_token(sd, f"block.downsample_list.{i}.", x, ds.M[i], ds.K,
                               ds.bin.num_bins[i], states[i], ds.bin.sample_mode[i],
                               force_idx=(_FORCE.ds_idx[i] if _FORCE is not None and i < len(_FORCE.ds_idx) else None))
        if record is not None:
            record[f"ds{i}"] = out
        x = n2p_attention(sd, f"block.feature_learning_layer_list.{i + 1}.", out["x_ds"],
                          att.K[i + 1], att.num_heads[i + 1])
        xyz = gather_by_idx(xyz, out["idx"])
        xs.append(x), xyzs.append(xyz), idxs.append(out["idx"])
    return xs, xyzs, idxs


def seg_forward(sd: SD, config, x: Tensor, category_id: Tensor, states: Sequence[DSState],
                record: Optional[dict] = None) -> Tensor:
    """models/seg_model.py:176-224 (+ FeatureLearningBlock.forward :96-133).
    x (B,3,N), category_id (B,16,1) -> logits (B,50,N)."""
    cfg = config.feature_learning_block
    B, _, N = x.shape
    if cfg.STN:
        x0, _ = group(x, 32, "center_diff")
        x = torch.bmm(x.transpose(2, 1), stn(sd, "STN.", x0)).transpose(2, 1)
    xs, xyzs, _ = _block_down(sd, cfg, x, states, record)
    att = cfg.attention
    L = len(cfg.downsample.M)
    split = (len(att.K) - 1) // 2
    cur, cur_xyz = xs.pop(), xyzs.pop()
    for j in range(L):
        skip = xs.pop()
        up_xyz = xyzs[len(xyzs) - 1 - j]
        cur = upsample_interpolation(sd, f"block.upsample_list.{j}.", skip, cur, up_xyz, cur_xyz,
                                     cfg.upsample.interpolation.K[j])
        cur = n2p_attention(sd, f"block.feature_learning_layer_list.{j + 1 + split}.", cur,
                            att.K[j + 1 + split], att.num_heads[j + 1 + split])
        cur_xyz = up_xyz
    f = cur
    g = _cbl(sd, "conv", f)
    g = torch.cat([g.max(dim=-1, keepdim=True)[0], g.mean(dim=-1, keepdim=True),
                   _cbl(sd, "conv1", category_id)], dim=1).repeat(1, 1, N)
    y = _cbl(sd, "conv3", _cbl(sd, "conv2", torch.cat([g, f], dim=1)))
    return F.conv1d(y, sd["conv4.weight"])


def cls_forward(sd: SD, config, x: Tensor, states: Sequence[DSState],
                record: Optional[dict] = None) -> Tensor:
    """models/cls_model.py:102-139,185-205 with res_link on (cls.yaml:98-99). -> (B,40)."""
    cfg = config.feature_learning_block
    xs, _, _ = _block_down(sd, cfg, x, states, record)
    pooled = [F.conv1d(t, sd[f"block.conv_list.{i}.weight"]).max(dim=-1)[0] for i, t in enumerate(xs)]
    y = torch.cat(pooled, dim=1)
    for name in ("linear1", "linear2"):
        y = F.linear(y, sd[f"{name}.0.weight"], sd[f"{name}.0.bias"])
        y = _lrelu(_bn(sd, f"{name}.1", y))
    return F.linear(y, sd["linear3.weight"], sd["linear3.bias"])
