"""Shared test/bench helpers: synthetic clouds, deterministic weights, tie-aware comparators.

Nothing at module level touches the oracle or the reference; it only produces inputs and
compares outputs, so both the product tests and the golden-vector generator use it.  The two
DownSampleToken judges at the end (amp_excusing_knn_ties, judge_against_reference_scores) import
the oracle and the native ops when called: they serve the GPU tests only.
"""
from __future__ import annotations

import math
import zlib
from typing import Dict, Tuple

import numpy as np
import torch

Tensor = torch.Tensor


def synthetic_clouds(B: int, N: int, seed: int = 0) -> Tuple[Tensor, Tensor]:
    """ShapeNetPart-shaped input (SURVEY 8d): xyz ~ U(-1,1)^3 as (B,3,N) fp32 and a
    one-hot category (B,16,1) with class b mod 16.  CPU tensors."""
    g = torch.Generator().manual_seed(seed)
    xyz = torch.rand(B, 3, N, generator=g, dtype=torch.float32) * 2 - 1
    cat = torch.zeros(B, 16, 1)
    cat[torch.arange(B), torch.arange(B) % 16, 0] = 1.0
    return xyz, cat


def synthetic_features(B: int, C: int, N: int, seed: int = 0) -> Tensor:
    """x ~ N(0,1) (B,C,N): the micro-bench / parity input for feature-space kernels."""
    g = torch.Generator().manual_seed(seed)
    return torch.randn(B, C, N, generator=g, dtype=torch.float32)


def fill_state_dict_(sd: Dict[str, Tensor], seed: int = 0, sharpen: float = 1.0) -> Dict[str, Tensor]:
    """Overwrite every entry of a state_dict in place with values that depend only on
    (seed, entry name, shape), so two differently-constructed models (the reference's
    nn.Modules here, ours on the GPU box) hold identical weights without shipping them.

    weights ~ N(0, 1/fan_in) (x `sharpen` for the DownSample q/k projections: SURVEY 8d's
    "sharpened" variant), BN weight ~ U(0.5,1.5), BN bias/running_mean ~ N(0,0.1),
    running_var ~ U(0.5,1.5), so eval-mode BN is not the identity."""
    for name, t in sd.items():
        g = torch.Generator().manual_seed((zlib.crc32(name.encode()) ^ (seed * 0x9E3779B1)) & 0x7FFFFFFF)
        if name.endswith("num_batches_tracked"):
            t.fill_(1)
            continue
        if name.endswith("running_var"):
            v = torch.rand(t.shape, generator=g) + 0.5
        elif name.endswith("running_mean"):
            v = torch.randn(t.shape, generator=g) * 0.1
        elif t.dim() == 1 and name.endswith("weight"):          # BN scale
            v = torch.rand(t.shape, generator=g) + 0.5
        elif t.dim() == 1:                                       # biases
            v = torch.randn(t.shape, generator=g) * 0.1
        elif name.endswith("bin_tokens"):
            v = torch.randn(t.shape, generator=g) / (t.shape[1] ** 0.5)
        else:
            fan_in = t[0].numel()
            v = torch.randn(t.shape, generator=g) / (fan_in ** 0.5)
            if sharpen != 1.0 and "downsample_list" in name and (".q_conv." in name or ".k_conv." in name):
                v = v * sharpen
        if name.endswith("transform.weight"):
            v = v * 0.05          # keep the STN near identity like its zero-init (embedding.py:73-74)
        if name.endswith("transform.bias"):
            v = torch.eye(3).reshape(-1) + v * 0.05
        t.copy_(v.to(t.dtype))
    return sd


# --------------------------------------------------------------------------
# comparators (SURVEY 8c protocol step 5)
# --------------------------------------------------------------------------


def knn_parity(idx: Tensor, ref_idx: Tensor, a: Tensor, b: Tensor, rel_band: float = 2e-5, cancel_ulps: float = 8.0) -> dict:
    """Tie-aware kNN comparison.  a (B,Nq,C), b (B,Nr,C) are the RAW inputs.

    Exact position-wise match rate is reported; every mismatching row must agree as
    a SET except for members whose fp64 squared distance (raw units; the reference's
    normalisation is a per-cloud similarity transform, so order is unaffected) lies
    within `rel_band` (relative) of that row's k-th distance -- i.e. the swap is an
    fp32 near-tie that no two fp32 implementations are obliged to order alike.
    """
    idx, ref_idx = idx.cpu().long(), ref_idx.cpu().long()
    B, Nq, k = ref_idx.shape
    exact = (idx == ref_idx)
    bad_rows = (~exact.all(dim=-1)).nonzero()
    a64, b64 = a.double().cpu(), b.double().cpu()
    mu = a64.mean(dim=1, keepdim=True)                              # the reference centres both clouds on a's mean (ops.py:23-29)
    na, nb_ = ((a64 - mu) ** 2).sum(-1), ((b64 - mu) ** 2).sum(-1)   # |a'|^2, |b'|^2 up to the common scale
    unexplained = 0
    for bi, qi in bad_rows.tolist():
        d = ((b64[bi] - a64[bi, qi]) ** 2).sum(-1)                  # (Nr,)
        mine, ref = idx[bi, qi], ref_idx[bi, qi]
        if len(set(mine.tolist())) != k:
            unexplained += 1
            continue
        kth = torch.sort(d)[0][k - 1]
        # two sources of fp32 indecision: a relative near-tie, and the cancellation of the reference's own distance
        # formula |a|^2 + |b|^2 - 2ab (ops.py:35, torch.cdist's GEMM form): a few roundings of |a'|^2 + |b'|^2
        band = max(rel_band * max(float(kth), 1e-30), cancel_ulps * 2.0 ** -24 * float(na[bi, qi] + nb_[bi].max()))
        # every element either side must be no worse than the k-th distance + band,
        # and the sequence must be sorted up to the band
        ok = bool((d[mine] <= kth + band).all()) and bool((d[ref] <= kth + band).all())
        dm = d[mine]
        ok = ok and bool((dm[1:] - dm[:-1] >= -band).all())
        unexplained += 0 if ok else 1
    return dict(exact_rate=float(exact.float().mean()), rows=B * Nq, mismatch_rows=len(bad_rows),
                unexplained_rows=unexplained)


def sampled_index_parity(idx: Tensor, ref_idx: Tensor, score: Tensor, k_per_bin: Tensor) -> dict:
    """Tie-aware sampler comparison.  idx/ref_idx (B,1,M) int64, score (B,1,N) is the
    REFERENCE score, k_per_bin (B,nb).  Indices must be equal except inside groups of
    exactly equal reference score (sort order among equals is implementation-defined)."""
    idx, ref_idx, score = idx.cpu(), ref_idx.cpu(), score.cpu()
    B, _, M = ref_idx.shape
    exact = idx == ref_idx
    unexplained = 0
    for b in range(B):
        if bool(exact[b].all()):
            continue
        s = score[b, 0]
        off = 0
        for kb in k_per_bin[b].tolist():
            seg_m, seg_r = idx[b, 0, off:off + kb], ref_idx[b, 0, off:off + kb]
            off += kb
            if torch.equal(seg_m, seg_r):
                continue
            # same multiset of scores in the same order == only ties were permuted
            if not torch.equal(s[seg_m], s[seg_r]) or len(set(seg_m.tolist())) != kb:
                unexplained += 1
    return dict(exact_rate=float(exact.float().mean()), clouds=B, unexplained_bins=unexplained)


def ds_scores_fp64(x: Tensor, wq: Tensor, wk: Tensor, tokens: Tensor, knn_idx: Tensor) -> Tuple[Tensor, Tensor]:
    """fp64 statement of DownSampleToken's point score (models/downsample.py:124-153, 300-344) for the GIVEN
    neighbour sets: x (B,C,N), wq/wk (D,C), tokens (C,nb), knn_idx (B,N,K) -> (score (B,N), amp (B,N)).
    `amp[j]` = the largest sum_c |q_ic k_jc| / sqrt(D) over the edges i->j that enter score[j] and over the dominant
    logit of those rows: the condition number that turns a relative fp32 dot-product error into a relative error of
    score[j] (the softmax exponentiates the logit error)."""
    B, C, N = x.shape
    D = wq.shape[0]
    wq, wk, tok = wq.double().cpu(), wk.double().cpu(), tokens.double().cpu()
    scores, amps = [], []
    for b in range(B):
        xb = x[b].double().cpu()                                   # (C,N)
        q = (wq @ xb).t()                                          # (N,D)
        kk = (wk @ torch.cat([xb, tok], dim=1)).t()                # (N+nb,D)
        logits = q @ kk.t() / (D ** 0.5)
        amap = torch.softmax(logits, dim=-1)[:, :N]
        idx = knn_idx[b].long().cpu()
        mask = torch.zeros(N, N, dtype=torch.float64).scatter_(1, idx, 1.0)
        indeg = mask.sum(0) + 1e-8
        s = (amap * mask).sum(0) / indeg / indeg
        s[torch.isnan(s)] = 0
        scores.append(s)
        mag = (q.abs() @ kk.abs().t()) / (D ** 0.5)                # sum_c |q_ic k_jc| / sqrt(D)
        row_dom = mag.gather(1, logits.argmax(dim=1, keepdim=True))[:, 0]          # magnitude at each row's largest logit
        edge = torch.maximum(mag[:, :N], row_dom[:, None]) * mask
        amps.append(edge.max(dim=0)[0])
    return torch.stack(scores), torch.stack(amps)


def ds_parity(score64: Tensor, amp: Tensor, cuts: Tensor, idx: Tensor, bin_mask: Tensor, k_per_bin: Tensor,
              ulps: float = 64.0) -> dict:
    """fp64 adjudication of one DownSampleToken decision (the twin of knn_parity).

    score64/amp from ds_scores_fp64; cuts (nb-1,) the frozen z-score thresholds (descending); idx (B,1,M), bin_mask
    (B,1,N,nb) bool, k_per_bin (B,nb): the decision under test.  Any fp32 evaluation of the score carries a relative
    error of about  eps_j = ulps * 2^-24 * amp_j  (dot-product rounding exponentiated by the softmax), so
      * a point may sit in another bin than its fp64 z-score says only if that z is within eps_j*score_j/std of a cut;
      * inside a bin, a chosen point may score below an unchosen one only if both are within eps of the bin's k-th score.
    Everything else is counted as unexplained (must be 0)."""
    score64, amp, idx = score64.double().cpu(), amp.double().cpu(), idx.cpu().long()
    bin_mask, k_per_bin, cuts = bin_mask.cpu(), k_per_bin.cpu().long(), cuts.double().cpu().reshape(-1)
    B, N = score64.shape
    nb = bin_mask.shape[-1]
    eps = ulps * 2.0 ** -24 * amp.clamp_min(1.0)                                     # (B,N) relative score tolerance
    mu, sd = score64.mean(1, keepdim=True), score64.std(1, unbiased=False, keepdim=True)
    z = (score64 - mu) / sd
    upper = torch.cat([torch.tensor([float("inf")], dtype=torch.float64), cuts])
    lower = torch.cat([cuts, torch.tensor([float("-inf")], dtype=torch.float64)])
    bin64 = ((z.unsqueeze(-1) < upper) & (z.unsqueeze(-1) >= lower)).double().argmax(-1)     # (B,N)
    mine = bin_mask[:, 0]
    assert bool((mine.sum(-1) == 1).all()), "every point must sit in exactly one bin"
    my_bin = mine.double().argmax(-1)
    # + the fp32 evaluation of z itself: (s - mean) / std with mean, std and the difference each rounded to fp32
    zband = eps * score64.abs() / sd + 32 * 2.0 ** -24 * (mu.abs() / sd + z.abs() + 1.0)
    d_cut = (z.unsqueeze(-1) - cuts).abs().min(-1)[0] if cuts.numel() else torch.full_like(z, float("inf"))
    flips = my_bin != bin64
    bad_flips = flips & (d_cut > zband)
    # points the reference's fp32 z-score cannot tell apart (equal scores -- e.g. 0 for every point no neighbourhood
    # contains -- or scores far below mean/std's resolution) sit at ONE fp32 z and flip together
    s32 = score64.float()
    z32 = (s32 - s32.mean(1, keepdim=True)) / s32.std(1, unbiased=False, keepdim=True)
    flip_groups = max([len(set(z32[b][flips[b]].tolist())) for b in range(B)] + [0])
    swaps = bad_swaps = wrong_bin = dup = 0
    for b in range(B):
        off = 0
        for j in range(nb):
            kj = int(k_per_bin[b, j])
            seg = idx[b, 0, off:off + kj]
            off += kj
            members = (my_bin[b] == j).nonzero()[:, 0]
            if kj == 0:
                continue
            if len(set(seg.tolist())) != kj:
                dup += 1
            if not bool(mine[b, seg, j].all()):
                wrong_bin += int((~mine[b, seg, j]).sum())      # (k > bin size: the reference then takes non-members too)
                continue
            # the sampler orders by key = fl32(score + 1e-8) (utils/ops.py:478): two keys closer than one fp32 rounding
            # of the key are a tie (every score below ~6e-16 collapses onto 1e-8), on top of the score's own tolerance
            s = score64[b, members]
            key = s + 1e-8
            order = torch.sort(key, descending=True)[0]
            kth = float(order[min(kj, len(order)) - 1])
            chosen = torch.zeros(N, dtype=torch.bool)
            chosen[seg] = True
            ch = chosen[members]
            tol = eps[b, members] * s.abs() + 2.0 ** -23 * key
            low = ch & (key < kth)                   # chosen although below the fp64 k-th key
            high = (~ch) & (key > kth)               # passed over although above it
            swaps += int(low.sum()) + int(high.sum())
            bad_swaps += int((low & (key < kth - tol - 2.0 ** -23 * kth)).sum()) + int((high & (key > kth + tol + 2.0 ** -23 * kth)).sum())
    return dict(points=B * N, bin_flips=int(flips.sum()), distinct_flipped_z_per_cloud=flip_groups,
                unexplained_bin_flips=int(bad_flips.sum()), topk_swaps=swaps,
                unexplained_topk_swaps=bad_swaps, chosen_outside_bin=wrong_bin, duplicate_rows=dup,
                max_eps=float(eps.max()), median_eps=float(eps.median()))


def amp_excusing_knn_ties(x: Tensor, sd: Dict[str, Tensor], pre: str, cheap: bool = False):
    """(fp64 scores, amplification, touched columns) of one DownSampleToken layer for ds_parity.  Columns whose in-edge
    set differs between the native kNN and the oracle's (an fp32 near-tie of two distances, adjudicated by the kNN tests)
    get an unbounded tolerance: one neighbour more or less changes such a score by ~3 % (score = colsum / indeg^2), which
    says nothing about the scoring kernels.  Runs the native kNN on cuda:0 and the oracle's on the CPU."""
    from oracle import samble_oracle as O
    from samble_b200 import ops

    C = x.shape[1]
    mine = ops.knn_indices(x.to("cuda:0"), 32).cpu().long()
    _, theirs = O.knn(x.transpose(1, 2), x.transpose(1, 2), 32)
    if cheap:             # large clouds: skip the fp64 N x N pass, take a typical amplification for sharpened logits
        s64, amp = None, torch.full((x.shape[0], x.shape[2]), 100.0, dtype=torch.float64)
    else:
        s64, amp = ds_scores_fp64(x, sd[pre + "q_conv.weight"].view(C, C), sd[pre + "k_conv.weight"].view(C, C), sd[pre + "bin_tokens"][0], mine)
    B, N = amp.shape
    a = torch.zeros(B, N, N, dtype=torch.bool).scatter_(2, mine, True)
    b = torch.zeros(B, N, N, dtype=torch.bool).scatter_(2, theirs, True)
    touched = (a != b).any(dim=1)                                   # (B,N) columns
    return s64, torch.where(touched, torch.full_like(amp, 1e15), amp), touched


def judge_against_reference_scores(ds, idx: Tensor, x_ds: Tensor, ref_score: Tensor, ref_idx: Tensor, ref_k: Tensor,
                                   ref_x_ds: Tensor, amp: Tensor, max_flip_groups=8) -> dict:
    """One DownSampleToken decision against the REFERENCE's own fp32 scores of the same input (golden file or oracle):
    every bin membership and every per-bin choice must be the one those scores dictate, except where they cannot
    decide: a z-score within fp32 rounding of a cut (a freshly calibrated cut IS some point's z), keys closer than one
    rounding of score + 1e-8, or scores closer than the reference's OWN fp32 error (16 roundings x the softmax's
    amplification `amp`, ds_scores_fp64; measured 1e-5 for the reference, 3e-6 for the native kernels).
    Rows of x_ds are compared wherever the same point was chosen, unconditionally.  `max_flip_groups` bounds the distinct
    fp32 z-scores among the (explained) bin flips of a cloud; None leaves every flip to the band alone.  Returns the
    ds_parity report."""
    cuts = ds.bin_boundaries[0].reshape(-1)[1:].cpu()
    rep = ds_parity(ref_score[:, 0].double(), amp, cuts, idx, ds.bin_points_mask, ds.k_point_to_choose, ulps=16.0)
    print(rep)
    assert rep["unexplained_bin_flips"] == 0 and rep["unexplained_topk_swaps"] == 0, rep
    assert rep["chosen_outside_bin"] == 0 and rep["duplicate_rows"] == 0, rep
    if max_flip_groups is not None:     # only points (nearly) tied with a cut flip -- as whole tie groups
        assert rep["distinct_flipped_z_per_cloud"] <= max_flip_groups, rep
    k_mine = ds.k_point_to_choose.cpu().long()
    assert int((k_mine - ref_k.long()).abs().max()) <= 1 and bool((k_mine.sum(1) == idx.shape[-1]).all())
    same = idx.cpu() == ref_idx                              # (B,1,M)
    key = ref_score + 1e-8                                   # the reference's fp32 sort key: equal keys are ordered arbitrarily
    tie = key.gather(2, idx.cpu()) == key.gather(2, ref_idx)
    assert float((same | tie).float().mean()) >= 0.98, float((same | tie).float().mean())
    ok = ((x_ds.cpu().double() - ref_x_ds.double()).abs() <= 2e-4 + 2e-4 * ref_x_ds.double().abs())       # (B,C,M)
    assert bool(ok[same.expand_as(ok)].all()), "x_ds rows of identically chosen points differ"
    return rep


def n2p_attend_literal(qkv: Tensor, idx: Tensor, heads: int) -> Tensor:
    """The reference's Neighbor2Point attention core in its own gathered-difference form (models/attention.py:165-185,
    207-250): k_ij = k_j - k_i, v_ij = v_j - v_i, out_i = sum_j softmax_j(q_i . k_ij / sqrt(d)) v_ij per head, on the
    hoisted projections qkv (B,N,3C) = [q|k|v] and idx (B,N,K).  Runs in qkv's dtype and device and is differentiable, so
    fp64 autograd of it is the gradient reference of ops.n2p_attend."""
    B, N, C3 = qkv.shape
    C, K = C3 // 3, idx.shape[-1]
    D = C // heads
    q, k, v = qkv[..., :C], qkv[..., C:2 * C], qkv[..., 2 * C:]
    flat = idx.long().reshape(B, -1, 1).expand(-1, -1, C)
    kd = (torch.gather(k, 1, flat).view(B, N, K, C) - k[:, :, None, :]).view(B, N, K, heads, D)
    vd = (torch.gather(v, 1, flat).view(B, N, K, C) - v[:, :, None, :]).view(B, N, K, heads, D)
    att = torch.softmax(torch.einsum("bnhd,bnkhd->bnhk", q.reshape(B, N, heads, D), kd) / math.sqrt(D), dim=-1)
    return torch.einsum("bnhk,bnkhd->bnhd", att, vd).reshape(B, N, C)


def max_abs_rel(x: Tensor, ref: Tensor) -> Tuple[float, float]:
    x, ref = x.detach().double().cpu(), ref.detach().double().cpu()
    err = (x - ref).abs()
    return float(err.max()), float((err / (ref.abs() + 1e-6)).max())


def to_numpy_tree(d: dict) -> Dict[str, np.ndarray]:
    return {k: (v.detach().cpu().numpy() if isinstance(v, torch.Tensor) else np.asarray(v)) for k, v in d.items()}
