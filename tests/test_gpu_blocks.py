"""GPU parity of the fused block cores, the four blocks and the whole models against the CPU oracle
and the committed golden vectors (outputs of the unmodified reference).

Tolerances (fp32 throughout; the native path re-associates sums and hoists the linear k/v
projections, so results are not bitwise):
  activations / logits : |err| <= 2e-4 + 2e-4*|ref| on clouds/points whose neighbour sets agree
  point scores         : rtol 2e-5 on columns unaffected by a kNN near-tie
  indices              : exact except provable fp32 near-ties / exact-score ties (SURVEY 8c)
"""
import math
import os

import numpy as np
import pytest
import torch

from oracle import samble_oracle as O
from samble_b200 import blocks, models, ops
from samble_b200.config import cls_config, seg_config
from oracle import harness
from samble_b200.testing import (amp_excusing_knn_ties, fill_state_dict_, judge_against_reference_scores, sampled_index_parity,
                                 synthetic_clouds, synthetic_features)
from tests.golden import make_golden as G

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def cu(t):
    return t.to(DEV)


def close_frac(x, ref, atol=2e-4, rtol=2e-4):
    x, ref = x.detach().cpu().double(), ref.detach().cpu().double()
    return float(((x - ref).abs() <= atol + rtol * ref.abs()).double().mean())


# ---------------------------------------------------------------- DownSample stages, teacher-forced


@pytest.mark.parametrize("B,N,nb,sharp", [(2, 512, 4, 1.0), (2, 2048, 4, 4.0), (1, 1000, 6, 2.0), (1, 4096, 4, 8.0)])
def test_ds_row_stats_and_edge_score(B, N, nb, sharp):
    D, K = 128, 32
    g = torch.Generator().manual_seed(N + nb)
    q = torch.randn(B, N, D, generator=g) * sharp
    k = torch.randn(B, N, D, generator=g)
    k_tok = torch.randn(nb, D, generator=g)
    x = synthetic_features(B, D, N, 3)
    _, idx = O.knn(x.transpose(1, 2), x.transpose(1, 2), K)
    # CPU statement of models/downsample.py:139-153, 300-344 on the same q/k/idx (fp64 for the reference value)
    logits = torch.cat([q.double() @ k.double().transpose(1, 2), q.double() @ k_tok.double().t()], -1) / math.sqrt(D)
    amap = torch.softmax(logits, -1)
    mask = torch.zeros(B, N, N, dtype=torch.float64).scatter_(2, idx, 1.0)
    indeg = mask.sum(1)
    score_ref = ((amap[..., :N] * mask).sum(1) / (indeg + 1e-8) / (indeg + 1e-8))
    from samble_b200 import _lib as L
    m_ref = logits.max(-1)[0]
    L.lib().samble_set_ds_mode(1)                      # exact FFMA tile kernel
    try:
        rm_f, rs_f, tok_f = ops.ds_row_stats(cu(q), cu(k), cu(k_tok))
    finally:
        L.lib().samble_set_ds_mode(0)
    torch.testing.assert_close(rm_f.cpu().double(), m_ref, atol=1e-4, rtol=1e-5)
    torch.testing.assert_close(rs_f.cpu().double(), torch.exp(logits - m_ref.unsqueeze(-1)).sum(-1), atol=1e-5, rtol=1e-4)
    rowmax, rowsum, tok = ops.ds_row_stats(cu(q), cu(k), cu(k_tok))      # tcgen05 3xTF32 kernel
    assert torch.equal(tok, tok_f)                     # token columns: exact fp32 in both
    print(f"row stats tc vs fp64: max|dm| {(rowmax.cpu().double() - m_ref).abs().max():.2e}, max rel ds "
          f"{((rowsum.cpu().double() * torch.exp(rowmax.cpu().double() - m_ref)) / torch.exp(logits - m_ref.unsqueeze(-1)).sum(-1) - 1).abs().max():.2e}")
    torch.testing.assert_close(rowmax.cpu().double(), m_ref, atol=3e-4, rtol=1e-5)
    # the pair (max, sum) matters only through logsumexp = max + log(sum)
    lse_ref = torch.logsumexp(logits, -1)
    lse = rowmax.cpu().double() + torch.log(rowsum.cpu().double())
    torch.testing.assert_close(lse, lse_ref, atol=2e-4, rtol=1e-5)
    torch.testing.assert_close(tok.cpu().double(), logits[..., N:], atol=1e-4, rtol=1e-5)
    # the two tensor-core kernels (linear_tma.cu row-statistics epilogue vs ds_rowstats_tc.cu) agree
    ops._DS_FAST = not ops._DS_FAST
    try:
        rm_o, rs_o, tok_o = ops.ds_row_stats(cu(q), cu(k), cu(k_tok))
    finally:
        ops._DS_FAST = not ops._DS_FAST
    assert torch.equal(tok_o, tok)
    torch.testing.assert_close(rm_o.cpu().double() + torch.log(rs_o.cpu().double()), lse, atol=2e-5, rtol=1e-6)
    for bits in (torch.int64, torch.int32):
        score = ops.ds_edge_score(cu(q), cu(k), rowmax, rowsum, cu(idx.to(bits)))
        torch.testing.assert_close(score.cpu().double(), score_ref, atol=1e-12, rtol=2e-4)
    # determinism: fixed accumulation order => bitwise repeatable
    again = ops.ds_edge_score(cu(q), cu(k), rowmax, rowsum, cu(idx))
    assert torch.equal(again, ops.ds_edge_score(cu(q), cu(k), rowmax, rowsum, cu(idx)))
    # strided (row stride 3D) views as the block passes them
    qkv = torch.cat([q, k, torch.zeros_like(q)], -1).to(DEV)
    rm2, rs2, _ = ops.ds_row_stats(qkv[..., :D], qkv[..., D:2 * D], cu(k_tok))
    assert torch.equal(rm2, rowmax) and torch.equal(rs2, rowsum)


@pytest.mark.parametrize("B,N,nb,M", [(4, 2048, 4, 1024), (4, 1024, 4, 512), (3, 1024, 6, 512), (2, 777, 6, 300), (1, 8192, 4, 4096),
                                      (1, 16384, 4, 8192)])
def test_ds_sample_vs_oracle(B, N, nb, M):
    g = torch.Generator().manual_seed(N * nb + M)
    score = torch.rand(B, N, generator=g) ** 3 * 1e-3
    tok = torch.randn(B, N, nb, generator=g)
    bnd, _ = O.bin_partition(score.unsqueeze(1), None, True, 0.99, nb)          # calibrated, monotone cuts
    cuts = bnd[0].reshape(-1)[1:].clone()
    bnd, mask = O.bin_partition(score.unsqueeze(1), bnd, False, 0.99, nb)
    w_raw = ((tok.unsqueeze(1) * mask).sum(2) / (torch.count_nonzero(mask, dim=2) + 1e-8)).squeeze(1)
    counts = mask.squeeze(1).sum(1)
    k_ref = O.calculate_num_points_to_choose(torch.relu(w_raw), counts, M)
    idx_ref = O.generating_downsampled_index(M, score.unsqueeze(1), mask, "topk", None, k_ref)
    z_ref = (score - score.mean(1, keepdim=True)) / score.std(1, unbiased=False, keepdim=True)
    s = ops.ds_sample(cu(score), cu(tok), cu(cuts), M, want_z=True)
    torch.testing.assert_close(s["z"].cpu(), z_ref, atol=2e-6, rtol=2e-6)
    bin_ref = mask.squeeze(1).float().argmax(-1)
    flips = int((s["bin_id"].cpu().long() != bin_ref).sum())
    assert flips <= 2, flips                                                    # z within an ulp of a cut
    if flips == 0:
        assert torch.equal(s["counts"].cpu().long(), counts)
        torch.testing.assert_close(s["w_raw"].cpu(), w_raw, atol=1e-6, rtol=1e-5)
        # k: the reference truncates fp32 values that sit ON integers whenever a bin saturates or has zero
        # weight (e.g. 225*(1-1e-12)), so a last-ulp difference in the bin weight (ours is an fp64 sum, the
        # reference an fp32 one) moves one point between two bins.  Same inputs => same k is pinned bit-exact
        # by test_num_points_to_choose; here a unit transfer is accepted and the take is checked against OUR k.
        k_mine = s["k"].cpu()
        assert int((k_mine - k_ref).abs().max()) <= 1 and int((k_mine - k_ref).abs().sum()) <= 2 * B, (k_mine, k_ref)
        idx_tf = O.generating_downsampled_index(M, score.unsqueeze(1), mask, "topk", None, k_mine)
        rep = sampled_index_parity(s["idx"].unsqueeze(1), idx_tf, score.unsqueeze(1), k_mine)
        # (exact score ties -- a few at N = 16384 with 2^24 distinct random floats -- are ordered lower index first here,
        # arbitrarily by torch.sort: sampled_index_parity counts only differences it cannot attribute to them)
        assert rep["unexplained_bins"] == 0 and rep["exact_rate"] >= (1.0 if N < 8192 else 0.999), rep
    assert bool((s["k"].sum(1) == M).all())
    for b in range(B):
        assert len(set(s["idx"][b].tolist())) == M                              # a sample, not a multiset


# ---------------------------------------------------------------- blocks


def _sd(N, M=None, seed=5, sharpen=4.0):
    cfg = seg_config(M=M or (N // 2, N // 4))
    m = models.ShapeNetModel(cfg)
    sd = fill_state_dict_(m.state_dict(), seed=seed, sharpen=sharpen)
    m.load_state_dict(sd)
    return cfg, m.eval().to(DEV), sd


def test_blocks_golden():
    """the reference's own block outputs (tests/golden/blocks_small.npz)."""
    gold = np.load(os.path.join(GOLD, "blocks_small.npz"))
    N = G.BLOCK_N
    cfg, m, sd = _sd(N)
    x3, x64, x128 = synthetic_features(2, 3, N, 61), synthetic_features(2, 64, N, 63), synthetic_features(2, 128, N, 62)
    with torch.no_grad():
        assert close_frac(m.block.embedding_list[0](cu(x3)), torch.from_numpy(gold["edgeconv0"])) == 1.0
        assert close_frac(m.block.embedding_list[1](cu(x64)), torch.from_numpy(gold["edgeconv1"])) == 1.0
        assert close_frac(m.block.feature_learning_layer_list[0](cu(x128)), torch.from_numpy(gold["n2p0"])) >= 0.999
        ds = m.block.downsample_list[0]
        for tag in ("calib", "frozen"):
            (x_ds, idx), _ = ds(cu(x128))
            torch.testing.assert_close(ds.bin_boundaries[0].cpu(), torch.from_numpy(gold[f"ds0.{tag}.upper"]), rtol=1e-5, atol=1e-6)
            gscore = torch.from_numpy(gold[f"ds0.{tag}.score"])
            torch.testing.assert_close(ds.bin_weights_beforerelu.cpu(), torch.from_numpy(gold[f"ds0.{tag}.w"]), atol=1e-5, rtol=1e-4)
            _, amp, touched = amp_excusing_knn_ties(x128, sd, "block.downsample_list.0.")
            ok = (ds.attention_point_score.cpu()[:, 0] - gscore[:, 0]).abs() <= 5e-5 * gscore[:, 0].abs() + 1e-30
            assert bool((ok | touched).all()) and int(touched.sum()) <= 8, (int((~ok).sum()), int(touched.sum()))
            judge_against_reference_scores(ds, idx, x_ds, gscore, torch.from_numpy(gold[f"ds0.{tag}.idx"]),
                                            torch.from_numpy(gold[f"ds0.{tag}.k"]), torch.from_numpy(gold[f"ds0.{tag}.x_ds"]), amp)
            ds.dynamic_boundaries_enable = False
        xyz_up, xyz_dn = synthetic_features(2, 3, N, 64), synthetic_features(2, 3, N // 2, 65)
        dn = synthetic_features(2, 128, N // 2, 66)
        up = m.block.upsample_list[0](cu(x128), ((cu(dn), None, cu(xyz_dn)), (None, None)), cu(xyz_up))
        assert close_frac(up, torch.from_numpy(gold["upsample0"])) == 1.0


@pytest.mark.parametrize("N", [512, 2048])
def test_blocks_vs_oracle(N):
    cfg, m, sd = _sd(N, seed=9, sharpen=4.0)
    B = 2
    x3, x64, x128 = synthetic_features(B, 3, N, 71), synthetic_features(B, 64, N, 72), synthetic_features(B, 128, N, 73)
    with torch.no_grad():
        assert close_frac(m.block.embedding_list[0](cu(x3)), O.edgeconv(sd, "block.embedding_list.0.", x3, 32)) >= 0.9995
        assert close_frac(m.block.embedding_list[1](cu(x64)), O.edgeconv(sd, "block.embedding_list.1.", x64, 32)) >= 0.9995
        y = m.block.feature_learning_layer_list[0](cu(x128))
        assert close_frac(y, O.n2p_attention(sd, "block.feature_learning_layer_list.0.", x128, 32)) >= 0.9995
        ds, st = m.block.downsample_list[0], O.DSState(True)
        pre = "block.downsample_list.0."
        for it in range(2):
            (x_ds, idx), _ = ds(cu(x128))
            ref = O.downsample_token(sd, pre, x128, N // 2, 32, 4, st)
            torch.testing.assert_close(ds.bin_boundaries[0].cpu(), ref["boundaries"][0], rtol=1e-5, atol=1e-6)
            assert tuple(ds.bin_points_mask.shape) == tuple(ref["mask"].shape) and ds.bin_points_mask.dtype == torch.bool
            assert close_frac(ds.attention_bins_beforesoftmax, ref["token_logits"]) == 1.0
            # the exact-product GEMM (csrc/xgemm.cu) puts the native score within a few fp32 roundings of the fp64 value
            s64, amp, touched = amp_excusing_knn_ties(x128, sd, pre)
            big = s64 > 1e-30                                 # (below that the fp32 probabilities underflow)
            rel = (ds.attention_point_score.cpu().double()[:, 0] - s64).abs()[big] / s64[big]
            assert float(rel.max()) <= 2e-5, float(rel.max())
            judge_against_reference_scores(ds, idx, x_ds, ref["score"], ref["idx"], ref["k"], ref["x_ds"], amp)
            ds.dynamic_boundaries_enable, st.dynamic = False, False
        M = N // 2
        xyz_up, xyz_dn, dn = synthetic_features(B, 3, N, 74), synthetic_features(B, 3, M, 75), synthetic_features(B, 128, M, 76)
        up = m.block.upsample_list[0](cu(x128), ((cu(dn), None, cu(xyz_dn)), (None, None)), cu(xyz_up))
        assert close_frac(up, O.upsample_interpolation(sd, "block.upsample_list.0.", x128, dn, xyz_up, xyz_dn, 3)) == 1.0


@pytest.mark.parametrize("N", [8192, 16384])
def test_downsample_block_large_clouds(N):
    """BASELINE config 4 sizes: one DownSampleToken layer (N -> N/2) against the oracle, which needs ~6 GB of dense
    N x N temporaries at 16384 where the native path needs O(N K)."""
    cfg = seg_config(M=(N // 2, N // 4))
    m = models.ShapeNetModel(cfg)
    sd = fill_state_dict_(m.state_dict(), seed=9, sharpen=4.0)
    m.load_state_dict(sd)
    ds = m.block.downsample_list[0].eval().to(DEV)
    x = synthetic_features(1, 128, N, 77)
    pre = "block.downsample_list.0."
    st = O.DSState(True)
    with torch.no_grad():
        for it in range(2):
            (x_ds, idx), _ = ds(cu(x))
            ref = O.downsample_token(sd, pre, x, N // 2, 32, 4, st)
            torch.testing.assert_close(ds.bin_boundaries[0].cpu(), ref["boundaries"][0], rtol=1e-5, atol=1e-6)
            _, amp, touched = amp_excusing_knn_ties(x, sd, pre, cheap=True)
            ok = (ds.attention_point_score.cpu()[:, 0] - ref["score"][:, 0]).abs() <= 2e-4 * ref["score"][:, 0].abs() + 1e-30
            assert bool((ok | touched).all()), int((~(ok | touched)).sum())
            judge_against_reference_scores(ds, idx, x_ds, ref["score"], ref["idx"], ref["k"], ref["x_ds"], amp)
            ds.dynamic_boundaries_enable, st.dynamic = False, False


@pytest.mark.parametrize("B,N,K,Cin,C1,C2,gt", [(2, 300, 32, 3, 64, 64, "center_diff"), (1, 515, 16, 64, 64, 128, "center_diff"),
                                                (2, 128, 7, 8, 32, 32, "diff"), (1, 200, 20, 16, 64, 64, "center_neighbor"),
                                                (2, 2048, 32, 3, 64, 128, "center_diff"), (1, 1023, 32, 64, 128, 64, "center_diff"),
                                                (1, 64, 32, 6, 16, 32, "neighbor")])
def test_fused_edge_mlp_vs_unfused(B, N, K, Cin, C1, C2, gt):
    """csrc/edgeconv.cu against the literal group -> conv -> BN -> LeakyReLU -> conv -> BN -> LeakyReLU -> max
    (models/embedding.py:29-39) on CPU, teacher-forced with the same neighbour indices."""
    from torch import nn

    g = torch.Generator().manual_seed(N + K)
    x = torch.randn(B, Cin, N, generator=g)
    cin_t = 2 * Cin if gt.startswith("center") else Cin
    conv1, bn1, conv2, bn2 = nn.Conv2d(cin_t, C1, 1, bias=False), nn.BatchNorm2d(C1), nn.Conv2d(C1, C2, 1, bias=False), nn.BatchNorm2d(C2)
    sd = {f"{n}.{k}": v for n, mod in (("conv1", conv1), ("bn1", bn1), ("conv2", conv2), ("bn2", bn2)) for k, v in mod.state_dict().items()}
    fill_state_dict_(sd, seed=N)
    for mod in (conv1, bn1, conv2, bn2):
        mod.eval()
    _, idx = O.knn(x.transpose(1, 2), x.transpose(1, 2), K)
    pts = x.transpose(1, 2)
    nbr = O.index_points(pts, idx)
    if gt.endswith("diff"):
        nbr = nbr - pts.unsqueeze(2)
    grouped = nbr.permute(0, 3, 1, 2)
    if gt.startswith("center"):
        grouped = torch.cat([x.unsqueeze(-1).repeat(1, 1, 1, K), grouped], dim=1)
    with torch.no_grad():
        lrelu = torch.nn.functional.leaky_relu
        ref = lrelu(bn2(conv2(lrelu(bn1(conv1(grouped)), 0.2))), 0.2).max(dim=-1)[0]
        w = [t.to(DEV) for t in blocks.edge_mlp_weights(conv1, bn1, conv2, bn2, gt)]
        from samble_b200 import _lib as L
        for mode in (0, 1):                                # 0: tcgen05 where eligible, 1: FFMA kernel
            L.lib().samble_set_edge_mode(mode)
            try:
                for dt in (torch.int32, torch.int64):
                    out = blocks.fused_edge_mlp(cu(x), cu(idx.to(dt)), w)
                    assert close_frac(out, ref, atol=1e-4, rtol=1e-4) == 1.0, (mode, dt)
            finally:
                L.lib().samble_set_edge_mode(0)


def test_cuda_graph_replay_matches_eager():
    from samble_b200.runtime import GraphedForward

    cfg, m, _ = _sd(512, seed=4)
    x, cat = synthetic_clouds(3, 512, 8)
    x2, cat2 = synthetic_clouds(3, 512, 9)
    with torch.no_grad():
        m(cu(x), cu(cat))
        with pytest.raises(RuntimeError, match="frozen"):
            GraphedForward(m, cu(x), cu(cat))
        models.freeze_boundaries(m)
        y_eager, y2_eager = m(cu(x), cu(cat)).clone(), m(cu(x2), cu(cat2)).clone()
        idx2 = [ds.idx.clone() for ds in m.block.downsample_list]
        g = GraphedForward(m, cu(x), cu(cat))
        assert torch.equal(g(cu(x), cu(cat)), y_eager)
        assert torch.equal(g(cu(x2), cu(cat2)), y2_eager)            # new inputs through the same graph
        assert all(torch.equal(a, ds.idx) for a, ds in zip(idx2, m.block.downsample_list))


def test_grad_is_never_silently_dropped():
    """An input (or parameter) that requires grad sends a block down the differentiable path (tests/test_gpu_backward.py);
    the fused inference kernels themselves refuse such tensors instead of returning a detached result."""
    cfg, m, sd = _sd(128)
    x = cu(synthetic_features(1, 128, 128, 1)).requires_grad_(True)
    y = m.block.feature_learning_layer_list[0](x)
    assert y.requires_grad
    y.sum().backward()
    assert x.grad is not None and float(x.grad.abs().max()) > 0
    with pytest.raises(RuntimeError, match="forward-only"):
        ops.linear(x, m.block.feature_learning_layer_list[0].ff[0].weight, x_layout="bcn")


# ---------------------------------------------------------------- whole models


@pytest.mark.parametrize("which", ["seg", "cls"])
def test_models_golden(which):
    """logits + sampled indices of the unmodified reference (tests/golden/{seg,cls}_small.npz)."""
    c = G.MODEL_CASES[which]
    gold = np.load(os.path.join(GOLD, f"{which}_small.npz"))
    cfg = (seg_config if which == "seg" else cls_config)(M=c["M"])
    m = (models.ShapeNetModel if which == "seg" else models.ModelNetModel)(cfg)
    m.load_state_dict(fill_state_dict_(m.state_dict(), seed=c["wseed"], sharpen=4.0))
    m = m.eval().to(DEV)
    x, cat = synthetic_clouds(c["B"], c["N"], c["xseed"])
    with torch.no_grad():
        for tag in ("calib", "frozen"):
            y = m(cu(x), cu(cat)) if which == "seg" else m(cu(x))
            agree = True
            for i, ds in enumerate(m.block.downsample_list):
                ref_idx = torch.from_numpy(gold[f"{tag}.ds{i}.idx"])
                same = torch.equal(ds.idx.cpu(), ref_idx)
                overlap = np.mean([len(set(ds.idx[b, 0].tolist()) & set(ref_idx[b, 0].tolist())) / ref_idx.shape[-1]
                                   for b in range(c["B"])])
                assert overlap >= (0.97 if i == 0 else 0.9), (tag, i, overlap)   # chained: reported as a rate (SURVEY 8c step 7)
                agree &= same
            if agree:                                            # free-running chained agreement: logits match too
                assert close_frac(y, torch.from_numpy(gold[f"{tag}.logits"]), atol=2e-3, rtol=2e-3) >= 0.999
            models.freeze_boundaries(m)
    # ... and unconditionally: every decision adjudicated in fp64, every logit within tolerance once the decisions are
    # forced into the oracle (oracle/harness.py)
    sd = fill_state_dict_(m.cpu().state_dict(), seed=c["wseed"], sharpen=4.0)
    m = m.to(DEV)
    x2, cat2 = synthetic_clouds(c["B"], c["N"], c["xseed"] + 50)       # not the calibration batch: no cut sits on a z
    rep = harness.forward_parity(m, sd, cfg, x2, cat2, which=which)
    print(harness.brief(rep))
    harness.assert_report(rep)


@pytest.mark.parametrize("which,B,N,M", [("seg", 16, 2048, (1024, 512)), ("cls", 32, 1024, (512, 256))])
def test_full_size_forward_vs_oracle(which, B, N, M):
    """BASELINE configs 3 and 2 at full size against the CPU oracle (teacher-forced protocol, oracle/harness.py)."""
    cfg = (seg_config if which == "seg" else cls_config)(M=M)
    m = (models.ShapeNetModel if which == "seg" else models.ModelNetModel)(cfg)
    sd = fill_state_dict_(m.state_dict(), seed=3, sharpen=4.0)
    m.load_state_dict(sd)
    m = m.eval().to(DEV)
    xc, catc = synthetic_clouds(B, N, 105)
    x, cat = synthetic_clouds(B, N, 5)
    with torch.no_grad():
        m(cu(xc), cu(catc)) if which == "seg" else m(cu(xc))
    models.freeze_boundaries(m)
    rep = harness.forward_parity(m, sd, cfg, x, cat, which=which)
    print(harness.brief(rep))
    harness.assert_report(rep)
    for d in rep["ds"]:
        assert d["score_rel_err_vs_fp64"]["native_max"] <= 2e-5, d["score_rel_err_vs_fp64"]


def test_seg_forward_full_size_properties():
    """BASELINE config 3 size (B=16, N=2048): size-independent properties instead of a CPU oracle run:
    run-to-run determinism, valid samples, and batch-shard invariance (what lets the batch be split
    across GPUs with no collective, SURVEY 8e)."""
    cfg, m, _ = _sd(2048, M=(1024, 512), seed=3, sharpen=4.0)
    x, cat = synthetic_clouds(16, 2048, 5)
    x, cat = cu(x), cu(cat)
    xc, catc = synthetic_clouds(16, 2048, 105)
    with torch.no_grad():
        m(cu(xc), cu(catc))                                      # calibration batch (another one: no cut sits exactly on a z)
        models.freeze_boundaries(m)
        y1 = m(x, cat)
        idx1 = [ds.idx.clone() for ds in m.block.downsample_list]
        y2 = m(x, cat)
        assert torch.equal(y1, y2) and all(torch.equal(a, ds.idx) for a, ds in zip(idx1, m.block.downsample_list))
        assert tuple(y1.shape) == (16, 50, 2048) and bool(torch.isfinite(y1).all())
        for ds, M, N in zip(m.block.downsample_list, (1024, 512), (2048, 1024)):
            assert tuple(ds.idx.shape) == (16, 1, M) and int(ds.idx.min()) >= 0 and int(ds.idx.max()) < N
            assert all(len(set(ds.idx[b, 0].tolist())) == M for b in range(16))
            assert bool((ds.k_point_to_choose.sum(1) == M).all())
        ys = m(x[4:8], cat[4:8])                                 # a shard alone == the same clouds in the batch
        # every native kernel is per-cloud; the few library GEMMs left (STN / category vectors) may pick another split for
        # another batch size, so fp32 near-tie flips are possible (the reference shows the same B-dependence, SURVEY 8e
        # caveat 2): measured identical here, asserted >= 0.99
        for a, ds in zip(idx1, m.block.downsample_list):
            ov = np.mean([len(set(a[4 + b, 0].tolist()) & set(ds.idx[b, 0].tolist())) / a.shape[-1] for b in range(4)])
            assert ov >= 0.99, ov


@pytest.mark.parametrize("mode", ["random", "uniform"])
def test_stochastic_sample_modes_run_and_respect_bins(mode):
    """sample_mode 'random' (the reference's YAML default) / 'uniform', utils/ops.py:507-613: the scores, bins and the
    k per bin are the deterministic native path; the indices are torch.multinomial draws that must fall into their
    bin, be distinct, and number k per bin."""
    from samble_b200 import models
    from samble_b200.config import seg_config
    from samble_b200.testing import fill_state_dict_, synthetic_clouds

    B, N = 2, 512
    m = models.ShapeNetModel(seg_config(M=(N // 2, N // 4), sample_mode=mode))
    m.load_state_dict(fill_state_dict_(m.state_dict(), seed=1, sharpen=4.0))
    m = m.eval().cuda()
    x, cat = synthetic_clouds(B, N, 2)
    with torch.no_grad():
        y = m(x.cuda(), cat.cuda())
    assert tuple(y.shape) == (B, 50, N) and torch.isfinite(y).all()
    for ds in m.block.downsample_list:
        idx, mask, k = ds.idx.cpu(), ds.bin_points_mask.cpu(), ds.k_point_to_choose.cpu()
        nb = mask.shape[-1]
        for b in range(B):
            assert len(set(idx[b, 0].tolist())) == idx.shape[-1]              # bins are disjoint, draws without replacement
            off = 0
            for j in range(nb):
                seg = idx[b, 0, off:off + int(k[b, j])]
                assert bool(mask[b, 0, seg, j].all())
                off += int(k[b, j])
            assert off == idx.shape[-1]


def test_host_pipeline_returns_the_graph_results_in_order():
    """runtime.HostPipeline: pinned host inputs in, pinned host results out, D2H of a step overlapping the next step."""
    from samble_b200.runtime import GraphedForward, HostPipeline

    cfg, m, _ = _sd(512, seed=4)
    batches = [synthetic_clouds(2, 512, 20 + i) for i in range(5)]
    with torch.no_grad():
        m(cu(batches[0][0]), cu(batches[0][1]))
        models.freeze_boundaries(m)
        want = [m(cu(x), cu(c)).cpu() for x, c in batches]
        g = GraphedForward(m, cu(batches[0][0]), cu(batches[0][1]))
        pipe = HostPipeline(g)
        got = []
        for x, c in batches:
            host, done = pipe.submit(x.pin_memory(), c.pin_memory())
            pipe.wait_previous()
            done.synchronize()                      # a consumer reads a result only after its event
            got.append(host.clone())
        pipe.wait_all()
        torch.cuda.synchronize()
    for a, b in zip(got, want):
        assert torch.equal(a, b)


ATTEND_CASES = [(2, 2048, 1024, 4, 4.0, 128), (3, 1024, 512, 6, 2.0, 128), (1, 1000, 300, 4, 4.0, 128), (1, 8192, 4096, 4, 8.0, 128),
                (2, 256, 128, 4, 1.0, 128), (2, 1024, 512, 8, 4.0, 32), (2, 1000, 300, 8, 4.0, 64), (2, 2048, 1024, 8, 4.0, 96)]


@pytest.mark.parametrize("B,N,M,nb,sharp,D", ATTEND_CASES,
                         ids=["-".join(map(str, c[:5])) + ("" if c[5] == 128 else f"-D{c[5]}") for c in ATTEND_CASES])
def test_ds_attend_rows_vs_fp64(B, N, M, nb, sharp, D):
    """The flash-style selected-row attention (csrc/ds_attend.cu) against the literal statement of
    models/downsample.py:242-252 in fp64: softmax rows of the selected points over the N point and nb token columns, times
    [v ; v_tok].  No (B,M,N) tensor on the device side.  D = C below 128 are the widths DownSampleToken's exact path takes
    for narrower layers (C % 32 == 0)."""
    C = D
    g = torch.Generator().manual_seed(N + M)
    q = (torch.randn(B, N, D, generator=g) * sharp)
    k = torch.randn(B, N, D, generator=g)
    v = torch.randn(B, N, C, generator=g)
    k_tok, v_tok = torch.randn(nb, D, generator=g), torch.randn(nb, C, generator=g)
    idx = torch.stack([torch.randperm(N, generator=g)[:M] for _ in range(B)])
    qkv = torch.cat([q, k, v], -1).to(DEV)                          # the (B,N,3C) buffer the block slices
    qg, kg, vg = qkv[..., :D], qkv[..., D:2 * D], qkv[..., 2 * D:]
    qd, kd = ops.digits(qg), ops.digits(kg)
    rowmax, rowsum, tok = ops.ds_row_stats_exact(qd, kd, qg, cu(k_tok))
    out = ops.ds_attend_rows(qd, kd, vg, cu(idx), rowmax, rowsum, tok, cu(v_tok))
    again = ops.ds_attend_rows(qd, kd, vg, cu(idx), rowmax, rowsum, tok, cu(v_tok))
    assert torch.equal(out, again)                                   # (the two-way key split adds commutatively)
    logits = torch.cat([q.double() @ k.double().transpose(1, 2), q.double() @ k_tok.double().t()], -1) / math.sqrt(D)
    amap = torch.softmax(logits, -1).gather(1, idx.unsqueeze(-1).expand(-1, -1, N + nb))          # (B,M,N+nb)
    ref = amap @ torch.cat([v.double(), v_tok.double().unsqueeze(0).expand(B, -1, -1)], 1)
    err = (out.cpu().double() - ref).abs()
    print(f"ds_attend_rows B={B} N={N} M={M} D={D}: max abs err {err.max():.2e} on values of magnitude {ref.abs().max():.1f}")
    assert bool((err <= 5e-5 + 1e-4 * ref.abs()).all()), float(err.max())


@pytest.mark.parametrize("B,N,M,nb,D,C,sliced", [(2, 1024, 512, 4, 64, 128, False), (1, 1000, 301, 1, 128, 128, True),
                                                 (2, 777, 301, 8, 48, 48, True), (3, 512, 8, 6, 256, 256, False)])
def test_ds_select_rows_vs_fp64(B, N, M, nb, D, C, sliced):
    """samble_ds_select_rows (the gather in front of DownSampleToken's 3xTF32 row GEMMs) against fp64: q_sel, m_sel and
    s_sel are the gathered values exactly; tok_mix is sum_t exp(tok - m) / s * v_tok[t], the token columns' share of
    models/downsample.py:242-252.  M = 301 leaves the kernel's last block of 8 rows partly empty; `sliced` passes q as a
    column slice of a (B,N,3C) buffer, as the block does."""
    g = torch.Generator().manual_seed(N + M + D)
    q = torch.randn(B, N, D, generator=g) * 2
    rowmax = torch.randn(B, N, generator=g) + 3
    rowsum = torch.rand(B, N, generator=g) * 10 + 1
    tok = torch.randn(B, N, nb, generator=g)
    v_tok = torch.randn(nb, C, generator=g)
    idx = torch.stack([torch.randperm(N, generator=g)[:M] for _ in range(B)])
    if sliced:
        buf = torch.randn(B, N, 3 * C, generator=g)
        buf[..., :D] = q
        qg = cu(buf)[..., :D]
    else:
        qg = cu(q)
    q_sel, m_sel, s_sel, tok_mix = ops.ds_select_rows(qg, cu(rowmax), cu(rowsum), cu(tok), cu(v_tok), cu(idx))
    gat = lambda t: torch.gather(t, 1, idx.view(B, M, *([1] * (t.dim() - 2))).expand(-1, -1, *t.shape[2:]))
    assert torch.equal(q_sel.cpu(), gat(q))
    assert torch.equal(m_sel.cpu(), gat(rowmax)) and torch.equal(s_sel.cpu(), gat(rowsum))
    p = torch.exp(gat(tok).double() - gat(rowmax).double().unsqueeze(-1)) / gat(rowsum).double().unsqueeze(-1)     # (B,M,nb)
    ref = p @ v_tok.double()
    err = (tok_mix.cpu().double() - ref).abs()
    print(f"ds_select_rows tok_mix: max abs err {err.max():.2e} on values of magnitude {ref.abs().max():.2e}")
    assert bool((err <= 1e-6 + 1e-5 * ref.abs()).all()), float(err.max())


def test_checkpoint_and_eval_harness(tmp_path):
    """SURVEY 8 row f4: a reference-format checkpoint ({"model_state_dict" with DDP prefix, "bin_boundaries"}) restores a
    model that reproduces the source model's predictions and sampled indices bit for bit through the evaluation loop."""
    from torch.utils.data import DataLoader

    from samble_b200 import checkpoint, evaluate

    cfg = seg_config(M=(128, 64))
    src = models.ShapeNetModel(cfg)
    src.load_state_dict(fill_state_dict_(src.state_dict(), seed=12, sharpen=2.0))
    src = src.eval().to(DEV)
    xc, catc = synthetic_clouds(4, 256, 31)
    with torch.no_grad():
        src(cu(xc), cu(catc))                                     # calibrates the dynamic boundaries (EMA state outside the state_dict)
    path = str(tmp_path / "checkpoint.pt")
    checkpoint.save(src, path)
    dst = checkpoint.load(models.ShapeNetModel(cfg).to(DEV), path, map_location=DEV)
    models.freeze_boundaries(src)
    data = evaluate.SyntheticShapeNetPart(8, N=256, seed=3)
    a = evaluate.evaluate_seg(src, DataLoader(data, batch_size=4), device=DEV)
    b = evaluate.evaluate_seg(dst, DataLoader(data, batch_size=4), device=DEV)
    assert a["pred"].shape == (8, 256) and a["seg_label"].shape == (8, 256) and len(a["ds_idx"]) == 2
    assert a["ds_idx"][0].shape == (8, 1, 128) and a["ds_idx"][1].shape == (8, 1, 64)
    assert np.array_equal(a["pred"], b["pred"]) and all(np.array_equal(x, y) for x, y in zip(a["ds_idx"], b["ds_idx"]))
    assert 0.0 <= a["point_accuracy"] <= 1.0
    ccfg = cls_config(M=(128, 64))
    cm = models.ModelNetModel(ccfg)
    cm.load_state_dict(fill_state_dict_(cm.state_dict(), seed=13))
    cm = cm.eval().to(DEV)
    r = evaluate.evaluate_cls(cm, DataLoader(evaluate.SyntheticModelNet(6, N=256), batch_size=3), device=DEV)
    assert r["pred"].shape == (6,) and 0.0 <= r["accuracy"] <= 1.0


@pytest.mark.needs_reference
@pytest.mark.parametrize("which", ["seg", "cls"])
def test_unmodified_reference_wiring_with_the_patch_installed(which):
    """The drop-in claim end to end: the reference's OWN models/seg_model.py / cls_model.py (unmodified, imported from
    the checkout named by SAMBLE_REFERENCE) with samble_b200.patch installed, against the wiring mirror the other tests
    use.  Needs a reference checkout next to a GPU: it runs wherever a maintainer has both, and is skipped otherwise."""
    from samble_b200 import patch
    from tests.golden import ref_loader as R

    B, N, M = 2, 512, (256, 128)
    with patch.installed():
        over = {"downsample.M": list(M), "downsample.bin.sample_mode": ["topk", "topk"]}
        ref = R.build_model(which, R.reference_config(which, **over))
    cfg = (seg_config if which == "seg" else cls_config)(M=M)
    mine = (models.ShapeNetModel if which == "seg" else models.ModelNetModel)(cfg)
    sd = fill_state_dict_(mine.state_dict(), seed=21, sharpen=2.0)
    mine.load_state_dict(sd)
    ref.load_state_dict(sd)
    mine, ref = mine.eval().to(DEV), ref.eval().to(DEV)
    x, cat = synthetic_clouds(B, N, 41)
    args = (cu(x), cu(cat)) if which == "seg" else (cu(x),)
    with torch.no_grad(), patch.installed():
        for net in (mine, ref):
            net(*args)                                               # calibrate the boundaries
            for ds in net.block.downsample_list:
                ds.dynamic_boundaries_enable = False
        y_ref, y = ref(*args), mine(*args)
    assert all(isinstance(ds, blocks.DownSampleToken) for ds in ref.block.downsample_list)
    for a, b in zip(ref.block.downsample_list, mine.block.downsample_list):
        assert torch.equal(a.idx, b.idx)
    assert close_frac(y, y_ref) == 1.0


@pytest.mark.parametrize("B,N,C,K,H", [(2, 2048, 128, 32, 4), (1, 1000, 128, 32, 4), (3, 77, 64, 20, 4), (1, 300, 128, 17, 1), (2, 130, 64, 32, 8)])
def test_n2p_attend_eight_lane_kernel_vs_warp_per_point_and_fp64(B, N, C, K, H):
    """The two gather-attend kernels (csrc/attention.cu) against each other and against the literal fp64 statement of
    models/attention.py:207-250 on the hoisted projections, incl. the fused residual + folded-BN tail."""
    from samble_b200 import _lib as L
    g = torch.Generator().manual_seed(N + C + K)
    qkv = torch.randn(B, N, 3 * C, generator=g)
    idx = torch.stack([torch.stack([torch.randperm(N, generator=g)[:K] for _ in range(N)]) for _ in range(B)])
    res, sc, sh = torch.randn(B, N, C, generator=g), torch.rand(C, generator=g) + 0.5, torch.randn(C, generator=g)
    D = C // H
    q, k, v = (qkv.double()[..., i * C:(i + 1) * C] for i in range(3))
    gat = lambda t: torch.gather(t, 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, N, K, C)
    att = torch.softmax(torch.einsum("bnhd,bnkhd->bnhk", q.reshape(B, N, H, D), gat(k).view(B, N, K, H, D)) / math.sqrt(D), dim=-1)
    ref = torch.einsum("bnhk,bnkhd->bnhd", att, (gat(v) - v[:, :, None, :]).view(B, N, K, H, D)).reshape(B, N, C)
    ref_tail = (ref + res.double()) * sc.double() + sh.double()
    outs = {}
    for mode in (0, 1):
        L.lib().samble_set_n2p_mode(mode)
        try:
            for dt in (torch.int32, torch.int64):
                y = ops.n2p_attend(cu(qkv), cu(idx).to(dt), H)
                yt = ops.n2p_attend(cu(qkv), cu(idx).to(dt), H, residual=cu(res), scale=cu(sc), shift=cu(sh))
                assert close_frac(y, ref, 2e-5, 2e-5) == 1.0 and close_frac(yt, ref_tail, 2e-5, 2e-5) == 1.0, (mode, dt)
            outs[mode] = (y, yt)
        finally:
            L.lib().samble_set_n2p_mode(0)
    assert close_frac(outs[0][0], outs[1][0].cpu(), 1e-5, 1e-5) == 1.0


@pytest.mark.parametrize("D,K", [(64, 32), (192, 20), (32, 8)])
def test_ds_edge_score_other_widths(D, K):
    """ADVICE r1: samble_ds_edge_score accepts any D % 4 == 0; widths whose 16-byte chunk count is not a multiple of 32
    (D = 64: 16 chunks, D = 192: 48) leave some lanes without a chunk -- the neighbour-index broadcasts must not sit in that
    divergent loop.  Checked against the fp64 statement of models/downsample.py:300-344."""
    B, N, nb = 2, 384, 4
    g = torch.Generator().manual_seed(D + K)
    q, k = torch.randn(B, N, D, generator=g), torch.randn(B, N, D, generator=g)
    idx = torch.stack([torch.stack([torch.randperm(N, generator=g)[:K] for _ in range(N)]) for _ in range(B)])
    logits = q.double() @ k.double().transpose(1, 2) / math.sqrt(D)
    m = logits.max(-1)[0]
    ssum = torch.exp(logits - m.unsqueeze(-1)).sum(-1)
    amap = torch.exp(logits - m.unsqueeze(-1)) / ssum.unsqueeze(-1)
    mask = torch.zeros(B, N, N, dtype=torch.float64).scatter_(2, idx, 1.0)
    indeg = mask.sum(1)
    ref = (amap * mask).sum(1) / (indeg + 1e-8) / (indeg + 1e-8)
    ref = torch.where(torch.isnan(ref), torch.zeros_like(ref), ref)
    for bits in (torch.int32, torch.int64):
        score = ops.ds_edge_score(cu(q), cu(k), cu(m.float()), cu(ssum.float()), cu(idx.to(bits)))
        torch.testing.assert_close(score.cpu().double(), ref, atol=1e-12, rtol=2e-4)
