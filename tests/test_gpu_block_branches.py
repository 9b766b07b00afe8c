"""The four blocks at widths and sizes off the shipped configurations, against the CPU oracle.

Each block's eval forward picks one of several native branches (or an ATen fallback) from the widths and sizes it is
given; the model-level tests only reach the branch the shipped seg / cls configurations take.  Every case here builds
one block from the config helpers, fills it with fill_state_dict_, compares it with the oracle's block function at the
bar the model-level tests use, and checks through the library's launch profiler (samble_b200._lib.profile) that the
branch it is about actually ran, so that a later change to a gate cannot silently move a case onto another branch.
"""
import pytest
import torch

from oracle import samble_oracle as O
from samble_b200 import blocks, ops
from samble_b200.config import Cfg, _attention, _downsample
from samble_b200.testing import (amp_excusing_knn_ties, fill_state_dict_, judge_against_reference_scores, launched,
                                 synthetic_features)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def cu(t):
    return t.to(DEV)


def close_frac(x, ref, atol=2e-4, rtol=2e-4):
    x, ref = x.detach().cpu().double(), ref.detach().cpu().double()
    return float(((x - ref).abs() <= atol + rtol * ref.abs()).double().mean())


def filled(block, seed, sharpen=1.0):
    """block with fill_state_dict_ weights (q/k projections of a DownSampleToken x sharpen, as in the model tests), moved
    to the GPU in eval mode, and its CPU state_dict for the oracle (prefix "")."""
    sd = block.state_dict()
    prefix = "block.downsample_list.0." if isinstance(block, blocks.DownSampleToken) else ""
    fill_state_dict_({prefix + k: v for k, v in sd.items()}, seed=seed, sharpen=sharpen)     # fills sd's tensors in place
    sd = {k: v.clone() for k, v in sd.items()}
    block.load_state_dict(sd)
    return block.eval().to(DEV), sd


# ---------------------------------------------------------------- DownSampleToken

DS_CASES = [  # C, N, M, nb, switches, row statistics kernel, rows of the selected points
    (32, 512, 256, 8, {}, "exact", "attend"),
    (64, 1000, 300, 4, {}, "exact", "attend"),                     # N and M not multiples of 128
    (96, 2048, 1024, 6, {}, "exact", "attend"),
    (48, 1024, 512, 4, {}, "fast", "cloud_matmul"),                 # C % 32 != 0: 3xTF32
    (80, 1000, 300, 4, {}, "ffma", "eager"),
    (128, 2048, 1024, 4, {"DS_EXACT": False}, "fast", "cloud_matmul"),
    (128, 2048, 1024, 4, {"DS_EXACT": False, "_DS_FAST": False}, "tc", "cloud_matmul"),
    (128, 4096, 2048, 4, {"DS_EXACT": False}, "fast", "cloud_matmul"),      # cloud_matmul at its 4096-key limit
    (128, 1000, 300, 6, {"DS_EXACT": False}, "tc", "eager"),
    (256, 1024, 512, 4, {}, "fast", "cloud_matmul"),                # C > 128: 3xTF32, feature kNN on the exact tile kernel
]
ROW_STATS_KERNEL = {"exact": "xgemm_rowstat_kernel", "fast": "ds_rowstats_finalize_kernel", "ffma": "ds_row_stats_kernel",
                    "tc": "ds_row_stats_tc_kernel"}
# Max relative error of the point score against fp64, calibrating forward, measured on a B200:
#   exact:  C=32 N=512 1.1e-5, C=64 N=1000 7.6e-6, C=96 N=2048 1.4e-5 (asserted <= 2e-5)
#   3xTF32: C=48 N=1024 2.0e-4, C=80 N=1000 1.6e-4, C=128 N=2048 3.0e-4 (either row-statistics kernel), C=128 N=4096 2.9e-4,
#           C=128 N=1000 2.5e-4, C=256 N=1024 3.8e-4.
# That is ~20x the exact path's error, exponentiated logit error of the tf32 splits: the sharpened logits put most points'
# scores far below the mean, and those land on a handful of fp32 z-scores that several cuts can split (up to 22 such tie
# groups per cloud).  On these rows the fp64 band of ds_parity adjudicates every flip and swap; the count of tie groups
# is bounded on the exact rows only.


def _switch(mod, name, value):
    old = getattr(mod, name)
    setattr(mod, name, value)
    return lambda: setattr(mod, name, old)


def _check_ds_branch(k, C, stats, rows):
    for kind, name in ROW_STATS_KERNEL.items():
        if kind != "fast" or stats != "exact":        # (the exact statistics end in the same finalize kernel)
            assert (name in k) == (kind == stats), (stats, sorted(k))
    assert ("ds_attend_rows_kernel" in k) == (rows == "attend"), sorted(k)
    assert ("ds_select_rows_kernel" in k) == (rows != "attend"), sorted(k)
    if rows != "attend":
        # the [q|k|v] projection, the fast row statistics, and the two per-cloud GEMMs of cloud_matmul
        want = 1 + (stats == "fast") + 2 * (rows == "cloud_matmul")
        assert k.get("linear_tma_kernel", 0) == want, (rows, k.get("linear_tma_kernel"))
    tc_knn = any(name.startswith("knn_tc_") for name in k)
    assert tc_knn == (C <= 128) and (("knn_feat_kernel" in k) == (C > 128)), sorted(k)


@pytest.mark.parametrize("C,N,M,nb,switches,stats,rows", DS_CASES,
                         ids=[f"C{c[0]}_N{c[1]}_M{c[2]}_nb{c[3]}_" + ("_".join(f"{k}{int(v)}" for k, v in c[4].items()) or "default")
                              for c in DS_CASES])
def test_downsample_token_branch_vs_oracle(C, N, M, nb, switches, stats, rows):
    """One DownSampleToken layer (B = 2) on each of its branches against O.downsample_token: a calibrating forward then
    a frozen one, asserting what test_blocks_vs_oracle asserts (boundaries, token logits, the fp64-adjudicated decision
    with 0 unexplained flips / swaps, x_ds rows of identically chosen points)."""
    B = 2
    ds, sd = filled(blocks.DownSampleToken(Cfg(_downsample([M], nb, "topk", C=C)), 0), seed=C + N, sharpen=4.0)
    x = synthetic_features(B, C, N, C * 7 + N)
    st = O.DSState(True)
    restore = [_switch(blocks if name == "DS_EXACT" else ops, name, v) for name, v in switches.items()]
    try:
        with torch.no_grad():
            for it in range(2):
                ((x_ds, idx), _), k = launched(lambda: ds(cu(x)))
                _check_ds_branch(k, C, stats, rows)
                ref = O.downsample_token(sd, "", x, M, 32, nb, st)
                torch.testing.assert_close(ds.bin_boundaries[0].cpu(), ref["boundaries"][0], rtol=1e-5, atol=1e-6)
                assert tuple(ds.bin_points_mask.shape) == tuple(ref["mask"].shape) and ds.bin_points_mask.dtype == torch.bool
                assert close_frac(ds.attention_bins_beforesoftmax, ref["token_logits"]) == 1.0
                s64, amp, _ = amp_excusing_knn_ties(x, sd, "")
                big = s64 > 1e-30                                 # (below that the fp32 probabilities underflow)
                rel = float(((ds.attention_point_score.cpu().double()[:, 0] - s64).abs()[big] / s64[big]).max())
                print(f"DownSampleToken C={C} N={N} {stats}/{rows}: max rel score error vs fp64 {rel:.2e}")
                if stats == "exact":
                    assert rel <= 2e-5, rel
                judge_against_reference_scores(ds, idx, x_ds, ref["score"], ref["idx"], ref["k"], ref["x_ds"], amp,
                                               max_flip_groups=max(8, 3 * (nb - 1)) if stats == "exact" else None)
                ds.dynamic_boundaries_enable, st.dynamic = False, False
    finally:
        for r in restore:
            r()


# ---------------------------------------------------------------- Neighbor2PointAttention

N2P_CASES = [  # C, heads, K, FUSED_MLP2
    (64, 4, 32, True),           # mlp2 not eligible at an output width of 64: two `linear` launches
    (32, 2, 16, True),
    (128, 8, 20, True),
    (128, 1, 32, True),
    (128, 4, 32, False),
]


@pytest.mark.parametrize("N", [300, 1024])
@pytest.mark.parametrize("C,H,K,fused", N2P_CASES, ids=[f"C{c[0]}_H{c[1]}_K{c[2]}_mlp2{int(c[3])}" for c in N2P_CASES])
def test_n2p_attention_branch_vs_oracle(C, H, K, fused, N):
    att, sd = filled(blocks.Neighbor2PointAttention(Cfg(_attention(1, C=C, K=K, heads=H)), 0), seed=C + H + K)
    x = synthetic_features(2, C, N, C + N)
    restore = _switch(ops, "FUSED_MLP2", fused)
    try:
        with torch.no_grad():
            y, k = launched(lambda: att(cu(x)))
    finally:
        restore()
    mlp2 = fused and ops.mlp2_eligible(C, 4 * C, C)
    assert ("mlp2_kernel" in k) == mlp2, sorted(k)
    assert k.get("linear_tma_kernel", 0) == (1 if mlp2 else 3), k          # [q|k|v] (+ the two feed-forward layers)
    eight = C == 128 and H == 4
    assert ("n2p_attend8_kernel" in k) == eight and ("n2p_attend_kernel" in k) == (not eight), sorted(k)
    assert close_frac(y, O.n2p_attention(sd, "", x, K, H)) >= 0.9995


# ---------------------------------------------------------------- EdgeConv

EDGE_CASES = [  # Cin, C1, C2, K, group_type, normal_channel, kernel (None: group + ATen convolutions), out_rows slice
    (3, 64, 128, 32, "center_diff", False, "edge_mlp_tc_kernel", True),
    (16, 48, 64, 32, "center_neighbor", False, "edge_mlp_max_kernel", False),
    (64, 64, 32, 16, "diff", False, "edge_mlp_max_kernel", False),
    (6, 64, 64, 20, "neighbor", True, "edge_mlp_tc_kernel", False),
    (8, 64, 96, 16, "center_diff", False, None, True),             # C2 = 96
    (8, 30, 64, 16, "diff", False, None, False),                   # C1 = 30
]


def _edgeconv(Cin, C1, C2, K, gt, normal):
    cin_t = 2 * Cin if gt.startswith("center") else Cin
    cfg = Cfg(K=[K], group_type=[gt], normal_channel=normal, conv1_in=[cin_t], conv1_out=[C1], conv2_in=[C1], conv2_out=[C2])
    return filled(blocks.EdgeConv(cfg, 0), seed=Cin + C1 + C2 + K)


@pytest.mark.parametrize("Cin,C1,C2,K,gt,normal,kernel,slot", EDGE_CASES,
                         ids=[f"{c[0]}-{c[1]}-{c[2]}_K{c[3]}_{c[4]}" + ("_normal" if c[5] else "") for c in EDGE_CASES])
def test_edgeconv_branch_vs_oracle(Cin, C1, C2, K, gt, normal, kernel, slot):
    """EdgeConv against O.group -> O._cbl -> O._cbl -> max (models/embedding.py:29-39).  With `slot` the result is written
    into a column slice of a wider NaN-filled row buffer (the concatenated embedding of seg_model.py:98-102)."""
    B, N = 2, 512
    ec, sd = _edgeconv(Cin, C1, C2, K, gt, normal)
    x = synthetic_features(B, Cin, N, Cin + K)
    buf = torch.full((B, N, C2 + 40), float("nan"), device=DEV) if slot else None
    out_rows = buf[..., 8:8 + C2] if slot else None
    with torch.no_grad():
        y, k = launched(lambda: ec(cu(x), out_rows=out_rows))
    fused = {"edge_mlp_tc_kernel", "edge_mlp_max_kernel"}
    assert fused & set(k) == ({kernel} if kernel else set()), sorted(k)
    if kernel is None:
        assert "group_rows_kernel" in k or "group_center_kernel" in k, sorted(k)
    g, _ = O.group(x, K, gt, normal_channel=normal)
    ref = O._cbl(sd, "conv2", O._cbl(sd, "conv1", g)).max(dim=-1)[0]
    assert close_frac(y, ref) >= 0.9995
    if slot:
        assert torch.equal(out_rows.transpose(1, 2), y)
        assert bool(buf[..., :8].isnan().all()) and bool(buf[..., 8 + C2:].isnan().all()), "wrote outside its columns"


def test_edgeconv_more_than_32_neighbours_is_refused():
    """K > 32 sends EdgeConv to its unfused branch, whose neighbour search is the native kNN: that kernel keeps at most
    32 neighbours and refuses more instead of returning a different grouping."""
    ec, _ = _edgeconv(8, 64, 64, 40, "center_diff", False)
    with torch.no_grad(), pytest.raises(ValueError, match=r"k=40 outside \[1,32\]"):
        ec(cu(synthetic_features(1, 8, 256, 3)))


# ---------------------------------------------------------------- UpSampleInterpolation

UP_CASES = [  # B, N, M, q_in, v_out, branch
    (2, 4096, 2049, 128, 128, "rows"),            # the search's second 2048-candidate chunk
    (1, 8192, 4100, 128, 128, "rows"),            # seg at N = 8192 upsamples from M = 4096 and more
    (2, 1024, 512, 128, 50, "channels"),          # feature rows of 50 floats: not 16-byte chunks
    (2, 1024, 512, 30, 64, "rows"),               # an input width that is not a multiple of 4 does not matter
]


@pytest.mark.parametrize("B,N,M,q_in,v_out,branch", UP_CASES, ids=[f"N{c[1]}_M{c[2]}_{c[3]}to{c[4]}" for c in UP_CASES])
def test_upsample_interpolation_branch_vs_oracle(B, N, M, q_in, v_out, branch):
    cfg = Cfg(interpolation=dict(distance_type=["xyz"], K=[3]), q_in=[q_in], v_out=[v_out])
    up, sd = filled(blocks.UpSampleInterpolation(cfg, 0), seed=q_in + v_out)
    pcd_up, sel = synthetic_features(B, v_out, N, N + 1), synthetic_features(B, q_in, M, M + 2)
    xyz_up, xyz_sel = synthetic_features(B, 3, N, N + 3), synthetic_features(B, 3, M, M + 4)
    with torch.no_grad():
        y, k = launched(lambda: up(cu(pcd_up), ((cu(sel), None, cu(xyz_sel)), (None, None)), cu(xyz_up)))
    assert "interpolate3_kernel" in k and ("interp3_rows_kernel" in k) == (branch == "rows"), sorted(k)
    assert close_frac(y, O.upsample_interpolation(sd, "", pcd_up, sel, xyz_up, xyz_sel, 3)) == 1.0
