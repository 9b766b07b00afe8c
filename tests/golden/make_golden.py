"""Mint golden vectors from the UNMODIFIED reference.

    SAMBLE_REFERENCE=<checkout of upstream SAMBLE> python tests/golden/make_golden.py

The reference ships no tests or known-answer files (SURVEY 4), so the fixtures
that pin the oracle are outputs of the reference itself, imported from
the SAMBLE_REFERENCE checkout and run on CPU in eval()/no_grad with
  * inputs from samble_b200.testing.synthetic_clouds / synthetic_features (seeded),
  * weights from samble_b200.testing.fill_state_dict_ (a pure function of the entry
    name and a seed, so no weights need to be stored),
  * sample_mode 'topk', boundaries calibrated on the first call then frozen
    (SURVEY 8c protocol).
Only OUTPUTS are stored (inputs regenerate from their seeds); files stay < 1 MB.
"""
from __future__ import annotations

import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from samble_b200.config import cls_config, seg_config  # noqa: E402
from samble_b200.testing import fill_state_dict_, synthetic_clouds, synthetic_features  # noqa: E402
from tests.golden import ref_loader as R  # noqa: E402

# ---- the cases; tests/test_oracle_golden.py reads these same tables ----
KNN_CASES = [  # (name, B, Nq, Nr, C, k, seed)
    ("xyz_self", 2, 96, 96, 3, 8, 11),
    ("xyz_cross", 2, 80, 40, 3, 3, 12),
    ("feat64_self", 2, 64, 64, 64, 16, 13),
    ("feat128_self", 1, 160, 160, 128, 32, 14),
    ("tiny_exact_path", 1, 20, 20, 3, 4, 15),       # <=25 rows: cdist's non-GEMM path
]
GROUP_CASES = [  # (name, B, C, N, K, seed)
    ("c3", 2, 3, 64, 8, 21),
    ("c64", 1, 64, 48, 16, 22),
]
KALLOC_CASES = [  # (name, B, nb, M, N, seed)
    ("nb4", 64, 4, 128, 256, 31),
    ("nb6", 64, 6, 96, 256, 32),
    ("nb4_sat", 64, 4, 200, 256, 33),
]
MODEL_CASES = dict(seg=dict(B=2, N=256, M=(128, 64), wseed=1, xseed=2),
                   cls=dict(B=2, N=256, M=(128, 64), wseed=3, xseed=4))
BLOCK_N = 128


def kalloc_inputs(B, nb, M, N, seed):
    g = torch.Generator().manual_seed(seed)
    w = torch.relu(torch.randn(B, nb, generator=g))
    w[::7] = 0.0                                                  # all-zero weight rows
    cuts = torch.sort(torch.rand(B, nb - 1, generator=g), dim=1)[0]
    edges = torch.cat([torch.zeros(B, 1), cuts, torch.ones(B, 1)], 1)
    cnt = ((edges[:, 1:] - edges[:, :-1]) * N).long()
    cnt[:, -1] += N - cnt.sum(1)
    return w, cnt


def main() -> None:
    torch.set_num_threads(max(1, (os.cpu_count() or 2) // 2))
    ops, embedding, attention, downsample, upsample, seg_model, cls_model = R.modules()
    out_ops: dict = {}
    with torch.no_grad():
        for name, B, Nq, Nr, C, k, seed in KNN_CASES:
            a = synthetic_features(B, Nq, C, seed)                # (B,Nq,C)
            b = a if name.endswith("self") or name.startswith("tiny") else synthetic_features(B, Nr, C, seed + 100)
            d, i = ops.knn(a, b, k)
            out_ops[f"knn.{name}.dist"], out_ops[f"knn.{name}.idx"] = d.numpy(), i.numpy()
        for name, B, C, N, K, seed in GROUP_CASES:
            x = synthetic_features(B, C, N, seed)
            for gt in ("neighbor", "diff", "center_neighbor", "center_diff"):
                g, i = ops.group(x, K, gt)
                out_ops[f"group.{name}.{gt}"] = g.contiguous().numpy()
            out_ops[f"group.{name}.idx"] = i.numpy()
            out_ops[f"mask.{name}"] = np.packbits(ops.neighbor_mask(x, K).numpy().astype(bool), axis=-1)
            sel = torch.stack([torch.randperm(N, generator=torch.Generator().manual_seed(seed + b))[: N // 2]
                               for b in range(B)]).unsqueeze(1)
            out_ops[f"gather.{name}"] = ops.gather_by_idx(x, sel).numpy()
        # three-NN interpolation neighbours
        unk, kn = synthetic_features(2, 3, 96, 41), synthetic_features(2, 3, 40, 42)
        feat = synthetic_features(2, 16, 40, 43)
        nbr, i, d = ops.select_neighbors_interpolate(unk, kn, feat, 3)
        out_ops["interp.nbr"], out_ops["interp.idx"], out_ops["interp.d"] = nbr.contiguous().numpy(), i.numpy(), d.numpy()
        # water-filling k allocation
        for name, B, nb, M, N, seed in KALLOC_CASES:
            w, cnt = kalloc_inputs(B, nb, M, N, seed)
            out_ops[f"kalloc.{name}"] = ops.calculate_num_points_to_choose(w, cnt, M).numpy()
        # bin partition (static + dynamic) and per-bin top-k
        score = torch.rand(3, 1, 200, generator=torch.Generator().manual_seed(51)) * 1e-3
        bnd, mask = ops.bin_partition(score, None, True, 0.99, 4)
        out_ops["bin.dyn_init.upper"], out_ops["bin.dyn_init.mask"] = bnd[0].numpy(), mask.numpy()
        score2 = torch.rand(3, 1, 200, generator=torch.Generator().manual_seed(52)) * 1e-3
        bnd2, mask2 = ops.bin_partition(score2, [t.clone() for t in bnd], True, 0.99, 4)
        out_ops["bin.dyn_ema.upper"], out_ops["bin.dyn_ema.mask"] = bnd2[0].numpy(), mask2.numpy()
        _, mask3 = ops.bin_partition(score2, bnd, False, 0.99, 4)
        out_ops["bin.static.mask"] = mask3.numpy()
        cnt = mask3.squeeze(1).sum(1)
        w = torch.rand(3, 4, generator=torch.Generator().manual_seed(53))
        kk = ops.calculate_num_points_to_choose(w, cnt, 100)
        out_ops["bin.static.k"] = kk.numpy()
        out_ops["bin.static.idx"] = ops.generating_downsampled_index(100, score2, mask3, "topk", 0.1, kk).numpy()
    np.savez_compressed(os.path.join(HERE, "ops_small.npz"), **out_ops)

    # ---- blocks, pulled out of a filled reference seg model ----
    out_blk: dict = {}
    rcfg = R.reference_config("seg")
    rcfg.feature_learning_block.downsample.M = [BLOCK_N // 2, BLOCK_N // 4]
    rcfg.feature_learning_block.downsample.bin.sample_mode = ["topk", "topk"]
    m = R.build_model("seg", rcfg).eval()
    m.load_state_dict(fill_state_dict_(m.state_dict(), seed=5, sharpen=4.0))
    with torch.no_grad():
        x3, x128 = synthetic_features(2, 3, BLOCK_N, 61), synthetic_features(2, 128, BLOCK_N, 62)
        out_blk["edgeconv0"] = m.block.embedding_list[0](x3).numpy()
        out_blk["edgeconv1"] = m.block.embedding_list[1](synthetic_features(2, 64, BLOCK_N, 63)).numpy()
        out_blk["n2p0"] = m.block.feature_learning_layer_list[0](x128).numpy()
        ds = m.block.downsample_list[0]
        for tag in ("calib", "frozen"):
            (x_ds, idx), _ = ds(x128)
            out_blk[f"ds0.{tag}.x_ds"], out_blk[f"ds0.{tag}.idx"] = x_ds.numpy(), idx.numpy()
            out_blk[f"ds0.{tag}.score"] = ds.attention_point_score.numpy()
            out_blk[f"ds0.{tag}.k"] = ds.k_point_to_choose.numpy()
            out_blk[f"ds0.{tag}.w"] = ds.bin_weights_beforerelu.numpy()
            out_blk[f"ds0.{tag}.upper"] = ds.bin_boundaries[0].numpy().copy()
            ds.dynamic_boundaries_enable = False
        xyz_up, xyz_dn = synthetic_features(2, 3, BLOCK_N, 64), synthetic_features(2, 3, BLOCK_N // 2, 65)
        dn = synthetic_features(2, 128, BLOCK_N // 2, 66)
        out_blk["upsample0"] = m.block.upsample_list[0](x128, ((dn, None, xyz_dn), (None, None)), xyz_up).numpy()
    np.savez_compressed(os.path.join(HERE, "blocks_small.npz"), **out_blk)

    # ---- whole models ----
    for which, c in MODEL_CASES.items():
        rcfg = R.reference_config(which)
        rcfg.feature_learning_block.downsample.M = list(c["M"])
        rcfg.feature_learning_block.downsample.bin.sample_mode = ["topk", "topk"]
        m = R.build_model(which, rcfg).eval()
        m.load_state_dict(fill_state_dict_(m.state_dict(), seed=c["wseed"], sharpen=4.0))
        x, cat = synthetic_clouds(c["B"], c["N"], c["xseed"])
        out: dict = {}
        with torch.no_grad():
            for tag in ("calib", "frozen"):
                y = m(x, cat) if which == "seg" else m(x)
                out[f"{tag}.logits"] = y.numpy()
                for i, ds in enumerate(m.block.downsample_list):
                    out[f"{tag}.ds{i}.idx"] = ds.idx.numpy()
                    out[f"{tag}.ds{i}.k"] = ds.k_point_to_choose.numpy()
                    out[f"{tag}.ds{i}.upper"] = ds.bin_boundaries[0].numpy().copy()
                    ds.dynamic_boundaries_enable = False
        np.savez_compressed(os.path.join(HERE, f"{which}_small.npz"), **out)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")


if __name__ == "__main__":
    main()
