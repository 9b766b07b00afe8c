"""Live pin of the oracle (and of our config / state_dict mirrors) against the UNMODIFIED reference.
Runs only where SAMBLE_REFERENCE names a checkout of upstream SAMBLE; skipped otherwise (tests/test_oracle_golden.py
keeps the oracle pinned to the reference's stored outputs)."""
import pytest
import torch

from oracle import samble_oracle as O
from samble_b200 import models
from samble_b200.config import cls_config, seg_config
from samble_b200.testing import fill_state_dict_, synthetic_clouds
from tests.golden import ref_loader as R

pytestmark = pytest.mark.needs_reference


@pytest.mark.parametrize("which", ["seg", "cls"])
def test_full_forward_bit_exact(which):
    M = (96, 48)
    rcfg = R.reference_config(which)
    rcfg.feature_learning_block.downsample.M = list(M)
    rcfg.feature_learning_block.downsample.bin.sample_mode = ["topk", "topk"]
    ref = R.build_model(which, rcfg).eval()
    sd = fill_state_dict_(ref.state_dict(), seed=11, sharpen=8.0)
    ref.load_state_dict(sd)
    cfg = (seg_config if which == "seg" else cls_config)(M=M)
    x, cat = synthetic_clouds(3, 192, seed=12)
    states = [O.DSState(True), O.DSState(True)]
    with torch.no_grad():
        for it in range(3):
            if it == 2:                              # freeze after two EMA steps
                for ds in ref.block.downsample_list:
                    ds.dynamic_boundaries_enable = False
                for s in states:
                    s.dynamic = False
            rec = {}
            yr = ref(x, cat) if which == "seg" else ref(x)
            yo = O.seg_forward(sd, cfg, x, cat, states, rec) if which == "seg" else O.cls_forward(sd, cfg, x, states, rec)
            assert torch.equal(yr, yo)
            for i, ds in enumerate(ref.block.downsample_list):
                assert torch.equal(ds.idx, rec[f"ds{i}"]["idx"])
                assert torch.equal(ds.k_point_to_choose, rec[f"ds{i}"]["k"])
                assert torch.equal(ds.attention_point_score, rec[f"ds{i}"]["score"])
                assert torch.equal(ds.bin_points_mask, rec[f"ds{i}"]["mask"])


def test_config_and_state_dict_mirrors():
    for which, mine_cfg, cls_ in (("seg", seg_config(sample_mode="random"), models.ShapeNetModel),
                                  ("cls", cls_config(M=(1024, 512), sample_mode="random"), models.ModelNetModel)):
        rcfg = R.reference_config(which)
        ref = R.build_model(which, rcfg)
        mine = cls_(mine_cfg)
        a = {k: tuple(v.shape) for k, v in ref.state_dict().items()}
        b = {k: tuple(v.shape) for k, v in mine.state_dict().items()}
        assert a == b and list(a) == list(b)
        mine.load_state_dict(ref.state_dict())       # a reference checkpoint loads as is
        rf, mf = rcfg.feature_learning_block, mine_cfg.feature_learning_block
        for blk in ("embedding", "downsample", "attention") + (("upsample",) if which == "seg" else ()):
            for key, val in mf[blk].items():
                if key in ("bin",):
                    for k2, v2 in val.items():
                        if k2 != "bin_boundaries":
                            assert rf[blk][key][k2] == v2, (blk, key, k2)
                elif key != "asm" or blk != "attention":
                    assert rf[blk][key] == val, (blk, key)


def test_patch_swaps_the_reference_entry_points():
    from samble_b200 import blocks, ops, patch

    ref_ops, embedding, attention, downsample, upsample, _, _ = R.modules()
    with patch.installed():
        assert ref_ops.group is ops.group and ref_ops.knn is ops.knn
        assert downsample.bin_partition is ops.bin_partition          # bound by name at import (downsample.py:8-12)
        assert downsample.DownSampleToken is blocks.DownSampleToken
        assert attention.Neighbor2PointAttention is blocks.Neighbor2PointAttention
        assert embedding.EdgeConv is blocks.EdgeConv and upsample.UpSampleInterpolation is blocks.UpSampleInterpolation
        m = R.build_model("seg", R.reference_config("seg"))          # reference wiring builds OUR blocks
        assert isinstance(m.block.downsample_list[0], blocks.DownSampleToken)
    assert ref_ops.group is not ops.group and downsample.DownSampleToken is not blocks.DownSampleToken


@pytest.mark.parametrize("mode,bt", [("uniform", 0.1), ("random", 0.1), ("random", "mode_1"), ("random", "mode_3"), ("random", 0.05)])
def test_stochastic_sampling_modes_match_the_reference_under_the_same_rng(mode, bt):
    """utils/ops.py:507-613: with the CPU generator in the same state the oracle draws the reference's indices, which
    pins its sampling distributions bit for bit (torch.multinomial consumes them directly)."""
    import torch

    from oracle import samble_oracle as O

    ref_ops = R.modules()[0]
    g = torch.Generator().manual_seed(11)
    B, N, nb, M = 3, 256, 4, 96
    score = torch.rand(B, 1, N, generator=g) * 1e-3
    bins = torch.randint(0, nb, (B, 1, N, 1), generator=g)
    mask = bins == torch.arange(nb).view(1, 1, 1, nb)
    k = O.calculate_num_points_to_choose(torch.rand(B, nb, generator=g), mask.squeeze(1).sum(1), M)
    torch.manual_seed(5)
    want = ref_ops.generating_downsampled_index(M, score.clone(), mask, mode, bt, k)
    torch.manual_seed(5)
    got = O.generating_downsampled_index(M, score.clone(), mask, mode, bt, k)
    assert torch.equal(want, got)

