"""GPU parity of the L0 ops (utils/ops.py drop-ins) against the CPU oracle, through the C ABI.
Integer/index outputs: bit-exact up to provable fp32 near-ties (tie-aware comparators, SURVEY 8c);
float outputs: stated tolerance."""
import os

import numpy as np
import pytest
import torch

from oracle import samble_oracle as O
from samble_b200 import ops
from samble_b200.testing import knn_parity, sampled_index_parity, synthetic_clouds, synthetic_features
from tests.golden import make_golden as G

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def cu(t):
    return t.to(DEV)


# ---------------------------------------------------------------- kNN

KNN_SHAPES = [  # (B, Nq, Nr, C, k, seed)   Nr == 0 -> self
    (4, 512, 0, 3, 32, 1),
    (2, 2048, 0, 3, 32, 2),          # BASELINE seg size, xyz
    (3, 333, 0, 3, 7, 3),            # ragged, small k
    (2, 300, 150, 3, 3, 4),          # cross (upsample shape)
    (2, 2048, 1024, 3, 3, 5),
    (1, 40, 0, 3, 32, 6),            # k close to N
    (2, 512, 0, 64, 32, 7),
    (2, 2048, 0, 128, 32, 8),        # BASELINE seg size, features
    (2, 1000, 0, 128, 32, 9),        # ragged
    (1, 700, 260, 20, 5, 10),        # odd channel count, cross
    (1, 8192, 0, 3, 32, 11),         # BASELINE config 4
    (1, 8192, 0, 128, 32, 12),
    (2, 64, 0, 6, 16, 13),
    (1, 3000, 0, 3, 1, 14),          # candidate chunking (> 2048) and k = 1
    (1, 16384, 0, 3, 32, 15),        # BASELINE config 4, largest size
    (1, 16384, 0, 128, 32, 16),
]


@pytest.mark.parametrize("shape", KNN_SHAPES, ids=[f"B{s[0]}_N{s[1]}x{s[2] or s[1]}_C{s[3]}_k{s[4]}" for s in KNN_SHAPES])
def test_knn_vs_oracle(shape):
    B, Nq, Nr, C, k, seed = shape
    a = synthetic_features(B, Nq, C, seed)                     # point-major (B,N,C) like ops.knn takes
    if C == 3:
        a = a * 0.3 + torch.tensor([0.5, -1.0, 2.0])          # off-centre: exercises the normalisation
    b = a if Nr == 0 else synthetic_features(B, Nr, C, seed + 100)
    d_ref, i_ref = O.knn(a, b, k)
    d, i = ops.knn(cu(a), cu(b), k)
    assert i.dtype == torch.int64 and tuple(i.shape) == (B, Nq, k)
    rep = knn_parity(i, i_ref, a, b)
    assert rep["unexplained_rows"] == 0, rep
    assert rep["exact_rate"] >= 0.995, rep
    # distances: fp32 GEMM-form cancellation noise is ~1e-3 absolute at d=0 (SURVEY 7 hard part 2)
    same = (i.cpu() == i_ref)
    err = (d.cpu() - d_ref).abs()[same]
    assert float(err.max()) < (5e-3 if C <= 3 else 3e-2), float(err.max())
    assert float(err.mean()) < 1e-4


def test_knn_channel_major_int32_path_matches_int64_path():
    x = synthetic_features(2, 128, 777, 21)                    # (B,C,N)
    i32 = ops.knn_indices(cu(x), 32)
    _, i64 = ops.knn(cu(x).transpose(1, 2), cu(x).transpose(1, 2), 32)
    assert i32.dtype == torch.int32 and torch.equal(i32.long(), i64)


def test_knn_duplicate_points_and_errors():
    a = synthetic_features(1, 100, 3, 22)
    a[0, 50:] = a[0, :50]                                      # every point has an exact duplicate
    _, i = ops.knn(cu(a), cu(a), 4)
    i = i.cpu()
    d = torch.cdist(a.double(), a.double())[0]
    for q in range(100):                                       # distance-0 pair first, lower index first
        assert set(i[0, q, :2].tolist()) == {q % 50, q % 50 + 50} and i[0, q, 0] < i[0, q, 1]
        assert torch.all(d[q, i[0, q]][1:] >= d[q, i[0, q]][:-1] - 1e-6)
    with pytest.raises(RuntimeError):
        ops.knn(cu(a), cu(a), 101)                             # torch.topk raises too
    with pytest.raises(ValueError):
        ops.knn(cu(a), cu(a), 33)                              # documented limit of the native path


@pytest.mark.parametrize("case", G.KNN_CASES, ids=[c[0] for c in G.KNN_CASES])
def test_knn_golden(case):
    name, B, Nq, Nr, C, k, seed = case
    gold = np.load(os.path.join(GOLD, "ops_small.npz"))
    a = synthetic_features(B, Nq, C, seed)
    b = a if name.endswith("self") or name.startswith("tiny") else synthetic_features(B, Nr, C, seed + 100)
    d, i = ops.knn(cu(a), cu(b), k)
    rep = knn_parity(i, torch.from_numpy(gold[f"knn.{name}.idx"]), a, b)
    assert rep["unexplained_rows"] == 0 and rep["exact_rate"] >= 0.99, rep


# ---------------------------------------------------------------- gathers / grouping


@pytest.mark.parametrize("B,C,N,K", [(2, 3, 512, 32), (2, 64, 300, 16), (1, 128, 1024, 32), (1, 6, 100, 8)])
def test_group_all_types(B, C, N, K):
    x = synthetic_features(B, C, N, 31)
    xg = cu(x)
    for gt in ("neighbor", "diff", "center_neighbor", "center_diff"):
        g, idx = ops.group(xg, K, gt)
        g_ref, idx_ref = O.group(x, K, gt)
        assert tuple(g.shape) == tuple(g_ref.shape) and g.stride() == g_ref.stride()      # same view layout
        rep = knn_parity(idx, idx_ref, x.transpose(1, 2), x.transpose(1, 2))
        assert rep["unexplained_rows"] == 0 and rep["exact_rate"] >= 0.995, rep
        # teacher-forced: the gather itself must be exact given OUR indices
        pts = x.transpose(1, 2)
        nbr = O.index_points(pts, idx.cpu())
        if gt.endswith("diff"):
            nbr = nbr - pts.unsqueeze(2)
        exp = nbr.permute(0, 3, 1, 2)
        if gt.startswith("center"):
            exp = torch.cat([x.unsqueeze(-1).repeat(1, 1, 1, K), exp], dim=1)
        assert torch.equal(g.cpu(), exp)
    with pytest.raises(ValueError):
        ops.group(xg, K, "nope")
    if C == 6:
        _, i_n = ops.group(xg, K, "neighbor", normal_channel=True)
        _, i_ref = O.group(x, K, "neighbor", normal_channel=True)
        assert knn_parity(i_n, i_ref, x[:, :3].transpose(1, 2), x[:, :3].transpose(1, 2))["unexplained_rows"] == 0


def test_index_points_gather_mask():
    B, N, C, M, K = 2, 500, 128, 77, 5
    pts = synthetic_features(B, N, C, 41)
    idx = torch.randint(0, N, (B, M, K), generator=torch.Generator().manual_seed(42))
    assert torch.equal(ops.index_points(cu(pts), cu(idx)).cpu(), O.index_points(pts, idx))
    pts3 = synthetic_features(B, N, 3, 43)                                        # non-float4 rows
    assert torch.equal(ops.index_points(cu(pts3), cu(idx)).cpu(), O.index_points(pts3, idx))
    pcd = synthetic_features(B, 3, N, 44)
    sel = torch.stack([torch.randperm(N, generator=torch.Generator().manual_seed(45 + b))[:200] for b in range(B)]).unsqueeze(1)
    assert torch.equal(ops.gather_by_idx(cu(pcd), cu(sel)).cpu(), O.gather_by_idx(pcd, sel))
    x = synthetic_features(B, 16, 300, 46)
    m, m_ref = ops.neighbor_mask(cu(x), 8).cpu(), O.neighbor_mask(x, 8)
    assert m.dtype == torch.float32 and float(m.sum()) == B * 300 * 8
    assert float((m != m_ref).float().mean()) < 1e-4


def test_select_neighbors_interpolate():
    unk, kn, feat = synthetic_features(2, 3, 400, 51), synthetic_features(2, 3, 150, 52), synthetic_features(2, 32, 150, 53)
    nbr, idx, d = ops.select_neighbors_interpolate(cu(unk), cu(kn), cu(feat), 3)
    nbr_r, idx_r, d_r = O.select_neighbors_interpolate(unk, kn, feat, 3)
    assert torch.equal(idx.cpu(), idx_r) and nbr.stride() == nbr_r.stride()
    assert torch.equal(nbr.cpu(), nbr_r)
    torch.testing.assert_close(d.cpu(), d_r, atol=1e-4, rtol=1e-5)
    out, idx3, d3 = ops.interpolate3(cu(unk), cu(kn), cu(feat), want_idx=True)
    assert torch.equal(idx3.cpu(), idx_r)
    w = 1.0 / (d_r + 1e-8)
    w = w / w.sum(-1, keepdim=True)
    torch.testing.assert_close(out.cpu(), (nbr_r * w.unsqueeze(1)).sum(-1), atol=2e-5, rtol=1e-4)


# ---------------------------------------------------------------- bins, k per bin, per-bin top-k


@pytest.mark.parametrize("case", G.KALLOC_CASES + [("nb5", 512, 5, 300, 1024, 7), ("nb8", 300, 8, 700, 2048, 8)],
                         ids=lambda c: c[0])
def test_num_points_to_choose(case):
    name, B, nb, M, N, seed = case
    w, cnt = G.kalloc_inputs(B, nb, M, N, seed)
    k = ops.calculate_num_points_to_choose(cu(w), cu(cnt), M)
    assert k.dtype == torch.int32
    assert torch.equal(k.cpu(), O.calculate_num_points_to_choose(w, cnt, M))



def _assert_only_cut_ties_flip(score, mask, mask_ref, bnd):
    """mask/mask_ref (B,1,N,nb) bool; bnd the [upper, lower] pair both used.  Points whose membership differs must have a
    reference z-score within 8 fp32 roundings (of the z computation's magnitude) of a cut."""
    z = (score - score.mean(dim=2, keepdim=True)) / score.std(dim=2, unbiased=False, keepdim=True)      # the reference's fp32 z
    cuts = bnd[0].reshape(-1)[1:]
    flipped = (mask != mask_ref).any(-1)[:, 0]                                   # (B,N)
    mag = z.abs()[:, 0] + (score.mean(dim=2, keepdim=True) / score.std(dim=2, unbiased=False, keepdim=True)).abs()[:, 0] + 1
    dist = (z[:, 0].unsqueeze(-1) - cuts).abs().min(-1)[0]
    assert bool((dist[flipped] <= 8 * 2.0 ** -24 * mag[flipped]).all()), float((dist[flipped] / mag[flipped]).max())
    for b in range(score.shape[0]):
        assert len(set(z[b, 0][flipped[b]].tolist())) <= cuts.numel(), "more than one tie group per cut flipped"


@pytest.mark.parametrize("N,nb,M", [(200, 4, 100), (2048, 4, 1024), (1024, 6, 512), (777, 6, 300), (8192, 4, 4096), (16384, 4, 8192)])
def test_bin_partition_and_topk_ops(N, nb, M):
    B = 3
    g = torch.Generator().manual_seed(N + nb)
    score = torch.rand(B, 1, N, generator=g) * 1e-3
    score[:, :, ::17] = score[:, :, 5:6]                       # exact score ties across the cloud
    bnd_ref, mask_ref = O.bin_partition(score, None, True, 0.99, nb)          # dynamic init
    bnd, mask = ops.bin_partition(cu(score), None, True, 0.99, nb)
    torch.testing.assert_close(bnd[0].cpu(), bnd_ref[0], rtol=2e-6, atol=1e-6)
    torch.testing.assert_close(bnd[1].cpu(), bnd_ref[1], rtol=2e-6, atol=1e-6)           # [upper, lower], +-inf sentinels included
    # a dynamic cut IS some point's z (ops.py:189), so points tied with it flip on a last-ulp difference of z (ours comes
    # from an fp64 mean / std, the reference's from fp32 ones): every flipped point must sit within a few roundings
    # of a cut, and only whole tie groups may flip (at most one distinct z per cut and cloud)
    _assert_only_cut_ties_flip(score, mask.cpu(), mask_ref, bnd_ref)
    # static partition with the REFERENCE boundaries, EMA step, then k allocation and per-bin top-k
    _, mask_s = ops.bin_partition(cu(score), [t.clone() for t in bnd_ref], False, 0.99, nb)
    _, mask_s_ref = O.bin_partition(score, bnd_ref, False, 0.99, nb)
    assert mask_s.dtype == torch.bool
    _assert_only_cut_ties_flip(score, mask_s.cpu(), mask_s_ref, bnd_ref)
    bnd2_ref, _ = O.bin_partition(score * 1.1, [t.clone() for t in bnd_ref], True, 0.99, nb)
    bnd2, _ = ops.bin_partition(cu(score * 1.1), [t.clone() for t in bnd_ref], True, 0.99, nb)
    torch.testing.assert_close(bnd2[0].cpu(), bnd2_ref[0], rtol=2e-6, atol=1e-6)
    torch.testing.assert_close(bnd2[1].cpu(), bnd2_ref[1], rtol=2e-6, atol=1e-6)
    w = torch.rand(B, nb, generator=g)
    cnt = mask_s_ref.squeeze(1).sum(1)
    kk = O.calculate_num_points_to_choose(w, cnt, M)
    idx_ref = O.generating_downsampled_index(M, score, mask_s_ref, "topk", 0.1, kk)
    idx = ops.generating_downsampled_index(M, cu(score), cu(mask_s_ref), "topk", 0.1, cu(kk))
    assert idx.dtype == torch.int64 and tuple(idx.shape) == (B, 1, M)
    # torch.sort's order among EQUAL scores is implementation-defined (unstable by default, probed on
    # CPU); ours is "lower index first".  Everything outside exact-tie groups must be identical.
    rep = sampled_index_parity(idx, idx_ref, score, kk)
    assert rep["unexplained_bins"] == 0 and rep["exact_rate"] > 0.5, rep
    score_nt = torch.rand(B, 1, N, generator=g) * 1e-3                          # no ties: bit-exact
    idx_nt = ops.generating_downsampled_index(M, cu(score_nt), cu(mask_s_ref), "topk", 0.1, cu(kk))
    idx_nt_ref = O.generating_downsampled_index(M, score_nt, mask_s_ref, "topk", 0.1, kk)
    if N < 8192:
        assert torch.equal(idx_nt.cpu(), idx_nt_ref)
    else:                                      # 2^24 distinct random floats: a few collide among >= 8192 draws
        rep = sampled_index_parity(idx_nt, idx_nt_ref, score_nt, kk)
        assert rep["unexplained_bins"] == 0 and rep["exact_rate"] > 0.999, rep
    # stochastic modes: same distributions as the oracle; draws come from the right bin, distinct, k per bin
    for mode, bt in (("uniform", 0.1), ("random", 0.1), ("random", "mode_1"), ("random", "mode_2")):
        p = ops.sampling_probabilities(cu(score), cu(mask_s_ref), mode, bt)
        torch.testing.assert_close(p.cpu(), O.sampling_probabilities(score, mask_s_ref, mode, bt), rtol=2e-5, atol=1e-9)
        idx_r = ops.generating_downsampled_index(M, cu(score), cu(mask_s_ref), mode, bt, cu(kk)).cpu()
        assert tuple(idx_r.shape) == (B, 1, M)
        for b in range(B):
            off = 0
            for j in range(nb):
                seg = idx_r[b, 0, off:off + int(kk[b, j])]
                assert len(set(seg.tolist())) == len(seg) and bool(mask_s_ref[b, 0, seg, j].all())
                off += int(kk[b, j])
    with pytest.raises(ValueError):
        ops.generating_downsampled_index(M, cu(score), cu(mask_s_ref), "bogus", 0.1, cu(kk))


def test_bin_golden():
    gold = np.load(os.path.join(GOLD, "ops_small.npz"))
    score2 = torch.rand(3, 1, 200, generator=torch.Generator().manual_seed(52)) * 1e-3
    mask3 = torch.from_numpy(gold["bin.static.mask"])
    kk = torch.from_numpy(gold["bin.static.k"])
    idx = ops.generating_downsampled_index(100, cu(score2), cu(mask3), "topk", 0.1, cu(kk))
    np.testing.assert_array_equal(idx.cpu().numpy(), gold["bin.static.idx"])
    w = torch.rand(3, 4, generator=torch.Generator().manual_seed(53))
    np.testing.assert_array_equal(ops.calculate_num_points_to_choose(cu(w), cu(mask3.squeeze(1).sum(1)), 100).cpu().numpy(),
                                  gold["bin.static.k"])


# ---------------------------------------------------------------- tensor-core kNN == exact kNN


def _knn_both(a, b, k):
    from samble_b200 import _lib as L

    lib = L.lib()
    try:
        lib.samble_set_knn_mode(1)
        d1, i1 = ops.knn(a, b, k)
        torch.cuda.synchronize()
    finally:
        lib.samble_set_knn_mode(0)
    d0, i0 = ops.knn(a, b, k)
    torch.cuda.synchronize()
    return (d0, i0), (d1, i1)


def _same_sets_any_order(a, b, k, i_ref):
    """SAMBLE_KNN_ANY_ORDER (knn_select_kernel): the same neighbour set per row, order free."""
    i_any = ops._knn_strided(a, b, k, "bnc", False, torch.int32, ordered=False)[1]
    torch.cuda.synchronize()
    return torch.equal(i_any.long().sort(-1).values, i_ref.sort(-1).values)


TC_SHAPES = [(2, 2048, 0, 128, 32), (2, 2048, 0, 64, 32), (3, 1000, 0, 128, 32), (2, 512, 0, 128, 16), (1, 700, 260, 20, 5),
             (2, 130, 0, 8, 32), (1, 64, 0, 128, 32), (1, 40, 33, 64, 32), (1, 4096, 0, 128, 32), (4, 300, 1200, 96, 3)]


@pytest.mark.parametrize("shape", TC_SHAPES, ids=[f"B{s[0]}_N{s[1]}x{s[2] or s[1]}_C{s[3]}_k{s[4]}" for s in TC_SHAPES])
def test_tensor_core_knn_is_bit_identical_to_exact_kernel(shape):
    """csrc/knn_tc.cu (tcgen05 tf32 candidates + fp32 re-rank) must reproduce csrc/knn.cu's exact FFMA kernel
    bit for bit: same indices in the same order, same distances."""
    B, Nq, Nr, C, k = shape
    a = cu(synthetic_features(B, Nq, C, 100 + Nq))
    b = a if Nr == 0 else cu(synthetic_features(B, Nr, C, 200 + Nr))
    (d0, i0), (d1, i1) = _knn_both(a, b, k)
    assert torch.equal(i0, i1)
    assert torch.equal(d0, d1)
    assert _same_sets_any_order(a, b, k, i1)


def test_tensor_core_knn_hard_cases():
    g = torch.Generator().manual_seed(5)
    # (1) tight clusters + duplicated points: near-zero distances, exact ties, candidate-buffer overflow -> repair kernel
    centers = torch.randn(1, 8, 128, generator=g) * 4
    a = (centers[:, torch.randint(0, 8, (1024,), generator=g)] + 1e-3 * torch.randn(1, 1024, 128, generator=g))
    a[:, 512:768] = a[:, 256:512]
    a = cu(a.contiguous())
    (d0, i0), (d1, i1) = _knn_both(a, a, 32)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    assert _same_sets_any_order(a, a, 32, i1)
    # (2) wildly different norms (margin driven by the largest candidate norm)
    s = cu(synthetic_features(2, 600, 64, 7) * (1 + 50 * (torch.rand(2, 600, 1, generator=g) > 0.97).float()))
    (d0, i0), (d1, i1) = _knn_both(s, s, 32)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    assert _same_sets_any_order(s, s, 32, i1)
    # (3) low intrinsic dimension (a curve embedded in 128-d): many candidates near the threshold
    tt = torch.linspace(0, 1, 2048).view(1, 2048, 1)
    curve = cu(torch.cat([torch.sin(tt * (i + 1)) for i in range(128)], dim=-1).contiguous())
    (d0, i0), (d1, i1) = _knn_both(curve, curve, 32)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    assert _same_sets_any_order(curve, curve, 32, i1)
    # (4) k duplicates and more of every point: the clamp-to-zero tie rule decides, nothing is "certainly in"
    base = synthetic_features(1, 40, 64, 11)
    dup = cu(base.repeat(1, 40, 1).contiguous())          # 1600 points, each present 40 times
    (d0, i0), (d1, i1) = _knn_both(dup, dup, 32)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    assert _same_sets_any_order(dup, dup, 32, i1)


@pytest.mark.parametrize("shape", [(2, 2048, 0, 3, 32), (3, 1000, 0, 3, 20), (1, 300, 700, 2, 5), (2, 5000, 0, 3, 32), (1, 256, 0, 3, 32)],
                         ids=lambda s: f"B{s[0]}_N{s[1]}x{s[2] or s[1]}_C{s[3]}_k{s[4]}")
def test_two_pass_xyz_knn_is_bit_identical_to_kset_kernel(shape):
    """knn_xyz2_kernel (group-minima threshold -> short list -> rank counting) vs knn_xyz_kernel (running k-set)."""
    B, Nq, Nr, C, k = shape
    a = cu(synthetic_features(B, Nq, C, 300 + Nq))
    b = a if Nr == 0 else cu(synthetic_features(B, Nr, C, 400 + Nr))
    (d0, i0), (d1, i1) = _knn_both(a, b, k)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)


def test_two_pass_xyz_knn_duplicates_overflow_fallback():
    # 300 copies of each of 8 points: every list overflows (all duplicates tie at distance 0) -> k-set fallback
    base = synthetic_features(1, 8, 3, 5)
    a = cu(base.repeat(1, 300, 1).contiguous())
    (d0, i0), (d1, i1) = _knn_both(a, a, 32)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)
    # a regular grid: many exact ties at the k-th distance
    g = torch.stack(torch.meshgrid(torch.arange(16.), torch.arange(16.), torch.arange(8.), indexing="ij"), -1).reshape(1, -1, 3)
    g = cu(g.contiguous())
    (d0, i0), (d1, i1) = _knn_both(g, g, 32)
    assert torch.equal(i0, i1) and torch.equal(d0, d1)


def test_transpose12():
    x = torch.randn(3, 1000, 130, generator=torch.Generator().manual_seed(1))
    assert torch.equal(ops.transpose12(cu(x)).cpu(), x.transpose(1, 2).contiguous())
    wide = torch.randn(2, 257, 384, generator=torch.Generator().manual_seed(2))
    sl = cu(wide)[..., 128:256]                                     # column slice of a wider row-major buffer
    assert torch.equal(ops.transpose12(sl).cpu(), wide[..., 128:256].transpose(1, 2).contiguous())
    bcn = cu(torch.randn(2, 64, 300, generator=torch.Generator().manual_seed(3)))
    assert torch.equal(ops.transpose12(bcn), bcn.transpose(1, 2).contiguous())


@pytest.mark.parametrize("seed", [0, 1, 2, 3])
def test_tensor_core_knn_margin_stress(seed):
    """The bf16x2 candidate passes keep a rigorous superset under heavy-tailed, badly scaled and low-rank features
    (the error margin knn_margin is relative to |a||b|): ordered and any-order results equal the exact kernel's."""
    g = torch.Generator().manual_seed(1000 + seed)
    B, N, C = 3, 2048, (128, 96, 64, 36)[seed]
    base = torch.randn(B, N, C, generator=g)
    heavy = base * torch.exp(1.5 * torch.randn(B, N, 1, generator=g))              # norms spread over ~3 decades
    lowrank = (torch.randn(B, N, 5, generator=g) @ torch.randn(5, C, generator=g)) + 1e-3 * base
    chan = base * torch.logspace(-3, 2, C).view(1, 1, C)                           # channel scales 1e-3 .. 1e2
    for x in (heavy, lowrank, chan):
        a = cu(x.contiguous())
        (d0, i0), (d1, i1) = _knn_both(a, a, 32)
        assert torch.equal(i0, i1) and torch.equal(d0, d1)
        assert _same_sets_any_order(a, a, 32, i1)


@pytest.mark.parametrize("B,C,N,K,normal", [(2, 3, 400, 16, False), (1, 6, 300, 8, True), (2, 64, 256, 32, False)])
def test_select_neighbors(B, C, N, K, normal):
    """utils/ops.py:47-65 through the C ABI: same (B,C,N,K) view of (B,N,K,C) storage, same neighbours (tie-aware), exact
    gather / difference given the indices."""
    x = synthetic_features(B, C, N, 91)
    for nt in ("neighbor", "diff"):
        g, idx = ops.select_neighbors(cu(x), K, nt, normal_channel=normal)
        g_ref, idx_ref = O.select_neighbors(x, K, nt, normal_channel=normal)
        assert idx.dtype == torch.int64 and tuple(g.shape) == tuple(g_ref.shape) and g.stride() == g_ref.stride()
        key = (x[:, :3] if (normal and C == 6) else x).transpose(1, 2)
        rep = knn_parity(idx, idx_ref, key, key)
        assert rep["unexplained_rows"] == 0 and rep["exact_rate"] >= 0.995, rep
        pts = x.transpose(1, 2)
        nbr = O.index_points(pts, idx.cpu())
        if nt == "diff":
            nbr = nbr - pts.unsqueeze(2)
        assert torch.equal(g.cpu(), nbr.permute(0, 3, 1, 2))
    with pytest.raises(ValueError):
        ops.select_neighbors(cu(x), K, "center_diff")


def test_sampler_bin_asked_for_more_points_than_it_holds():
    """The remainder rule (utils/ops.py:427-430) can hand a bin more points than it has when every bin is nearly full: the
    reference's per-bin sort then continues with NON-members (masked value 0), ours in index order -- never index 0
    by default, never a member of the bin twice."""
    N, nb, M = 64, 4, 62
    g = torch.Generator().manual_seed(3)
    score = (torch.rand(1, N, generator=g) + 0.1) * 1e-3
    tok = torch.ones(1, N, nb)
    bnd, mask = O.bin_partition(score.unsqueeze(1), None, True, 0.99, nb)            # quantile cuts: 17/16/16/15 points per bin
    for t in bnd:                 # a fresh cut IS a point's z (a last-ulp matter, tested elsewhere): move the cuts off the points
        t[torch.isfinite(t)] -= 1e-3
    bnd, mask = O.bin_partition(score.unsqueeze(1), bnd, False, 0.99, nb)
    counts = mask.squeeze(1).sum(1)
    k_ref = O.calculate_num_points_to_choose(torch.ones(1, nb), counts, M)
    assert int((k_ref - counts).max()) > 0, (k_ref, counts)                          # the case this test is about
    s = ops.ds_sample(cu(score), cu(tok), cu(bnd[0].reshape(-1)[1:].clone()), M)
    assert torch.equal(s["k"].cpu(), k_ref) and torch.equal(s["counts"].cpu().long(), counts)
    idx_ref = O.generating_downsampled_index(M, score.unsqueeze(1), mask, "topk", None, k_ref)
    mine = s["idx"].cpu()
    off = 0
    for j in range(nb):
        kj, cj = int(k_ref[0, j]), int(counts[0, j])
        seg, seg_ref = mine[0, off:off + kj], idx_ref[0, 0, off:off + kj]
        assert torch.equal(seg[:min(kj, cj)], seg_ref[:min(kj, cj)])                 # the members, best first
        if kj > cj:
            extra = seg[cj:]
            assert not bool(mask[0, 0, extra, j].any())                              # non-members, as in the reference ...
            assert not bool(mask[0, 0, seg_ref[cj:], j].any())
            non = (~mask[0, 0, :, j]).nonzero()[:, 0]
            assert torch.equal(extra, non[:kj - cj])                                 # ... lowest index first
        off += kj
    # the unfused op takes the same path
    idx_op = ops.generating_downsampled_index(M, cu(score.unsqueeze(1)), cu(mask), "topk", None, cu(k_ref))
    assert torch.equal(idx_op.cpu()[0, 0], mine[0])


def test_index_topk_with_negative_and_zero_scores():
    """generating_downsampled_index accepts any score (utils/ops.py:476-505): a member whose score + 1e-8 is negative sorts
    AFTER the non-members (whose masked value is 0), zero scores tie with them."""
    N, nb, M = 40, 2, 30
    g = torch.Generator().manual_seed(4)
    score = torch.randn(1, 1, N, generator=g)                                          # about half negative
    mask = torch.zeros(1, 1, N, nb, dtype=torch.bool)
    mask[0, 0, :20, 0] = True
    mask[0, 0, 20:, 1] = True
    k = torch.tensor([[15, 15]], dtype=torch.int32)                                    # more than the positive members of a bin
    idx = ops.generating_downsampled_index(M, cu(score), cu(mask), "topk", None, cu(k)).cpu()
    for j in range(nb):
        v = ((score + 1e-8).unsqueeze(3) * mask)[0, 0, :, j]                           # the reference's sort key
        seg = idx[0, 0, j * 15:(j + 1) * 15]
        got = v[seg]
        assert bool((got[1:] <= got[:-1]).all())                                       # descending
        rest = torch.ones(N, dtype=torch.bool)
        rest[seg] = False
        assert float(got.min()) >= float(v[rest].max())                                # nothing better was left out


@pytest.mark.parametrize("B,N,C,M,K", [(2, 2048, 128, 2048, 32), (3, 300, 64, 77, 5), (1, 1000, 16, 1000, 3), (2, 500, 1024, 33, 2), (2, 100, 12, 50, 7)])
def test_index_points_copy_engine_vs_thread_copy(B, N, C, M, K):
    """samble_index_points: the cp.async.bulk staged gather (tiles of rows loaded by the copy engine, one bulk store per
    tile) and the thread-copy kernel both equal torch.gather (utils/ops.py:5-14), int32 and int64 indices."""
    from samble_b200 import _lib as L
    g = torch.Generator().manual_seed(B * N + C)
    pts = torch.randn(B, N, C, generator=g)
    idx = torch.randint(0, N, (B, M, K), generator=g)
    ref = torch.gather(pts, 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, M, K, C)
    for mode in (0, 1):
        L.lib().samble_set_gather_mode(mode)
        try:
            for dt in (torch.int64, torch.int32):
                assert torch.equal(ops.index_points(cu(pts), cu(idx).to(dt)).cpu(), ref), (mode, dt)
        finally:
            L.lib().samble_set_gather_mode(0)


# ---------------------------------------------------------------- 3-NN interpolation: the three entry points


def _interp_clouds(B, N, M, C, seed):
    """an up cloud and a selected cloud of different offset and scale (the search normalises both by the UP cloud's
    statistics), features (B,C,M)"""
    g = torch.Generator().manual_seed(seed)
    up = (torch.rand(B, 3, N, generator=g) * 2 - 1) * 0.7 + torch.tensor([0.5, -1.0, 2.0]).view(1, 3, 1)
    sel = (torch.rand(B, 3, M, generator=g) * 2 - 1) * 0.9 + torch.tensor([0.4, -0.8, 2.1]).view(1, 3, 1)
    return up, sel, torch.randn(B, C, M, generator=g)


def _interp_all(up, sel, feat, pad=8):
    """interpolate3 (channel-major), interpolate3_rows and interpolate3_search + interpolate3_gather_rows, the two row
    forms writing into column slices of NaN-filled (B,N,C+pad) buffers -> (out (B,N,C) x3, idx int64, dist, nn_w, bufs)"""
    B, C, N = up.shape[0], feat.shape[1], up.shape[2]
    feat_rows = cu(feat.transpose(1, 2).contiguous())
    out3, idx3, d3 = ops.interpolate3(cu(up), cu(sel), cu(feat), want_idx=True)
    bufs = [torch.full((B, N, C + pad), float("nan"), device=DEV) for _ in range(2)]
    ops.interpolate3_rows(cu(up), cu(sel), feat_rows, bufs[0][..., 4:4 + C])
    nn_idx, nn_w = ops.interpolate3_search(cu(up), cu(sel))
    ops.interpolate3_gather_rows(nn_idx, nn_w, feat_rows, bufs[1][..., 4:4 + C])
    assert torch.equal(nn_idx.long(), idx3)
    for buf in bufs:
        assert bool(buf[..., :4].isnan().all()) and bool(buf[..., 4 + C:].isnan().all()), "wrote outside its columns"
    return (out3.transpose(1, 2), bufs[0][..., 4:4 + C], bufs[1][..., 4:4 + C]), idx3, d3, nn_w


@pytest.mark.parametrize("M", [3, 2047, 2048, 2049, 4100])
@pytest.mark.parametrize("N", [1, 33, 5000])
@pytest.mark.parametrize("C", [4, 20, 132])
def test_interpolate3_entry_points_vs_fp64(M, N, C):
    """models/upsample.py:194-212 through its three native entry points.  The per-element arithmetic of the channel-major
    kernel and the row kernel is the same (csrc/upsample.cu), so all three give the same bits; the 3-NN sets match the
    oracle's up to fp32 near-ties (knn_parity), and the output equals the fp64 weighted sum over the native neighbours
    and distances.  M = 2048 / 2049 / 4100 cross the search's 2048-candidate shared-memory chunks."""
    B = 2
    up, sel, feat = _interp_clouds(B, N, M, C, seed=M + N + C)
    outs, idx, dist, nn_w = _interp_all(up, sel, feat)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    idx = idx.cpu()
    assert int(idx.min()) >= 0 and int(idx.max()) < M
    assert bool((idx[..., 0] != idx[..., 1]).all() & (idx[..., 1] != idx[..., 2]).all() & (idx[..., 0] != idx[..., 2]).all())
    if N == 1:
        # the reference normalises by the unbiased std of the up cloud, undefined for one point (its distances are NaN);
        # the native search then sees every candidate at distance 0 and takes the lowest indices -- finite, in range
        assert bool(torch.isfinite(outs[0]).all())
        return
    _, idx_r, _ = O.select_neighbors_interpolate(up, sel, feat, 3)
    rep = knn_parity(idx, idx_r, up.transpose(1, 2), sel.transpose(1, 2))
    assert rep["unexplained_rows"] == 0 and rep["exact_rate"] >= 0.99, rep
    # distances in the reference's normalised units (centred and scaled by the up cloud's statistics, utils/ops.py:23-35)
    up64, sel64 = up.double().transpose(1, 2), sel.double().transpose(1, 2)
    sigma = up64.std(dim=1, keepdim=True).mean(dim=2, keepdim=True)
    d64 = torch.linalg.norm(up64.unsqueeze(2) - sel64.gather(1, idx.view(B, -1, 1).expand(-1, -1, 3)).view(B, N, 3, 3), dim=-1)
    d64 = d64 / sigma
    assert float((dist.cpu().double() - d64).abs().max()) < 5e-3              # GEMM-form cancellation, as test_knn_vs_oracle
    w = 1.0 / (dist.cpu().double() + 1e-8)
    w = w / w.sum(-1, keepdim=True)
    torch.testing.assert_close(nn_w.cpu().double(), w, atol=1e-6, rtol=1e-6)
    nbr = feat.double().transpose(1, 2).gather(1, idx.view(B, -1, 1).expand(-1, -1, C)).view(B, N, 3, C)
    ref = (nbr * w.unsqueeze(-1)).sum(2)                                        # (B,N,C)
    torch.testing.assert_close(outs[0].cpu().double(), ref, atol=2e-5, rtol=1e-4)


def test_interpolate3_coincident_and_duplicate_points():
    B, N, M, C = 1, 300, 64, 8
    up, sel, feat = _interp_clouds(B, N, M, C, seed=7)
    # (1) two selected points at identical coordinates: a tie broken towards the lower index in every entry point
    sel[:, :, 40] = sel[:, :, 10]
    up[:, :, 100] = sel[:, :, 10] + 1e-3
    # (2) up points ON selected points: finite output, that point carries (almost) all of the weight
    up[:, :, :M] = sel
    outs, idx, dist, nn_w = _interp_all(up, sel, feat)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[0], outs[2])
    assert bool(torch.isfinite(outs[0]).all())
    idx, nn_w = idx.cpu(), nn_w.cpu()
    own = torch.arange(M).view(1, M, 1)
    share = (nn_w[:, :M] * (idx[:, :M] == own)).sum(-1)                          # weight of the coincident point
    for i in (10, 40):                                                            # (10 and 40 coincide)
        share[:, i] = (nn_w[:, i] * ((idx[:, i] == 10) | (idx[:, i] == 40))).sum(-1)
    print(f"coincident points: min weight share {float(share.min()):.6f}")
    assert float(share.min()) >= 0.99
    assert idx[0, 100, :2].tolist() == [10, 40] and float(dist[0, 100, 0]) == float(dist[0, 100, 1])
    assert idx[0, 10, :2].tolist() == [10, 40] and idx[0, 40, :2].tolist() == [10, 40]
    # fewer than three selected points: refused by all three
    for fn in (lambda: ops.interpolate3(cu(up), cu(sel[..., :2]), cu(feat[..., :2])),
               lambda: ops.interpolate3_rows(cu(up), cu(sel[..., :2]), cu(feat[..., :2].transpose(1, 2).contiguous()),
                                             torch.empty(B, N, C, device=DEV)),
               lambda: ops.interpolate3_search(cu(up), cu(sel[..., :2]))):
        with pytest.raises(ValueError, match="at least 3"):
            fn()


# ---------------------------------------------------------------- dynamic bin boundaries, bit for bit


def _aten_boundary_update(old, total, world, num_bins, momentum):
    """utils/ops.py:198-233 as the reference states it (the oracle's update_sampling_score_bin_boundary after the
    all_reduce), evaluated by ATen on whatever device `total` lives on"""
    cut = total / world
    if old is not None:
        upper, lower = old[0].clone(), old[1].clone()
        cut = upper[0, 0, 0, 1:] * momentum + (1 - momentum) * cut
        upper[0, 0, 0, 1:] = cut
        lower[0, 0, 0, :-1] = cut
        return [upper, lower]
    inf = torch.full((1,), float("inf"), device=total.device)
    return [torch.cat([inf, cut]).reshape(1, 1, 1, num_bins), torch.cat([cut, -inf]).reshape(1, 1, 1, num_bins)]


@pytest.mark.parametrize("nb", [2, 4, 6, 8])
def test_boundary_update_bit_exact_vs_aten_on_the_gpu(nb):
    """ops._quantile_pick + ops._boundary_ema (csrc/sampler.cu) against the reference's statement of utils/ops.py:182-233
    run by ATen on the same GPU (the reference trains there), torch.equal: every rank count the bench shards over, fresh
    pairs and EMA steps, two momentum factors, cloud sizes the bin count does not divide.  The ranks' local quantiles are
    summed once and handed to both sides, as torch.distributed.all_reduce hands one sum to every rank."""
    g = torch.Generator().manual_seed(nb)
    cpu_diff = 0
    for world in (1, 2, 3, 6, 8):
        for n in (nb * 97 + 1, 1001, 2048 * 3 + nb - 1):
            if n % nb == 0:
                continue
            for momentum in (0.99, 0.9):
                state_native = state_aten = state_cpu = None
                for step in range(3):                                          # fresh pair, then two EMA steps
                    zs = [cu(torch.randn(n, generator=g) * (1 + step)) for _ in range(world)]
                    ranked = [torch.sort(z, descending=True)[0] for z in zs]
                    pos = (torch.arange(1, nb) / nb * n).int().long()         # utils/ops.py:182-189
                    picks = [ops._quantile_pick(r, nb) for r in ranked]
                    for p, r in zip(picks, ranked):
                        assert torch.equal(p, r[pos.to(DEV)])
                    total = picks[0].clone()
                    for p in picks[1:]:
                        total += p
                    state_native = ops._boundary_ema(total, world, state_native, nb, momentum)
                    state_aten = _aten_boundary_update(state_aten, total, world, nb, momentum)
                    for a, b in zip(state_native, state_aten):
                        assert torch.equal(a, b), (world, n, momentum, step, (a - b)[torch.isfinite(b)].abs().max().item())
                    state_cpu = _aten_boundary_update(state_cpu, total.cpu(), world, nb, momentum)
                    cpu_diff += sum(int((a.cpu() != b).sum()) for a, b in zip(state_aten, state_cpu))
                    state_cpu = [t.cpu() for t in state_aten]                  # keep the CPU chain on the GPU's inputs
    # ATen on the CPU divides by world; on CUDA it multiplies by the fp32 reciprocal: the CPU statement that stands in for
    # the kernels in tests/test_distributed_cpu.py differs in the last bits of some boundaries (measured: 8 / 36 / 54 / 62
    # values for nb = 2 / 4 / 6 / 8 over this sweep)
    print(f"nb={nb}: CPU vs CUDA ATen statement: {cpu_diff} differing boundary values")
