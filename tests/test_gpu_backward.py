"""SURVEY 8 row f1: the differentiable path (samble_b200/autograd.py, csrc/backward.cu) against ATen autograd.

Op level: each native backward against torch.autograd of the reference's literal formula (utils/ops.py:5-112,136-145,
models/attention.py:207-250) evaluated in fp64 on the same indices.  Model level: one backward pass of the whole seg / cls
model against the CPU oracle's autograd with the discrete decisions forced (oracle/harness.gradient_parity), in eval mode
(running-statistics BatchNorm) and in train mode (batch statistics).

Tolerance: |g - g_ref|_inf <= 1e-4 * |g_ref|_inf per tensor (fp32 sums in another order; atomics)."""

import pytest
import torch
from torch import nn

from oracle import harness
from samble_b200 import blocks, models, ops
from samble_b200.config import cls_config, seg_config
from samble_b200.testing import fill_state_dict_, n2p_attend_literal, synthetic_clouds, synthetic_features

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
TOL = 1e-4


def rel(g, r):
    g, r = g.detach().cpu().double(), r.detach().cpu().double()
    return float((g - r).abs().max() / r.abs().max().clamp_min(1e-30))


def rand_idx(B, R, N, seed):
    return torch.randint(0, N, (B, R), generator=torch.Generator().manual_seed(seed))


def test_index_points_backward():
    B, N, C, M, K = 2, 300, 24, 200, 7
    p = synthetic_features(B, N, C, 1).requires_grad_(True)               # (B,N,C)
    idx = rand_idx(B, M * K, N, 2).view(B, M, K)
    probe = torch.randn(B, M, K, C, generator=torch.Generator().manual_seed(3))
    ref = torch.gather(p.double(), 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, M, K, C)
    (g_ref,) = torch.autograd.grad((ref * probe.double()).sum(), p)
    for dt in (torch.int64, torch.int32):
        pc = p.detach().to(DEV).requires_grad_(True)
        out = ops.index_points(pc, idx.to(DEV, dt))
        assert torch.equal(out.detach().cpu(), ref.float())
        (g,) = torch.autograd.grad((out * probe.to(DEV)).sum(), pc)
        assert rel(g, g_ref) <= 1e-6


def _group_ref(pcd, idx, group_type):
    """utils/ops.py:47-65, 83-112 given the indices (fp64)."""
    B, C, N = pcd.shape
    pts = pcd.permute(0, 2, 1)
    nbr = torch.gather(pts, 1, idx.reshape(B, -1, 1).expand(-1, -1, C)).view(B, N, idx.shape[-1], C)
    if group_type in ("diff", "center_diff"):
        nbr = nbr - pts[:, :, None, :]
    out = nbr.permute(0, 3, 1, 2)
    if group_type.startswith("center"):
        out = torch.cat([pcd[:, :, :, None].expand(-1, -1, -1, idx.shape[-1]), out], dim=1)
    return out


@pytest.mark.parametrize("group_type", ["neighbor", "diff", "center_neighbor", "center_diff"])
@pytest.mark.parametrize("C", [3, 64])
def test_group_backward(group_type, C):
    B, N, K = 2, 256, 32
    x = synthetic_features(B, C, N, 5)
    xc = x.to(DEV).requires_grad_(True)
    out, idx = ops.group(xc, K, group_type)
    assert idx.dtype == torch.int64 and not idx.requires_grad
    xr = x.double().requires_grad_(True)
    ref = _group_ref(xr, idx.cpu(), group_type)
    assert torch.equal(out.detach().cpu(), ref.detach().float()) or rel(out, ref) <= 1e-6
    assert out.stride() == ops.group(x.to(DEV), K, group_type)[0].stride()         # same layout as the forward-only path
    probe = torch.randn(ref.shape, generator=torch.Generator().manual_seed(6))
    (g_ref,) = torch.autograd.grad((ref * probe.double()).sum(), xr)
    (g,) = torch.autograd.grad((out * probe.to(DEV)).sum(), xc)
    assert rel(g, g_ref) <= 1e-5
    # select_neighbors shares the machinery
    if group_type in ("neighbor", "diff"):
        xc2 = x.to(DEV).requires_grad_(True)
        out2, idx2 = ops.select_neighbors(xc2, K, group_type)
        (g2,) = torch.autograd.grad((out2 * probe.to(DEV)).sum(), xc2)
        assert torch.equal(idx2, idx) and rel(g2, g_ref) <= 1e-5


def test_gather_by_idx_backward():
    B, C, N, M = 3, 128, 512, 200
    x = synthetic_features(B, C, N, 7)
    idx = torch.stack([torch.randperm(N, generator=torch.Generator().manual_seed(b))[:M] for b in range(B)]).view(B, 1, M)
    xr = x.double().requires_grad_(True)
    ref = torch.gather(xr, 2, idx.expand(-1, C, -1))
    probe = torch.randn(B, C, M, generator=torch.Generator().manual_seed(8))
    (g_ref,) = torch.autograd.grad((ref * probe.double()).sum(), xr)
    xc = x.to(DEV).requires_grad_(True)
    out = ops.gather_by_idx(xc, idx.to(DEV))
    assert torch.equal(out.detach().cpu(), ref.detach().float())
    (g,) = torch.autograd.grad((out * probe.to(DEV)).sum(), xc)
    assert rel(g, g_ref) <= 1e-6


@pytest.mark.parametrize("B,N,C,K,H", [(2, 256, 128, 32, 4), (1, 200, 64, 20, 4), (1, 128, 32, 8, 1)])
def test_n2p_attend_backward_matches_the_literal_form(B, N, C, K, H):
    """The reference forms k_ij = Wk(x_j - x_i), v_ij = Wv(x_j - x_i) on gathered (B,C,N,K) tensors
    (models/attention.py:165-185) and lets autograd differentiate softmax(q.k_ij/sqrt(d)) v_ij; the native kernels work on
    the hoisted per-point projections.  Same value, same gradients w.r.t. q, k and v."""
    g = torch.Generator().manual_seed(N + C)
    qkv = torch.randn(B, N, 3 * C, generator=g)
    idx = torch.stack([torch.stack([torch.randperm(N, generator=g)[:K] for _ in range(N)]) for _ in range(B)])     # (B,N,K)
    probe = torch.randn(B, N, C, generator=g)
    r = qkv.double().requires_grad_(True)
    ref = n2p_attend_literal(r, idx, H)
    (g_ref,) = torch.autograd.grad((ref * probe.double()).sum(), r, retain_graph=True)
    for dt in (torch.int32, torch.int64):
        rc = qkv.to(DEV).requires_grad_(True)
        out = ops.n2p_attend(rc, idx.to(DEV, dt), H)
        assert rel(out, ref) <= 2e-5
        (gq,) = torch.autograd.grad((out * probe.to(DEV)).sum(), rc)
        for name, sl in (("q", slice(0, C)), ("k", slice(C, 2 * C)), ("v", slice(2 * C, 3 * C))):
            assert rel(gq[..., sl], g_ref[..., sl]) <= 2e-5, name
    # the fused tail (residual, folded BatchNorm) in differentiable form
    rc = qkv.to(DEV).requires_grad_(True)
    res = torch.randn(B, N, C, generator=g).to(DEV).requires_grad_(True)
    sc, sh = torch.rand(C, generator=g).to(DEV) + 0.5, torch.randn(C, generator=g).to(DEV)
    out = ops.n2p_attend(rc, idx.to(DEV), H, residual=res, scale=sc, shift=sh)
    with torch.no_grad():
        fused = ops.n2p_attend(rc.detach(), idx.to(DEV), H, residual=res.detach(), scale=sc, shift=sh)
    assert rel(out, fused) <= 1e-6
    g1, g2 = torch.autograd.grad((out * probe.to(DEV)).sum(), (rc, res))
    res_r = res.detach().cpu().double().requires_grad_(True)
    ref2 = (ref + res_r) * sc.cpu().double() + sh.cpu().double()
    g1_ref, g2_ref = torch.autograd.grad((ref2 * probe.double()).sum(), (r, res_r))
    assert rel(g1, g1_ref) <= 2e-5 and rel(g2, g2_ref) <= 1e-6


def _knn_ref_dist(a, b, idx):
    """utils/ops.py:17-44 distances of the selected pairs, differentiable (fp64)."""
    mu = a.mean(dim=1, keepdim=True)
    a0, b0 = a - mu, b - mu
    sg = a0.std(dim=1, keepdim=True).mean(dim=2, keepdim=True)
    return torch.cdist(a0 / sg, b0 / sg).gather(2, idx)


@pytest.mark.parametrize("C,k,same", [(3, 3, False), (3, 32, True), (64, 16, False)])
def test_knn_distance_gradient(C, k, same):
    B, Nq, Nr = 2, 300, 300 if same else 160
    a = synthetic_features(B, Nq, C, 11)                                    # (B,Nq,C)
    b = a.clone() if same else a[:, torch.randperm(Nq, generator=torch.Generator().manual_seed(1))[:Nr]].clone()
    ac, bc = a.to(DEV).requires_grad_(True), b.to(DEV).requires_grad_(True)
    neg, idx = ops.knn(ac, bc, k)
    assert neg.requires_grad and not idx.requires_grad
    ar, br = a.double().requires_grad_(True), b.double().requires_grad_(True)
    d_ref = _knn_ref_dist(ar, br, idx.cpu())
    probe = torch.randn(B, Nq, k, generator=torch.Generator().manual_seed(2))
    probe = probe * (d_ref.detach() > 1e-3)              # coincident pairs: d is fp32 cancellation noise, its gradient is 0 * x/0
    ga_ref, gb_ref = torch.autograd.grad((d_ref * probe.double()).sum(), (ar, br))
    ga, gb = torch.autograd.grad((-neg * probe.to(DEV)).sum(), (ac, bc))
    assert rel(ga, ga_ref) <= TOL and rel(gb, gb_ref) <= TOL


def test_select_neighbors_interpolate_gradients():
    """models/upsample.py:194-212 end to end: gradients w.r.t. the features AND both xyz sets (the path by which the seg
    model's STN is trained, models/seg_model.py:187-192)."""
    B, N, M, C = 2, 512, 256, 32
    xyz, _ = synthetic_clouds(B, N, 3)
    sel = torch.stack([torch.randperm(N, generator=torch.Generator().manual_seed(b))[:M] for b in range(B)])
    xyz_s = torch.gather(xyz, 2, sel.unsqueeze(1).expand(-1, 3, -1)) + 0.01 * torch.randn(B, 3, M, generator=torch.Generator().manual_seed(9))
    feat = synthetic_features(B, C, M, 4)
    probe = torch.randn(B, C, N, generator=torch.Generator().manual_seed(5))

    def interp(nbr, d):
        w = 1.0 / (d + 1e-8)
        w = w / torch.sum(w, dim=-1, keepdim=True)
        return torch.sum(nbr * w.unsqueeze(1), dim=-1)

    uc, kc, fc = (t.to(DEV).requires_grad_(True) for t in (xyz, xyz_s, feat))
    nbr, idx, d = ops.select_neighbors_interpolate(uc, kc, fc, K=3)
    out = interp(nbr, d)
    g = torch.autograd.grad((out * probe.to(DEV)).sum(), (uc, kc, fc))
    ur, kr, fr = (t.double().requires_grad_(True) for t in (xyz, xyz_s, feat))
    d_ref = _knn_ref_dist(ur.permute(0, 2, 1), kr.permute(0, 2, 1), idx.cpu())
    # the VALUES of small distances carry the GEMM form's fp32 cancellation error (utils/ops.py:35; any fp32 implementation
    # has it) and 1/d^2 amplifies it in the gradient: take the native values, keep the fp64 graph (as the oracle's forcing does)
    d_ref = d_ref + (d.detach().cpu().double() - d_ref).detach()
    nbr_ref = torch.gather(fr.permute(0, 2, 1), 1, idx.cpu().reshape(B, -1, 1).expand(-1, -1, C)).view(B, N, 3, C).permute(0, 3, 1, 2)
    ref = interp(nbr_ref, d_ref)
    g_ref = torch.autograd.grad((ref * probe.double()).sum(), (ur, kr, fr))
    assert rel(out, ref) <= 5e-4
    for a, r, name in zip(g, g_ref, ("unknown xyz", "known xyz", "features")):
        assert rel(a, r) <= 2e-4, name


def test_fused_kernels_still_refuse_gradients():
    x = synthetic_features(1, 128, 256, 1).to(DEV).requires_grad_(True)
    w = torch.randn(64, 128, device=DEV)
    with pytest.raises(RuntimeError, match="forward-only"):
        ops.linear(x, w, x_layout="bcn")
    with pytest.raises(RuntimeError, match="forward-only"):
        ops.interpolate3(torch.rand(1, 3, 64, device=DEV, requires_grad=True), torch.rand(1, 3, 32, device=DEV), torch.rand(1, 8, 32, device=DEV))


def _prepared(which, B, N, M, seed, train):
    cfg = (seg_config if which == "seg" else cls_config)(M=M)
    m = (models.ShapeNetModel if which == "seg" else models.ModelNetModel)(cfg)
    sd = fill_state_dict_(m.state_dict(), seed=seed, sharpen=2.0)
    m.load_state_dict(sd)
    m = m.eval().to(DEV)
    xc, catc = synthetic_clouds(B, N, 100 + seed)
    with torch.no_grad():
        m(xc.to(DEV), catc.to(DEV)) if which == "seg" else m(xc.to(DEV))
    models.freeze_boundaries(m)
    if train:
        m.train()
        for mod in m.modules():
            if isinstance(mod, nn.Dropout):
                mod.eval()                       # the only random layer of the head (seg_model.py:212-216): off for a comparable step
    return m, sd, cfg


@pytest.mark.parametrize("which,train", [("seg", False), ("seg", True), ("cls", False), ("cls", True)])
def test_model_backward_vs_oracle_autograd(which, train):
    """One backward pass through the whole model: every parameter gradient and the input gradient against the oracle's
    autograd (the reference's formulas), neighbour sets / 3-NN distances / sampled indices forced."""
    B, N, M = (8 if (train and which == "cls") else 2), 256, (128, 64)     # (cls head: BatchNorm1d over the B clouds themselves)
    m, sd, cfg = _prepared(which, B, N, M, seed=4, train=train)
    x, cat = synthetic_clouds(B, N, 6)
    rep = harness.gradient_parity(m, sd, cfg, x, cat, which=which)
    allp = list(rep["params"].items()) + [("<input>", rep["input"])]
    worst = sorted(allp, key=lambda kv: -kv[1]["rel"])[:4]
    print(which, "train" if train else "eval", "tensors", rep["n_params"], "logits", rep["logits_close_frac"], rep["logits_close_frac_fp64"],
          "LeakyReLU sides forced:", rep["lrelu_flips_vs_fp64"], "of", rep["lrelu_elements"])
    for n, e in worst:
        print(f"  {n}: rel {e['rel']:.2e} (reference fp32 autograd: {e['rel_oracle32']:.2e}) own scale {e['own_scale']:.2e}")
    print("  median rel native", sorted(e["rel"] for _, e in allp)[len(allp) // 2], "oracle32", sorted(e["rel_oracle32"] for _, e in allp)[len(allp) // 2])
    assert rep["logits_close_frac_fp64"] == 1.0
    assert rep["n_params"] >= 60
    harness.assert_gradient_report(rep, tol=TOL)


def test_eval_mode_with_frozen_parameters_keeps_the_fused_path():
    """grad mode on, nothing requires grad -> the fused inference kernels; a parameter that requires grad -> the
    differentiable path (ADVICE round 1: no silently detached outputs)."""
    m, sd, cfg = _prepared("seg", 2, 256, (128, 64), seed=2, train=False)
    x, cat = synthetic_clouds(2, 256, 8)
    from samble_b200 import _lib as L
    with torch.no_grad():
        y0 = m(x.to(DEV), cat.to(DEV))
    for p in m.parameters():
        p.requires_grad_(False)
    L.lib().samble_reset_launch_count()
    y1 = m(x.to(DEV), cat.to(DEV))
    assert not y1.requires_grad and torch.equal(y0, y1)
    n2p = m.block.feature_learning_layer_list[0]
    n2p.q_conv.weight.requires_grad_(True)
    y2 = m(x.to(DEV), cat.to(DEV))
    assert y2.requires_grad
    y2.sum().backward()
    assert n2p.q_conv.weight.grad is not None and float(n2p.q_conv.weight.grad.abs().max()) > 0
    assert harness.close_frac(y2, y0.cpu()) == 1.0
