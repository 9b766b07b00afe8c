"""The tensor-core linear kernels at schedules where one CTA computes several output tiles, against fp64.

linear_tma_kernel (csrc/linear_tma.cu: ops.linear on row-major x, ops.linear_pool, ops.cloud_matmul) and linear_tc_kernel
(csrc/linear_tc.cu: ops.linear on channel-major x with fewer than 32 channels) are persistent, grid = min(tiles, 148).
linear_tma_kernel gives CTA c a contiguous run of the n-major tile order (lt_range); linear_tc_kernel walks tiles c,
c + grid, ...  Past 148 tiles a CTA alternates between two TMEM accumulator sets (or reuses its one set when
2 * nacc * NT > 512), double-buffers its TMA stores across tiles, and reloads its resident weight slice where its run
crosses an n-tile or, in cloud_matmul, a cloud.  The op-level cases of tests/test_gpu_tc.py launch at most 128 tiles, so
every CTA there computes one tile and none of this runs.

schedule() restates the host planning for one call; the case ids are built from it, so a failure names its schedule
cell, and test_case_tables_cover_their_cells checks (without a GPU) that the tables reach every cell they claim.  Each
case is compared with the fp64 statement computed on the GPU, at the bar of test_linear_3xtf32_matches_fp64:
max|y - ref| < 2e-5 * max(1, max|ref|).  Each case is also run twice and on a sub-range of its rows (128-aligned row
blocks, or whole clouds): same K and Nout give the same NT, plan and epilogue, so only the grid and each CTA's tile run
change, and the kernels compute the same products in the same order -- the bits must not move.
"""
from collections import namedtuple

import pytest
import torch

from samble_b200 import _lib as L

gpu = pytest.mark.gpu
DEV = "cuda"
SMS = 148
TOL = 2e-5

# ---------------------------------------------------------------- the host's schedule, restated

Sched = namedtuple("Sched", "kernel NT nacc nsets w_res epi tiles per_cta crossings")


def schedule(M, K, Nout, op="linear", npc=0, x_cm=False, out_cm=False, res_cm=False):
    """The launch one call gets.  op: "linear" (samble_linear), "pool" (samble_linear_pool) or "cloud_matmul"
    (samble_cloud_matmul, npc = rows per cloud); x_cm: channel-major x, which ops.linear sends to linear_tc_kernel when
    K < 32.  crossings = CTAs whose tiles use more than one weight slice (n-tile, and cloud for per-cloud weights)."""
    nkb = -(-K // 32)
    chain = 16 if op == "cloud_matmul" and K > 1024 else 8                 # samble_cloud_matmul; kLinChain elsewhere
    nacc = -(-nkb // chain)
    NT = 128 if Nout > 64 and nacc * 128 <= 512 else 64                   # samble_linear, launch_linear_tma_auto
    nsets = 2 if 2 * nacc * NT <= 512 else 1                              # both kernels
    mt, nt = -(-M // 128), -(-Nout // NT)
    tiles = mt * nt
    grid = min(tiles, SMS)
    if x_cm:                                                             # linear_tc_kernel: tile = m_tile * nt + n_tile
        runs = [[t % nt for t in range(c, tiles, grid)] for c in range(grid)]
        return Sched("linear_tc_kernel", NT, nacc, nsets, False, "direct", tiles, max(map(len, runs)),
                     sum(len(set(r)) > 1 for r in runs))
    wbytes = 2 * nkb * NT * 128                                          # lt_resident_ok, lt_plan (kLtFixed = 1.5 KB)
    w_res = wbytes + 3 * 32768 + 1536 <= 227 * 1024
    room = 227 * 1024 - 1536 - (wbytes if w_res else 0)
    stage = 32768 if w_res else 32768 + 2 * NT * 128
    stages = min(4, room // stage)
    staged = room - stages * stage >= 32768 or stages == 4               # a 4th stage is given up for the store slab
    if op == "pool":                                                     # samble_linear_pool: pool_rows 128 -> EPI 5
        epi = "pool_swapped" if NT == 128 and npc % 128 == 0 else "pool_rows"
    else:                                                                # launch_linear_tma: tma_out (ldo = Nout here)
        epi = "tma_store" if staged and not out_cm and not res_cm and Nout % 4 == 0 else "direct"
    runs = [[(t // mt, (t % mt) * 128 // npc if op == "cloud_matmul" else 0)             # lt_range; the wkey of a tile
             for t in range(c * tiles // grid, (c + 1) * tiles // grid)] for c in range(grid)]
    return Sched("linear_tma_kernel", NT, nacc, nsets, w_res, epi, tiles, max(map(len, runs)),
                 sum(len(set(r)) > 1 for r in runs))


def sched_id(s):
    return (f"NT{s.NT}-acc{s.nacc}-{s.nsets}set-{'resW' if s.w_res else 'streamW'}-{s.epi}-{s.tiles}t-"
            f"{s.per_cta}perCTA-{s.crossings}cross")


# ---------------------------------------------------------------- case tables

Case = namedtuple("Case", "B P K N cell out scale shift lrelu res res_first")


def case(B, P, K, N, cell, out="rows", scale=None, shift=None, lrelu=False, res=None, res_first=False):
    """scale: None / True / "off1" (a view 1 float into its storage); shift: None / "shared" / "off1" / "cloud" (B, N);
    res: None / "rows" / "ldr" (column slice of a wider row buffer) / "off4" / "off1" (slice 4 or 1 floats in) / "bcn"."""
    return Case(B, P, K, N, cell, out, scale, shift, lrelu, res, res_first)


def lin_sched(c, x_cm=False):
    return schedule(c.B * c.P, c.K, c.N, x_cm=x_cm, out_cm=c.out == "bcn", res_cm=c.res == "bcn")


# ops.linear, row-major x -> linear_tma_kernel.  Cell name -> what its schedule must be.
TMA_CELLS = {
    "resident NT128 2-set direct, n-tile crossings":
        lambda s: s.NT == 128 and s.w_res and s.nsets == 2 and s.epi == "direct" and s.crossings > 0,
    "streamed NT128 TMA-store": lambda s: s.NT == 128 and not s.w_res and s.nacc == 1 and s.epi == "tma_store",
    "nacc 2 TMA-store": lambda s: s.NT == 128 and s.nacc == 2 and s.nsets == 2 and s.epi == "tma_store",
    "one accumulator set NT128": lambda s: s.NT == 128 and s.nsets == 1,
    "NT64 K > 1024, one set": lambda s: s.NT == 64 and s.nacc > 4 and s.nsets == 1,
    "NT64 resident, Nout <= 64": lambda s: s.NT == 64 and s.w_res,
    "K tail": lambda s: True,
}
TMA_CASES = [
    case(19, 1000, 128, 384, "resident NT128 2-set direct, n-tile crossings", scale=True, shift="shared", lrelu=True, res="off4"),
    case(3, 3000, 128, 1000, "resident NT128 2-set direct, n-tile crossings", out="bcn", scale=True, shift="cloud", lrelu=True,
         res="bcn"),
    case(7, 1100, 256, 520, "streamed NT128 TMA-store", scale=True, shift="shared", res="ldr"),
    case(5, 2000, 512, 300, "nacc 2 TMA-store", scale=True, shift="shared", lrelu=True, res="rows", res_first=True),
    case(9, 1000, 1024, 260, "one accumulator set NT128", scale="off1", shift="off1", lrelu=True),
    case(6, 1000, 1152, 200, "NT64 K > 1024, one set", scale=True, shift="cloud"),
    case(3, 2100, 2048, 130, "NT64 K > 1024, one set", lrelu=True, res="off1"),
    case(20, 1000, 256, 64, "NT64 resident, Nout <= 64", shift="cloud", res="ldr"),
    case(40, 600, 64, 36, "NT64 resident, Nout <= 64", scale=True, shift="shared", lrelu=True),
    case(10, 1000, 129, 200, "K tail", scale=True, res="rows", res_first=True),               # K % 32 = 1
    case(12, 1000, 36, 256, "K tail", shift="shared", res="off1"),                             # K % 32 = 4
    case(30, 700, 60, 100, "K tail", scale="off1", lrelu=True),                                # K % 32 = 28
]

# ops.linear, channel-major x with K < 32 -> linear_tc_kernel (the first EdgeConv projection: xyz, K = 3 or 6)
TC_CASES = [
    case(16, 2048, 3, 128, "first EdgeConv projection", out="bcn", scale=True, shift="shared", lrelu=True),
    case(20, 1000, 31, 64, "NT64", shift="cloud", res="rows"),
    case(40, 300, 1, 50, "NT64", out="bcn", scale=True, res="bcn"),
    case(10, 999, 6, 200, "NT128", scale=True, shift="cloud", lrelu=True, res="ldr"),
]

# ops.linear_pool: (B, P, K, N, shift kind)
POOL_CASES = [
    (40, 512, 128, 1024, "cloud"),        # swapped orientation, 1280 tiles
    (150, 96, 64, 200, "cloud"),          # row-per-thread (P % 128 != 0), NT 128
    (100, 256, 256, 64, "cloud"),         # row-per-thread (Nout <= 64), NT 64
    (24, 1024, 512, 256, "shared"),       # swapped, streamed weights, nacc 2
]

# ops.cloud_matmul: (B, R, K, N, epilogue)
CM_CASES = [
    (16, 1024, 128, 2048, "softmax"),     # resident per-cloud weights, every CTA crosses clouds
    (16, 512, 100, 384, "residual"),      # K tail, resident, cloud crossings
    (20, 1024, 2048, 128, "residual"),    # 16-block chains, one accumulator set, streamed
]


def pool_sched(c):
    B, P, K, N, _ = c
    return schedule(B * P, K, N, op="pool", npc=P)


def cm_sched(c):
    B, R, K, N, _ = c
    return schedule(B * R, K, N, op="cloud_matmul", npc=R)


def test_case_tables_cover_their_cells():
    """Runs without a GPU: every case reaches the schedule its table claims, with more than 148 tiles where a CTA is
    meant to run several of them."""
    for c in TMA_CASES:
        s = lin_sched(c)
        assert TMA_CELLS[c.cell](s), (c, s)
        assert s.kernel == "linear_tma_kernel" and s.tiles > SMS and s.per_cta >= 2, (c, s)
    assert {c.cell for c in TMA_CASES} == set(TMA_CELLS)
    assert {lin_sched(c).nacc for c in TMA_CASES} >= {1, 2, 4, 5, 8}
    assert {c.K % 32 for c in TMA_CASES if lin_sched(c).per_cta >= 2} >= {1, 4, 28}
    assert sum(lin_sched(c).crossings for c in TMA_CASES if lin_sched(c).w_res) > 0
    assert any(c.shift == "cloud" and c.P % 128 and c.out == "bcn" and lin_sched(c).w_res for c in TMA_CASES)
    # the epilogue's load paths: a 4-float offset residual takes the 16-byte path, which only the direct epilogue has
    assert any(c.res == "off4" and lin_sched(c).epi == "direct" for c in TMA_CASES)
    assert {c.res for c in TMA_CASES} >= {"ldr", "off4", "off1", "bcn", "rows"}
    assert any(c.res == "ldr" and lin_sched(c).epi == "tma_store" for c in TMA_CASES)
    assert any(c.scale == "off1" for c in TMA_CASES) and any(c.shift == "off1" for c in TMA_CASES)
    assert any(c.N % 4 and lin_sched(c).epi == "direct" for c in TMA_CASES)            # scalar stores
    assert any(c.res_first for c in TMA_CASES)

    tc = [lin_sched(c, x_cm=True) for c in TC_CASES]
    assert all(s.kernel == "linear_tc_kernel" for s in tc)
    assert {c.K for c in TC_CASES} == {1, 3, 6, 31} and {c.N for c in TC_CASES} == {50, 64, 128, 200}
    assert sum(s.tiles > SMS and s.per_cta >= 2 for s in tc) >= 2
    assert any(c.P % 128 for c in TC_CASES) and {c.out for c in TC_CASES} == {"rows", "bcn"}
    assert any(c.shift == "cloud" for c in TC_CASES) and {c.res for c in TC_CASES} >= {"rows", "bcn"}

    ps = [pool_sched(c) for c in POOL_CASES]
    assert all(s.tiles > SMS and s.per_cta >= 2 for s in ps)
    assert {(s.epi, s.NT) for s in ps} >= {("pool_swapped", 128), ("pool_rows", 128), ("pool_rows", 64)}
    assert all(any(c[4] == "cloud" for c, s in zip(POOL_CASES, ps) if s.epi == e) for e in ("pool_swapped", "pool_rows"))

    cs = [cm_sched(c) for c in CM_CASES]
    assert all(s.tiles > SMS and s.per_cta >= 2 for s in cs)
    assert any(s.w_res and s.crossings > 0 and c[4] == "softmax" for c, s in zip(CM_CASES, cs))
    assert any(c[2] % 32 and s.w_res and s.crossings > 0 for c, s in zip(CM_CASES, cs))
    assert any(c[2] > 1024 and s.nsets == 1 and c[4] == "residual" for c, s in zip(CM_CASES, cs))


def test_schedule_restates_the_modelled_layers():
    """The seg config's layers at B = 16, N = 2048, as the host code plans them."""
    qkv = schedule(16 * 2048, 128, 384)
    assert (qkv.tiles, qkv.per_cta, qkv.crossings, qkv.w_res, qkv.epi) == (768, 6, 2, True, "direct")
    pool = schedule(16 * 2048, 128, 1024, op="pool", npc=2048)
    assert (pool.tiles, pool.per_cta, pool.epi) == (2048, 14, "pool_swapped")
    edge = schedule(16 * 2048, 3, 128, x_cm=True, out_cm=True)
    assert (edge.kernel, edge.tiles) == ("linear_tc_kernel", 256)
    att = schedule(16 * 1024, 128, 2048, op="cloud_matmul", npc=1024)
    assert att.tiles == 2048 and att.w_res and att.crossings == SMS
    assert schedule(1000, 2048, 100).nacc == 8 and schedule(1024, 4096, 128, op="cloud_matmul", npc=1024).nacc == 8


# ---------------------------------------------------------------- helpers


def launched(fn):
    """(fn(), {kernel name: launches}) over the native launches fn makes."""
    torch.cuda.synchronize()
    L.profile_report()                                   # drop anything recorded earlier
    L.profile(True)
    try:
        out = fn()
        torch.cuda.synchronize()
    finally:
        L.profile(False)
    return out, {name: n for name, (n, _) in L.profile_report().items()}


def gen(seed):
    return torch.Generator(device=DEV).manual_seed(seed)


def randn(g, *shape):
    return torch.randn(*shape, generator=g, device=DEV)


def fp64_statement(x, w, scale=None, shift=None, lrelu=False, res=None, res_first=False):
    """x (B,P,K) rows -> (B,P,N) in fp64: x W^T [+res] * scale + shift -> LeakyReLU(0.2) [+res]."""
    ref = x.double() @ w.double().t()
    if res is not None and res_first:
        ref = ref + res.double()
    if scale is not None:
        ref = ref * scale.double()
    if shift is not None:
        ref = ref + (shift.double() if shift.dim() == 1 else shift.double().unsqueeze(1))
    if lrelu:
        ref = torch.where(ref > 0, ref, 0.2 * ref)
    if res is not None and not res_first:
        ref = ref + res.double()
    return ref


def check_fp64(y, ref, what):
    err = (y.double() - ref).abs().max().item()
    amax = ref.abs().max().item()
    print(f"{what}: max|y - fp64| = {err:.3e}, / max|ref| = {err / max(amax, 1e-30):.3e} (max|ref| = {amax:.3g})")
    assert err < TOL * max(1.0, amax), f"{what}: max err {err:.3e} vs bar {TOL * max(1.0, amax):.3e}"


def lin_inputs(c, x_cm=False):
    """x as ops.linear is to get it, the fp64 reference in (B,P,N) rows, and linear's keyword arguments."""
    B, P, K, N = c.B, c.P, c.K, c.N
    g = gen(B * 100003 + P * 101 + K * 7 + N)
    x_rows = randn(g, B, P, K) * 2
    w = randn(g, N, K) / K ** 0.5
    scale = None if c.scale is None else torch.rand(N + 1, generator=g, device=DEV) + 0.5
    scale = None if scale is None else (scale[1:] if c.scale == "off1" else scale[:N].clone())
    shift = {None: lambda: None, "shared": lambda: randn(g, N), "off1": lambda: randn(g, N + 1)[1:],
             "cloud": lambda: randn(g, B, N)}[c.shift]()
    res_rows = res_arg = None
    if c.res is not None:
        M = B * P
        if c.res == "bcn":
            res_arg = randn(g, B, N, P)
            res_rows = res_arg.transpose(1, 2)
        else:
            lo, width = {"rows": (0, N), "ldr": (0, N + 8), "off4": (4, N + 8), "off1": (1, N + 1)}[c.res]
            res_arg = randn(g, M, width)[:, lo:lo + N]
            res_rows = res_arg.reshape(B, P, N)
    ref = fp64_statement(x_rows, w, scale, shift, c.lrelu, res_rows, c.res_first)
    x = x_rows.transpose(1, 2).contiguous() if x_cm else x_rows
    kw = dict(x_layout="bcn" if x_cm else "rows", out_layout=c.out, scale=scale, shift=shift, lrelu=c.lrelu,
              residual=res_arg, residual_first=c.res_first, residual_layout="bcn" if c.res == "bcn" else "rows")
    return x, w, ref, kw


def as_rows(y, c):
    return y.transpose(1, 2) if c.out == "bcn" else y


def run_linear_case(c, x_cm):
    from samble_b200 import ops

    x, w, ref, kw = lin_inputs(c, x_cm)
    y, names = launched(lambda: ops.linear(x, w, **kw))
    s = lin_sched(c, x_cm)
    assert names.get(s.kernel, 0) == 1 and sum(n for k, n in names.items() if k.startswith("linear_t")) == 1, names
    assert tuple(as_rows(y, c).shape) == (c.B, c.P, c.N)
    check_fp64(as_rows(y, c), ref, sched_id(s))
    assert torch.equal(ops.linear(x, w, **kw), y), "second run differs"


def slice_kw(kw, c, b0, b1):
    """linear's keyword arguments for clouds b0:b1."""
    kw = dict(kw)
    if c.shift == "cloud":
        kw["shift"] = kw["shift"][b0:b1]
    if c.res is not None:
        r = kw["residual"]
        kw["residual"] = r[b0:b1] if c.res == "bcn" else r[b0 * c.P:b1 * c.P]
    return kw


def row_blocks(M):
    """a few 128-aligned row blocks: the first tile, a run from the middle, and the tail block."""
    mt = -(-M // 128)
    return [(0, 128), (128 * (mt // 3), 128 * (mt // 3 + 5)), (128 * (mt - 2), M)]


def cloud_blocks(B):
    return [(0, 1), (B // 2, B // 2 + 2), (B - 1, B)]


def check_linear_slices(c, x_cm):
    from samble_b200 import ops

    x, w, _, kw = lin_inputs(c, x_cm)
    y = ops.linear(x, w, **kw)
    for b0, b1 in cloud_blocks(c.B):
        yb = ops.linear(x[b0:b1], w, **slice_kw(kw, c, b0, b1))
        assert torch.equal(yb, y[b0:b1]), f"clouds {b0}:{b1}"
    if x_cm or c.out == "bcn" or c.shift == "cloud" or c.res == "bcn":
        return
    M = c.B * c.P                       # row-major everywhere: any 128-aligned row block is a call of its own
    x2, y2 = x.reshape(M, c.K), y.reshape(M, c.N)
    for r0, r1 in row_blocks(M):
        kr = dict(kw)
        if c.res is not None:
            kr["residual"] = kw["residual"][r0:r1]
        assert torch.equal(ops.linear(x2[r0:r1], w, **kr), y2[r0:r1]), f"rows {r0}:{r1}"


# ---------------------------------------------------------------- ops.linear on linear_tma_kernel


@gpu
@pytest.mark.parametrize("c", TMA_CASES, ids=[f"B{c.B}_P{c.P}_K{c.K}_N{c.N}-" + sched_id(lin_sched(c)) for c in TMA_CASES])
def test_linear_tma_several_tiles_per_cta_matches_fp64(c):
    run_linear_case(c, x_cm=False)


@gpu
@pytest.mark.parametrize("c", TMA_CASES, ids=[f"B{c.B}_P{c.P}_K{c.K}_N{c.N}-" + sched_id(lin_sched(c)) for c in TMA_CASES])
def test_linear_tma_is_bit_identical_on_row_blocks_and_cloud_slices(c):
    check_linear_slices(c, x_cm=False)


@gpu
def test_linear_refuses_k_past_2048():
    from samble_b200 import ops

    g = gen(2049)
    w = randn(g, 70, 2049)
    x = randn(g, 2, 128, 2049)
    with pytest.raises(ValueError, match="too large"):
        ops.linear(x, w)
    ops.linear(x[..., :2048], w[:, :2048].contiguous())              # the longest contraction it takes


# ---------------------------------------------------------------- ops.linear on linear_tc_kernel (channel-major x, K < 32)


@gpu
@pytest.mark.parametrize("c", TC_CASES, ids=[f"B{c.B}_P{c.P}_K{c.K}_N{c.N}_{c.out}-" + sched_id(lin_sched(c, True)) for c in TC_CASES])
def test_linear_channel_major_matches_fp64(c):
    run_linear_case(c, x_cm=True)


@gpu
@pytest.mark.parametrize("c", TC_CASES, ids=[f"B{c.B}_P{c.P}_K{c.K}_N{c.N}_{c.out}-" + sched_id(lin_sched(c, True)) for c in TC_CASES])
def test_linear_channel_major_is_bit_identical_on_cloud_slices(c):
    check_linear_slices(c, x_cm=True)


# ---------------------------------------------------------------- ops.linear_pool


def pool_inputs(c):
    B, P, K, N, shift_kind = c
    g = gen(B * 7919 + P * 31 + K + N)
    x = randn(g, B, P, K) * 2
    w = randn(g, N, K) / K ** 0.5
    scale = torch.rand(N, generator=g, device=DEV) + 0.5
    shift = randn(g, B, N) if shift_kind == "cloud" else randn(g, N)
    return x, w, dict(scale=scale, shift=shift, lrelu=True)


@gpu
@pytest.mark.parametrize("c", POOL_CASES, ids=[f"B{c[0]}_P{c[1]}_K{c[2]}_N{c[3]}-" + sched_id(pool_sched(c)) for c in POOL_CASES])
def test_linear_pool_several_tiles_per_cta_matches_fp64(c):
    from samble_b200 import ops

    x, w, kw = pool_inputs(c)
    (mx, mean), names = launched(lambda: ops.linear_pool(x, w, **kw))
    assert names.get("linear_tma_kernel", 0) == 1, names
    ref = fp64_statement(x, w, **kw)
    sid = sched_id(pool_sched(c))
    check_fp64(mx, ref.amax(dim=1), f"max {sid}")
    check_fp64(mean, ref.mean(dim=1), f"mean {sid}")
    mx2, mean2 = ops.linear_pool(x, w, **kw)
    assert torch.equal(mx, mx2) and torch.equal(mean, mean2), "second run differs"
    for b0, b1 in cloud_blocks(c[0]):
        kb = dict(kw, shift=kw["shift"][b0:b1] if kw["shift"].dim() == 2 else kw["shift"])
        mxb, meanb = ops.linear_pool(x[b0:b1], w, **kb)
        assert torch.equal(mxb, mx[b0:b1]) and torch.equal(meanb, mean[b0:b1]), f"clouds {b0}:{b1}"


# ---------------------------------------------------------------- ops.cloud_matmul


def cm_inputs(c):
    """Each cloud's weights at a different scale (0.5, 1, 1.5, 2, ...): a tile multiplied by the previous cloud's slice
    is off by O(1), not by a near miss."""
    B, R, K, N, _ = c
    g = gen(B * 131 + R + K * 3 + N)
    x = randn(g, B, R, K)
    cloud_scale = 0.5 + 0.5 * (torch.arange(B, device=DEV) % 4).float()
    w = randn(g, B, N, K) / K ** 0.5 * cloud_scale.view(B, 1, 1)
    res = randn(g, B, R, N)
    return x, w, res


@gpu
@pytest.mark.parametrize("c", CM_CASES, ids=[f"B{c[0]}_R{c[1]}_K{c[2]}_N{c[3]}_{c[4]}-" + sched_id(cm_sched(c)) for c in CM_CASES])
def test_cloud_matmul_several_tiles_per_cta_matches_fp64(c):
    from samble_b200 import ops

    x, w, res = cm_inputs(c)
    sid = sched_id(cm_sched(c))
    prod = torch.matmul(x.double(), w.double().transpose(1, 2))
    if c[4] == "softmax":
        div = 3.0
        logits = prod / div
        rmax = logits.amax(dim=-1)
        rsum = torch.exp(logits - rmax.unsqueeze(-1)).sum(-1)
        kw = dict(row_max=rmax.float(), row_sum=rsum.float(), logit_div=div)
        ref = torch.softmax(logits, dim=-1)
        y, names = launched(lambda: ops.cloud_matmul(x, w, **kw))
        check_fp64(ops.cloud_matmul(x, w), prod, f"product {sid}")
    else:
        kw = dict(residual=res)
        ref = prod + res.double()
        y, names = launched(lambda: ops.cloud_matmul(x, w, **kw))
    assert names.get("linear_tma_kernel", 0) == 1, names
    check_fp64(y, ref, f"{c[4]} {sid}")
    assert torch.equal(ops.cloud_matmul(x, w, **kw), y), "second run differs"
    for b0, b1 in cloud_blocks(c[0]):
        kb = {k: (v[b0:b1] if isinstance(v, torch.Tensor) else v) for k, v in kw.items()}
        assert torch.equal(ops.cloud_matmul(x[b0:b1], w[b0:b1], **kb), y[b0:b1]), f"clouds {b0}:{b1}"


# ---------------------------------------------------------------- the weight-split cache (ops._split_weight)


@gpu
def test_split_weight_of_column_slices_matches_contiguous_copy():
    """The seg head passes w2[:, ng:, 0] (a strided column slice: split with torch bit ops in place of the split kernel);
    a slice at an odd column offset is copied into a padded, aligned buffer.  Both give the contiguous copy's bits."""
    from samble_b200 import ops

    g = gen(2240)
    w2 = randn(g, 1024, 2240, 1) / 128 ** 0.5                 # conv2 of the seg head: 2112 pooled + 128 point channels
    x = randn(g, 4, 1000, 128)
    shift = randn(g, 4, 1024)
    for ng in (2112, 2111):
        view = w2[:, ng:ng + 128, 0]
        w, lo = ops._split_weight(view)
        assert (w.data_ptr() == view.data_ptr()) == (ng % 4 == 0), "the aligned slice is split in place, the odd one copied"
        wc, loc = ops._split_weight(view.contiguous())
        assert torch.equal(w, wc) and torch.equal(lo, loc)
        y = ops.linear(x, view, shift=shift, lrelu=True)
        assert torch.equal(y, ops.linear(x, view.contiguous(), shift=shift, lrelu=True))
        check_fp64(y, fp64_statement(x, view, shift=shift, lrelu=True), f"column slice at {ng}")


@gpu
def test_split_weight_cache_follows_in_place_updates_and_views():
    from samble_b200 import ops

    g = gen(77)
    x = randn(g, 3, 700, 96)
    base = randn(g, 256, 96) / 96 ** 0.5
    y = ops.linear(x, base)
    with torch.no_grad():
        base.mul_(2.0)                                           # a power of two: every product and sum doubles exactly
    y2 = ops.linear(x, base)
    assert torch.equal(y2, 2 * y), "the split of the old weight values was reused after an in-place update"
    # two views of one base with the same shape and strides, and a view sharing the first one's address
    top, bottom, half = base[:128], base[128:], base[:64]
    yt, yb, yh = ops.linear(x, top), ops.linear(x, bottom), ops.linear(x, half)
    assert torch.equal(yt, ops.linear(x, top.clone())) and torch.equal(yb, ops.linear(x, bottom.clone()))
    assert torch.equal(yh, ops.linear(x, half.clone())) and yh.shape[-1] == 64
    check_fp64(yb, fp64_statement(x, bottom), "second view")
    with torch.no_grad():
        bottom.mul_(0.5)                                         # through a view: the base's version moves too
    assert torch.equal(ops.linear(x, bottom), 0.5 * yb)
    assert torch.equal(ops.linear(x, top), yt)
