"""Every dispatch branch of the neighbour search (samble_knn, csrc/knn.cu knn_impl) against an fp64 referee, at its edges.

The tensor-core path is elsewhere judged mostly against the exact FFMA kernel, and both read the same channel statistics
and the same normalised copy, so a fault in those shared stages would go unseen there.  Here every case is judged by an
fp64 search on the raw inputs that shares nothing with the library, at the widths, sizes, index ranges, list capacities,
tile tails and input layouts where each branch changes behaviour.  Each case also checks, through the library's launch
profiler, that the kernels which ran are the ones of the branch it names, so a gate change that moves a case onto
another branch fails here.

The case table is built from the constants of csrc/knn.cu and csrc/knn_tc.cu (parsed, not copied), so the capacity and
tail cases follow a retune.  The gates of knn_impl are restated below; the CPU-only tests check the restatement against
the sources and the case table against the cells it must cover.
"""
import os
import re
from dataclasses import dataclass

import pytest
import torch

from samble_b200.testing import launched

DEV = "cuda:0"
CSRC = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "samble_b200", "csrc")


def _source(name):
    with open(os.path.join(CSRC, name)) as f:
        return f.read()


def _const(src, name):
    m = re.search(rf"constexpr int {name} = (\d+);", src)
    assert m, f"constexpr int {name} not found"
    return int(m.group(1))


_KNN, _KNN_TC, _TILE = _source("knn.cu"), _source("knn_tc.cu"), _source("gemm_tile.cuh")
K_TC_ROWS, K_TC_TILE, K_TC_CAP = (_const(_KNN_TC, n) for n in ("kTcRows", "kTcTile", "kTcCap"))
K_XYZ_CAP, K_XYZ_CHUNK, K_XYZ_QW = (_const(_KNN, n) for n in ("kXyzCap", "kXyzChunk", "kXyzQW"))
XYZ_CTA_QUERIES = 8 * K_XYZ_QW                 # 8 warps of kXyzQW queries per xyz CTA
_two_pass = re.search(r"if \(g_knn_mode != 1 && Nr >= (\d+)\)", _KNN)
XYZ_TWO_PASS_MIN = int(_two_pass.group(1)) if _two_pass else -1

# ------------------------------------------------------------------ the gates of knn_impl, restated
# (test_restated_gates_match_the_sources pins each line these restate)
GATE_LINES = {
    "knn.cu": [
        "p.xyz = C <= 3;",
        "p.Cp = p.xyz ? 4 : (int)align_up(C, 32);",
        "bool knn_stats_point_major(long long sc, int C) { return sc == 1 && C >= 8; }",
        "return sc == 1 && C % 4 == 0 && sn % 4 == 0 && sb % 4 == 0 && (uintptr_t)x % 16 == 0;",
        "const bool fuse_stats = !plan.xyz && C <= 512 && knn_stats_point_major(a_sc, C) && prep_point_major(a, a_sb, a_sn, a_sc, C) &&\n"
        "                          (self || prep_point_major(b, b_sb, b_sn, b_sc, C));",
        "const bool self = (a == b) && a_sb == b_sb && a_sn == b_sn && a_sc == b_sc && Nq == Nr;",
        "const bool use_tc = g_knn_mode != 1 && knn_tc_eligible(Nq, Nr, C, k);",
        "const bool big = (long long)ceil_div(Nq, 128) * B >= 2 * 148 && knn_feat_smem<DotTileCfg<8>>(Cp) <= 200 * 1024;",
        "return (Cfg::smem_floats(Cp) + 2 * Cfg::TQ * 32 + Cfg::TQ) * sizeof(float);",
        'SAMBLE_REQUIRE(C <= 512, "samble_knn: C=%d > 512", C);',
        'SAMBLE_REQUIRE(B <= 65535, "samble_knn: B=%d > 65535", B);',
    ],
    "knn_tc.cu": ["return C >= 4 && Cp <= 128 && k <= 32 && Nr <= 65535 && Nr >= k;"],
    "gemm_tile.cuh": [
        "static constexpr int MN = 8;",
        "static constexpr int TQ = 16 * MQ;",
        "static constexpr int TN = 16 * MN;",
        "static constexpr int KC = 16;",
        "static constexpr int LDB = KC + 4;",
        "static constexpr int LDS_ = TN + 4;",
        "static __host__ __device__ int lda(int Cp) { return Cp + 4; }",
        "return (size_t)TQ * lda(Cp) + 2 * TN * LDB + (size_t)TQ * LDS_;",
    ],
}
NUM_SMS = 148


def padded_width(C):
    return 4 if C <= 3 else -(-C // 32) * 32


def feat_smem_bytes(mq, Cp):
    """knn_feat_smem<DotTileCfg<mq>>(Cp) (knn.cu, gemm_tile.cuh)."""
    tq, tn, kc = 16 * mq, 16 * 8, 16
    smem_floats = tq * (Cp + 4) + 2 * tn * (kc + 4) + tq * (tn + 4)
    return (smem_floats + 2 * tq * 32 + tq) * 4


def tc_eligible(Nq, Nr, C, k):
    return C >= 4 and padded_width(C) <= 128 and k <= 32 and Nr <= 65535 and Nr >= k


def predicted_path(B, Nq, Nr, C, k):
    """The branch knn_impl takes in auto mode: xyz / xyz2 / tc / tile8 (DotTileCfg<8>) / tile4 (DotTileCfg<4>)."""
    if C <= 3:
        return "xyz2" if Nr >= XYZ_TWO_PASS_MIN else "xyz"
    if tc_eligible(Nq, Nr, C, k):
        return "tc"
    big = -(-Nq // 128) * B >= 2 * NUM_SMS and feat_smem_bytes(8, padded_width(C)) <= 200 * 1024
    return "tile8" if big else "tile4"


# layouts: (B,N,C) logical view -> element strides (sb, sn, sc) and the element offset of its first value in its buffer
LAYOUTS = {
    "pm": lambda B, N, C: ((N * C, C, 1), 0),                   # contiguous point-major
    "slice384": lambda B, N, C: ((N * 384, 384, 1), 128),       # columns 128:128+C of a (B,N,384) row buffer
    "offset4": lambda B, N, C: ((N * (C + 4), C + 4, 1), 1),    # columns 1:1+C of a (B,N,C+4) buffer: 4-byte offset
    "cm": lambda B, N, C: ((C * N, 1, N), 0),                   # channel-major (B,C,N)
    "cstride": lambda B, N, C: ((N * 2 * C, 2 * C, 2), 0),      # every other column of a (B,N,2C) buffer
}


def _prep_point_major(strides, off, C):
    sb, sn, sc = strides
    return sc == 1 and C % 4 == 0 and sn % 4 == 0 and sb % 4 == 0 and off % 4 == 0   # (buffers are 16-byte aligned)


def predicted_stats(case):
    """fused (point-major slice statistics combined inside the prep kernel), combine (the same slices plus
    knn_stats_combine_kernel) or strided (the one-pass strided statistics kernel)."""
    a_strides, a_off = LAYOUTS[case.layout_a](case.B, case.Nq, case.C)
    b_strides, b_off = LAYOUTS[case.layout_b](case.B, case.Nr, case.C)
    pm_stats = a_strides[2] == 1 and case.C >= 8
    fuse = (case.C > 3 and case.C <= 512 and pm_stats and _prep_point_major(a_strides, a_off, case.C)
            and (case.self_ or _prep_point_major(b_strides, b_off, case.C)))
    return "fused" if fuse else ("combine" if pm_stats else "strided")


def expected_kernels(path, stats, ordered):
    if path in ("xyz", "xyz2"):
        return {"knn_stats_kernel", "knn_prep_xyz_kernel", "knn_xyz_kernel" if path == "xyz" else "knn_xyz2_kernel"}
    k = {"knn_stats_kernel", "knn_prep_feat_kernel"} | ({"knn_stats_combine_kernel"} if stats == "combine" else set())
    if path == "tc":
        return k | {"knn_tc_threshold_kernel", "knn_tc_collect_kernel", "knn_rerank_kernel" if ordered else "knn_select_kernel"}
    return k | {"knn_feat_kernel"}


# ------------------------------------------------------------------ the case table


@dataclass(frozen=True)
class Case:
    cell: str
    B: int
    Nq: int
    Nr: int
    C: int
    k: int
    self_: bool
    path: str                  # the branch this case is about (asserted against predicted_path and the profiler)
    stats: str = ""            # "" -> fused / strided as the layout gives; asserted against predicted_stats
    layout: str = "pm"         # pm | slice384 | offset4 | cm | pm_cm (a point-major, b channel-major) | cstride
    data: str = "randn"        # randn | straddle | plant | dup | offset | scaled
    m: int = 0                 # dup: copies of one point
    judge: int = 0             # 0: judge every row; else that many seeded rows besides the tile boundaries
    seed: int = 0

    @property
    def layout_a(self):
        return "pm" if self.layout == "pm_cm" else self.layout

    @property
    def layout_b(self):
        return "cm" if self.layout == "pm_cm" else self.layout

    @property
    def generic(self):         # random data without constructed ties: counts toward the exact-order rate
        return self.data != "dup"

    @property
    def id(self):
        shape = f"N{self.Nq}" if self.self_ else f"Nq{self.Nq}-Nr{self.Nr}"
        extra = "" if self.data == "randn" else f"-{self.data}{self.m or ''}"
        lay = "" if self.layout == "pm" else f"-{self.layout}"
        return f"{self.cell}-C{self.C}-B{self.B}-{'self' if self.self_ else 'cross'}-{shape}-k{self.k}{extra}{lay}"


def _c(cell, B, Nq, Nr, C, k, path, **kw):
    """Nr = None: self search."""
    self_ = Nr is None
    return Case(cell, B, Nq, Nq if self_ else Nr, C, k, self_, path, **kw)


def build_cases():
    R, T, cap, xcap, ch, qc, two = K_TC_ROWS, K_TC_TILE, K_TC_CAP, K_XYZ_CAP, K_XYZ_CHUNK, XYZ_CTA_QUERIES, XYZ_TWO_PASS_MIN
    cases = [
        # xyz: one-pass below the two-pass switch, two-pass at it; candidate chunk tails with neighbours planted across
        # the chunk edges; query counts around one CTA; k = 1 and 32; C = 1, 2, 3; cross and self
        _c("xyz", 1, two - 1, None, 3, 32, "xyz"),
        _c("xyz", 1, two, None, 3, 32, "xyz2"),
        _c("xyz", 2, two - 1, None, 1, 1, "xyz"),
        _c("xyz", 2, qc + 1, None, 2, 32, "xyz"),
        _c("xyz", 1, qc + 1, two - 1, 3, 32, "xyz"),
        _c("xyz", 2, qc + 1, two, 2, 32, "xyz2"),
        _c("xyz", 1, qc - 1, ch - 1, 3, 32, "xyz2", data="straddle"),
        _c("xyz", 1, qc, ch, 3, 32, "xyz2", data="straddle"),
        _c("xyz", 2, qc + 1, ch + 1, 2, 1, "xyz2", data="straddle"),
        _c("xyz", 1, qc, 2 * ch + 1, 1, 32, "xyz2", data="straddle"),
        _c("xyz", 1, 2 * ch + 1, None, 3, 32, "xyz2", data="straddle"),
        _c("xyz", 1, ch + 1, None, 1, 32, "xyz2", data="straddle"),
        # the two-pass CTA's per-query list: m copies of one far point, m = kXyzCap - 1, kXyzCap (fits), kXyzCap + 1 (the
        # CTA falls back to the k-set algorithm)
        *[_c("xyz-cap", 1, 1024, None, 3, 32, "xyz2", data="dup", m=m) for m in (xcap - 1, xcap, xcap + 1)],
        # tensor core, width steps: Cp 32 / 64 / 96 / 128, half-filled 64-wide K tiles, strided statistics below C = 8,
        # strided prep for C % 4 != 0
        *[_c("tc-width", 2, 600, None, C, 32, "tc", seed=C) for C in (4, 5, 7, 8, 31, 32, 33, 63, 64, 65, 100, 127, 128)],
        # tensor core, query-tile and candidate-tile tails
        _c("tc-tail", 1, 2, 1000, 64, 32, "tc"),
        _c("tc-tail", 2, R - 1, T, 64, 31, "tc"),
        _c("tc-tail", 2, R, T - 1, 64, 2, "tc"),
        _c("tc-tail", 1, R + 1, T + 1, 16, 1, "tc"),
        _c("tc-tail", 1, R + 1, 1000, 64, 32, "tc"),
        _c("tc-tail", 1, 2 * R + 1, 32, 64, 32, "tc"),             # Nr = k = 32: every candidate is in
        _c("tc-tail", 2, R - 1, 2, 32, 2, "tc"),                   # Nr = k = 2
        _c("tc-tail", 2, 2, T + 1, 96, 31, "tc"),
        _c("tc-tail", 1, R + 1, None, 32, 32, "tc"),
        # tensor core, candidate indices with bit 15 set (the list word keeps 16 index bits); queries planted on the
        # candidates at and around 32767 / 32768 and at the end
        *[_c("tc-idx16", 1, 3 * R, Nr, 32, 32, "tc", data="plant") for Nr in (32767, 32768, 32769, 65535)],
        _c("tc-idx16", 1, 65535, None, 32, 32, "tc", judge=256),
        # tensor core, the candidate list's capacity: m copies of one far point, kTcCap - 1 (re-ranked), kTcCap and
        # kTcCap + 1 (saturated: the row's warp searches it exactly)
        *[_c("tc-cap", 1, 1024, None, 32, 32, "tc", data="dup", m=m) for m in (cap - 1, cap, cap + 1)],
        # the exact tile kernel past the tensor-core widths (C <= 512 is samble_knn's limit)
        _c("tile-wide", 2, 300, None, 129, 32, "tile4"),
        _c("tile-wide", 1, 200, 2500, 160, 16, "tile4"),
        _c("tile-wide", 1, 1000, None, 256, 32, "tile4"),
        _c("tile-wide", 1, 300, 500, 384, 8, "tile4"),
        _c("tile-wide", 1, 257, None, 511, 32, "tile4"),
        _c("tile-wide", 1, 130, 700, 512, 32, "tile4"),
        # the exact tile kernel past the tensor core's 16-bit candidate indices
        _c("tile-bigN", 1, 65536, None, 32, 32, "tile8", judge=256),
        _c("tile-bigN", 1, 300, 70000, 64, 32, "tile4", data="plant"),
        # input layouts: the statistics and prep variants
        _c("layout", 2, 700, None, 64, 32, "tc"),
        _c("layout", 2, 500, None, 128, 32, "tc", layout="slice384"),
        _c("layout", 2, 500, None, 128, 32, "tc", layout="offset4"),
        _c("layout", 2, 700, None, 64, 32, "tc", layout="cm"),
        _c("layout", 1, 1000, None, 3, 32, "xyz2", layout="cm"),
        _c("layout", 2, 300, 900, 64, 32, "tc", layout="pm_cm"),
        _c("layout", 2, 400, None, 16, 32, "tc", layout="cstride"),
        # grid.y = B at its limit
        _c("grid", 65535, 40, None, 3, 16, "xyz", judge=64),
        _c("grid", 65535, 40, None, 16, 16, "tc", judge=64),
        # a large common offset (normalisation cancels it) and badly scaled channels / clouds
        _c("spread", 2, 800, None, 64, 32, "tc", data="offset"),
        _c("spread", 2, 800, None, 3, 32, "xyz2", data="offset"),
        _c("spread", 2, 800, None, 64, 32, "tc", data="scaled"),
        _c("spread", 2, 800, None, 3, 32, "xyz2", data="scaled"),
    ]
    return [c if c.stats else Case(**{**c.__dict__, "stats": predicted_stats(c)}) for c in cases]


CASES = build_cases()

# refusals: (id, B, Nq, Nr, C, k, exception)
REFUSALS = [
    ("C513", 1, 40, 40, 513, 8, ValueError),
    ("B65536-xyz", 65536, 4, 4, 3, 2, ValueError),
    ("B65536-tc", 65536, 4, 4, 16, 2, ValueError),
    ("k33", 1, 40, 40, 16, 33, ValueError),
    ("k-over-Nr", 1, 40, 20, 16, 21, RuntimeError),
]
CELLS = ["xyz", "xyz-cap", "tc-width", "tc-tail", "tc-idx16", "tc-cap", "tile-wide", "tile-bigN", "layout", "grid", "spread",
         "refusal"]


# ------------------------------------------------------------------ inputs


def _raw(case, N, seed):
    """(B,N,C) fp32 CPU cloud of the case's kind; a per-case seeded torch.Generator."""
    g = torch.Generator().manual_seed(seed)
    B, C = case.B, case.C
    x = torch.randn(B, N, C, generator=g)
    if case.data == "offset":
        x = x + 1e3
    elif case.data == "scaled":                            # cloud 0: channel scales 1e-3 .. 1e2; cloud 1: x 1e4
        x[0] *= torch.logspace(-3, 2, C)
        x[1:] *= 1e4
    return x


def _far(C, t):
    return torch.full((C,), 4.0 + 3.0 * t)


def make_inputs(case):
    """Logical (B,Nq,C) / (B,Nr,C) fp32 CPU clouds: a, b (b is a for a self search)."""
    a = _raw(case, case.Nq, 1000 + case.seed + 7 * case.C + case.Nq)
    b = a if case.self_ else _raw(case, case.Nr, 2000 + case.seed + 7 * case.C + case.Nr)
    g = torch.Generator().manual_seed(3000 + case.Nr)
    if case.data == "straddle":
        # tight far clusters over indices [e - 16, e + 16) for every candidate-chunk edge e and the cloud's end, and
        # queries inside them: the true neighbours straddle the chunk edge
        edges = [e for e in range(K_XYZ_CHUNK, case.Nr, K_XYZ_CHUNK)] + [case.Nr]
        for t, e in enumerate(edges):
            lo, hi = max(0, e - 16), min(case.Nr, e + 16)
            b[:, lo:hi] = _far(case.C, t) + 0.05 * torch.randn(case.B, hi - lo, case.C, generator=g)
            if not case.self_:
                a[:, 2 * t:2 * t + 2] = _far(case.C, t) + 0.05 * torch.randn(case.B, 2, case.C, generator=g)
    elif case.data == "plant":
        # the last queries sit next to candidates whose indices set bit 15 or 16, and next to the last candidate
        js = [j for j in (32766, 32767, 32768, 32769, 65534, 65535, 65536, case.Nr - 2, case.Nr - 1) if j < case.Nr]
        for t, j in enumerate(sorted(set(js))):
            a[:, case.Nq - 1 - t] = b[:, j] + 0.01 * torch.randn(case.B, case.C, generator=g)
    elif case.data == "dup":
        # m bitwise-identical copies of one far point at seeded scattered indices
        where = torch.randperm(case.Nr, generator=g)[:case.m]
        b[:, where] = _far(case.C, 1)
    return a, b


def to_layout(x, layout):
    """x (B,N,C) CPU -> the same values on the GPU as a (B,N,C) view with the layout's strides."""
    B, N, C = x.shape
    if layout == "pm":
        return x.to(DEV)
    if layout == "slice384":
        buf = torch.zeros(B, N, 384)
        buf[..., 128:128 + C] = x
        return buf.to(DEV)[..., 128:128 + C]
    if layout == "offset4":
        buf = torch.zeros(B, N, C + 4)
        buf[..., 1:1 + C] = x
        return buf.to(DEV)[..., 1:1 + C]
    if layout == "cm":
        return x.transpose(1, 2).contiguous().to(DEV).transpose(1, 2)
    if layout == "cstride":
        buf = torch.zeros(B, N, 2 * C)
        buf[..., ::2] = x
        return buf.to(DEV)[..., ::2]
    raise ValueError(layout)


def judged_rows(case, seed=77):
    """(cloud, row) pairs the referee judges: every row, or for large searches the rows at every 128-row tile boundary,
    the last tile, the rows around 32768 and a seeded sample (for a wide batch: whole clouds, the last ones included)."""
    B, Nq = case.B, case.Nq
    if not case.judge:
        return torch.arange(B * Nq)
    g = torch.Generator().manual_seed(seed)
    if B > 1:
        clouds = torch.cat([torch.arange(4), torch.arange(B - 4, B), torch.randint(0, B, (case.judge,), generator=g)]).unique()
        return (clouds[:, None] * Nq + torch.arange(Nq)[None]).reshape(-1)
    tile = torch.arange(0, Nq, K_TC_ROWS)
    rows = torch.cat([tile, (tile + K_TC_ROWS - 1).clamp(max=Nq - 1), torch.arange(int(tile[-1]), Nq),
                      torch.arange(32766, 32770), torch.randint(0, Nq, (case.judge,), generator=g)])
    return rows[rows < Nq].unique()


# ------------------------------------------------------------------ the fp64 referee
#
# Squared distances in fp64 on the raw inputs, centred on a's per-cloud mean (the library's normalisation is a per-cloud
# similarity transform, so it changes no order).  Per judged row i with kth the k-th smallest fp64 distance:
#
#   band_i = max(2e-5 * kth, (Cp + 8) * 2^-23 * (|a'_i|^2 + max_j |b'_j|^2))
#
# The second term bounds the error of the library's fp32 distance, u = 2^-24, S = |a'|^2 + |b'|^2 (scaled alike):
#   the dot product, one FMA chain over Cp channels:       Cp u sum_c |a_c b_c| <= Cp u S / 2, times 2 ........ Cp u S
#   |a'|^2 and |b'|^2, Cp rounded products and sums each: ....................................................... Cp u S
#   the sum of the norms and the final FMA (|result| <= 2 S): ................................................... 3 u S
#   the prep, (x - mean) / sigma rounded twice per coordinate (relative 2u): |d(a~,b~) - d(a,b)| <= 8 u S ....... 8 u S
# together (2 Cp + 11) u S <= (Cp + 8) 2^-23 S.  The xyz path's five-term distance is the Cp = 4 case of the same count.
# The first term is the relative fp32 near-tie band of knn_parity.
#
# The returned distance is -sqrt(d) of the normalised points; with sigma64 the oracle's scale:
#   |dist^2 - d64 / sigma64^2| <= band_i / sigma64^2 + 2^-21 d64 / sigma64^2
# where 2^-21 = 8u covers sqrtf, the square and the fp32 sigma (a C-term sum whose typical error grows as sqrt(C) u;
# at large C the band's second term, >= (Cp + 8) u d64, dominates).


class Referee:
    def __init__(self, case, a, b, idx, dist, rows):
        self.case, self.a, self.b, self.idx, self.dist, self.rows = case, a, b, idx, dist, rows
        self.matches = 0
        self.total = 0
        self.failures = []

    def fail(self, what, bad, rows):
        if bool(bad.any()):
            r = rows[bad.nonzero()[0, 0]]
            self.failures.append(f"{what}: {int(bad.sum())} rows, first (cloud {int(r) // self.case.Nq}, row {int(r) % self.case.Nq})")

    def run(self):
        c = self.case
        k, Cp = c.k, padded_width(c.C)
        rows = self.rows.to(DEV)
        clouds = (rows // c.Nq).unique().tolist()
        for bi in clouds:
            rb = rows[rows // c.Nq == bi]
            a64 = self.a[bi].double()
            b64 = self.b[bi].double()
            mu = a64.mean(0)
            sigma2 = float(a64.std(0).mean()) ** 2
            a0, b0 = a64 - mu, b64 - mu
            nb_max = float((b0 * b0).sum(-1).max())
            self.tie_groups(bi, rb, b64)
            chunk = max(1, (1 << 25) // c.Nr)                       # <= 256 MB of fp64 distances at a time
            for s in range(0, rb.numel(), chunk):
                rr = rb[s:s + chunk]
                q = rr % c.Nq
                d = torch.cdist(a0[q], b0, compute_mode="donot_use_mm_for_euclid_dist") ** 2      # (R, Nr) fp64
                ref_d, ref_i = d.topk(k, dim=1, largest=False, sorted=True)
                kth = ref_d[:, -1:]
                na = (a0[q] * a0[q]).sum(-1, keepdim=True)
                band = torch.maximum(2e-5 * kth, (Cp + 8) * 2.0 ** -23 * (na + nb_max))
                idx = self.idx.view(-1, k)[rr].long()
                in_range = ((idx >= 0) & (idx < c.Nr)).all(1)
                self.fail("index outside [0, Nr)", ~in_range, rr)
                idx = idx.clamp(0, c.Nr - 1)
                srt = idx.sort(1).values
                self.fail("repeated index", (srt[:, 1:] == srt[:, :-1]).any(1), rr)
                dl = d.gather(1, idx)
                self.fail("returned neighbour beyond kth + band", (dl > kth + band).any(1), rr)
                # every candidate nearer than kth - band must be returned (the returned indices are distinct)
                n_near = (d < kth - band).sum(1)
                self.fail("a clearly nearer candidate is missing", (dl < kth - band).sum(1) != n_near, rr)
                self.fail("returned order not ascending up to the band", (dl[:, 1:] - dl[:, :-1] < -band).any(1), rr)
                self.matches += int((idx == ref_i).sum())
                self.total += idx.numel()
                dist = self.dist.view(-1, k)[rr].double()
                err = (dist * dist - dl / sigma2).abs()
                self.fail("returned distance off", (err > band / sigma2 + 2.0 ** -21 * dl / sigma2).any(1), rr)
                del d
        return self

    def tie_groups(self, bi, rb, b64):
        """The tie rule, strictly: among returned members whose raw rows are bitwise identical, indices ascend with the
        position, and a group of identical points cut at k keeps its lowest indices."""
        c, k = self.case, self.case.k
        bits = self.b[bi].contiguous().view(torch.int32)
        _, inv = torch.unique(bits, dim=0, return_inverse=True)
        order = torch.argsort(inv, stable=True)
        counts = torch.bincount(inv)
        starts = torch.cumsum(counts, 0) - counts
        rank = torch.empty_like(inv)
        rank[order] = torch.arange(c.Nr, device=inv.device) - starts[inv[order]]      # earlier members of the own group
        if int(counts.max()) == 1:
            return
        idx = self.idx.view(-1, k)[rb].long().clamp(0, c.Nr - 1)
        gid = inv[idx]
        same = gid[:, :, None] == gid[:, None, :]
        earlier = idx[:, None, :] < idx[:, :, None]
        self.fail("a tie group cut at k did not keep its lowest indices", ((same & earlier).sum(-1) != rank[idx]).any(1), rb)
        later_pos = torch.ones(k, k, dtype=torch.bool, device=idx.device).triu(1)
        self.fail("tied indices out of ascending order", (same & later_pos & ~earlier.transpose(1, 2)).any(-1).any(-1), rb)


# ------------------------------------------------------------------ running a case


def _ordered(case, a, b):
    """Ordered search through the public op: (-dist, int64 idx)."""
    from samble_b200 import ops

    if case.layout == "cm":                                 # channel-major (B,C,N) self search
        x = a.transpose(1, 2)
        return ops._knn_strided(x, x, case.k, "bcn", True)
    return ops.knn(a, b, case.k)


def _any_order(case, a, b):
    from samble_b200 import ops

    if case.layout == "cm":
        return ops.knn_indices(a.transpose(1, 2), case.k, ordered=False)
    return ops._knn_strided(a, b, case.k, "bnc", False, torch.int32, ordered=False)[1]


_ORDER_RATE = {}      # case id -> (position-wise matches with the fp64 order, returned entries), generic cases only


@pytest.mark.gpu
@pytest.mark.parametrize("case", CASES, ids=[c.id for c in CASES])
def test_knn_dispatch_vs_fp64(case):
    from samble_b200 import _lib as L
    from samble_b200 import ops

    assert predicted_path(case.B, case.Nq, case.Nr, case.C, case.k) == case.path
    a_cpu, b_cpu = make_inputs(case)
    a = to_layout(a_cpu, case.layout_a)
    b = a if case.self_ else to_layout(b_cpu, case.layout_b)
    for t, lay, N in ((a, case.layout_a, case.Nq), (b, case.layout_b, case.Nr)):
        strides, off = LAYOUTS[lay](case.B, N, case.C)
        assert t.stride() == strides and t.storage_offset() == off and t.data_ptr() % 4 == 0

    (neg, idx), ran = launched(lambda: _ordered(case, a, b))
    assert set(ran) == expected_kernels(case.path, case.stats, True), sorted(ran)
    assert idx.dtype == torch.int64 and tuple(idx.shape) == (case.B, case.Nq, case.k) and neg.shape == idx.shape
    any_idx, ran = launched(lambda: _any_order(case, a, b))
    assert set(ran) == expected_kernels(case.path, case.stats, False), sorted(ran)
    assert any_idx.dtype == torch.int32
    assert torch.equal(any_idx.long().sort(-1).values, idx.sort(-1).values), "any-order set differs from the ordered set"
    if case.layout == "cm":                                 # the blocks' own entry point: int32, no distances
        assert torch.equal(ops.knn_indices(a.transpose(1, 2), case.k).long(), idx)

    if case.path in ("tc", "xyz2"):                         # the exact FFMA / k-set kernels, bit for bit
        lib = L.lib()
        try:
            lib.samble_set_knn_mode(1)
            neg1, idx1 = _ordered(case, a, b)
            torch.cuda.synchronize()
        finally:
            lib.samble_set_knn_mode(0)
        assert torch.equal(idx, idx1) and torch.equal(neg, neg1), "differs from the exact kernel (mode 1)"

    rows = judged_rows(case)
    a_dev = a_cpu.to(DEV)
    ref = Referee(case, a_dev, a_dev if case.self_ else b_cpu.to(DEV), idx, -neg, rows).run()
    assert not ref.failures, ref.failures
    if case.generic:
        _ORDER_RATE[case.id] = (ref.matches, ref.total)


@pytest.mark.gpu
@pytest.mark.parametrize("rid,B,Nq,Nr,C,k,exc", REFUSALS, ids=[r[0] for r in REFUSALS])
def test_knn_refusals(rid, B, Nq, Nr, C, k, exc):
    from samble_b200 import ops

    a = torch.zeros(B, Nq, C, device=DEV)
    a[:, :, 0] = torch.arange(Nq, dtype=torch.float32, device=DEV)
    b = a if Nq == Nr else torch.zeros(B, Nr, C, device=DEV)
    with pytest.raises(exc):
        ops.knn(a, b, k)


@pytest.mark.gpu
def test_exact_order_rate_over_generic_cases():
    """Position-wise agreement with the fp64 order over this file's generic random cases (the bar of test_knn_vs_oracle).
    Runs after the case tests; alone it has nothing to judge."""
    if not _ORDER_RATE:
        pytest.skip("no generic case ran in this session")
    m = sum(v[0] for v in _ORDER_RATE.values())
    n = sum(v[1] for v in _ORDER_RATE.values())
    worst = sorted(_ORDER_RATE.items(), key=lambda kv: kv[1][0] / kv[1][1])[:3]
    assert m / n >= 0.995, (m / n, worst)


# ------------------------------------------------------------------ CPU-side: the table and its restated gates


def test_restated_gates_match_the_sources():
    sources = {"knn.cu": _KNN, "knn_tc.cu": _KNN_TC, "gemm_tile.cuh": _TILE}
    for name, lines in GATE_LINES.items():
        for line in lines:
            assert line in sources[name], f"{name} no longer has: {line}"
    assert XYZ_TWO_PASS_MIN > 0, "the two-pass switch of knn_impl moved"
    assert K_TC_ROWS == K_TC_TILE == 128           # knn_impl's 128-row tile arithmetic (ceil_div(Nq, 128), align_up(Nr, 128))
    assert "Cfg::MQ == 4 ? 2 : 1" in _KNN          # DotTileCfg<4> / <8> are the only forms launched


def test_dot_tile_form_of_every_exact_case():
    """DotTileCfg<8> needs two CTAs of 128 rows per SM and its smem under 200 KB; Cp > 128 never fits it."""
    assert feat_smem_bytes(8, 128) <= 200 * 1024 < feat_smem_bytes(8, 160)
    assert feat_smem_bytes(4, 512) <= 227 * 1024
    exact = [c for c in CASES if c.path.startswith("tile")]
    assert {c.path for c in exact} == {"tile4", "tile8"}
    for c in exact:
        assert not tc_eligible(c.Nq, c.Nr, c.C, c.k), c.id
        assert predicted_path(c.B, c.Nq, c.Nr, c.C, c.k) == c.path, c.id


def test_case_table_covers_every_cell():
    ids = [c.id for c in CASES]
    assert len(ids) == len(set(ids))
    assert {c.cell for c in CASES} | {"refusal"} == set(CELLS)
    for c in CASES:
        assert predicted_path(c.B, c.Nq, c.Nr, c.C, c.k) == c.path, c.id
        assert c.Nq >= 2 and c.k <= c.Nr and c.B <= 65535 and c.C <= 512, c.id
    cell = lambda name: [c for c in CASES if c.cell == name]
    # xyz
    xyz = cell("xyz")
    assert {c.C for c in xyz} == {1, 2, 3} and {c.k for c in xyz} >= {1, 32} and {c.self_ for c in xyz} == {True, False}
    assert {"xyz", "xyz2"} == {c.path for c in xyz}
    assert {XYZ_TWO_PASS_MIN - 1, XYZ_TWO_PASS_MIN} <= {c.Nr for c in xyz}
    ch = K_XYZ_CHUNK
    assert {ch - 1, ch, ch + 1, 2 * ch + 1} <= {c.Nr for c in xyz if c.data == "straddle"}
    assert {XYZ_CTA_QUERIES - 1, XYZ_CTA_QUERIES, XYZ_CTA_QUERIES + 1} <= {c.Nq for c in xyz}
    assert sorted(c.m for c in cell("xyz-cap")) == [K_XYZ_CAP - 1, K_XYZ_CAP, K_XYZ_CAP + 1]
    assert all(c.path == "xyz2" and c.k == 32 and c.m <= c.Nr for c in cell("xyz-cap"))
    # tensor core
    width = cell("tc-width")
    assert {c.C for c in width} == {4, 5, 7, 8, 31, 32, 33, 63, 64, 65, 100, 127, 128}
    assert {padded_width(c.C) for c in width} == {32, 64, 96, 128}
    assert {c.stats for c in width} == {"fused", "combine", "strided"}
    tail = cell("tc-tail")
    assert {2, K_TC_ROWS - 1, K_TC_ROWS, K_TC_ROWS + 1, 2 * K_TC_ROWS + 1} <= {c.Nq for c in tail}
    assert {K_TC_TILE - 1, K_TC_TILE, K_TC_TILE + 1, 1000} <= {c.Nr for c in tail}
    assert any(c.Nr == c.k == 32 for c in tail) and any(c.Nr == c.k != 32 for c in tail)
    assert {1, 2, 31, 32} <= {c.k for c in tail}
    assert any(c.Nq < c.Nr for c in tail) and any(c.Nq > c.Nr for c in tail)
    idx16 = cell("tc-idx16")
    assert {32767, 32768, 32769, 65535} <= {c.Nr for c in idx16 if not c.self_ and c.B == 1 and c.Nq == 3 * K_TC_ROWS}
    assert any(c.self_ and c.Nr == 65535 and c.C == 32 for c in idx16)
    assert sorted(c.m for c in cell("tc-cap")) == [K_TC_CAP - 1, K_TC_CAP, K_TC_CAP + 1]
    # exact tile kernel
    wide = cell("tile-wide")
    assert {c.C for c in wide} == {129, 160, 256, 384, 511, 512}
    assert {c.self_ for c in wide} == {True, False} and any(c.Nr > ch for c in wide)
    big = cell("tile-bigN")
    assert {(c.self_, c.Nr, c.C, c.path) for c in big} == {(True, 65536, 32, "tile8"), (False, 70000, 64, "tile4")}
    # layouts, grid, spreads
    lay = cell("layout")
    assert {c.layout for c in lay} == {"pm", "slice384", "offset4", "cm", "pm_cm", "cstride"}
    assert {(c.layout, c.stats) for c in lay if c.path == "tc"} >= {
        ("pm", "fused"), ("slice384", "fused"), ("offset4", "combine"), ("cm", "strided"), ("pm_cm", "combine"),
        ("cstride", "strided")}
    assert {(c.B, c.path) for c in cell("grid")} == {(65535, "xyz"), (65535, "tc")}
    assert {(c.data, c.C) for c in cell("spread")} == {("offset", 64), ("offset", 3), ("scaled", 64), ("scaled", 3)}
    # refusals
    assert {(r[4] > 512, r[1] > 65535, r[5] > 32, r[5] > r[3]) for r in REFUSALS} >= {
        (True, False, False, False), (False, True, False, False), (False, False, True, False), (False, False, False, True)}


def test_cap_and_tail_cases_follow_the_parsed_constants():
    """A retune of kTcCap / kXyzCap / the tile and chunk sizes moves the edge cases with it."""
    assert sorted(c.m for c in build_cases() if c.cell == "tc-cap") == [K_TC_CAP + d for d in (-1, 0, 1)]
    assert all(K_TC_CAP + 1 <= c.Nr for c in CASES if c.cell == "tc-cap")
    assert all(c.m + 1 <= c.Nr for c in CASES if c.data == "dup")
