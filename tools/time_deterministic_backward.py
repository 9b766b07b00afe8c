"""Cost of the ordered (deterministic) backward against the atomic one, in one run with the two modes alternating.

  python tools/time_deterministic_backward.py [--reps 20] [--warmup 3] [--json out.json]

Times with CUDA events, after warm-up, the backward of the three ops whose scatters the mode changes, at the shipped
shapes (B = 16 clouds of N = 2048 points):
  group       center_diff, K = 32, C = 64             (the EdgeConv train path; index_points_bwd_kernel)
  n2p         Neighbor2Point core, C = 128, 4 heads, K = 32
  gather      gather_by_idx, C = 128, M = 1024
the worst case of the ordered fold, a hub (index_points with all 2048 * 32 edges of a cloud on one point, C = 64), and one
seg training step (train mode, forward + backward, B = 16, N = 2048).  Each row prints the median per call of
both modes; `atomic` is torch.use_deterministic_algorithms(False), `ordered` is True (warn_only, so an ATen op without a
deterministic implementation warns instead of stopping the measurement).  The card name and its power limit go beside
the numbers.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import warnings

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from samble_b200 import models, ops  # noqa: E402
from samble_b200.config import seg_config  # noqa: E402
from samble_b200.testing import fill_state_dict_, synthetic_clouds, synthetic_features  # noqa: E402

DEV = "cuda:0"


def card() -> str:
    name = torch.cuda.get_device_name(0)
    try:
        p = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=60)
        power = p.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return f"{name}, power limit {power}"


def set_mode(ordered: bool) -> None:
    torch.use_deterministic_algorithms(ordered, warn_only=True)


def timed(fn, reps: int) -> list:
    """ms of each of reps calls of fn(), each between its own pair of events."""
    ts = []
    for _ in range(reps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1))
    return ts


def median(v: list) -> float:
    v = sorted(v)
    return 0.5 * (v[(len(v) - 1) // 2] + v[len(v) // 2])


def op_cases():
    B, N = 16, 2048
    g = torch.Generator().manual_seed(0)
    cases = {}
    x = synthetic_features(B, 64, N, 1).to(DEV).requires_grad_(True)
    out, _ = ops.group(x, 32, "center_diff")
    probe = torch.randn(out.shape, generator=g).to(DEV)
    cases["group center_diff B16 N2048 K32 C64"] = lambda: torch.autograd.grad(out, x, probe, retain_graph=True)
    qkv = torch.randn(B, N, 384, generator=g).to(DEV).requires_grad_(True)
    idx = ops.knn_indices(synthetic_features(B, 128, N, 2).to(DEV), 32, ordered=False)
    att = ops.n2p_attend(qkv, idx, 4)
    p2 = torch.randn(att.shape, generator=g).to(DEV)
    cases["n2p B16 N2048 C128 H4 K32"] = lambda: torch.autograd.grad(att, qkv, p2, retain_graph=True)
    pcd = synthetic_features(B, 128, N, 3).to(DEV).requires_grad_(True)
    sel = torch.stack([torch.randperm(N, generator=g)[:1024] for _ in range(B)]).view(B, 1, 1024).to(DEV)
    gat = ops.gather_by_idx(pcd, sel)
    p3 = torch.randn(gat.shape, generator=g).to(DEV)
    cases["gather_by_idx B16 N2048 C128 M1024"] = lambda: torch.autograd.grad(gat, pcd, p3, retain_graph=True)
    hub_pts = synthetic_features(B, N, 64, 4).to(DEV).requires_grad_(True)
    hub = ops.index_points(hub_pts, torch.zeros(B, N, 32, dtype=torch.int64, device=DEV))
    p4 = torch.randn(hub.shape, generator=g).to(DEV)
    cases["index_points hub: all 65536 edges on one point, C64"] = lambda: torch.autograd.grad(hub, hub_pts, p4, retain_graph=True)
    return cases


def seg_step_case():
    B, N = 16, 2048
    cfg = seg_config()
    m = models.ShapeNetModel(cfg)
    m.load_state_dict(fill_state_dict_(m.state_dict(), seed=1, sharpen=2.0))
    m = m.to(DEV).train()
    x, cat = synthetic_clouds(B, N, 4)
    x, cat = x.to(DEV), cat.to(DEV)
    with torch.no_grad():
        m(x, cat)                                          # first dynamic boundary estimate

    def step():
        m.zero_grad(set_to_none=True)
        m(x, cat).square().mean().backward()
    return {"seg train step B16 N2048 (forward + backward)": step}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--json", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_deterministic_backward.py measures on a GPU; none is visible")
    warnings.simplefilter("ignore", UserWarning)           # warn_only: ATen's notices would flood the output
    cases = {**op_cases(), **seg_step_case()}
    res = {}
    for name, fn in cases.items():
        for mode in (False, True, False, True):            # warm both modes
            set_mode(mode)
            for _ in range(a.warmup):
                fn()
        torch.cuda.synchronize()
        t = {False: [], True: []}
        for r in range(4):                                 # alternate: atomic, ordered, atomic, ...
            for mode in (False, True):
                set_mode(mode)
                t[mode] += timed(fn, max(1, a.reps // 4))
        set_mode(False)
        res[name] = {"atomic_ms": median(t[False]), "ordered_ms": median(t[True]),
                     "atomic_all_ms": t[False], "ordered_all_ms": t[True]}
    info = card()
    print(f"# {info}; torch {torch.__version__}; medians of {a.reps} calls per mode, modes alternating")
    print(f"{'backward':<56} {'atomic ms':>10} {'ordered ms':>11} {'ratio':>6}")
    for name, r in res.items():
        print(f"{name:<56} {r['atomic_ms']:>10.3f} {r['ordered_ms']:>11.3f} {r['ordered_ms'] / r['atomic_ms']:>6.2f}")
    if a.json:
        with open(a.json, "w") as f:
            json.dump({"card": info, "torch": torch.__version__, "results": res}, f, indent=1)


if __name__ == "__main__":
    main()
