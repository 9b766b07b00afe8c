#!/usr/bin/env python
"""Benchmark of the SAMBLE hot path on B200 (contract: README of the task / DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--workload seg|cls|knn_ds] [--batch B | --global-batch G] [--points N]
                  [--dump-outputs DIR]
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...
  python bench.py --impl reference ...        # the reference's CPU algorithm (oracle port) on host cores

Workloads (BASELINE.json configs):
  seg     (default; configs 3 and 5) one SAMBLE ShapeNetPart segmentation forward: per-GPU batch of B=16 clouds
          (or --global-batch G split over the ranks: config 5, strong scaling), N=2048, k=32, 2048->1024->512
  cls     (config 2) one SAMBLE ModelNet40 classification forward, B=32/GPU, N=1024, 1024->512->256, nb=6
  knn_ds  (config 4) micro-benchmark at N=8192 and N=16384: ops.knn (C=3 and C=128, k=32) and one DownSampleToken
          layer (N -> N/2), us per batch with the roofline of each, the CPU oracle beside it at B=1
All in eval mode with frozen bin boundaries and topk sampling, on synthetic clouds with seeded weights.
`value` = clouds/s with inputs resident in HBM (whole step replayed as one CUDA graph); `e2e` = the same forward fed
from HOST (pinned) buffers with a host copy of the result, every copy inside the timed region.  The batch is sharded
by cloud across ranks with no collective on the path.  One JSON line is printed by rank 0.
`--steps K` is the number of timed steps (graph replays for knn_ds) of every arm.
--dump-outputs DIR (seg / cls, native): the logits of the last timed step, all ranks' clouds in order, go to
DIR/logits.npy.  Inputs, weights and the calibration batch are seeded, so two builds run with the same arguments can be
compared output for output.
"""
from __future__ import annotations

import argparse
import json
import os
import sys
import threading
import time

import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRICS = {"seg": "clouds/sec SAMBLE seg fwd (N=2048)", "cls": "clouds/sec SAMBLE cls fwd (N=1024)",
           "knn_ds": "kNN+sampling us/batch (N=8192, 16384)"}
UNIT = "clouds/s"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--workload", default="seg", choices=["seg", "cls", "knn_ds"])
    ap.add_argument("--batch", type=int, default=None, help="clouds per GPU per step (default 16 seg / 32 cls)")
    ap.add_argument("--global-batch", type=int, default=None, help="total clouds per step, split over the ranks (strong scaling)")
    ap.add_argument("--points", type=int, default=None)
    ap.add_argument("--impl", default="native", choices=["native", "reference"])
    ap.add_argument("--cpu-steps", type=int, default=2)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="launch kernel by kernel instead of replaying a CUDA graph")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the logits of the last timed step as DIR/logits.npy (float32)")
    a = ap.parse_args()
    a.points = a.points or (1024 if a.workload == "cls" else 2048)
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "native" or a.workload == "knn_ds"):
        ap.error("--dump-outputs writes the logits of the native seg / cls forward")
    return a


def per_rank_batch(args, world):
    if args.global_batch is not None:
        if args.global_batch % world:
            raise SystemExit(f"--global-batch {args.global_batch} is not divisible by {world} ranks")
        return args.global_batch // world
    return args.batch or (32 if args.workload == "cls" else 16)


def workload_config(args, world, B):
    N = args.points
    if args.workload == "seg":
        w = (f"SAMBLE ShapeNetPart seg forward, B={B}/GPU N={N} k=32 M=[{N // 2},{N // 4}] nb=4, eval, frozen boundaries, "
             f"sample_mode=topk")
    elif args.workload == "cls":
        w = (f"SAMBLE ModelNet40 cls forward, B={B}/GPU N={N} k=32 M=[{N // 2},{N // 4}] nb=6, eval, frozen boundaries, "
             f"sample_mode=topk")
    else:
        w = "kNN (C=3, C=128; k=32) + DownSampleToken (N -> N/2) micro-benchmark at N=8192 and N=16384"
    return {"workload": w, "global_batch": B * world, "points": N, "parallelism": f"cloud-sharded x{world}",
            "l2": "256 MiB scratch write between timed steps (L2 flush)"}


def build_model(workload, N):
    from samble_b200 import models
    from samble_b200.config import cls_config, seg_config
    from samble_b200.testing import fill_state_dict_

    cfg = (seg_config if workload == "seg" else cls_config)(M=(N // 2, N // 4))
    model = (models.ShapeNetModel if workload == "seg" else models.ModelNetModel)(cfg)
    sd = fill_state_dict_(model.state_dict(), seed=1, sharpen=4.0)
    model.load_state_dict(sd)
    return cfg, model, sd


# ------------------------------------------------------------------------------- CPU arm


def cpu_reference_rate(workload, batch, points, steps, warmup):
    """The reference's algorithm (oracle port: dense cdist/topk/softmax on ATen CPU) on host cores."""
    from oracle import samble_oracle as O
    from samble_b200.testing import synthetic_clouds

    # torchrun exports OMP_NUM_THREADS=1; the CPU arm is entitled to every host core it can use
    torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    cfg, _, sd = build_model(workload, points)
    x, cat = synthetic_clouds(batch, points, seed=2)
    states = [O.DSState(True), O.DSState(True)]
    fwd = (lambda: O.seg_forward(sd, cfg, x, cat, states)) if workload == "seg" else (lambda: O.cls_forward(sd, cfg, x, states))
    times = []
    with torch.no_grad():
        fwd()                                           # calibration
        for s in states:
            s.dynamic = False
        for i in range(warmup + steps):
            t0 = time.perf_counter()
            fwd()
            if i >= warmup:
                times.append(time.perf_counter() - t0)
    dt = sum(times) / len(times)
    return batch / dt, dt


def cpu_knn_ds(N, reps=1):
    """oracle ops.knn (C=3, C=128) and downsample_token at B=1 (the reference needs ~6 GB of N x N temporaries per cloud
    at N=16384): seconds per call."""
    from oracle import samble_oracle as O
    from samble_b200.testing import synthetic_features

    torch.set_num_threads(max(1, len(os.sched_getaffinity(0))))
    _, _, sd = build_model("seg", N)
    out = {}
    with torch.no_grad():
        for C in (3, 128):
            a = synthetic_features(1, N, C, 3)
            t0 = time.perf_counter()
            for _ in range(reps):
                O.knn(a, a, 32)
            out[f"knn_c{C}_s"] = (time.perf_counter() - t0) / reps
        x = synthetic_features(1, 128, N, 4)
        st = O.DSState(True)
        t0 = time.perf_counter()
        for _ in range(reps):
            O.downsample_token(sd, "block.downsample_list.0.", x, N // 2, 32, 4, st)
        out["downsample_token_s"] = (time.perf_counter() - t0) / reps
    return out


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    world = max(1, args.gpus)
    B = per_rank_batch(args, world)
    cores = max(1, len(os.sched_getaffinity(0)))
    if args.workload == "knn_ds":
        res = {str(N): cpu_knn_ds(N, reps=args.steps) for N in (8192, 16384)}
        line = {"impl": "reference", "metric": METRICS["knn_ds"], "value": res["8192"]["downsample_token_s"] * 1e6, "unit": "us/batch",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": 0, "higher_is_better": False, "scaling": "weak", "vs_baseline": None,
                "dtype": "f32", "data": "synthetic", "config": workload_config(args, world, 1), "results_s_per_call_B1": res,
                "cpu_baseline": {"value": res["8192"]["downsample_token_s"] * 1e6, "unit": "us/batch", "cores": cores, "kind": "port",
                                 "sample": f"oracle knn (C=3, C=128) and downsample_token at B=1, N=8192 and 16384, {args.steps} calls each"},
                "e2e": {"value": res["8192"]["downsample_token_s"] * 1e6, "unit": "us/batch", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line), flush=True)
        return
    # the SAME per-GPU batch as the native arm (a CPU step takes seconds at the default size: pass a small --steps)
    steps, warmup = args.steps, 1
    rate, dt = cpu_reference_rate(args.workload, B, args.points, steps, warmup)
    line = {"impl": "reference", "metric": METRICS[args.workload], "value": rate, "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
            "warmup": warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
            "scaling": "strong" if args.global_batch is not None else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, world, B),
            "cpu_baseline": {"value": rate, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                             "sample": f"{args.workload} forward of B={B} clouds N={args.points} per step (one rank's share), {steps} timed "
                                       f"steps after {warmup} warm-up (reference is pure Python/ATen; its CPU path = the oracle port, "
                                       f"bit-exact to it)"},
            "e2e": {"value": rate, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------- clocks


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.samples, self.reasons, self.max_mhz, self.stop_flag = [], set(), None, False
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    NAMES = {0x8: "hw_slowdown", 0x40: "hw_thermal_slowdown", 0x20: "sw_thermal_slowdown", 0x4: "sw_power_cap",
             0x80: "hw_power_brake", 0x2: "applications_clocks_setting", 0x100: "display_clock_setting"}

    def run(self):
        if self.nv is None:
            return
        while not self.stop_flag:
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                mask = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                for bit, name in self.NAMES.items():
                    if mask & bit:
                        self.reasons.add(name)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


# ------------------------------------------------------------------------------- native arm


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return d, "measured (MEASURED_PEAKS.json)"
    return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0}, "fallback (B200_PROFILING.md)"


def linear_census(run_model):
    """Algorithmic bytes / FLOPs of the point-wise linear layers of one forward: every call of ops.linear /
    ops.linear_pool is intercepted once and its operands counted (activations in + weights + activations out
    (+ residual); 2*M*K*Nout FLOPs)."""
    from samble_b200 import ops

    tot = {"bytes": 0.0, "flops": 0.0, "calls": 0}
    real_linear, real_pool = ops.linear, ops.linear_pool

    def lin(xx, w, **kw):
        y = real_linear(xx, w, **kw)
        nout, k = w.shape[0], w[0].numel()
        m = xx.numel() // k
        res = kw.get("residual")
        tot["bytes"] += 4.0 * (xx.numel() + w.numel() + y.numel() + (res.numel() if res is not None else 0))
        tot["flops"] += 2.0 * m * k * nout
        tot["calls"] += 1
        return y

    def pool(xx, w, **kw):
        r = real_pool(xx, w, **kw)
        nout, k = w.shape[0], w[0].numel()
        m = xx.numel() // k
        tot["bytes"] += 4.0 * (xx.numel() + w.numel() + 2 * (m // 32) * nout)     # partial max/sum rows instead of y
        tot["flops"] += 2.0 * m * k * nout
        tot["calls"] += 1
        return r

    real_mlp2 = ops.mlp2

    def mlp2(xx, w1, w2, **kw):
        y = real_mlp2(xx, w1, w2, **kw)
        hd, k = w1.shape[0], w1[0].numel()
        m = xx.numel() // k
        res = kw.get("residual")
        # the hidden (m x hd) activation is neither written nor read: it is not part of the algorithmic bytes any more
        tot["bytes"] += 4.0 * (xx.numel() + w1.numel() + w2.numel() + y.numel() + (res.numel() if res is not None else 0))
        tot["flops"] += 2.0 * m * hd * (k + w2.shape[0])
        tot["calls"] += 1
        return y

    ops.linear, ops.linear_pool, ops.mlp2 = lin, pool, mlp2
    try:
        run_model()
        torch.cuda.synchronize()
    finally:
        ops.linear, ops.linear_pool, ops.mlp2 = real_linear, real_pool, real_mlp2
    return tot


def ds_flops(n, m, d=128, nb=4, k=32):
    """SURVEY 8d: feature kNN 2 N^2 C + q/k/v 6 N D^2 + QK^T 2 N (N+nb) D + edge pass 2 N K D + selected rows 2 M (N+nb) D."""
    return 2.0 * n * n * d + 6.0 * n * d * d + 2.0 * n * (n + nb) * d + 2.0 * n * k * d + 2.0 * m * (n + nb) * d


def graphed_us(fn, reps=20, flush=None):
    """device time of fn() replayed as ONE CUDA graph (median of reps), us"""
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side), torch.no_grad():
        for _ in range(2):
            fn()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.no_grad(), torch.cuda.graph(g):
        fn()
    for _ in range(3):
        g.replay()
    ts = []
    for _ in range(reps):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        g.replay()
        e1.record()
        e1.synchronize()
        ts.append(e0.elapsed_time(e1) * 1e3)
    ts.sort()
    return ts[len(ts) // 2]


def knn_sampling_path(model, run_model, B, N, nb, pk, pk_src, flush):
    """The north-star path (BASELINE.json's secondary metric, SURVEY 8d's 'kNN + DownSample path'): both DownSampleToken
    blocks of the step -- feature kNN + q/k/v + QK^T row statistics + edge scores + bins / k / per-bin top-k + selected
    rows x V -- replayed as one CUDA graph on the inputs they see inside the model."""
    ds_list = list(model.block.downsample_list)
    seen = {}
    hooks = [ds.register_forward_pre_hook(lambda mod, a, i=i: seen.__setitem__(i, tuple(t.detach().clone() if torch.is_tensor(t) else t for t in a)))
             for i, ds in enumerate(ds_list)]
    try:
        run_model()
    finally:
        for h in hooks:
            h.remove()

    def both():
        for i, ds in enumerate(ds_list):
            ds(*seen[i])

    us = graphed_us(both, flush=flush)
    flops = (ds_flops(N, N // 2, nb=nb) + ds_flops(N // 2, N // 4, nb=nb)) * B
    ach = flops / (us * 1e-6) / 1e12
    bf16 = pk["bf16_tflops_sustained"]
    # what the tensor pipe actually executes per algorithmic product: the kNN runs 1 + 3 bf16 passes (threshold, collect),
    # the exact-product GEMMs 10 digit products (q/k/v projection and QK^T), the selected-row attention 3 tf32 (= 6 bf16-rate) units
    def executed(n, m, d=128):
        return 4 * 2.0 * n * n * d + 10 * (6.0 * n * d * d + 2.0 * n * n * d) + 6 * 2.0 * m * n * d * 2
    ex = (executed(N, N // 2) + executed(N // 2, N // 4)) * B / (us * 1e-6) / 1e12
    return {"kernel": "kNN + DownSampleToken path (both blocks, CUDA-graph replay)", "bound": "tensor", "achieved": ach, "peak": bf16,
            "unit": "TFLOP/s", "frac": ach / bf16, "traffic": None, "peak_source": pk_src + ", bf16 sustained (every MMA on this path is kind::f16)",
            "us_per_batch": us, "clouds": B, "algorithmic_gflop_per_batch": flops / 1e9,
            "executed_bf16_tflops": ex, "executed_frac_of_peak": ex / bf16,
            "note": "achieved = ALGORITHMIC fp32 FLOPs (SURVEY 8d: 3.68 GFLOP per seg cloud) / graph-replayed device time. The path is "
                    "fp32-exact by construction: the tensor pipe executes 4x (kNN: bf16 split passes) to 10x (exact-product digit GEMMs) "
                    "the algorithmic products, so `executed_frac_of_peak` is the pipe utilisation and `frac` the price of exactness"}


def ncu_traffic(family):
    """DRAM bytes per step of one kernel family from the committed `ncu --set full` capture of the seg step
    (profiles/r2_traffic.json, written by tools/ncu_table.py); None when the file is absent."""
    try:
        with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "profiles", "r2_traffic.json")) as f:
            return json.load(f)["families"][family]
    except Exception:
        return None


def linear_roofline(ms, census, pk, workload="seg"):
    """The point-wise linear layers (linear_tma_kernel): 3xTF32 => fp32-equivalent tensor peak = tf32 peak / 3."""
    sec = ms * 1e-3
    tf32 = pk["bf16_tflops_sustained"] / 2
    ach = census["flops"] / sec / 1e12
    tr = None
    if workload == "seg":
        fams = [f for f in (ncu_traffic("linear_tma_kernel"), ncu_traffic("mlp2_kernel")) if f]
        if fams:
            tr = {"dram_bytes_per_step": sum(f["dram_bytes_per_step"] for f in fams), "launches_per_step": sum(f["launches_per_step"] for f in fams)}
    return {"kernel": "linear_tma_kernel + mlp2_kernel (all point-wise linear layers of the step)", "bound": "tensor", "achieved": ach, "peak": tf32 / 3,
            "unit": "TFLOP/s (fp32-equivalent)", "frac": ach / (tf32 / 3), "ms_per_step": ms, "calls_per_step": census["calls"],
            "algorithmic_gb_per_step": census["bytes"] / 1e9, "hbm_gbs": census["bytes"] / sec / 1e9,
            "flop_per_byte": census["flops"] / census["bytes"],
            "traffic": (tr["dram_bytes_per_step"] / tr["launches_per_step"]) if tr else None,
            "traffic_note": "DRAM read+write bytes per launch (ncu --set full, profiles/r2r_final_full.md), average over the two families' "
                            f"{tr['launches_per_step']} launches of the seg step; algorithmic bytes per launch: "
                            f"{census['bytes'] / max(census['calls'], 1):.0f}" if tr else None,
            "note": "3 kind::tf32 MMAs per fp32-class product: peak = (bf16 sustained / 2) / 3; the layers sit above the 3xTF32 ridge "
                    "(35 FLOP/B), so the tensor pipe is the binding roof"}


def run_knn_ds(args, dev, pk, pk_src, flush):
    """BASELINE config 4."""
    from samble_b200 import blocks, ops
    from samble_b200.config import seg_config
    from samble_b200.testing import fill_state_dict_, synthetic_features
    from samble_b200 import models

    out = {}
    bf16 = pk["bf16_tflops_sustained"]
    for N in (8192, 16384):
        B = 8 if N == 8192 else 4                       # >= 2 waves of 128-row tiles on 148 SMs
        res = {"B": B}
        for C in (3, 128):
            a = synthetic_features(B, N, C, 3).to(dev)
            us = graphed_us(lambda: ops.knn(a, a, 32), reps=args.steps, flush=flush)
            flops = 2.0 * N * N * C * B
            res[f"knn_c{C}"] = {"us_per_batch": us, "algorithmic_tflops": flops / (us * 1e-6) / 1e12,
                                 "bound": "fp32 pipe" if C == 3 else "tensor",
                                 "frac": (N * N * (C + 1) * B / (us * 1e-6)) / (148 * 128 * pk.get("sm_max_mhz", 1965.0) * 1e6) if C == 3
                                 else flops / (us * 1e-6) / 1e12 / bf16}
        cfg = seg_config(M=(N // 2, N // 4))
        m = models.ShapeNetModel(cfg)
        m.load_state_dict(fill_state_dict_(m.state_dict(), seed=1, sharpen=4.0))
        ds = m.block.downsample_list[0].eval().to(dev)
        x = synthetic_features(B, 128, N, 4).to(dev)
        with torch.no_grad():
            ds(x)
        ds.dynamic_boundaries_enable = False
        us = graphed_us(lambda: ds(x), reps=args.steps, flush=flush)
        fl = ds_flops(N, N // 2) * B
        res["downsample_token"] = {"us_per_batch": us, "algorithmic_tflops": fl / (us * 1e-6) / 1e12, "bound": "tensor",
                                   "frac": fl / (us * 1e-6) / 1e12 / bf16}
        out[str(N)] = res
    return out


DUMP_BYTES = 64 * 10**6


def dump_outputs(directory, name, y):
    """Write y (clouds along dim 0) as <directory>/<name>.npy in float32.  When that would exceed DUMP_BYTES, a fixed
    seeded sample of whole clouds is written instead and their indices (ascending) go to <name>_clouds.npy (float64)."""
    import numpy as np

    y = y.float().cpu()
    os.makedirs(directory, exist_ok=True)
    if y.numel() * 4 > DUMP_BYTES:
        keep = (DUMP_BYTES - 1024) // (y[0].numel() * 4 + 8)    # room for both .npy headers and the indices
        idx = torch.randperm(y.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        y = y[idx]
        np.save(os.path.join(directory, f"{name}_clouds.npy"), idx.double().numpy())
    np.save(os.path.join(directory, f"{name}.npy"), y.numpy())


def run_native(args):
    import torch.distributed as dist

    from samble_b200 import _lib as L
    from samble_b200 import models
    from samble_b200.testing import synthetic_clouds

    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the native path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    torch.backends.cuda.matmul.allow_tf32 = False          # stock GEMMs stay true fp32 (SURVEY 8c)
    torch.backends.cudnn.allow_tf32 = False
    pk, pk_src = peaks()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lib = L.lib()

    if args.workload == "knn_ds":
        if rank == 0:
            sampler = ClockSampler(local)
            sampler.start()
            res = run_knn_ds(args, dev, pk, pk_src, flush)
            sampler.stop_flag = True
            sampler.join()
            line = {"metric": METRICS["knn_ds"], "value": res["8192"]["downsample_token"]["us_per_batch"], "unit": "us/batch", "n_gpus": 1,
                    "steps": args.steps, "warmup": 5, "higher_is_better": False, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                    "data": "synthetic", "config": workload_config(args, 1, res["8192"]["B"]), "clocks": sampler.result(),
                    "results": res, "gpu_launches": int(lib.samble_launch_count())}
            if not args.no_cpu_baseline:
                cpu = {str(N): cpu_knn_ds(N) for N in (8192, 16384)}
                line["cpu_baseline"] = {"value": cpu["8192"]["downsample_token_s"] * 1e6, "unit": "us/batch (B=1)",
                                        "cores": torch.get_num_threads(), "kind": "port", "results_s_per_call_B1": cpu,
                                        "sample": "oracle knn (C=3, C=128) and downsample_token at B=1, one call each"}
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    B, N = per_rank_batch(args, world), args.points
    seg = args.workload == "seg"
    cfg, model, _ = build_model(args.workload, N)
    model = model.eval().to(dev)
    nb = cfg.feature_learning_block.downsample.bin.num_bins[0]
    # every rank owns its own shard of the global batch: clouds [rank*B, (rank+1)*B)
    xh, cath = synthetic_clouds(B * world, N, seed=2)
    xh, cath = xh[rank * B:(rank + 1) * B].contiguous().pin_memory(), cath[rank * B:(rank + 1) * B].contiguous().pin_memory()
    xc, catc = synthetic_clouds(B, N, seed=1002)            # calibration batch
    x, cat = xh.to(dev), cath.to(dev)
    ins = (x, cat) if seg else (x,)
    ins_h = (xh, cath) if seg else (xh,)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(step_fn, steps, tail_fn=None):
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
        barrier()
        lib.samble_reset_launch_count()
        for i, (s, e) in enumerate(evs):
            flush.zero_()                                  # evict L2 between timed steps
            s.record()
            step_fn()
            if tail_fn is not None and i == steps - 1:
                tail_fn()                                  # e.g. the last step's own D2H: nothing escapes the timed regions
            e.record()
        barrier()
        ms = sum(s.elapsed_time(e) for s, e in evs)
        mine = torch.tensor([ms], dtype=torch.float64, device=dev)
        allms = [torch.zeros_like(mine) for _ in range(world)]
        if world > 1:
            dist.all_gather(allms, mine)
        else:
            allms = [mine]
        per_rank = [float(t.item()) for t in allms]
        return max(per_rank), per_rank, int(lib.samble_launch_count())

    with torch.no_grad():
        model(xc.to(dev), catc.to(dev)) if seg else model(xc.to(dev))      # calibration batch (dynamic boundaries)
        models.freeze_boundaries(model)
        lib.samble_reset_launch_count()
        y = model(*ins)
        launches_per_step = int(lib.samble_launch_count())
        out_h = torch.empty(y.shape, dtype=torch.float32).pin_memory()
        run = model
        pipe = None
        if not args.no_graph:
            from samble_b200.runtime import GraphedForward, HostPipeline

            run = GraphedForward(model, *ins)              # whole step = one graph launch
            pipe = HostPipeline(run)       # the serving loop a host-resident caller uses: D2H of step i overlaps step i+1

        last = {}

        def step_resident():
            last["y"] = run(*ins)

        def step_e2e():
            # every timed step contains: H2D of its inputs, the forward, and the wait for the PREVIOUS step's D2H (which
            # ran beside this step's compute); the last step also waits for its own (tail_fn) -- all copies are timed
            if pipe is None:
                yy = model(*[t.to(dev, non_blocking=True) for t in ins_h])
                out_h.copy_(yy, non_blocking=True)
            else:
                pipe.submit(*ins_h)
                pipe.wait_previous()

        for _ in range(max(3, args.warmup)):
            step_resident()
        sampler = ClockSampler(local)
        sampler.start()
        ms, per_rank, launches = timed(step_resident, args.steps)
        # (the graph's output buffer is overwritten by the e2e steps below)
        y_last = last["y"].clone() if args.dump_outputs else None
        for _ in range(2):
            step_e2e()
        ms_e2e, per_rank_e2e, _ = timed(step_e2e, args.steps, tail_fn=(pipe.wait_all if pipe is not None else None))
        sampler.stop_flag = True
        sampler.join()
        # every rank samples ITS OWN GPU: a rank that runs slower than its peers shows here whether clocks / a power or
        # thermal cap explain it (the job is timed as the maximum over ranks)
        clocks_all = [sampler.result()]
        if world > 1:
            clocks_all = [None] * world
            dist.all_gather_object(clocks_all, sampler.result())

        # per-kernel device time of one profiled forward (CUDA events around every launch of ours); the concurrent branches
        # (ops.fork: neighbour search beside the projections) are serialised for this census so that every event pair
        # times its kernel alone -- the timed steps above ran with them on
        from samble_b200 import ops as _ops
        _ops.CONCURRENT_BRANCHES = False
        L.profile(True)
        torch.cuda.synchronize()
        t0 = torch.cuda.Event(enable_timing=True)
        t1 = torch.cuda.Event(enable_timing=True)
        t0.record()
        for _ in range(3):
            model(*ins)
        t1.record()
        torch.cuda.synchronize()
        prof = L.profile_report()
        L.profile(False)
        census = linear_census(lambda: model(*ins))
        _ops.CONCURRENT_BRANCHES = True
        north = knn_sampling_path(model, lambda: model(*ins), B, N, nb, pk, pk_src, flush) if rank == 0 else None

    value = B * world * args.steps / (ms / 1e3)
    e2e_value = B * world * args.steps / (ms_e2e / 1e3)
    if args.dump_outputs:
        ys = [y_last]
        if world > 1:
            ys = [torch.empty_like(y_last) for _ in range(world)]
            dist.all_gather(ys, y_last)
        if rank == 0:
            dump_outputs(args.dump_outputs, "logits", torch.cat(ys))
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    native_ms = {k: v[1] / 3 for k, v in prof.items()}
    step_ms = ms / args.steps                     # the graph-replayed step the kernels' event-timed durations are set against
    north["share_of_step"] = north["us_per_batch"] * 1e-3 / step_ms
    line = {"metric": METRICS[args.workload], "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(3, args.warmup), "ms_per_step": step_ms, "higher_is_better": True,
            "scaling": "strong" if args.global_batch is not None else "weak", "vs_baseline": None,
            "dtype": "f32", "data": "synthetic", "config": workload_config(args, world, B), "clocks": sampler.result(),
            "per_rank_ms_per_step": [round(t / args.steps, 4) for t in per_rank],
            "per_rank_clocks": [{"sm_mhz": c["sm_mhz"], "reasons": c["reasons"]} for c in clocks_all],
            "e2e": {"value": e2e_value, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "per_rank_ms_per_step": [round(t / args.steps, 4) for t in per_rank_e2e],
                    "h2d_bytes_per_step": int(sum(t.numel() * 4 for t in ins_h)), "d2h_bytes_per_step": int(out_h.numel() * 4)},
            "gpu_launches": launches_per_step * args.steps, "launch_mode": "eager" if args.no_graph else "cuda_graph",
            "roofline": north,
            "roofline_linear": linear_roofline((native_ms.get("linear_tma_kernel", 0.0) + native_ms.get("mlp2_kernel", 0.0)) or 1e-9, census, pk, args.workload),
            "kernels_ms_per_step": {k: round(v, 4) for k, v in sorted(native_ms.items(), key=lambda kv: -kv[1])},
            "native_share_of_step": min(1.0, sum(native_ms.values()) / step_ms)}
    if not args.no_cpu_baseline and world == 1:
        bs = min(B, 16)
        rate, dt = cpu_reference_rate(args.workload, bs, N, args.cpu_steps, 1)
        line["cpu_baseline"] = {"value": rate, "unit": UNIT, "cores": torch.get_num_threads(), "kind": "port",
                                "sample": f"oracle {args.workload} forward, B={bs} N={N}, {args.cpu_steps} timed steps after 1 warm-up"}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    a = parse()
    # stdout carries exactly ONE JSON line.  Native libraries write banners there on some boxes (NCCL prints "NCCL version ..." at communicator
    # creation whatever NCCL_DEBUG_FILE says): file descriptor 1 points at stderr while the benchmark runs and is restored for the result line.
    sys.stdout.flush()
    _real_stdout = os.dup(1)
    os.dup2(2, 1)
    _print = print

    def print(*args, **kw):          # noqa: A001  (the result lines below go to the real stdout)
        sys.stdout.flush()
        os.dup2(_real_stdout, 1)
        try:
            _print(*args, **kw)
            sys.stdout.flush()
        finally:
            os.dup2(2, 1)

    if a.impl == "reference":
        run_reference(a)
    else:
        run_native(a)
