"""ctypes binding of libsamble_b200.so (the C ABI declared in include/samble_b200.h).

There is deliberately no fallback: if the library is missing, or a tensor is not on a
CUDA device, every entry point raises.  PyTorch is used only to own device memory and
to name the current stream.
"""
from __future__ import annotations

import ctypes as C
import os
import re
from typing import Dict, Tuple

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(HERE, "_lib", "libsamble_b200.so")
HEADER = os.path.join(HERE, "..", "include", "samble_b200.h")

_p, _i, _ll, _sz, _f = C.c_void_p, C.c_int, C.c_longlong, C.c_size_t, C.c_float

# name -> (restype, argtypes); mirrors include/samble_b200.h one to one (tests/test_abi.py
# parses the header and checks that nothing is missing on either side).
PROTOTYPES: Dict[str, Tuple[object, tuple]] = {
    "samble_abi_version": (_i, ()),
    "samble_last_error": (C.c_char_p, ()),
    "samble_launch_count": (_ll, ()),
    "samble_reset_launch_count": (None, ()),
    "samble_profile_enable": (None, (_i,)),
    "samble_profile_report": (_i, (C.c_char_p, _sz)),
    "samble_selftest_tc_gemm": (_i, (_p, _p, _i, _p, _p, _p, _p)),
    "samble_selftest_tc_gemm_ts": (_i, (_p, _p, _i, _p, _i, _i, _p, _p)),
    "samble_selftest_tc_gemm_ts_bf16": (_i, (_p, _p, _i, _p, _i, _i, _p, _i, _p)),
    "samble_selftest_mma_rate": (_i, (_i, _i, _i, _p, _p)),
    "samble_selftest_mma_rate_ex": (_i, (_i, _i, _i, _i, _i, _i, _p, _p)),
    "samble_set_knn_mode": (None, (_i,)),
    "samble_knn_workspace_bytes": (_sz, (_i, _i, _i, _i)),
    "samble_knn": (_i, (_p, _ll, _ll, _ll, _p, _ll, _ll, _ll, _i, _i, _i, _i, _i, _p, _i, _p, _i, _p, _sz, _p)),
    "samble_index_points": (_i, (_p, _p, _i, _i, _i, _i, _i, _p, _p)),
    "samble_group": (_i, (_p, _p, _i, _i, _i, _i, _i, _i, _p, _p)),
    "samble_gather_by_idx": (_i, (_p, _p, _i, _i, _i, _i, _i, _p, _p)),
    "samble_index_points_backward": (_i, (_p, _p, _i, _i, _i, _i, _i, _p, _p)),
    "samble_gather_by_idx_backward": (_i, (_p, _p, _i, _i, _i, _i, _i, _p, _p)),
    "samble_n2p_attend_backward": (_i, (_p, _p, _p, _ll, _p, _i, _i, _i, _i, _i, _i, _p, _ll, _p, _p, _p, _ll, _p)),
    "samble_reverse_index_workspace_bytes": (_sz, (_i, _i)),
    "samble_reverse_index": (_i, (_p, _i, _i, _i, _i, _p, _p, _p, _sz, _p)),
    "samble_scatter_rows_ordered": (_i, (_p, _ll, _ll, _ll, _i, _p, _i, _p, _p, _p, _ll, _ll, _i, _i, _i, _i, _p, _ll, _ll, _ll, _p)),
    "samble_n2p_attend_backward_edges": (_i, (_p, _p, _p, _ll, _p, _i, _i, _i, _i, _i, _i, _p, _ll, _p, _ll, _p, _p, _p)),
    "samble_transpose": (_i,(_p, _ll, _ll, _i, _i, _i, _p, _p)),
    "samble_neighbor_mask": (_i, (_p, _i, _i, _i, _i, _p, _p)),
    "samble_split_tf32": (_i, (_p, _p, _ll, _p)),
    "samble_ds_row_stats_fast_workspace_bytes": (_sz, (_i, _i)),
    "samble_ds_row_stats_fast": (_i, (_p, _ll, _p, _p, _ll, _p, _i, _i, _i, _i, _p, _p, _p, _p, _sz, _p)),
    "samble_cloud_matmul": (_i, (_p, _ll, _p, _p, _ll, _i, _i, _i, _i, _p, _p, C.c_float, _p, _ll, _p, _ll, _p)),
    "samble_ds_select_rows": (_i, (_p, _ll, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _p, _p, _p)),
    "samble_linear_pool_workspace_bytes": (_sz, (_i, _i)),
    "samble_linear_pool": (_i, (_p, _ll, _p, _p, _ll, _p, _p, _ll, _i, _i, _i, _i, _i, _p, _p, _p, _sz, _p)),
    "samble_linear": (_i, (_p, _ll, _i, _p, _p, _ll, _p, _p, _ll, _i, _p, _ll, _i, _i, _p, _ll, _i, _i, _i, _i, _i, _p)),
    "samble_mlp2": (_i, (_p, _ll, _i, _i, _p, _p, _ll, _i, _p, _p, _ll, _i, _p, _p, _ll, _i, _p, _p, _ll, _i, _p, _ll, _i, _p, _ll, _i, _p)),
    "samble_set_mlp2_debug": (None, (_i,)),
    "samble_set_mlp2_probe": (None, (_p,)),
    "samble_set_edge_mode": (None, (_i,)),
    "samble_set_edge_debug": (None, (_i,)),
    "samble_edge_mlp_max": (_i, (_p, _ll, _p, _i, _p, _p, _i, _i, _i, _i, _i, _p, _ll, _p)),
    "samble_n2p_attend": (_i, (_p, _p, _p, _ll, _p, _i, _i, _i, _i, _i, _i, _p, _ll, _p, _p, _p, _ll, _p)),
    "samble_set_ds_mode": (None, (_i,)),
    "samble_set_n2p_mode": (None, (_i,)),
    "samble_set_gather_mode": (None, (_i,)),
    "samble_set_linear_debug": (None, (_i,)),
    "samble_set_knn_debug": (None, (_i,)),
    "samble_set_knn_probe": (None, (_p,)),
    "samble_ds_row_stats": (_i, (_p, _ll, _p, _ll, _p, _i, _i, _i, _i, _p, _p, _p, _p)),
    "samble_digits_bytes": (_sz, (_i, _i, _i)),
    "samble_digits": (_i, (_p, _ll, _ll, _i, _i, _i, _p, _i, _p, _p, _p, _p)),
    "samble_xgemm": (_i, (_p, _p, _i, _i, _p, _p, _i, _i, _i, _p, _ll, _p, _i, _i, _p)),
    "samble_ds_row_stats_exact_workspace_bytes": (_sz, (_i, _i)),
    "samble_ds_row_stats_exact": (_i, (_p, _p, _p, _p, _p, _ll, _p, _i, _i, _i, _i, _p, _p, _p, _p, _sz, _p)),
    "samble_ds_attend_rows_workspace_bytes": (_sz, (_i, _i, _i)),
    "samble_ds_attend_rows": (_i, (_p, _p, _p, _p, _p, _ll, _p, _p, _p, _p, _p, _i, _i, _i, _i, _i, _i, _p, _p, _sz, _p)),
    "samble_ds_edge_score_workspace_bytes": (_sz, (_i, _i)),
    "samble_ds_edge_score": (_i, (_p, _ll, _p, _ll, _p, _p, _p, _i, _i, _i, _i, _i, _p, _p, _sz, _p)),
    "samble_zscore": (_i, (_p, _i, _i, _p, _p)),
    "samble_bin_mask": (_i, (_p, _p, _p, _i, _i, _i, _p, _p)),
    "samble_num_points_to_choose": (_i, (_p, _p, _i, _i, _i, _p, _p)),
    "samble_downsample_index_topk": (_i, (_p, _p, _p, _i, _i, _i, _i, _p, _p)),
    "samble_ds_sample": (_i, (_p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _p, _p, _p)),
    "samble_sampling_probabilities": (_i, (_p, _p, _i, _i, _i, _i, _f, _f, _p, _p)),
    "samble_quantile_pick": (_i, (_p, _ll, _i, _p, _p)),
    "samble_boundary_ema": (_i, (_p, _i, C.c_double, _i, _i, _p, _p, _p)),
    "samble_interpolate3_workspace_bytes": (_sz, (_i, _i, _i)),
    "samble_interpolate3": (_i, (_p, _p, _p, _i, _i, _i, _i, _p, _p, _p, _p, _sz, _p)),
    "samble_interpolate3_search": (_i, (_p, _p, _i, _i, _i, _p, _p, _p, _sz, _p)),
    "samble_interpolate3_gather_rows": (_i, (_p, _p, _p, _ll, _i, _i, _i, _i, _p, _ll, _p)),
    "samble_interpolate3_rows": (_i, (_p, _p, _p, _ll, _i, _i, _i, _i, _p, _ll, _p, _sz, _p)),
}

_lib = None


def header_symbols() -> set:
    with open(HEADER) as f:
        text = re.sub(r"/\*.*?\*/", "", f.read(), flags=re.S)
    return set(re.findall(r"\b(samble_[a-z0-9_]+)\s*\(", text))


def lib() -> C.CDLL:
    """The loaded library; raises (never falls back) when it has not been built."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise RuntimeError(
                f"samble_b200: native library {LIB_PATH} is missing. Build it with "
                "`python -m samble_b200._build` (needs nvcc); there is no CPU or PyTorch fallback.")
        handle = C.CDLL(LIB_PATH)
        for name, (res, args) in PROTOTYPES.items():
            fn = getattr(handle, name)
            fn.restype, fn.argtypes = res, list(args)
        _lib = handle
    return _lib


def check(rc: int, what: str) -> None:
    if rc == 0:
        return
    msg = lib().samble_last_error().decode() or what
    if rc == -1:
        raise ValueError(msg)
    raise RuntimeError(f"{what} failed ({rc}): {msg}")


def need_cuda(*tensors: torch.Tensor) -> torch.device:
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("samble_b200 runs on CUDA tensors only (no CPU path); got a tensor on " + str(t.device))
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"samble_b200: tensors on different devices ({dev} vs {t.device})")
    if dev is not None and dev.index is not None and dev.index != torch.cuda.current_device():
        # kernels are launched on the calling thread's current device, on that device's current stream
        raise RuntimeError(f"samble_b200: tensors live on {dev} but the current CUDA device is cuda:{torch.cuda.current_device()}; "
                           "call torch.cuda.set_device(...) or wrap the call in `with torch.cuda.device(...)`")
    return dev


def no_grad_check(*tensors: torch.Tensor) -> None:
    """The fused inference kernels have no backward: refuse rather than return silently wrong gradients.  (The
    differentiable path is samble_b200.autograd; the blocks pick it whenever a gradient could be asked for.)"""
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise RuntimeError("samble_b200: this fused kernel is forward-only and a tensor (or module parameter) that requires "
                           "grad reached it; run under torch.no_grad(), or use the differentiable path")


def ptr(t) -> C.c_void_p:
    return C.c_void_p(0 if t is None else t.data_ptr())


def stream() -> C.c_void_p:
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


_workspaces: Dict[Tuple[int, int], torch.Tensor] = {}


def workspace(nbytes: int, device: torch.device) -> torch.Tensor:
    """Grow-only scratch per (device, stream): stream order makes reuse across calls safe, and a
    stable pointer keeps CUDA-graph replays valid (size it by one eager warm-up first)."""
    key = (device.index if device.index is not None else torch.cuda.current_device(),
           torch.cuda.current_stream(device).cuda_stream)
    ws = _workspaces.get(key)
    if ws is None or ws.numel() < nbytes:
        # (during CUDA-graph capture this allocation comes from the graph's private pool and stays
        # valid for every replay as long as this cache holds the tensor)
        ws = torch.empty(max(nbytes, 1 << 20), dtype=torch.uint8, device=device)
        _workspaces[key] = ws
    return ws


def profile(enable: bool) -> None:
    lib().samble_profile_enable(1 if enable else 0)


def profile_report() -> dict:
    """{kernel: (launches, total_ms)} of the launches recorded since profiling was enabled."""
    buf = C.create_string_buffer(1 << 16)
    check(lib().samble_profile_report(buf, len(buf)), "samble_profile_report")
    out = {}
    for line in buf.value.decode().splitlines():
        name, n, ms = line.rsplit(",", 2)
        out[name] = (int(n), float(ms))
    return out
