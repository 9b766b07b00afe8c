"""world_size-2 gloo tests (CPU): the only collective on the path is the reference's (nb-1)-float all_reduce in the
dynamic bin-boundary update (utils/ops.py:191-199); and the bench's batch sharding covers the global batch exactly once."""
import os

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from oracle import samble_oracle as O
from samble_b200 import ops


def _cpu_quantile_pick(ranked, num_bins):
    """the oracle's statement of utils/ops.py:182-189 (stands in for the native launch: this box has no GPU)"""
    n = ranked.nelement()
    pos = (torch.arange(1, num_bins) / num_bins * n).int().long()
    return ranked[pos].clone()


def _cpu_boundary_ema(cut_sum, world, old, num_bins, momentum):
    """the oracle's statement of utils/ops.py:198-233"""
    cut = cut_sum / world
    if old is not None:
        upper, lower = old[0].detach().clone(), old[1].detach().clone()
        cut = upper[0, 0, 0, 1:] * momentum + (1 - momentum) * cut
        upper[0, 0, 0, 1:] = cut
        lower[0, 0, 0, :-1] = cut
        return [upper, lower]
    inf = torch.full((1,), float("inf"))
    return [torch.cat([inf, cut]).reshape(1, 1, 1, num_bins), torch.cat([cut, -inf]).reshape(1, 1, 1, num_bins)]


def _worker(rank, world, port, z_all, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    # host logic under test: sort -> local quantiles -> ONE all_reduce of nb-1 floats -> / world -> EMA, state threaded
    # through calls.  The two native launches are GPU-only; their CPU statements stand in here.  The kernels are checked
    # bit for bit against the same statements run by ATen on the GPU, for 1 to 8 ranks, by
    # tests/test_gpu_ops.py::test_boundary_update_bit_exact_vs_aten_on_the_gpu.  ATen on the CPU rounds `cut / world`
    # differently from ATen on CUDA (a true division on the CPU, a product with the fp32 reciprocal on CUDA), so these stand-ins
    # match the GPU to the last bit of the division only -- hence the tolerance below.
    ops._quantile_pick, ops._boundary_ema = _cpu_quantile_pick, _cpu_boundary_ema
    try:
        z = z_all[rank]
        bnd = ops.update_sampling_score_bin_boundary(None, z, 4, 0.99)                    # init: rank-mean of local quantiles
        bnd = ops.update_sampling_score_bin_boundary(bnd, z * 1.5, 4, 0.99)               # EMA step
        out[rank] = torch.stack([bnd[0].flatten(), bnd[1].flatten()])
    finally:
        dist.destroy_process_group()


def test_dynamic_boundary_allreduce_matches_reference_semantics():
    world = 2
    g = torch.Generator().manual_seed(0)
    z_all = [torch.randn(3, 1, 200, 1, generator=g) for _ in range(world)]
    out = mp.Manager().dict()
    mp.spawn(_worker, args=(world, 29531, z_all, out), nprocs=world, join=True)

    def fake_all_reduce(scale):
        # what torch.distributed.all_reduce(SUM) would hand every rank: the sum of the ranks' local quantiles
        def f(cut):
            n = z_all[0].nelement()
            pos = (torch.arange(1, 4) / 4 * n).int().long()
            total = sum(torch.sort((z * scale).flatten(), descending=True)[0][pos] for z in z_all)
            return total, world
        return f

    ref = O.update_sampling_score_bin_boundary(None, z_all[0], 4, 0.99, fake_all_reduce(1.0))
    ref = O.update_sampling_score_bin_boundary(ref, z_all[0] * 1.5, 4, 0.99, fake_all_reduce(1.5))
    expect = torch.stack([ref[0].flatten(), ref[1].flatten()])
    for r in range(world):
        torch.testing.assert_close(out[r], expect, rtol=1e-6, atol=1e-7)       # every rank ends with the same boundaries
    assert torch.equal(out[0], out[1])


def test_bench_sharding_is_a_partition():
    """bench.py gives rank r the clouds [r*B, (r+1)*B) of one seeded global batch: disjoint and complete."""
    from samble_b200.testing import synthetic_clouds

    B, world, N = 4, 2, 64
    x, _ = synthetic_clouds(B * world, N, seed=2)
    shards = [x[r * B:(r + 1) * B] for r in range(world)]
    assert torch.equal(torch.cat(shards), x)
