"""world_size-2 gloo tests (CPU) of the multi-GPU host logic: tile ownership, source ranges, gradient/normal-equation
all-reduce.  The kernels themselves need a GPU (tests/test_multigpu_gpu.py); here the collectives and partitioning run."""
import os

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from gs_icp_slam_b200 import sharding


def test_tile_masks_and_ranges_partition():
    for world in (2, 3, 8):
        masks = [sharding.tile_owner_mask(480, 640, world, r) for r in range(world)]
        assert torch.equal(sum(masks), torch.ones(1, 480, 640))
        m = sharding.tile_owner_mask(50, 70, world, 0)
        assert m.shape == (1, 50, 70) and m[0, :16, :16].all()
        for n in (0, 1, 12416, 2000000, 7):
            r = [sharding.source_range(n, world, k) for k in range(world)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(r[k][1] == r[k + 1][0] for k in range(world - 1))


def _worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = torch.Generator().manual_seed(0)
        pred = torch.rand((3, 48, 64), generator=g, requires_grad=False)
        target = torch.rand((3, 48, 64), generator=g)
        w = torch.rand((3, 48, 64), generator=g).requires_grad_(True)
        b = torch.rand((5,), generator=g).requires_grad_(True)
        mask = sharding.tile_owner_mask(48, 64, world, rank)
        loss = sharding.sharded_l1(pred * w + b[:3, None, None], target, mask, pred.numel())
        loss.backward()
        sharding.allreduce_grads([w, b])
        # normal equations: rank partial sums -> all-reduce (what the GICP kernels' in-kernel exchange computes)
        rows = torch.arange(100, dtype=torch.float64)[:, None] * torch.ones(28, dtype=torch.float64)
        lo, hi = sharding.source_range(100, world, rank)
        part = rows[lo:hi].sum(0)
        dist.all_reduce(part)
        if rank == 0:
            torch.save(dict(gw=w.grad, gb=b.grad, part=part, loss=loss.detach()), out)
    finally:
        dist.destroy_process_group()


def test_gloo_world2_matches_single_process(tmp_path):
    out = str(tmp_path / "r0.pt")
    port = 29500 + (os.getpid() % 1000)
    mp.spawn(_worker, args=(2, port, out), nprocs=2, join=True)
    got = torch.load(out)
    g = torch.Generator().manual_seed(0)
    pred = torch.rand((3, 48, 64), generator=g)
    target = torch.rand((3, 48, 64), generator=g)
    w = torch.rand((3, 48, 64), generator=g).requires_grad_(True)
    b = torch.rand((5,), generator=g).requires_grad_(True)
    ((pred * w + b[:3, None, None] - target).abs().mean()).backward()
    assert torch.allclose(got["gw"], w.grad, atol=1e-7)
    assert torch.allclose(got["gb"], b.grad, atol=1e-6)
    assert torch.allclose(got["part"], torch.arange(100, dtype=torch.float64).sum() * torch.ones(28, dtype=torch.float64))
