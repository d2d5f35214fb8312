"""Multi-GPU parity (needs >= 2 GPUs; run with `gpurun --gpus 2 -- python -m pytest tests/test_multigpu_gpu.py -m gpu`):
tile-sharded rasterizer + point-sharded GICP must reproduce the single-GPU results through the library's in-kernel
exchange over peer memory (CUDA IPC / NVLink)."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

WORKER = r'''
import os, sys
import numpy as np, torch, torch.distributed as dist
sys.path.insert(0, os.environ["GSICP_ROOT"])
rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(rank); dev = torch.device("cuda", rank)
dist.init_process_group("nccl", device_id=dev)
from gs_icp_slam_b200 import rasterizer as R, sharding, synthetic as S
from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer
import pygicp
from tests.util import scene_tensors

def render(grp):
    shard = grp is not None
    if shard: grp.attach_rasterizer()
    g, cm, t, c, cam = scene_tensors(20000, 7, dev, size=(320, 240))
    for k in t: t[k].requires_grad_(True)
    m2 = torch.zeros_like(t["means3D"], requires_grad=True)
    rs = GaussianRasterizationSettings(240, 320, c["tanfovx"], c["tanfovy"], torch.zeros(3, device=dev), 1.0, c["viewmatrix"], c["projmatrix"], 0, c["campos"], False, False)
    out = []
    for rep in range(3 if shard else 1):   # repeated iterations: accumulators are cleared, barriers stay in step
        for k in t: t[k].grad = None
        depth, color, radii, used = GaussianRasterizer(rs)(means3D=t["means3D"], means2D=m2, opacities=t["opacities"], shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
        gt = torch.full_like(color, 0.5)
        if shard:
            mask = sharding.tile_owner_mask(240, 320, world, rank, dev)
            loss = sharding.sharded_l1(color, gt, mask, color.numel()) + 0.1 * sharding.sharded_l1(depth, gt[:1], mask, depth.numel())
            loss.backward()   # the render moments are exchanged inside the rasterizer's backward
            img = color.detach().clone(); dist.all_reduce(img)   # disjoint tiles, zeros elsewhere
        else:
            ((color - gt).abs().mean() + 0.1 * (depth - gt[:1]).abs().mean()).backward()
            img = color.detach()
        out.append((img, {k: t[k].grad.clone() for k in t}, radii))
    if shard: R.set_tile_shard(1, 0); R.set_comm(None)
    return out

tgt, src, T = S.gicp_pair(30000, 20000, 60, 61)
big_t, big_s, Tb = S.gicp_pair(150000, 150000, 62, 63, 0.001, scale=2.0)
def align(grp, host_lm, clouds=(tgt, src), corr_dist=0.05):
    r = pygicp.FastGICP(); r.set_max_correspondence_distance(corr_dist); r.set_max_knn_distance(99999)
    r.set_host_lm(host_lm)
    if grp is not None: grp.attach_gicp(r)
    r.set_input_target(clouds[0]); r.calculate_target_covariance_with_filter(); r.set_input_source(clouds[1])
    pose = r.align(np.eye(4))
    return pose, r.last_iterations, r.get_source_correspondence(), r.get_source_rotationsq(), r.get_source_scales()

img1, g1, r1 = render(None)[0]
p1 = align(None, False)
pb = align(None, False, (big_t, big_s), 0.1)
grp = sharding.ShardGroup(dev, world, rank)
for imgN, gN, rN in render(grp):
    assert torch.equal(r1, rN)
    assert torch.equal(img1, imgN), "sharded image differs"
    for k in g1:
        err = (g1[k] - gN[k]).abs().max() / (g1[k].abs().max() + 1e-30)
        assert err < 2e-4, (k, float(err))
for host_lm in (False, True):
    pN = align(grp, host_lm)
    assert p1[1] == pN[1] and np.abs(p1[0] - pN[0]).max() <= 1e-6, (host_lm, p1[1], pN[1], np.abs(p1[0] - pN[0]).max())
    assert np.array_equal(p1[2][0], pN[2][0]) and np.array_equal(p1[2][1], pN[2][1]), "sharded correspondences differ after the merge"
    assert np.array_equal(p1[3], pN[3]) and np.array_equal(p1[4], pN[4]), "sharded rotations / scales differ after the merge"
# above kLmPersistentMax points per rank: the full-occupancy kernels with in-kernel exchange
pN = align(grp, False, (big_t, big_s), 0.1)
assert pb[1] == pN[1] and np.abs(pb[0] - pN[0]).max() <= 1e-6
assert np.array_equal(pb[2][0], pN[2][0])
grp.close()
dist.barrier(); dist.destroy_process_group()
if rank == 0: print("MULTIGPU_OK")
'''


def test_two_gpu_sharding_matches_single(tmp_path):
    import torch

    if not torch.cuda.is_available() or torch.cuda.device_count() < 2:
        pytest.skip("needs >= 2 GPUs")
    w = tmp_path / "worker.py"
    w.write_text(WORKER)
    env = dict(os.environ, GSICP_ROOT=ROOT)
    p = subprocess.run([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", "--nproc-per-node=2", "--master-addr",
                        "127.0.0.1", "--master-port", "29611", str(w)], capture_output=True, text=True, env=env, cwd=ROOT,
                       timeout=900)
    assert "MULTIGPU_OK" in p.stdout, p.stdout[-3000:] + p.stderr[-3000:]
