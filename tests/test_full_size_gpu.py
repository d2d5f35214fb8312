"""BASELINE.json's full sizes, through properties that do not need an oracle run of the same size plus a direct comparison
with records of the reference's own CUDA code at the same sizes (tests/golden/raster_ref_records.npz):
  C3 640x480 / 300k Gaussians and C4 1280x960 / 1M Gaussians (rasterizer), C5-shape 2M x 2M points (GICP)."""
import numpy as np
import pytest
import torch

from gs_icp_slam_b200 import synthetic as S
from tests.refdigest import RASTER_RECORDS, Golden
from tests.util import rel_err, scene_tensors

pytestmark = pytest.mark.gpu


def _fw(R, t, c, H, W, bg):
    e = torch.Tensor([])
    return R.rasterize_gaussians(bg, t["means3D"], e, t["opacities"], t["scales"], t["rotations"], 1.0, e, c["viewmatrix"],
                                 c["projmatrix"], c["tanfovx"], c["tanfovy"], H, W, t["shs"], 0, c["campos"], False, False)


def _bw(R, t, c, bg, out, gdep, gcol):
    e = torch.Tensor([])
    n, depth, color, radii, is_used, geom, binning, img = out
    return R.rasterize_gaussians_backward(bg, t["means3D"], radii, e, t["scales"], t["rotations"], 1.0, e, c["viewmatrix"],
                                          c["projmatrix"], c["tanfovx"], c["tanfovy"], gdep, gcol, t["shs"], 0, c["campos"],
                                          geom, n, binning, img, False)


@pytest.mark.parametrize("P,size,scale", [(300000, (640, 480), 1.0), (1000000, (1280, 960), 2.0)])
def test_rasterizer_full_size_properties(cuda, P, size, scale):
    from gs_icp_slam_b200 import rasterizer as R

    g, cm, t, c, cam = scene_tensors(P, 3 if P == 300000 else 4, cuda, size=size, scale=scale)
    W, H = size
    bg = torch.tensor([0.05, 0.1, 0.15], device=cuda)
    out = _fw(R, t, c, H, W, bg)
    n, depth, color, radii, is_used, geom, binning, img = out
    pl, rg = R.export_binning(n, H, W, binning, img)
    cnt = rg[:, 1] - rg[:, 0]
    # binning: the ranges tile the instance list exactly; every listed Gaussian is visible; used implies visible
    assert n > P // 20 and int(cnt.sum()) == n and int(cnt.min()) >= 0
    ne = cnt > 0
    assert torch.equal(rg[ne][1:, 0], rg[ne][:-1, 1]) and int(rg[ne][0, 0]) == 0 and int(rg[ne][-1, 1]) == n
    assert bool((radii[pl] > 0).all()) and bool((radii[is_used] > 0).all())
    # sortedness: inside every tile the list is ordered by (view-space depth, index)
    view = c["viewmatrix"]
    z = (t["means3D"] @ view[:3, 2] + view[3, 2])[pl]
    tile_of = torch.repeat_interleave(torch.arange(rg.shape[0], device=cuda), cnt)
    same = tile_of[1:] == tile_of[:-1]
    dz = z[1:] - z[:-1]
    # (depth recomputed here in PyTorch float32: allow its rounding; exact ties are covered by the crowded-tile test)
    assert bool((dz[same] >= -1e-5 * z[1:][same].abs()).all())
    # image: finite, colour within [0, 1 + eps] for colours in [0,1], transmittance-weighted background
    assert bool(torch.isfinite(color).all()) and bool(torch.isfinite(depth).all())
    # determinism of the forward pass (no atomics on the image path)
    out2 = _fw(R, t, c, H, W, bg)
    assert out2[0] == n and torch.equal(out2[2], color) and torch.equal(out2[1], depth)
    # backward: linear in the incoming gradients
    gen = torch.Generator(device="cpu").manual_seed(1)
    g1c, g2c = (torch.randn((3, H, W), generator=gen).to(cuda) for _ in range(2))
    g1d, g2d = (torch.randn((1, H, W), generator=gen).to(cuda) for _ in range(2))
    a = _bw(R, t, c, bg, out, g1d, g1c)
    b = _bw(R, t, c, bg, out, g2d, g2c)
    ab = _bw(R, t, c, bg, out, 2.0 * g1d - 0.5 * g2d, 2.0 * g1c - 0.5 * g2c)
    for x, y, zz in zip(a, b, ab):
        if zz.numel():
            lin = (2.0 * x - 0.5 * y).cpu().numpy()
            assert rel_err(zz.cpu().numpy(), lin) <= 2e-4
    # invisible Gaussians receive exactly zero gradient
    inv = radii == 0
    for x in a:
        if x.numel():
            assert float(x[inv].abs().max()) == 0.0
    # the reference's own CUDA code at the same size: bit-exact lists and images
    gold, k = Golden(RASTER_RECORDS), f"full_{P}/"
    assert n == gold.scalar(k + "num_rendered") and gold.equal(k + "point_list", pl.to(torch.int64))
    assert gold.equal(k + "ranges", rg.to(torch.int64))
    assert gold.equal(k + "radii", radii) and gold.equal(k + "color", color) and gold.equal(k + "depth", depth)
    for name, o in zip(["means2D", "colors", "opacity", "means3D", "cov3D", "sh", "scales", "rotations"], a):
        assert gold.rel_err(k + "grad_" + name, o) <= 2e-4, name


def test_gicp_full_size_recovers_the_pose(cuda):
    """C5 shape: 2M x 2M points of the multi-room scene.  Properties: the known transform is recovered, every matched pair
    is within the correspondence threshold, the reported squared distances are those of the matched pairs."""
    import pygicp

    n = 2000000
    tgt, src, T = S.gicp_pair(n, n, 6, 7, 0.001, scale=5.0)
    r = pygicp.FastGICP()
    r.set_max_correspondence_distance(0.25)
    r.set_max_knn_distance(99999)
    r.set_input_target(tgt)
    r.calculate_target_covariance()
    r.set_input_source(src)
    pose = r.align(np.eye(4))
    assert r.has_converged() and np.abs(pose - T).max() < 1e-4
    corr, sqd = r.get_source_correspondence()
    assert corr.shape == (n,) and (corr >= -1).all() and (corr < n).all()
    m = corr >= 0
    assert m.mean() > 0.9 and (sqd[m] < 0.25 ** 2).all()
    idx = np.flatnonzero(m)[:: max(1, int(m.sum()) // 50000)]
    moved = (src[idx].astype(np.float32) @ pose[:3, :3].T.astype(np.float32) + pose[:3, 3].astype(np.float32))
    d2 = ((moved.astype(np.float64) - tgt[corr[idx]].astype(np.float32).astype(np.float64)) ** 2).sum(1)
    assert np.abs(d2 - sqd[idx]).max() <= 1e-5 + 1e-3 * sqd[idx].max()  # distances at the last linearisation point
    # nothing closer exists: brute force on a sample of queries
    sub = idx[:64]
    q = (src[sub].astype(np.float32) @ pose[:3, :3].T.astype(np.float32) + pose[:3, 3].astype(np.float32)).astype(np.float32)
    tt = torch.from_numpy(tgt.astype(np.float32)).to(cuda)
    qd = torch.from_numpy(q).to(cuda)
    best = np.array([float(((tt - qd[i]) ** 2).sum(1).min()) for i in range(len(sub))])  # exact differences, not cdist's GEMM form
    d2_sub = ((q.astype(np.float64) - tgt[corr[sub]].astype(np.float32).astype(np.float64)) ** 2).sum(1)
    # the matched target point is the nearest one (up to the last, sub-millimetre pose update after the search)
    assert (best <= d2_sub + 1e-7).all() and (best >= d2_sub - 1e-4).all()
