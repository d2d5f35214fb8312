"""GPU parity of the rasterizer: our CUDA path (through the C ABI) vs
  (1) the reference's own CUDA code compiled unmodified for sm_100a, through records of its outputs on these scenes
      (tests/golden/raster_ref_records.npz, written by tests/golden/make_raster_ref_records.py; tests/refdigest.py), and
  (2) the CPU restatement oracle/raster_oracle.c.
Tolerances (BASELINE.json north_star): indices bit-exact; rendered L1 <= 1e-4, PSNR within 0.01 dB.  Bit-exact
comparisons cover whole arrays; tolerance comparisons are evaluated on the recorded sample of the reference's output."""
import numpy as np
import pytest
import torch

from tests.refdigest import RASTER_RECORDS, Golden
from tests.util import psnr, rel_err, scene_tensors

pytestmark = pytest.mark.gpu
GRADS = ["means2D", "colors", "opacity", "means3D", "cov3D", "sh", "scales", "rotations"]


@pytest.fixture(scope="module")
def gold():
    return Golden(RASTER_RECORDS)


def _ours(t, c, H, W, bg, degree=0, colors=None, cov=None):
    from gs_icp_slam_b200 import rasterizer as R

    e = torch.Tensor([])
    return R.rasterize_gaussians(bg, t["means3D"], e if colors is None else colors, t["opacities"],
                                 e if cov is not None else t["scales"], e if cov is not None else t["rotations"], 1.0,
                                 e if cov is None else cov, c["viewmatrix"], c["projmatrix"], c["tanfovx"], c["tanfovy"],
                                 H, W, t["shs"] if colors is None else e, degree, c["campos"], False, False)


def _grad_pair(H, W, seed, cuda):
    gen = torch.Generator(device="cpu").manual_seed(seed)
    gcol = torch.randn((3, H, W), generator=gen).to(cuda)
    gdep = torch.randn((1, H, W), generator=gen).to(cuda)
    return gcol, gdep


def _check_indexing(gold, k, n, radii, is_used, pl, rg):
    assert n == gold.scalar(k + "num_rendered")
    assert gold.equal(k + "radii", radii) and gold.equal(k + "is_used", is_used)
    assert gold.equal(k + "ranges", rg.to(torch.int64))
    assert gold.equal(k + "point_list", pl.to(torch.int64))


# ---- scenes shared with tests/golden/make_raster_ref_records.py ----
def fb_scene(cuda, P, size, degree, seed):
    g, cm, t, c, cam = scene_tensors(P, seed, cuda, sh_degree=degree, size=size)
    bg = torch.tensor([0.1, 0.2, 0.3], device=cuda)
    return t, c, bg, _grad_pair(size[1], size[0], seed + 5, cuda)


def options_scene(cuda, active_degree, size):
    g, cm, t, c, cam = scene_tensors(15000, 40 + active_degree, cuda, sh_degree=3, size=size)
    bg = torch.tensor([0.7, 0.1, 0.4], device=cuda)
    return t, c, bg, _grad_pair(size[1], size[0], 77, cuda)


def degenerate_scene(cuda):
    """Finite but extreme inputs; returns the scene and the indices of the 40 modified Gaussians."""
    from gs_icp_slam_b200 import rasterizer as R

    g, cm, t, c, cam = scene_tensors(3000, 17, cuda, size=(200, 152))
    with torch.no_grad():
        vis = torch.nonzero(R.mark_visible(t["means3D"], c["viewmatrix"], c["projmatrix"])).flatten()
        a = vis[:40]
        t["scales"][a[0:8]] = 0.0
        t["scales"][a[8:12]] = 1000.0
        t["scales"][a[12:16], 0] = 1000.0           # needles
        t["opacities"][a[16:24]] = 40.0             # sigmoid -> 1 (alpha clamps at 0.99)
        t["opacities"][a[24:32]] = -40.0            # sigmoid -> 0 (never reaches 1/255)
        fwd = c["viewmatrix"][:3, 2]
        t["means3D"][a[32]] = c["campos"] + 0.2 * fwd            # exactly on the near plane (z <= 0.2 culls)
        t["means3D"][a[33]] = c["campos"] + 0.2000001 * fwd
        t["means3D"][a[34]] = c["campos"]                        # the camera centre
        t["rotations"][a[35]] = 0.0                              # zero quaternion (the reference does not normalise)
    bg = torch.tensor([0.3, 0.6, 0.9], device=cuda)
    return t, c, a, bg, _grad_pair(152, 200, 3, cuda)


def precomputed_scene(cuda):
    P, (W, H) = 30000, (320, 240)
    g, cm, t, c, cam = scene_tensors(P, 23, cuda, size=(W, H))
    gen = torch.Generator(device="cpu").manual_seed(1)
    colors = torch.rand((P, 3), generator=gen).to(cuda)
    # Sigma = Rm diag(s^2) Rm^T with Rm the rotation of the (x,y,z,w) quaternion (forward.cu:122-168), upper triangle
    q, s = t["rotations"].double(), t["scales"].double()
    x, y, z, w = q[:, 0], q[:, 1], q[:, 2], q[:, 3]
    Rm = torch.stack([1 - 2 * (y * y + z * z), 2 * (x * y - w * z), 2 * (x * z + w * y), 2 * (x * y + w * z),
                      1 - 2 * (x * x + z * z), 2 * (y * z - w * x), 2 * (x * z - w * y), 2 * (y * z + w * x),
                      1 - 2 * (x * x + y * y)], 1).view(P, 3, 3)
    Sg = Rm @ torch.diag_embed(s * s) @ Rm.transpose(1, 2)
    cov = torch.stack([Sg[:, 0, 0], Sg[:, 0, 1], Sg[:, 0, 2], Sg[:, 1, 1], Sg[:, 1, 2], Sg[:, 2, 2]], 1).float().contiguous()
    bg = torch.tensor([0.2, 0.1, 0.4], device=cuda)
    gcol = torch.randn((3, H, W), generator=gen).to(cuda)
    gdep = torch.randn((1, H, W), generator=gen).to(cuda)
    return t, c, colors, cov, bg, (gcol, gdep)


def crowded_scene(cuda, P):
    g, cm, t, c, cam = scene_tensors(P, 31, cuda, size=(160, 120))
    # pull every Gaussian towards a point 2 m in front of the camera so that a few tiles hold thousands of instances
    centre = c["campos"] + 2.0 * c["viewmatrix"][:3, 2]  # viewmatrix = (world->view)^T: column 2 is the optical axis
    t["means3D"] = (centre + 0.02 * (t["means3D"] - t["means3D"].mean(0))).contiguous()
    t["means3D"][100:200] = t["means3D"][300:400]  # exact duplicates: equal depth keys, order decided by the index
    return t, c, torch.zeros(3, device=cuda)


def autograd_scene(cuda, P, size, degree, seed):
    g, cm, t, c, cam = scene_tensors(P, seed, cuda, sh_degree=degree, size=size)
    bg = torch.tensor([0.1, 0.2, 0.3], device=cuda)
    active = max(degree - 1, 0) if degree == 3 else degree  # degree-3 table rendered at degree 2: the tail gets zero grads
    return t, c, bg, active, _grad_pair(size[1], size[0], 11, cuda)


def autograd_run(mod, t, c, bg, active, grads, H, W):
    """One module call + autograd.backward, then a second backward on the retained graph: (depth, color, radii, is_used,
    first gradients, second gradients)."""
    gcol, gdep = grads
    p = {k: v.detach().clone().requires_grad_(True) for k, v in t.items()}
    m2 = torch.zeros_like(p["means3D"], requires_grad=True)
    rs = mod.GaussianRasterizationSettings(H, W, c["tanfovx"], c["tanfovy"], bg, 1.0, c["viewmatrix"], c["projmatrix"],
                                           active, c["campos"], False, False)
    depth, color, radii, is_used = mod.GaussianRasterizer(rs)(means3D=p["means3D"], means2D=m2, opacities=p["opacities"],
                                                              shs=p["shs"], scales=p["scales"], rotations=p["rotations"])
    loss = (color * gcol).sum() + (depth * gdep).sum()
    loss.backward(retain_graph=True)
    g1 = {k: v.grad.clone() for k, v in p.items()}
    g1["means2D"] = m2.grad.clone()
    for v in p.values():
        v.grad = None
    m2.grad = None
    loss.backward()  # second backward on the same saved state
    g2 = {k: v.grad.clone() for k, v in p.items()}
    return depth.detach(), color.detach(), radii, is_used, g1, g2


@pytest.mark.parametrize("P,size,degree,seed", [(20000, (320, 240), 0, 2), (100000, (640, 480), 0, 3), (30000, (333, 211), 3, 5)])
def test_forward_backward_vs_reference_cuda(cuda, gold, P, size, degree, seed):
    from gs_icp_slam_b200 import rasterizer as R

    W, H = size
    t, c, bg, (gcol, gdep) = fb_scene(cuda, P, size, degree, seed)
    n, depth, color, radii, is_used, geom, binning, img = _ours(t, c, H, W, bg, degree)
    k = f"fb_{P}_{W}x{H}_{degree}_{seed}/"

    # ---- indexing: bit-exact ----
    pl, rg = R.export_binning(n, H, W, binning, img)
    _check_indexing(gold, k, n, radii, is_used, pl, rg)

    # ---- image: L1 / PSNR ----
    col, rcol, _ = gold.sample(k + "color", color)
    dep, rdep, _ = gold.sample(k + "depth", depth)
    assert np.abs(col - rcol).mean() <= 1e-4
    assert np.abs(col - rcol).max() <= 2e-3
    assert np.abs(dep - rdep).mean() <= 1e-4
    assert psnr(col, rcol) >= 80.0  # i.e. PSNR against any target differs by << 0.01 dB

    # ---- gradients (dL_dcolors: the reference returns it only as an internal when SHs are used) ----
    e = torch.Tensor([])
    ours = R.rasterize_gaussians_backward(bg, t["means3D"], radii, e, t["scales"], t["rotations"], 1.0, e, c["viewmatrix"],
                                          c["projmatrix"], c["tanfovx"], c["tanfovy"], gdep, gcol, t["shs"], degree,
                                          c["campos"], geom, n, binning, img, False)
    for name, o in zip(GRADS, ours):
        err = gold.rel_err(k + "grad_" + name, o)
        assert err <= 2e-4, f"grad {name}: rel err {err}"


@pytest.mark.parametrize("active_degree,scale_modifier,size", [(2, 0.7, (250, 190)), (1, 1.6, (96, 64)), (0, 1.0, (17, 33))])
def test_options_vs_reference_cuda(cuda, gold, active_degree, scale_modifier, size):
    """SH table larger than the active degree (the SLAM raises active_sh_degree over time), scale_modifier != 1, image
    sizes that are not multiples of the 16x16 tile, non-zero background."""
    from gs_icp_slam_b200 import rasterizer as R

    W, H = size
    t, c, bg, (gcol, gdep) = options_scene(cuda, active_degree, size)
    e = torch.Tensor([])
    n, depth, color, radii, is_used, geom, binning, img = R.rasterize_gaussians(
        bg, t["means3D"], e, t["opacities"], t["scales"], t["rotations"], scale_modifier, e, c["viewmatrix"], c["projmatrix"],
        c["tanfovx"], c["tanfovy"], H, W, t["shs"], active_degree, c["campos"], False, False)
    k = f"opt_{active_degree}_{scale_modifier}_{W}x{H}/"
    assert n > 0
    pl, rg = R.export_binning(n, H, W, binning, img)
    _check_indexing(gold, k, n, radii, is_used, pl, rg)
    assert gold.equal(k + "color", color) and gold.equal(k + "depth", depth)  # bit-identical images
    ours = R.rasterize_gaussians_backward(bg, t["means3D"], radii, e, t["scales"], t["rotations"], scale_modifier, e,
                                          c["viewmatrix"], c["projmatrix"], c["tanfovx"], c["tanfovy"], gdep, gcol, t["shs"],
                                          active_degree, c["campos"], geom, n, binning, img, False)
    for name, o in zip(GRADS, ours):
        assert gold.rel_err(k + "grad_" + name, o) <= 2e-4, name
    # SH coefficients above the active degree receive no gradient
    assert float(ours[5][:, (active_degree + 1) ** 2:, :].abs().max()) == 0.0
    # mark_visible (rasterize_points.cu:208-227) = the near-plane test of the forward pass
    vis = R.mark_visible(t["means3D"], c["viewmatrix"], c["projmatrix"])
    assert bool((vis | (radii == 0)).all())


def test_degenerate_gaussians_vs_reference_cuda(cuda, gold):
    """Finite but extreme inputs: zero scales (only the 0.3 px low-pass is left), 1 km scales (the rectangle is the whole
    screen), saturated and vanishing opacities, Gaussians exactly on the near plane and on the camera centre."""
    from gs_icp_slam_b200 import rasterizer as R

    W, H = 200, 152
    t, c, a, bg, (gcol, gdep) = degenerate_scene(cuda)
    n, depth, color, radii, is_used, geom, binning, img = _ours(t, c, H, W, bg)
    k = "degenerate/"
    pl, rg = R.export_binning(n, H, W, binning, img)
    _check_indexing(gold, k, n, radii, is_used, pl, rg)
    assert gold.equal(k + "color", color) and gold.equal(k + "depth", depth)  # bit patterns (robust to inf / nan)
    e = torch.Tensor([])
    ours = R.rasterize_gaussians_backward(bg, t["means3D"], radii, e, t["scales"], t["rotations"], 1.0, e, c["viewmatrix"],
                                          c["projmatrix"], c["tanfovx"], c["tanfovy"], gdep, gcol, t["shs"], 0, c["campos"],
                                          geom, n, binning, img, False)
    needles = set(a[12:16].tolist())
    slots = {int(v): j for j, v in enumerate(a.tolist())}
    for name, o in zip(GRADS, ours):
        assert gold.finite_equal(k + "grad_" + name, o), name
        a_, b_, smax = gold.sample(k + "grad_" + name, o)
        rows = gold.rows(k + "grad_" + name)
        fin = np.isfinite(b_)
        d = np.where(fin, np.abs(a_ - b_), 0.0).max(1, initial=0.0)
        scale_ = np.abs(np.where(fin, b_, 0.0)).max(1, initial=0.0)
        # the 1 km x 2 cm "needles" produce gradients of 1e9..1e10 out of terms that cancel to 7 digits: float32 noise
        # in both implementations (their forward output is still bit-identical); only their finiteness is compared
        d[[j for j, r in enumerate(rows) if int(r) in needles]] = 0.0
        bad = np.flatnonzero(d > 5e-4 * np.maximum(scale_, 1e-3 * smax))
        assert len(bad) == 0, (name, [(int(rows[i]), slots.get(int(rows[i]), -1), float(d[i]), float(scale_[i])) for i in bad[:8]])


def test_tile_shards_partition_the_frame(cuda):
    """Tile sharding on ONE GPU: rendering the shards one after the other reproduces the unsharded frame exactly and the
    per-shard instance counts add up (the multi-GPU path without the collective)."""
    from gs_icp_slam_b200 import rasterizer as R

    g, cm, t, c, cam = scene_tensors(20000, 8, cuda, size=(320, 240))
    bg = torch.tensor([0.2, 0.3, 0.1], device=cuda)
    full = _ours(t, c, 240, 320, bg)
    try:
        total, col, dep = 0, torch.zeros_like(full[2]), torch.zeros_like(full[1])
        for k in range(3):
            R.set_tile_shard(3, k)
            out = _ours(t, c, 240, 320, bg)
            total += out[0]
            col += out[2]
            dep += out[1]
            assert torch.equal(out[3], full[3])  # radii are computed for every Gaussian on every shard
    finally:
        R.set_tile_shard(1, 0)
    assert total == full[0]
    assert torch.equal(col, full[2]) and torch.equal(dep, full[1])


def test_precomputed_colors_and_cov3d_vs_reference_cuda(cuda, gold):
    """The alternative inputs of GaussianRasterizer.forward: colors_precomp instead of SHs, cov3D_precomp instead of
    scale/rotation (DGR/diff_gaussian_rasterization/__init__.py:189-222)."""
    from gs_icp_slam_b200 import rasterizer as R

    W, H = 320, 240
    t, c, colors, cov, bg, (gcol, gdep) = precomputed_scene(cuda)
    n, depth, color, radii, is_used, geom, binning, img = _ours(t, c, H, W, bg, 0, colors=colors, cov=cov)
    k = "precomputed/"
    assert n == gold.scalar(k + "num_rendered") and gold.equal(k + "radii", radii)
    assert gold.equal(k + "color", color) and gold.equal(k + "depth", depth)
    e = torch.Tensor([])
    ours = R.rasterize_gaussians_backward(bg, t["means3D"], radii, colors, e, e, 1.0, cov, c["viewmatrix"], c["projmatrix"],
                                          c["tanfovx"], c["tanfovy"], gdep, gcol, e, 0, c["campos"], geom, n, binning, img,
                                          False)
    for name, o in zip(GRADS[:5], ours[:5]):
        assert gold.rel_err(k + "grad_" + name, o) <= 2e-4, name
    assert ours[5].numel() == 0 and float(ours[6].abs().sum()) == 0 and float(ours[7].abs().sum()) == 0


@pytest.mark.parametrize("P,lo,hi", [(9000, 4096, 16384), (40000, 16384, 1 << 30)])
def test_crowded_tile_uses_segmented_sort_fallback(cuda, gold, P, lo, hi):
    """Crowded tiles: 1024..16384 instances go through the 1024-thread shared-memory sort, more than 16384 hand the whole
    frame over to the segmented radix sort; either way the sorted list must equal the reference's, including ties on equal
    depth (duplicated Gaussians)."""
    from gs_icp_slam_b200 import rasterizer as R

    t, c, bg = crowded_scene(cuda, P)
    n, depth, color, radii, is_used, geom, binning, img = _ours(t, c, 120, 160, bg)
    pl, rg = R.export_binning(n, 120, 160, binning, img)
    k = f"crowded_{P}/"
    assert lo < int((rg[:, 1] - rg[:, 0]).max()) <= hi, "scene does not exercise the intended sort path"
    assert n == gold.scalar(k + "num_rendered") and gold.equal(k + "ranges", rg.to(torch.int64))
    assert gold.equal(k + "point_list", pl.to(torch.int64))
    assert gold.equal(k + "color", color) and gold.equal(k + "depth", depth)


def test_cull_is_exact(cuda):
    """Sub-tile culling must not change a single bit of the output."""
    from gs_icp_slam_b200 import _lib

    g, cm, t, c, cam = scene_tensors(40000, 7, cuda, size=(320, 240))
    bg = torch.zeros(3, device=cuda)
    a = _ours(t, c, 240, 320, bg)
    _lib.lib.gsicp_test_set_render_cull(0)
    try:
        b = _ours(t, c, 240, 320, bg)
    finally:
        _lib.lib.gsicp_test_set_render_cull(1)
    assert a[0] == b[0]
    assert torch.equal(a[1], b[1]) and torch.equal(a[2], b[2])


def test_vs_cpu_oracle(cuda):
    from oracle import raster_oracle

    P, (W, H) = 3000, (160, 120)
    g, cm, t, c, cam = scene_tensors(P, 11, cuda, size=(W, H), sh_degree=1)
    bgn = np.array([0.0, 0.5, 1.0], np.float32)
    rng = np.random.default_rng(3)
    gcol = rng.normal(size=(3, H, W)).astype(np.float32)
    gdep = rng.normal(size=(1, H, W)).astype(np.float32)
    o = raster_oracle.forward_backward(g, cm, H, W, bgn, sh_degree=1, dL_dcolor=gcol, dL_ddepth=gdep)
    from gs_icp_slam_b200 import rasterizer as R

    bg = torch.from_numpy(bgn).to(cuda)
    n, depth, color, radii, is_used, geom, binning, img = _ours(t, c, H, W, bg, 1)
    # CPU and GPU round differently (fma contraction), so indices may differ for Gaussians that sit exactly on a
    # rounding boundary: demand exact equality here for this seed (it holds), and image closeness.
    assert np.array_equal(radii.cpu().numpy(), o.radii)
    assert n == o.num_rendered
    assert np.abs(color.cpu().numpy() - o.color).mean() <= 1e-4
    assert np.abs(depth.cpu().numpy() - o.depth).mean() <= 1e-4
    e = torch.Tensor([])
    ours = R.rasterize_gaussians_backward(bg, t["means3D"], radii, e, t["scales"], t["rotations"], 1.0, e, c["viewmatrix"],
                                          c["projmatrix"], c["tanfovx"], c["tanfovy"], torch.from_numpy(gdep).to(cuda),
                                          torch.from_numpy(gcol).to(cuda), t["shs"], 1, c["campos"], geom, n, binning, img,
                                          False)
    refs = [o.dL_dmeans2D, o.dL_dcolors, o.dL_dopacity, o.dL_dmeans3D, o.dL_dcov3D, o.dL_dsh, o.dL_dscales, o.dL_drotations]
    for name, a, b in zip(["means2D", "colors", "opacity", "means3D", "cov3D", "sh", "scales", "rotations"], ours, refs):
        assert rel_err(a.cpu().numpy().reshape(b.shape), b) <= 2e-4, name


def test_autograd_api(cuda):
    """The drop-in package: GaussianRasterizer(settings)(...) -> (depth, color, radii, is_used), backward fills grads."""
    from diff_gaussian_rasterization import GaussianRasterizationSettings, GaussianRasterizer

    g, cm, t, c, cam = scene_tensors(5000, 13, cuda, size=(160, 120))
    for k in ("means3D", "shs", "opacities", "scales", "rotations"):
        t[k].requires_grad_(True)
    means2D = torch.zeros_like(t["means3D"], requires_grad=True)
    rs = GaussianRasterizationSettings(120, 160, c["tanfovx"], c["tanfovy"], torch.zeros(3, device=cuda), 1.0,
                                       c["viewmatrix"], c["projmatrix"], 0, c["campos"], False, False)
    depth, color, radii, is_used = GaussianRasterizer(rs)(means3D=t["means3D"], means2D=means2D, opacities=t["opacities"],
                                                          shs=t["shs"], scales=t["scales"], rotations=t["rotations"])
    assert depth.shape == (1, 120, 160) and color.shape == (3, 120, 160)
    assert radii.dtype == torch.int32 and is_used.dtype == torch.bool
    (color.mean() + 0.1 * depth.mean()).backward()
    for k in ("means3D", "shs", "opacities", "scales", "rotations"):
        assert t[k].grad is not None and torch.isfinite(t[k].grad).all()
    assert means2D.grad is not None and means2D.grad.abs().sum() > 0
    with pytest.raises(Exception):
        GaussianRasterizer(rs)(means3D=t["means3D"], means2D=means2D, opacities=t["opacities"])
    vis = GaussianRasterizer(rs).markVisible(t["means3D"].detach())
    assert vis.dtype == torch.bool and vis.shape[0] == 5000


def test_empty_and_offscreen(cuda):
    from gs_icp_slam_b200 import rasterizer as R

    g, cm, t, c, cam = scene_tensors(100, 17, cuda, size=(64, 48))
    bg = torch.tensor([0.3, 0.2, 0.1], device=cuda)
    t0 = {k: v[:0] for k, v in t.items()}
    out = _ours(t0, c, 48, 64, bg)
    assert out[0] == 0 and out[2].abs().sum() == 0  # reference returns zero images when P == 0
    # everything behind the camera: background only
    t2 = dict(t)
    t2["means3D"] = t["means3D"] * 0 + torch.from_numpy(cm["campos"]).to(cuda) - 5.0 * c["viewmatrix"][:3, 2]
    out = _ours(t2, c, 48, 64, bg)
    assert out[0] == 0
    assert torch.allclose(out[2], bg.view(3, 1, 1).expand(3, 48, 64))
    assert torch.allclose(out[1], torch.full((1, 48, 64), 15.0, device=cuda))


@pytest.mark.parametrize("P,size,degree,seed", [(100000, (640, 480), 0, 3), (30000, (333, 211), 3, 5), (300000, (640, 480), 0, 3)])
def test_autograd_vs_reference_torch_extension(cuda, gold, P, size, degree, seed):
    """Drop-in parity at the Python API: this repo's diff_gaussian_rasterization against the REFERENCE's own package
    (unmodified sources built through their setup.py — rasterize_points.cu + ext.cpp, the stock path), same module call,
    same autograd.backward; includes a second backward on a retained graph and sh_degree below the SH table size."""
    import diff_gaussian_rasterization as ours

    W, H = size
    t, c, bg, active, grads = autograd_scene(cuda, P, size, degree, seed)
    o = autograd_run(ours, t, c, bg, active, grads, H, W)
    k = f"ext_{P}_{W}x{H}_{degree}_{seed}/"
    assert gold.equal(k + "radii", o[2]) and gold.equal(k + "is_used", o[3])
    assert gold.equal(k + "depth", o[0]) and gold.equal(k + "color", o[1])  # images bit-identical
    for name in o[4]:
        assert gold.rel_err(k + "g1_" + name, o[4][name]) <= 2e-4, name
    for name in o[5]:
        assert gold.rel_err(k + "g2_" + name, o[5][name]) <= 2e-4, ("second backward", name)
    if degree == 3:
        assert float(o[4]["shs"][:, (active + 1) ** 2:].abs().max()) == 0.0



@pytest.mark.parametrize("variant", [0, 1])
def test_backward_staging_variants_vs_reference_extension(cuda, gold, variant):
    """render_backward_kernel ships in two launch configurations (256-entry staging / 3 CTAs per SM, the default, and 128-entry
    staging / 4 CTAs per SM).  Each one must match the reference extension's gradients on its own."""
    from gs_icp_slam_b200 import _lib

    _lib.lib.gsicp_test_set_bwd_variant(variant)
    try:
        test_autograd_vs_reference_torch_extension(cuda, gold, 100000, (640, 480), 0, 3)
    finally:
        _lib.lib.gsicp_test_set_bwd_variant(0)
